"""`VideoCompressor` — drop-in for the reference's P-frame codec module
(reference main/model/pnet.py:15-83): same constructor, same `forward(input_image, refer_frames,
enabled_amp, is_compress=False)`, same return tuple, same state_dict key set (strict load both ways),
but every stage of the forward runs as hand-written sm_100a CUDA kernels behind the C-ABI of
include/tdvc_b200.h.  There is no CPU / PyTorch fallback: on a non-CUDA tensor `forward` raises.

Structure of this file
  * parameter containers that reproduce the reference's module tree (names only; no torch compute),
  * `_Packed`: device-side weight packing (implicit-GEMM layouts, GDN/entropy-model reparametrisations),
  * `_Plan`: static NHWC buffer plan for one (N, H, W) + the launch sequence of one P-frame.

Scope: inference (`eval()`), `is_compress=False`.  Training-mode quantisation noise / backward and the
rANS bitstream are "next" rows (SURVEY.md 8f) and raise NotImplementedError.

Per-GOP feature caches (`_Plan`): the features the reference recomputes for every P-frame from inputs that repeat
inside a GOP are keyed on a content hash of the reference slice and reused; `forward` stays stateless in its results.
"""
import ctypes as C
import itertools
import math
import os
import threading
import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F

from tdvc_b200 import lib as L

_LN2 = math.log(2.0)


# =============================================================================== parameter containers
_CDF_BUFFERS = ("_offset", "_quantized_cdf", "_cdf_length", "scale_table")   # written by update(); no packed weight reads them


class _ConvModule(nn.Module):  # mmcv ConvModule naming: `<name>.conv.weight`
    def __init__(self, i, o, k):
        super().__init__()
        self.conv = nn.Conv2d(i, o, k, 1, k // 2)


class _SE(nn.Module):  # reference main/model/inflate.py:159-208
    def __init__(self, c, ratio=16):
        super().__init__()
        self.conv1 = _ConvModule(c, int(c / ratio), 1)
        self.conv2 = _ConvModule(int(c / ratio), c, 1)


class _ResBlock(nn.Module):  # reference main/utils/utils.py:43-56
    def __init__(self, c=64):
        super().__init__()
        self.conv1 = nn.Conv2d(c, c, 3, 1, 1)
        self.conv2 = nn.Conv2d(c, c, 3, 1, 1)


def _res_stack(n, c=64):
    return nn.Sequential(*[_ResBlock(c) for _ in range(n)])


class _FeaExtra(nn.Module):  # pnet.py:86-96
    def __init__(self, nb):
        super().__init__()
        self.conv_first = nn.Conv2d(3, 64, 3, 1, 1)
        self.residual_layer = _res_stack(nb)


class _SPyNetLevel(nn.Module):  # flownet.py:178-238
    def __init__(self):
        super().__init__()
        self.basic_module = nn.Sequential(*[_ConvModule(i, o, 7) for i, o in
                                            ((8, 32), (32, 64), (64, 32), (32, 16), (16, 2))])


class _SPyNet(nn.Module):  # flownet.py:51-80 (mean/std buffers exist, unused)
    def __init__(self):
        super().__init__()
        self.basic_module = nn.ModuleList([_SPyNetLevel() for _ in range(6)])
        self.register_buffer("mean", torch.Tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1))
        self.register_buffer("std", torch.Tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1))


class _OffsetGen(nn.Module):  # pnet.py:99-129; SPyNet is built WITHOUT downloading weights (pretrained=None)
    def __init__(self, nf=64):
        super().__init__()
        self.offset_conv11 = nn.ModuleDict()
        self.offset_conv11_1 = nn.ModuleDict()
        self.offset_conv12 = nn.ModuleDict()
        self.feat_fusion = nn.ModuleDict()
        for i in (3, 2, 1):
            lv = f"l{i}"
            self.offset_conv11[lv] = nn.Conv2d(2 * nf, nf, 3, 1, 1)
            self.offset_conv11_1[lv] = nn.Conv2d(nf, nf, 3, 1, 1)
            self.offset_conv12[lv] = nn.Conv2d(nf, nf, 3, 1, 1)
            if i < 3:
                self.feat_fusion[lv] = nn.Conv2d(2 * nf, nf, 1, 1, 0)
        self.upsample_conv = nn.Conv2d(nf, nf, 3, 1, 1)
        self.conv_l2_1 = nn.Conv2d(nf, nf, 3, 2, 1)
        self.conv_l2_2 = nn.Conv2d(nf, nf, 3, 1, 1)
        self.conv_l3_1 = nn.Conv2d(nf, nf, 3, 2, 1)
        self.conv_l3_2 = nn.Conv2d(nf, nf, 3, 1, 1)
        self.spynet = _SPyNet()
        self.attn = _SE(64)
        self.feat_fusion_ = nn.Conv2d(nf, nf, 3, 1, 1)


class _DCN(nn.Module):  # dcn_v2_amp.py:125-217
    def __init__(self, cin, cout, dg):
        super().__init__()
        self.dg = dg
        self.weight = nn.Parameter(torch.Tensor(cout, cin, 3, 3))
        self.bias = nn.Parameter(torch.Tensor(cout))
        stdv = 1.0 / math.sqrt(cin * 9)
        self.weight.data.uniform_(-stdv, stdv)
        self.bias.data.zero_()
        self.conv_offset_mask = nn.Conv2d(cin, dg * 27, 3, 1, 1)
        self.conv_offset_mask.weight.data.zero_()
        self.conv_offset_mask.bias.data.zero_()


class _MCNet(nn.Module):  # pnet.py:170-177
    def __init__(self, nb):
        super().__init__()
        self.dconv = _DCN(64, 64, 8)
        self.recon_layer = _res_stack(nb)
        self.feat_down = nn.Conv2d(64, 3, 3, 1, 1)  # allocated, never executed
        self.conv = nn.Conv2d(128, 64, 3, 1, 1)


class _Bottleneck3D(nn.Module):  # pnet.py:296-307
    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv3d(64, 64, (1, 3, 3), padding=(0, 1, 1))
        self.spatial_conv3d = nn.Conv3d(64, 64, (1, 3, 3), padding=(0, 1, 1))
        self.temporal_conv3d = nn.Conv3d(64, 64, (3, 1, 1), stride=(3, 1, 1), bias=False)
        self.conv3 = nn.Conv3d(64, 64, (1, 3, 3), padding=(0, 1, 1))


class _LoopFilter(nn.Module):  # pnet.py:266-275 (attribute `mcfilter`)
    def __init__(self):
        super().__init__()
        self.conv01 = nn.Conv2d(3, 64, 3, 1, 1)
        self.conv02 = nn.Conv2d(64, 64, 3, 1, 1)
        self.conv1 = nn.Conv3d(64, 64, (1, 3, 3), padding=(0, 1, 1))
        self.layer1 = _Bottleneck3D()
        self.attn = _SE(64)
        self.feat_fusion = nn.Conv2d(256, 64, 1, 1)


class _FeatureExtract(nn.Module):  # pnet.py:320-326
    def __init__(self, cin, mid, nb):
        super().__init__()
        self.conv_first = nn.Conv2d(cin, mid, 3, 1, 1)
        self.body = _res_stack(nb, mid)
        self.conv_last = nn.Conv2d(mid, mid, 3, 1, 1)


class _FeatureFix(nn.Module):  # pnet.py:187-211 (attribute `loopfilter`)
    def __init__(self):
        super().__init__()
        self.FeatureExtract_input = _FeatureExtract(64, 64, 2)
        self.FeatureExtract_ref = _FeatureExtract(3, 64, 2)
        self.recon_layer = _res_stack(2)
        for nme, s in (("conv_10", 2), ("conv_11", 1), ("conv_12", 2), ("conv_13", 1)):  # never executed
            setattr(self, nme, nn.Conv2d(64, 64, 3, s, 1))
        self.featfusion = nn.Conv2d(128, 64, 3, 1, 1)
        self.featfusion2 = nn.Conv2d(128, 64, 3, 1, 1)
        self.featdown = nn.Conv2d(64, 3, 3, 1, 1)
        self.attn = _SE(64)


# ---- CompressAI-shaped containers (SURVEY.md App. A; names must match real checkpoints)
class _Bound(nn.Module):
    def __init__(self, b):
        super().__init__()
        self.register_buffer("bound", torch.Tensor([float(b)]))


class _Reparam(nn.Module):
    def __init__(self, minimum=0.0, offset=2 ** -18):
        super().__init__()
        self.register_buffer("pedestal", torch.Tensor([offset ** 2]))
        self.lower_bound = _Bound((minimum + offset ** 2) ** 0.5)

    def init(self, x):
        return torch.sqrt(torch.max(x + self.pedestal, self.pedestal))


class _GDN(nn.Module):
    def __init__(self, c, inverse=False, beta_min=1e-6, gamma_init=0.1):
        super().__init__()
        self.inverse = inverse
        self.beta_reparam = _Reparam(minimum=beta_min)
        self.beta = nn.Parameter(self.beta_reparam.init(torch.ones(c)))
        self.gamma_reparam = _Reparam()
        self.gamma = nn.Parameter(self.gamma_reparam.init(gamma_init * torch.eye(c)))


class _RBWithStride(nn.Module):
    def __init__(self, i, o, stride=2):
        super().__init__()
        self.conv1 = nn.Conv2d(i, o, 3, stride, 1)
        self.conv2 = nn.Conv2d(o, o, 3, 1, 1)
        self.gdn = _GDN(o)
        self.skip = nn.Conv2d(i, o, 1, stride)


class _RB(nn.Module):
    def __init__(self, i, o):
        super().__init__()
        self.conv1 = nn.Conv2d(i, o, 3, 1, 1)
        self.conv2 = nn.Conv2d(o, o, 3, 1, 1)


def _subpel(i, o, r):
    return nn.Sequential(nn.Conv2d(i, o * r * r, 3, padding=1), nn.PixelShuffle(r))


class _RBUpsample(nn.Module):
    def __init__(self, i, o, r=2):
        super().__init__()
        self.subpel_conv = _subpel(i, o, r)
        self.conv = nn.Conv2d(o, o, 3, 1, 1)
        self.igdn = _GDN(o, inverse=True)
        self.upsample = _subpel(i, o, r)


class _CdfBuffers(nn.Module):
    """compressai's entropy models carry their coding tables as buffers that `update()` resizes; a checkpoint saved after
    `update()` holds them filled.  Loading resizes ours to whatever arrives (compressai: `update_registered_buffers`)."""

    def _load_from_state_dict(self, state_dict, prefix, *args):
        for name in _CDF_BUFFERS:
            t = state_dict.get(prefix + name)
            buf = getattr(self, name, None)
            if t is not None and buf is not None and buf.shape != t.shape:
                setattr(self, name, torch.empty(t.shape, dtype=buf.dtype, device=buf.device))
        super()._load_from_state_dict(state_dict, prefix, *args)


class _EntropyBottleneck(_CdfBuffers):
    def __init__(self, channels, tail_mass=1e-9, init_scale=10, filters=(3, 3, 3, 3)):
        super().__init__()
        f = (1,) + tuple(filters) + (1,)
        scale = init_scale ** (1 / (len(filters) + 1))
        for i in range(len(filters) + 1):
            m = torch.Tensor(channels, f[i + 1], f[i]).fill_(math.log(math.expm1(1 / scale / f[i + 1])))
            self.register_parameter(f"_matrix{i}", nn.Parameter(m))
            self.register_parameter(f"_bias{i}", nn.Parameter(torch.Tensor(channels, f[i + 1], 1).uniform_(-0.5, 0.5)))
            if i < len(filters):
                self.register_parameter(f"_factor{i}", nn.Parameter(torch.zeros(channels, f[i + 1], 1)))
        self.quantiles = nn.Parameter(torch.Tensor([-init_scale, 0, init_scale]).repeat(channels, 1, 1))
        self.register_buffer("_offset", torch.IntTensor())
        self.register_buffer("_quantized_cdf", torch.IntTensor())
        self.register_buffer("_cdf_length", torch.IntTensor())
        t = math.log(2 / tail_mass - 1)
        self.register_buffer("target", torch.Tensor([-t, 0, t]))
        self.likelihood_lower_bound = _Bound(1e-9)


class _GaussianConditional(_CdfBuffers):
    def __init__(self):
        super().__init__()
        self.register_buffer("_offset", torch.IntTensor())
        self.register_buffer("_quantized_cdf", torch.IntTensor())
        self.register_buffer("_cdf_length", torch.IntTensor())
        self.register_buffer("scale_table", torch.Tensor())
        self.register_buffer("scale_bound", torch.Tensor([0.11]))
        self.likelihood_lower_bound = _Bound(1e-9)
        self.lower_bound_scale = _Bound(0.11)


class _MaskedConv(nn.Conv2d):
    def __init__(self, i, o):
        super().__init__(i, o, 5, 1, 2)
        self.register_buffer("mask", torch.ones_like(self.weight.data))
        self.mask[:, :, 2, 2:] = 0
        self.mask[:, :, 3:] = 0


class _Coder(nn.Module):
    """MVCoder / ResCoder (reference main/model/encoder_v3.py:14-69) = compressai Cheng2020Anchor(N=128)
    with the 64-channel g_a / g_s and SE blocks of the reference."""

    def __init__(self, N=128):
        super().__init__()
        lr = nn.LeakyReLU
        self.entropy_bottleneck = _EntropyBottleneck(N)
        self.g_a = nn.Sequential(_RBWithStride(64, N), _RB(N, N), _RBWithStride(N, N), _SE(N), _RB(N, N),
                                 _RBWithStride(N, N), _RB(N, N), nn.Conv2d(N, N, 3, 2, 1), _SE(N))
        self.h_a = nn.Sequential(nn.Conv2d(N, N, 3, 1, 1), lr(), nn.Conv2d(N, N, 3, 1, 1), lr(),
                                 nn.Conv2d(N, N, 3, 2, 1), lr(), nn.Conv2d(N, N, 3, 1, 1), lr(),
                                 nn.Conv2d(N, N, 3, 2, 1))
        self.h_s = nn.Sequential(nn.Conv2d(N, N, 3, 1, 1), lr(), _subpel(N, N, 2), lr(),
                                 nn.Conv2d(N, N * 3 // 2, 3, 1, 1), lr(), _subpel(N * 3 // 2, N * 3 // 2, 2), lr(),
                                 nn.Conv2d(N * 3 // 2, N * 2, 3, 1, 1))
        self.g_s = nn.Sequential(_SE(N), _RB(N, N), _RBUpsample(N, N), _RB(N, N), _RBUpsample(N, N), _SE(N),
                                 _RB(N, N), _RBUpsample(N, N), _RB(N, N), _subpel(N, 64, 2))
        self.entropy_parameters = nn.Sequential(nn.Conv2d(N * 4, N * 10 // 3, 1), lr(),
                                                nn.Conv2d(N * 10 // 3, N * 8 // 3, 1), lr(),
                                                nn.Conv2d(N * 8 // 3, N * 2, 1))
        self.context_prediction = _MaskedConv(N, 2 * N)
        self.gaussian_conditional = _GaussianConditional()


# =============================================================================== activations (NHWC views)
class Act:
    """A channels-last fp32 activation: element (n,y,x,c) at ptr + 4*(((n*H+y)*W+x)*ld + c)."""
    __slots__ = ("t", "ptr", "N", "H", "W", "C", "ld")

    def __init__(self, t, ptr, N, H, W, C, ld):
        self.t, self.ptr, self.N, self.H, self.W, self.C, self.ld = t, ptr, N, H, W, C, ld

    @staticmethod
    def alloc(N, H, W, C, device, ld=None, zero=False):
        ld = ld or C
        t = (torch.zeros if zero else torch.empty)((N, H, W, ld), device=device, dtype=torch.float32)
        return Act(t, t.data_ptr(), N, H, W, C, ld)

    @staticmethod
    def from_nchw(x, ld=None):
        """NHWC copy (torch permute; tests / plumbing only) of an NCHW tensor, channel-padded with zeros to ld."""
        N, C, H, W = x.shape
        a = Act.alloc(N, H, W, C, x.device, ld=ld, zero=True)
        a.t[..., :C] = x.permute(0, 2, 3, 1)
        return a

    def batch(self, i, n=1):
        return Act(self.t, self.ptr + 4 * i * self.H * self.W * self.ld, n, self.H, self.W, self.C, self.ld)

    def chan(self, c0, c):
        return Act(self.t, self.ptr + 4 * c0, self.N, self.H, self.W, c, self.ld)

    def nchw(self):
        """Torch NCHW copy of the logical channels (debug taps / tests)."""
        v = self.t.view(-1)
        off = (self.ptr - self.t.data_ptr()) // 4
        v = torch.as_strided(v, (self.N, self.H, self.W, self.C),
                             (self.H * self.W * self.ld, self.W * self.ld, self.ld, 1), off)
        return v.permute(0, 3, 1, 2).contiguous()


def _r(x, m):
    return (x + m - 1) // m * m


# =============================================================================== packed weights
class ConvW:
    __slots__ = ("w", "b", "cin", "cin_real", "cin_pad", "cout", "cout_pad", "k", "pad", "shuffle", "w_f16", "stride", "w_shift",
                 "w_f16_p1", "w_shift_p1", "p1_ok", "wmax")


def pack_conv(weight, bias, src_layout=None, shuffle=0, pad=None, stride=1):
    """(O, I, k, k) conv weight -> implicit-GEMM layout [k*k][cin_pad][cout_pad] fp32 (zero padded).
    src_layout: [(real_channels, stored_channels), ...] per concatenated source (stored >= real, % 4 == 0).
    shuffle=2 folds nn.PixelShuffle(2) into the output-channel order: co' = (dy*2+dx)*(O/4) + c."""
    O, I, k, _ = weight.shape
    dev = weight.device
    w = weight.detach().float()
    if shuffle == 2:
        cr = O // 4
        perm = torch.arange(O, device=dev).view(cr, 4).t().reshape(-1)  # co' -> original c*4 + q
        w = w[perm]
        bias = bias[perm] if bias is not None else None
    if src_layout is None:
        src_layout = [(I, _r(I, 4))]
    assert sum(r for r, _ in src_layout) == I
    cin = sum(s for _, s in src_layout)
    cin_pad, cout_pad = _r(cin, 8), _r(O, 16)
    out = torch.zeros(k * k, cin_pad, cout_pad, device=dev, dtype=torch.float32)
    wt = w.permute(2, 3, 1, 0).reshape(k * k, I, O)
    ri = si = 0
    for real, stored in src_layout:
        out[:, si:si + real, :O] = wt[:, ri:ri + real]
        ri += real
        si += stored
    cw = ConvW()
    cw.w = out.contiguous()
    cw.b = None
    if bias is not None:
        cw.b = torch.zeros(cout_pad, device=dev, dtype=torch.float32)
        cw.b[:O] = bias.detach().float()
    cw.cin, cw.cin_pad, cw.cout, cw.cout_pad, cw.k = cin, cin_pad, O, cout_pad, k
    cw.cin_real = I
    cw.pad = k // 2 if pad is None else pad
    cw.shuffle = shuffle
    cw.stride = stride   # the tcgen05 weight blocking depends on it (csrc/conv_tc.cu `choose`)
    cw.w_f16 = None
    cw.w_shift = 0
    cw.w_f16_p1 = None       # one-product fp16 blocks (tc.attach_f16), for the stages `precision = "mixed"` relaxes
    cw.w_shift_p1 = 0
    cw.p1_ok = False
    cw.wmax = None
    return cw


def _reparam(p, mod):
    """compressai NonNegativeParametrizer.forward: max(p, bound)^2 - pedestal."""
    p = p.detach()
    return torch.max(p, mod.lower_bound.bound.to(p.device)) ** 2 - mod.pedestal.to(p.device)


# stages that may run with ONE fp16 MMA product (`VideoCompressor.precision = "mixed"`): everything behind the last quantiser
# of the frame - the residual coder's synthesis transform and the in-loop filter on the reconstruction.  Measured budget:
# profiles/r02_precision_budget.txt (DESIGN.md, precision).  FeatureExtract_ref stays exact: it is cached per GOP.
_ONE_PRODUCT_PREFIXES = ("rs.gs", "lf.fe_in", "lf.featfusion", "lf.res", "lf.featdown")


class _Packed:
    """All packed weights of one VideoCompressor on one device.  Packing runs on the HOST from one copy of the parameters and
    goes to the device as a single flat fp32 buffer (one H2D copy; the fp16 blocks of the tensor-core kernels are then built
    from it by `pack_f16_kernel`), so loading a model issues no torch kernels."""

    def __init__(self, m, dev):
        c = {}
        cpu = {k: v.detach().to("cpu", torch.float32) for k, v in list(m.named_parameters()) + list(m.named_buffers())}

        def P(mod, name):   # host copy of a parameter / buffer of `mod`
            return cpu[self._names[id(getattr(mod, name))]]

        self._names = {id(v): k for k, v in list(m.named_parameters()) + list(m.named_buffers())}

        def cv(name, mod, **kw):
            c[name] = pack_conv(P(mod, "weight"), P(mod, "bias") if mod.bias is not None else None, **kw)

        def cv3d(name, mod):
            w = P(mod, "weight")
            c[name] = pack_conv(w.reshape(w.shape[0], w.shape[1], w.shape[3], w.shape[4]), P(mod, "bias"))

        def res(name, stack):
            for i, rb in enumerate(stack):
                cv(f"{name}.{i}.conv1", rb.conv1)
                cv(f"{name}.{i}.conv2", rb.conv2)

        def se(name, mod):
            w1, w2 = P(mod.conv1.conv, "weight"), P(mod.conv2.conv, "weight")
            c[name] = (w1.reshape(w1.shape[0], -1).contiguous(), P(mod.conv1.conv, "bias").contiguous(),
                       w2.reshape(w2.shape[0], -1).contiguous(), P(mod.conv2.conv, "bias").contiguous())

        img = [(3, 4)]
        cv("extra_fea.conv_first", m.extra_fea.conv_first, src_layout=img)
        res("extra_fea.res", m.extra_fea.residual_layer)
        me = m.motion_est
        for nme in ("conv_l2_1", "conv_l2_2", "conv_l3_1", "conv_l3_2", "upsample_conv", "feat_fusion_"):
            cv("me." + nme, getattr(me, nme), stride=getattr(me, nme).stride[0])
        for lv in ("l3", "l2", "l1"):
            cv(f"me.c11.{lv}", me.offset_conv11[lv], src_layout=[(64, 64), (64, 64)])
            cv(f"me.c11_1.{lv}", me.offset_conv11_1[lv])
            if lv == "l3":
                cv("me.c12.l3", me.offset_conv12[lv])
            else:
                cv(f"me.ff.{lv}", me.feat_fusion[lv], src_layout=[(64, 64), (64, 64)])
        se("me.attn", me.attn)
        for lvl in range(6):
            for i in range(5):
                cv(f"spy.{lvl}.{i}", me.spynet.basic_module[lvl].basic_module[i].conv)
        mc = m.mcnet
        cv("mc.offmask", mc.dconv.conv_offset_mask)
        wd = P(mc.dconv, "weight")  # (O, C, 3, 3) -> [C*9][O_pad], row = c*9 + tap
        O, Cc = wd.shape[0], wd.shape[1]
        opad = _r(O, 64)
        pk = torch.zeros(Cc * 9, opad, dtype=torch.float32)
        pk[:, :O] = wd.reshape(O, Cc * 9).t()
        c["mc.dcn.w"] = pk.contiguous()
        c["mc.dcn.b"] = P(mc.dconv, "bias").contiguous()
        cv("mc.conv", mc.conv, src_layout=[(64, 64), (64, 64)])
        res("mc.res", mc.recon_layer)
        mf = m.mcfilter
        cv("mf.conv01", mf.conv01, src_layout=img)
        cv("mf.conv02", mf.conv02)
        cv3d("mf.conv1", mf.conv1)
        cv3d("mf.l1.conv1", mf.layer1.conv1)
        cv3d("mf.l1.spatial", mf.layer1.spatial_conv3d)
        cv3d("mf.l1.conv3", mf.layer1.conv3)
        wt = P(mf.layer1.temporal_conv3d, "weight")  # (64, 64, 3, 1, 1): [o][c][t] -> 1x1 over (t, c)
        c["mf.l1.temporal"] = pack_conv(wt[:, :, :, 0, 0].permute(0, 2, 1).reshape(64, 192, 1, 1), None,
                                        src_layout=[(64, 64)] * 3)
        cv("mf.fusion", mf.feat_fusion, src_layout=[(64, 64)] * 4)
        se("mf.attn", mf.attn)
        lf = m.loopfilter
        for nme, fe, lay in (("lf.fe_in", lf.FeatureExtract_input, None), ("lf.fe_ref", lf.FeatureExtract_ref, img)):
            cv(nme + ".first", fe.conv_first, src_layout=lay)
            res(nme + ".body", fe.body)
            cv(nme + ".last", fe.conv_last)
        cv("lf.featfusion", lf.featfusion, src_layout=[(64, 64), (64, 64)])
        cv("lf.featfusion2", lf.featfusion2, src_layout=[(64, 64), (64, 64)])
        res("lf.res", lf.recon_layer)
        cv("lf.featdown", lf.featdown)
        se("lf.attn", lf.attn)
        for cn, cd in (("mv", m.mvCoder), ("rs", m.resCoder)):
            self._pack_coder(c, cn, cd, cv, se, P)
        for name, v in c.items():
            if isinstance(v, ConvW):
                v.p1_ok = name.startswith(_ONE_PRODUCT_PREFIXES)
        self.c = _upload(c, dev)
        del self._names

    @staticmethod
    def _pack_coder(c, cn, cd, cv, se, P):
        def gdn(name, g):
            C = g.beta.numel()
            gamma = _reparam(P(g, "gamma"), g.gamma_reparam)  # (C_out, C_in)
            beta = _reparam(P(g, "beta"), g.beta_reparam)
            c[name] = pack_conv(gamma.reshape(C, C, 1, 1), beta)

        ga, gs = cd.g_a, cd.g_s
        for i in (0, 2, 5):
            cv(f"{cn}.ga{i}.conv1", ga[i].conv1, stride=2)
            cv(f"{cn}.ga{i}.conv2", ga[i].conv2)
            cv(f"{cn}.ga{i}.skip", ga[i].skip, pad=0, stride=2)
            gdn(f"{cn}.ga{i}.gdn", ga[i].gdn)
        for i in (1, 4, 6):
            cv(f"{cn}.ga{i}.conv1", ga[i].conv1)
            cv(f"{cn}.ga{i}.conv2", ga[i].conv2)
        se(f"{cn}.ga3", ga[3])
        cv(f"{cn}.ga7", ga[7], stride=2)
        se(f"{cn}.ga8", ga[8])
        for i in (0, 2, 4, 6, 8):
            cv(f"{cn}.ha{i}", cd.h_a[i], stride=cd.h_a[i].stride[0])
        cv(f"{cn}.hs0", cd.h_s[0])
        cv(f"{cn}.hs2", cd.h_s[2][0], shuffle=2)
        cv(f"{cn}.hs4", cd.h_s[4])
        cv(f"{cn}.hs6", cd.h_s[6][0], shuffle=2)
        cv(f"{cn}.hs8", cd.h_s[8])
        se(f"{cn}.gs0", gs[0])
        se(f"{cn}.gs5", gs[5])
        for i in (1, 3, 6, 8):
            cv(f"{cn}.gs{i}.conv1", gs[i].conv1)
            cv(f"{cn}.gs{i}.conv2", gs[i].conv2)
        for i in (2, 4, 7):
            cv(f"{cn}.gs{i}.subpel", gs[i].subpel_conv[0], shuffle=2)
            cv(f"{cn}.gs{i}.conv", gs[i].conv)
            cv(f"{cn}.gs{i}.upsample", gs[i].upsample[0], shuffle=2)
            gdn(f"{cn}.gs{i}.igdn", gs[i].igdn)
        cv(f"{cn}.gs9", gs[9][0], shuffle=2)
        ctx = cd.context_prediction
        c[f"{cn}.ctx"] = pack_conv(P(ctx, "weight") * P(ctx, "mask"), P(ctx, "bias"))  # MaskedConv2d 'A' (12 live taps)
        ep = cd.entropy_parameters
        cv(f"{cn}.ep0", ep[0], src_layout=[(256, 256), (256, 256)])
        cv(f"{cn}.ep2", ep[2], src_layout=[(ep[2].in_channels, _r(ep[2].in_channels, 4))])
        cv(f"{cn}.ep4", ep[4], src_layout=[(ep[4].in_channels, _r(ep[4].in_channels, 4))])
        c[f"{cn}.eb"] = pack_entropy_bottleneck(cd.entropy_bottleneck, P)


def pack_entropy_bottleneck(eb, P=None):
    """Host tensors of one EntropyBottleneck as the kernels (and coding.eb_tables) read them: (softplus(matrices) [C][33],
    biases [C][13], tanh(factors) [C][12], medians [C], quantiles [C][3], target [3])."""
    if P is None:
        P = lambda mod, name: getattr(mod, name).detach().float().cpu()
    Cc = eb.quantiles.shape[0]
    mats = torch.cat([F.softplus(P(eb, f"_matrix{i}")).reshape(Cc, -1) for i in range(5)], 1)
    biases = torch.cat([P(eb, f"_bias{i}").reshape(Cc, -1) for i in range(5)], 1)
    factors = torch.cat([torch.tanh(P(eb, f"_factor{i}")).reshape(Cc, -1) for i in range(4)], 1)
    if mats.shape[1] != 33 or biases.shape[1] != 13 or factors.shape[1] != 12:
        raise RuntimeError("EntropyBottleneck: expected filters (3, 3, 3, 3)")
    return (mats.contiguous(), biases.contiguous(), factors.contiguous(),
            P(eb, "quantiles")[:, 0, 1].contiguous(), P(eb, "quantiles").reshape(Cc, 3).contiguous(),
            P(eb, "target").reshape(3).contiguous())


_PACK_GEN = itertools.count(1)


def _upload(c, dev):
    """Host-packed weights -> one flat device buffer (a single H2D copy); every tensor of `c` becomes a view into it."""
    slots = []   # (setter, host tensor)
    for name, v in c.items():
        if isinstance(v, ConvW):
            v.wmax = float(v.w.abs().max())   # the split / one-product schemes scale their fp16 blocks by it (tc.attach_f16)
            slots.append((lambda t, v=v: setattr(v, "w", t), v.w))
            if v.b is not None:
                slots.append((lambda t, v=v: setattr(v, "b", t), v.b))
        elif isinstance(v, tuple):
            lst = [None] * len(v)
            c[name] = lst
            for i, t in enumerate(v):
                slots.append((lambda t2, lst=lst, i=i: lst.__setitem__(i, t2), t))
        else:
            slots.append((lambda t, name=name: c.__setitem__(name, t), v))
    offs, total = [], 0
    for _, t in slots:
        offs.append(total)
        total += _r(t.numel(), 64)   # 256-byte aligned pieces
    flat = torch.zeros(total, dtype=torch.float32)
    for (_, t), o in zip(slots, offs):
        flat[o:o + t.numel()] = t.reshape(-1)
    flat = flat.to(dev)
    for (setter, t), o in zip(slots, offs):
        setter(flat[o:o + t.numel()].view(t.shape))
    c["_flat"] = flat
    c["_gen"] = next(_PACK_GEN)   # plans compare it to know that their cached features / graphs belong to these weights
    return c


def _param_key(m):
    bufs = [b for n, b in m.named_buffers() if n.rsplit(".", 1)[-1] not in _CDF_BUFFERS]
    return tuple((p.data_ptr(), p._version) for p in list(m.parameters()) + bufs)


# =============================================================================== the plan
class _Plan:
    """Static buffer plan + launch sequence of one P-frame for a fixed (N, H, W) on one device, and the per-GOP feature
    caches: everything the reference recomputes for every P-frame from inputs that repeat inside a GOP -
    FeatureExtract_ref(I-frame) with its pooled descriptors (reference pnet.py:213-217, 225-233) and, per previous
    reconstruction, the frame-wise front of the multi-frame fusion (conv01, conv02, conv1, layer1.conv1, layer1.spatial_conv3d
    act on each frame separately: pnet.py:277-290, 309-312) - is keyed on a 128-bit content hash of the reference slice it was
    computed from and reused while that hash matches.  Results are bit-identical to recomputing (same kernels, same inputs)."""

    GDN_SLOTS = {f"{cn}.{l}": i for i, (cn, l) in enumerate((cn, l) for cn in ("mv", "rs")
                                                            for l in ("ga0", "ga2", "ga5", "gs2", "gs4", "gs7"))}

    def __init__(self, N, H, W, device):
        self.N, self.H, self.W, self.dev = N, H, W, device
        self.lib = L.load()
        self.bufs = {}
        # per-frame device state, zeroed by one memset: [mv_y, mv_z, res_y, res_z] sum ln p (fp64) | abs-max of every GDN input (fp32)
        self.fstate = torch.zeros(4 + 8, device=device, dtype=torch.float64)
        self.acc = self.fstate[:4]
        self.bpp = torch.zeros(2, device=device, dtype=torch.float32)   # [bpp_mv, bpp_res]
        self.impl = L.IMPL_AUTO
        self.precision = "exact"
        self.launches = 0
        self.last_csum = None
        self.prof = None  # list of (label, macs, bytes, start_event, end_event) when instrumented (bench.py)
        self._order = 0
        self.alternate_order = os.environ.get("TDVC_B200_NO_ALTERNATE") is None   # developer A/B switch
        self.overlap_hyper = os.environ.get("TDVC_B200_NO_OVERLAP") is None       # developer A/B switch
        self._side = None
        # caches
        self.if_key = None                       # hash of the I-frame slice whose FeatureExtract_ref output is resident
        self.ring = [None, None, None]           # hash of the reference slice whose fusion front sits in ring entry e
        self.ring_used = [0, 0, 0]
        self.frame_no = 0
        self.hdev = torch.zeros(8 * N, device=device, dtype=torch.int64)
        self.hpin = torch.zeros(8 * N, dtype=torch.int64).pin_memory()
        self.graphs = {}
        self.cache_hits = 0
        self.weights_gen = None
        # training-mode forward (`VideoCompressor.train()`): noise quantisation, FeatureFix at scale 8, aux losses
        self.training = False
        self.noise = None                        # {"mv.z" | "mv.y" | "mv.y_lik" | "rs.z" | ...: NHWC Act of U(-0.5, 0.5) noise}
        self.aux = torch.zeros(2, device=device, dtype=torch.float32)   # [mv_aux_loss, res_aux_loss]

    def bind(self, W):
        """Cached features and captured graphs belong to one set of packed weights."""
        if self.weights_gen != W["_gen"]:
            self.invalidate()
            self.weights_gen = W["_gen"]

    def invalidate(self):
        """Forget every cached feature (weights changed / buffers were used by another entry point)."""
        self.if_key = None
        self.ring = [None, None, None]
        self.graphs = {}

    def _prof_begin(self):
        if self.prof is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record(torch.cuda.current_stream(self.dev))
        return e

    def _prof_end(self, e0, label, macs=0, nbytes=0, products=0):
        if e0 is None:
            return
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record(torch.cuda.current_stream(self.dev))
        self.prof.append((label, macs, nbytes, e0, e1, products))   # products: fp16 MMA products per MAC (0: no MMA)

    # ---------------------------------------------------------------- buffers
    def buf(self, name, N, H, W, C, ld=None, zero=False):
        key = (name, N, H, W, C, ld)
        a = self.bufs.get(key)
        if a is None:
            a = Act.alloc(N, H, W, C, self.dev, ld=ld, zero=zero)
            self.bufs[key] = a
        return a

    def raw(self, name, shape, dtype=torch.float32):
        key = (name, tuple(shape), dtype)
        t = self.bufs.get(key)
        if t is None:
            t = torch.zeros(shape, device=self.dev, dtype=dtype)
            self.bufs[key] = t
        return t

    def absmax_ptr(self, layer):
        return self.fstate.data_ptr() + 32 + 4 * self.GDN_SLOTS[layer]

    # ---------------------------------------------------------------- kernel wrappers
    def _st(self):
        return torch.cuda.current_stream(self.dev).cuda_stream

    def conv(self, srcs, cw, out, stride=1, act=L.ACT_NONE, slope=0.0, res1=None, res2=None, post=L.POST_NONE,
             mul=None, in_square=False, impl=None, planar=False, absmax_out=None, absmax_in=None, products=None, csum=False):
        """planar=True: `out` is a plain (N, cout, Ho, Wo) tensor written as NCHW planes (no shuffle / residual).
        products: None = by `self.precision` and the layer's stage (ConvW.p1_ok); 0 / 1 force the scheme.
        csum=True: also produce the per-channel partial sums of the output for a following squeeze-excitation (`self.se(...,
        csum=self.last_csum)`); `self.last_csum` stays None when the launch cannot (exact fp32 SIMT kernel)."""
        p = L.ConvParams()
        s0 = srcs[0]
        cin = 0
        for i, s in enumerate(srcs):
            if (s.N, s.H, s.W) != (s0.N, s0.H, s0.W):
                raise RuntimeError("conv: sources differ in shape")
            p.src[i] = s.ptr
            sc = _r(s.C, 4)
            p.src_c[i] = sc
            p.src_ld[i] = s.ld
            cin += sc
        if cin != cw.cin or stride != cw.stride:
            raise RuntimeError(f"conv: input channels / stride {cin}, {stride} do not match the packed weight ({cw.cin}, {cw.stride})")
        p.n_src = len(srcs)
        p.N, p.H, p.W = s0.N, s0.H, s0.W
        p.Ho = (s0.H + 2 * cw.pad - cw.k) // stride + 1
        p.Wo = (s0.W + 2 * cw.pad - cw.k) // stride + 1
        sh = 2 if cw.shuffle == 2 else 1
        if planar:
            if tuple(out.shape) != (s0.N, cw.cout, p.Ho, p.Wo) or not out.is_contiguous() or sh != 1:
                raise RuntimeError("conv: planar output tensor has the wrong shape")
        elif (out.N, out.H, out.W) != (s0.N, p.Ho * sh, p.Wo * sh) or out.C != (cw.cout // 4 if cw.shuffle == 2 else cw.cout):
            raise RuntimeError(f"conv: output {(out.N, out.H, out.W, out.C)} does not match {(s0.N, p.Ho * sh, p.Wo * sh, cw.cout)}")
        p.weight = cw.w.data_ptr()
        p.bias = cw.b.data_ptr() if cw.b is not None else None
        p.cin, p.cin_pad, p.cout, p.cout_pad = cw.cin, cw.cin_pad, cw.cout, cw.cout_pad
        p.kh = p.kw = cw.k
        p.stride, p.pad = stride, cw.pad
        p.in_square = 1 if in_square else 0
        p.act, p.slope, p.post = act, slope, post
        if mul is not None:
            p.mul, p.mul_ld = mul.ptr, mul.ld
        if res1 is not None:
            p.res1, p.res1_ld = res1.ptr, res1.ld
        if res2 is not None:
            p.res2, p.res2_ld = res2.ptr, res2.ld
        if planar:
            p.out, p.out_ld, p.out_planar = out.data_ptr(), 0, 1
        else:
            p.out, p.out_ld = out.ptr, out.ld
        p.shuffle = cw.shuffle
        p.impl = self.impl if impl is None else impl
        if products is None:
            products = 1 if (self.precision == "mixed" and cw.p1_ok and cw.w_f16_p1 is not None and p.impl != L.IMPL_SIMT) else 0
        if products == 1:
            if cw.w_f16_p1 is None:
                raise RuntimeError("conv: this layer has no one-product weight blocks")
            p.products, p.weight_f16, p.w_shift = 1, cw.w_f16_p1.data_ptr(), cw.w_shift_p1
        else:
            p.weight_f16 = cw.w_f16.data_ptr() if cw.w_f16 is not None else None
            p.w_shift = cw.w_shift
        p.out_absmax, p.in_absmax = absmax_out, absmax_in
        self.last_csum = None
        if csum and not planar:
            rows = self.lib.tdvc_conv2d_chan_sum_rows(p)
            if rows > 0:
                part = self.raw(("se_csum", cw.cout, rows), (rows * s0.N * cw.cout,))
                L.check(self.lib.tdvc_zero_bytes(part.data_ptr(), part.numel() * 4, self._st()), "zero_bytes")
                p.chan_sum = part.data_ptr()
                self.last_csum = (part, rows)
        self._order ^= 1          # alternate the tile walk direction between consecutive layers (L2 reuse)
        p.order = self._order if self.alternate_order else 0
        if p.chan_sum:            # the partial channel sums are per CTA: their summation order must not depend on how many
            p.order = 0           # layers ran before this one (cache hits skip layers), so these launches always walk forwards
        e0 = self._prof_begin()
        L.check(self.lib.tdvc_conv2d(p, self._st()), "conv2d")
        if e0 is not None:
            npx = s0.N * p.Ho * p.Wo
            gdn = post != L.POST_NONE and mul is not None and mul.ptr == s0.ptr   # x is both the conv input and the multiplier
            name = ("gdn" if post == L.POST_GDN else "igdn") if gdn else f"conv{cw.k}x{cw.k}s{stride}"
            prod = max(self.lib.tdvc_conv2d_products(p), 0)
            if prod == 1:
                name += "_p1"
            # algorithmic bytes: inputs + output (+ multiplier / residual rows); a GDN reads x once (SURVEY.md 8d: 1,024 B/px)
            self._prof_end(e0, f"{name}_{cw.cin}to{cw.cout}@{p.Ho}x{p.Wo}",
                           macs=npx * cw.cout * cw.cin_real * cw.k * cw.k,
                           nbytes=4 * (s0.N * s0.H * s0.W * cw.cin_real +
                                       npx * cw.cout * (1 + (mul is not None and not gdn) + (res1 is not None) + (res2 is not None))),
                           products=prod)
        self.launches += 1
        return out

    def se(self, x, w, out, act=L.ACT_NONE, slope=0.0, res=None, csum=None, sub_from=None, out2=None):
        """Squeeze-excitation (reference inflate.py:159-208).  csum = `self.last_csum` of the convolution that produced x: the
        channel sums were accumulated in its epilogue, the pass over x for the mean is skipped."""
        w1, b1, w2, b2 = w
        HW = x.H * x.W
        if csum is not None:
            part, nblk = csum
        else:
            nblk = max(1, min(592, HW // 64))
            part = self.raw(("se_part", x.C), (nblk * x.N * x.C,))
            e0 = self._prof_begin()
            L.check(self.lib.tdvc_se_partial_sums(x.ptr, x.ld, x.N, HW, x.C, part.data_ptr(), nblk, self._st()), "se_partial_sums")
            self._prof_end(e0, f"se_partial_sums_{x.C}ch@{x.H}x{x.W}", 0, 4 * x.N * HW * x.C)
            self.launches += 1
        e0 = self._prof_begin()
        L.check(self.lib.tdvc_se_apply(x.ptr, x.ld, part.data_ptr(), nblk, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                                       b2.data_ptr(), x.N, HW, x.C, w1.shape[0], act, slope,
                                       res.ptr if res is not None else None, res.ld if res is not None else 0,
                                       out.ptr, out.ld, sub_from.ptr if sub_from is not None else None,
                                       sub_from.ld if sub_from is not None else 0, out2.ptr if out2 is not None else None,
                                       out2.ld if out2 is not None else 0, self._st()), "se_apply")
        self._prof_end(e0, f"se_apply_{x.C}ch@{x.H}x{x.W}", 0,
                       4 * x.N * HW * x.C * (2 + (res is not None) + 2 * (sub_from is not None)))
        self.launches += 2   # gate (one block per image), apply
        return out

    def call(self, fn, *a, nbytes=0, tag=""):
        e0 = self._prof_begin()
        L.check(getattr(self.lib, fn)(*a, self._st()), fn)
        self._prof_end(e0, fn[5:] + tag, 0, nbytes)
        self.launches += 1

    # ---------------------------------------------------------------- blocks
    def res_stack(self, W, prefix, n, x, tag, last_res2=None, out_last=None):
        """n x [x + conv2(relu(conv1 x))]  (reference utils.py:43-56)."""
        for i in range(n):
            t = self.conv([x], W[f"{prefix}.{i}.conv1"], self.buf(tag + ".t", x.N, x.H, x.W, 64), act=L.ACT_RELU)
            o = out_last if (i == n - 1 and out_last is not None) else self.buf(f"{tag}.o{i % 2}", x.N, x.H, x.W, 64)
            x = self.conv([t], W[f"{prefix}.{i}.conv2"], o, res1=x, res2=last_res2 if i == n - 1 else None)
        return x

    def coder(self, W, cn, x, acc_off, taps, final_res=None, out=None):
        """Cheng2020Anchor.forward with the reference's g_a / g_s (SURVEY App. A; encoder_v3.py:14-69)."""
        y, yh = self.analysis(W, cn, x)
        # The hyperprior / context / entropy-parameter chain only feeds the bit count (x_hat depends on round(y) alone,
        # SURVEY.md App. A): ~17 small, latency-bound launches at H/16..H/64.  They run on a side stream, concurrently
        # with the (equally small) first layers of g_s, and are joined before this coder returns.  (Serialised when the
        # launches are being timed one by one: an event pair on the side stream would time the wait behind a main-stream kernel.)
        main = torch.cuda.current_stream(self.dev)
        side = self._side_stream() if (self.overlap_hyper and self.prof is None) else None
        if side is not None:
            side.wait_stream(main)
        with torch.cuda.stream(side if side is not None else main):
            gp, z, zh = self._hyper_path(W, cn, y, yh, acc_off)
        xh = self.synthesis(W, cn, yh, final_res=final_res, out=out)
        if side is not None:
            main.wait_stream(side)
        if taps is not None:
            nm = "mv" if cn == "mv" else "res"
            taps.update({f"{nm}.y": y.nchw(), f"{nm}.z": z.nchw(), f"{nm}.y_hat": yh.nchw(), f"{nm}.z_hat": zh.nchw(),
                         f"{nm}.scales_hat": gp.chan(0, 128).nchw(), f"{nm}.means_hat": gp.chan(128, 128).nchw()})
        return xh

    def _cbuf(self, cn, N):
        """Buffer allocator of coder `cn`'s layers: b(name, h, w, c=128, **kw) -> plan buffer "{cn}.{name}"."""
        return lambda nme, h, w, c=128, **kw: self.buf(f"{cn}.{nme}", N, h, w, c, **kw)

    def analysis(self, W, cn, x):
        """g_a of coder `cn` and the quantiser of the forward pass: x (N, H, W, 64) -> (y, y_hat) at H/16 x W/16, y_hat =
        round(y) (eval) or y + U(-0.5, 0.5) (training).  Only the bit count and forward's reconstruction use this y_hat: a
        decoder sees the autoregressive one (`launch_coding`'s `{cn}.ac.y_hat`), which `compress` synthesises from."""
        N, H, Wd = x.N, x.H, x.W
        lr = dict(act=L.ACT_LRELU, slope=0.01)
        b = self._cbuf(cn, N)

        # GDN: the layer that produces the GDN input also maintains max |t2| (one atomic per epilogue warp); the GDN
        # kernel pre-scales x*x by a power of two from it so that the fp16 operands cannot saturate (csrc/conv_tc.cu)
        def rb_stride(i, x, h, w):
            am = self.absmax_ptr(f"{cn}.ga{i}")
            idt = self.conv([x], W[f"{cn}.ga{i}.skip"], b(f"ga{i}.id", h, w), stride=2)
            t = self.conv([x], W[f"{cn}.ga{i}.conv1"], b(f"ga{i}.t", h, w), stride=2, **lr)
            t2 = self.conv([t], W[f"{cn}.ga{i}.conv2"], b(f"ga{i}.t2", h, w), absmax_out=am)
            return self.conv([t2], W[f"{cn}.ga{i}.gdn"], b(f"ga{i}.o", h, w), in_square=True, post=L.POST_GDN,
                             mul=t2, res1=idt, absmax_in=am, csum=(i == 2))

        rb = self._rb(W, cn, b, lr)
        a = rb_stride(0, x, H // 2, Wd // 2)
        a = rb("ga", 1, a)
        a = rb_stride(2, a, H // 4, Wd // 4)
        a = self.se(a, W[f"{cn}.ga3"], b("ga3.o", a.H, a.W), csum=self.last_csum)
        a = rb("ga", 4, a)
        a = rb_stride(5, a, H // 8, Wd // 8)
        a = rb("ga", 6, a)
        a = self.conv([a], W[f"{cn}.ga7"], b("ga7.o", H // 16, Wd // 16), stride=2, csum=True)
        y = self.se(a, W[f"{cn}.ga8"], b("y", a.H, a.W), csum=self.last_csum)
        yh = b("y_hat", y.H, y.W)
        if self.training:   # compressai quantize(y, "noise"): y + U(-0.5, 0.5)   (JointAutoregressiveHierarchicalPriors.forward)
            self.call("tdvc_axpby", y.ptr, self.noise[f"{cn}.y"].ptr, yh.ptr, y.N * y.H * y.W * 128, 1.0, 1.0)
        else:
            self.call("tdvc_round_half_even", y.ptr, yh.ptr, y.N * y.H * y.W * 128, nbytes=8 * y.N * y.H * y.W * 128)
        return y, yh

    def _rb(self, W, cn, b, lr):
        def rb(pfx, i, x):
            t = self.conv([x], W[f"{cn}.{pfx}{i}.conv1"], b(f"{pfx}{i}.t", x.H, x.W), **lr)
            return self.conv([t], W[f"{cn}.{pfx}{i}.conv2"], b(f"{pfx}{i}.o", x.H, x.W), res1=x, **lr)
        return rb

    def synthesis(self, W, cn, yh, final_res=None, out=None):
        """g_s of coder `cn` on a given y_hat (N, h, w, 128) -> x_hat (N, 16h, 16w, 64) (+ final_res, fused into the last
        convolution; written to `out` if given).  The one g_s of forward, compress and decompress."""
        N, H, Wd = yh.N, 16 * yh.H, 16 * yh.W
        lr = dict(act=L.ACT_LRELU, slope=0.01)
        b = self._cbuf(cn, N)
        rb = self._rb(W, cn, b, lr)

        # IGDN: as the GDN of g_a (analysis)
        def rb_up(i, x):
            h, w = 2 * x.H, 2 * x.W
            am = self.absmax_ptr(f"{cn}.gs{i}")
            t = self.conv([x], W[f"{cn}.gs{i}.subpel"], b(f"gs{i}.t", h, w), **lr)
            t2 = self.conv([t], W[f"{cn}.gs{i}.conv"], b(f"gs{i}.t2", h, w), absmax_out=am)
            idt = self.conv([x], W[f"{cn}.gs{i}.upsample"], b(f"gs{i}.id", h, w))
            return self.conv([t2], W[f"{cn}.gs{i}.igdn"], b(f"gs{i}.o", h, w), in_square=True, post=L.POST_IGDN,
                             mul=t2, res1=idt, absmax_in=am, csum=(i == 4))

        g = self.se(yh, W[f"{cn}.gs0"], b("gs0.o", yh.H, yh.W))
        g = rb("gs", 1, g)
        g = rb_up(2, g)
        g = rb("gs", 3, g)
        g = rb_up(4, g)
        g = self.se(g, W[f"{cn}.gs5"], b("gs5.o", g.H, g.W), csum=self.last_csum)
        g = rb("gs", 6, g)
        g = rb_up(7, g)
        g = rb("gs", 8, g)
        return self.conv([g], W[f"{cn}.gs9"], out if out is not None else b("x_hat", H, Wd, 64), res1=final_res)

    def _side_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(device=self.dev)
        return self._side

    def _hyper_path(self, W, cn, y, yh, acc_off):
        """h_a, factorised prior on z, h_s, context model, entropy parameters, conditional likelihood -> sum ln p."""
        lr = dict(act=L.ACT_LRELU, slope=0.01)
        b = self._cbuf(cn, y.N)
        # ---- h_a
        h = self.conv([y], W[f"{cn}.ha0"], b("ha0", y.H, y.W), **lr)
        h = self.conv([h], W[f"{cn}.ha2"], b("ha2", y.H, y.W), **lr)
        h = self.conv([h], W[f"{cn}.ha4"], b("ha4", y.H // 2, y.W // 2), stride=2, **lr)
        h = self.conv([h], W[f"{cn}.ha6"], b("ha6", h.H, h.W), **lr)
        z = self.conv([h], W[f"{cn}.ha8"], b("z", h.H // 2, h.W // 2), stride=2)
        # ---- factorised prior on z: quantise + likelihood + sum ln p in one pass
        zh = b("z_hat", z.H, z.W)
        mats, biases, factors, med, quantiles, target = W[f"{cn}.eb"]
        if self.training:
            self.call("tdvc_eb_bits_noise", z.ptr, self.noise[f"{cn}.z"].ptr, zh.ptr, mats.data_ptr(), biases.data_ptr(),
                      factors.data_ptr(), z.N * z.H * z.W, 128, self.acc.data_ptr() + 8 * (acc_off + 1))
            # EntropyBottleneck.loss() of this coder (reference pnet.py:35,59: `aux_loss()`)
            self.call("tdvc_eb_aux_loss", mats.data_ptr(), biases.data_ptr(), factors.data_ptr(), quantiles.data_ptr(),
                      target.data_ptr(), 128, self.aux.data_ptr() + 4 * (acc_off // 2))
        else:
            self.call("tdvc_eb_bits", z.ptr, zh.ptr, mats.data_ptr(), biases.data_ptr(), factors.data_ptr(), med.data_ptr(),
                      z.N * z.H * z.W, 128, self.acc.data_ptr() + 8 * (acc_off + 1))
        params = self.hyper_synthesis(W, cn, zh, b)
        # ---- context model, entropy parameters, conditional likelihood
        ctx = self.conv([yh], W[f"{cn}.ctx"], b("ctx", y.H, y.W, 256))
        c0, c2 = W[f"{cn}.ep0"].cout, W[f"{cn}.ep2"].cout
        e = self.conv([params, ctx], W[f"{cn}.ep0"], b("ep0", y.H, y.W, c0, ld=_r(c0, 8), zero=True), **lr)
        e = self.conv([e], W[f"{cn}.ep2"], b("ep2", y.H, y.W, c2, ld=_r(c2, 8), zero=True), **lr)
        gp = self.conv([e], W[f"{cn}.ep4"], b("gp", y.H, y.W, 256))
        if self.training:   # GaussianConditional.forward draws its own noise for the likelihood
            self.call("tdvc_gc_bits_noise", y.ptr, self.noise[f"{cn}.y_lik"].ptr, gp.ptr, gp.ld, y.N * y.H * y.W, 128,
                      self.acc.data_ptr() + 8 * acc_off)
        else:
            self.call("tdvc_gc_bits", y.ptr, gp.ptr, gp.ld, y.N * y.H * y.W, 128, self.acc.data_ptr() + 8 * acc_off,
                      nbytes=12 * y.N * y.H * y.W * 128)
        return gp, z, zh

    def hyper_synthesis(self, W, cn, zh, b):
        """h_s of coder `cn`: z_hat (N, H/64, W/64, 128) -> params (N, H/16, W/16, 256), the scales and means the entropy
        parameters start from.  The one h_s of both ends: the encoder runs it on its quantised z (`_hyper_path`), the decoder
        (`VideoCompressor.decompress_latents`) on the z_hat it decoded.  b(name, h, w, c=128, **kw) allocates the buffers."""
        lr = dict(act=L.ACT_LRELU, slope=0.01)
        s = self.conv([zh], W[f"{cn}.hs0"], b("hs0", zh.H, zh.W), **lr)
        s = self.conv([s], W[f"{cn}.hs2"], b("hs2", 2 * zh.H, 2 * zh.W), **lr)
        s = self.conv([s], W[f"{cn}.hs4"], b("hs4", s.H, s.W, 192), **lr)
        s = self.conv([s], W[f"{cn}.hs6"], b("hs6", 2 * s.H, 2 * s.W, 192), **lr)
        return self.conv([s], W[f"{cn}.hs8"], b("params", s.H, s.W, 256))

    # ---------------------------------------------------------------- cache keys and the variant of a frame
    def _variant(self, refs, cache, ref_keys=None):
        """Decide, from the content hashes of the four reference slices (or from the caller's own identities of them,
        `ref_keys`), what this frame has to compute.
        Returns (if_miss, assign, misses, keys): assign[j] = ring entry holding the fusion front of refer_frames[:, j + 1];
        misses = ((entry, j), ...) entries to compute from refer_frames[:, j + 1]."""
        N, H, Wd = self.N, self.H, self.W
        if not cache:
            return True, (0, 1, 2), ((0, 0), (1, 1), (2, 2)), [None] * 4
        if ref_keys is not None:
            keys = [("id", k) for k in ref_keys]
        else:
            fr = 3 * H * Wd
            L.check(self.lib.tdvc_slices_hash(refs.data_ptr(), fr, fr, 4 * N, self.hdev.data_ptr(), self._st()), "slices_hash")
            self.launches += 1
            self.hpin.copy_(self.hdev, non_blocking=True)
            torch.cuda.current_stream(self.dev).synchronize()
            hv = self.hpin.view(N, 4, 2).tolist()
            keys = [tuple((hv[n][j][0], hv[n][j][1]) for n in range(N)) for j in range(4)]
        if_miss = keys[0] != self.if_key
        if not any(k is not None and k in keys[1:] for k in self.ring):
            # nothing of the ring is referenced any more (a new GOP): start from the canonical empty state, so that every GOP
            # walks through the same sequence of launch variants (and replays the graphs captured for the first one)
            self.ring, self.ring_used = [None, None, None], [0, 0, 0]
        assign, misses, taken = [None] * 3, [], set()
        for j in range(3):
            for e in range(3):
                if self.ring[e] is not None and self.ring[e] == keys[j + 1]:
                    assign[j] = e
                    taken.add(e)
                    break
        for j in (2, 1, 0):   # newest first: refer_frames[:, 3] is converted to NHWC for the feature extractor anyway
            if assign[j] is not None:
                continue
            same = [e for (e, jj) in misses if keys[jj + 1] == keys[j + 1]]
            if same:
                assign[j] = same[0]
                continue
            free = [e for e in range(3) if e not in taken]
            e = min(free, key=lambda q: self.ring_used[q])
            taken.add(e)
            assign[j] = e
            misses.append((e, j))
        self.cache_hits += (0 if if_miss else 1) + (3 - len(misses))
        return if_miss, tuple(assign), tuple(misses), keys

    # ---------------------------------------------------------------- one P-frame
    def run(self, W, x_nchw, refs_nchw, taps=None, graph=False, cache=True, ref_keys=None):
        """reference pnet.py:26-83 (eval branch).  x (N,3,H,W), refs (N,4,3,H,W) contiguous fp32 CUDA.
        Returns the plan's static (recon (N,3,H,W), bpp [mv, res]) buffers."""
        N, H, Wd = self.N, self.H, self.W
        self.launches = 0
        if_miss, assign, misses, keys = self._variant(refs_nchw, cache, ref_keys)
        # ---- prologue (eager: reads the caller's tensors): NCHW -> NHWC (ld 4) of what this frame needs
        imgs = self.buf("imgs", 2 * N, H, Wd, 3, ld=4)        # [0:N] = input, [N:2N] = x^(t-1)
        self.call("tdvc_nchw_to_nhwc", x_nchw.data_ptr(), imgs.ptr, N, 3, H, Wd, 4, nbytes=28 * N * H * Wd)
        miss_imgs = self._load_refs(refs_nchw, if_miss, misses, imgs.batch(N, N))
        variant = (if_miss, assign, tuple((e, j) for e, j in misses), self.impl, self.precision)
        pre = self.launches
        if graph and taps is None and self.prof is None:
            g = self.graphs.get(variant)
            if g is None:
                # first frame of this variant: run it eagerly (allocates its buffers), then record it for the next time
                self.body(W, if_miss, assign, misses, miss_imgs, None)
                n_body = self.launches - pre
                graph_obj = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph_obj):
                    self.body(W, if_miss, assign, misses, miss_imgs, None)
                self.graphs[variant] = (graph_obj, n_body)
                self.launches = pre + n_body
            else:
                g[0].replay()
                self.launches = pre + g[1]
        else:
            self.body(W, if_miss, assign, misses, miss_imgs, taps)
        self._commit(cache, keys, assign, misses)
        return self.raw("recon", (N, 3, H, Wd)), self.bpp

    def _load_refs(self, refs_nchw, if_miss, misses, last):
        """NCHW -> NHWC (ld 4) of the reference slices a frame reads: refer_frames[:, 3] into `last` (N images) always, the
        I-frame and the references whose fusion front missed the ring only when they missed.  Returns {ring entry: images}."""
        N, H, Wd = self.N, self.H, self.W
        ifr = self.buf("iframe", N, H, Wd, 3, ld=4)
        fr = 3 * H * Wd * 4
        miss_imgs = {}
        for n in range(N):
            base = refs_nchw.data_ptr() + n * 4 * fr
            if if_miss:
                self.call("tdvc_nchw_to_nhwc", base, ifr.batch(n).ptr, 1, 3, H, Wd, 4, nbytes=28 * H * Wd)
            self.call("tdvc_nchw_to_nhwc", base + 3 * fr, last.batch(n).ptr, 1, 3, H, Wd, 4, nbytes=28 * H * Wd)
            for e, j in misses:
                if j == 2:
                    miss_imgs[e] = last
                else:
                    mi = miss_imgs.setdefault(e, self.buf(f"mf.img{j}", N, H, Wd, 3, ld=4))
                    self.call("tdvc_nchw_to_nhwc", base + (j + 1) * fr, mi.batch(n).ptr, 1, 3, H, Wd, 4, nbytes=28 * H * Wd)
        return miss_imgs

    def _commit(self, cache, keys, assign, misses):
        """The caches now hold what this frame computed."""
        self.frame_no += 1
        if cache:
            self.if_key = keys[0]
            for e, j in misses:
                self.ring[e] = keys[j + 1]
            for e in set(assign):
                self.ring_used[e] = self.frame_no
        else:
            self.if_key, self.ring = None, [None, None, None]

    def _frame_start(self, W, if_miss, misses, miss_imgs):
        """Per-frame state (bit sums, GDN maxima) to zero, then the per-GOP / per-reference features that missed their cache."""
        self._order = 0
        self.call("tdvc_zero_bytes", self.fstate.data_ptr(), self.fstate.numel() * 8)
        self.launches -= 1   # a memset node, not a kernel
        if if_miss:
            self.loopfilter_ref(W, self.buf("iframe", self.N, self.H, self.W, 3, ld=4))
        for e, j in misses:
            self.mcfilter_front(W, miss_imgs[e], e)

    def body(self, W, if_miss, assign, misses, miss_imgs, taps):
        """Everything of the frame that only touches plan buffers (graph-capturable)."""
        N, H, Wd = self.N, self.H, self.W
        self._frame_start(W, if_miss, misses, miss_imgs)
        imgs = self.buf("imgs", 2 * N, H, Wd, 3, ld=4)
        # ---- feature extraction on both images (pnet.py:29-30, 86-96)
        feats = self.features(W, imgs)
        in_f, ref_f = feats.batch(0, N), feats.batch(N, N)
        # ---- motion estimation (pnet.py:131-167)
        estmv = self.motion_est(W, feats, imgs, taps)
        # ---- motion coder (pnet.py:34-43)
        mv_xhat = self.coder(W, "mv", estmv, 0, taps)
        # ---- prediction (pnet.py:52-53); the residual input_feat - prediction of pnet.py:55 is written by the same pass
        resid = self.buf("resid", N, H, Wd, 64)
        pred1, pred = self.predict(W, mv_xhat, ref_f, assign, in_f, resid, taps)
        # ---- residual coder (pnet.py:55-67, 76)
        rec_f = self.coder(W, "rs", resid, 2, taps, final_res=pred, out=self.buf("rec_f", N, H, Wd, 64))
        self.finish(W, rec_f, taps)
        # ---- bpp (pnet.py:38-43, 62-67): sum ln p / (-ln2 * N*H*W), per coder
        self.call("tdvc_bpp_finish", self.acc.data_ptr(), self.bpp.data_ptr(), C.c_double(-1.0 / (_LN2 * N * H * Wd)))
        if taps is not None:
            self._stage_taps(taps, mv_xhat, pred1, pred, rec_f)
            taps.update({"input_feat": in_f.nchw(), "ref_feat": ref_f.nchw(), "estmv": estmv.nchw(),
                         "input_residual": resid.nchw()})

    @staticmethod
    def _stage_taps(taps, mv_xhat, pred1, pred, rec_f):
        taps.update({"mv.x_hat": mv_xhat.nchw(), "prediction1": pred1.nchw(), "prediction": pred.nchw(),
                     "recon_feat": rec_f.nchw()})

    def features(self, W, imgs, tag="fe", out="feats"):
        """extra_fea (pnet.py:86-96) on a batch of images (N, H, W, 3 in ld 4) -> (N, H, W, 64).  Every launch works on
        tiles of one image and picks its configuration from nothing but the layer's shape, so an image's features do not
        depend on what else is in the batch: the decoder's reference-only batch reproduces the encoder's [input; ref]."""
        f0 = self.conv([imgs], W["extra_fea.conv_first"], self.buf(tag + ".0", imgs.N, imgs.H, imgs.W, 64),
                       act=L.ACT_LRELU, slope=0.1)
        return self.res_stack(W, "extra_fea.res", 2, f0, tag, out_last=self.buf(out, imgs.N, imgs.H, imgs.W, 64))

    def predict(self, W, mv_xhat, ref_f, assign, sub_from=None, out2=None, taps=None):
        """The prediction from the decoded motion x_hat and the reference features: motion compensation (pnet.py:52,
        179-184; dcn_v2_amp.py:219-234) and the multi-frame fusion (:53, 277-293, 309-317) over the references of ring
        entries `assign`.  Returns (prediction1, prediction); with sub_from / out2 the fusion's last pass also writes
        out2 = sub_from - prediction (the residual of pnet.py:55)."""
        N, H, Wd = self.N, self.H, self.W
        lr1 = dict(act=L.ACT_LRELU, slope=0.1)
        dcn_out = self.buf("mc.dcn", N, H, Wd, 64)
        dp = L.DcnParams()
        wb = W.get("mc.dcn.w_f16")
        tc_dcn = self.impl != L.IMPL_SIMT and wb is not None
        if tc_dcn:
            # tcgen05 DCN (csrc/dcn_tc.cu): offsets / mask as NCHW planes straight from the offset conv's epilogue,
            # reference features regrouped to one 32-byte sector per (pixel, deformable group)
            om = self.raw("mc.om_planar", (N, 216, H, Wd))
            self.conv([mv_xhat], W["mc.offmask"], om, planar=True)
            ref_gp = self.raw("mc.ref_gp", (N * 8, H, Wd, 8))
            self.call("tdvc_nhwc_to_group_planar", ref_f.ptr, ref_f.ld, ref_gp.data_ptr(), N, H, Wd, 64,
                      nbytes=N * H * Wd * 512)
            dp.input_gp, dp.params_planar = ref_gp.data_ptr(), 1
            dp.offset, dp.off_ld = om.data_ptr(), 216
            dp.mask, dp.mask_ld, dp.mask_is_logit = om.data_ptr() + 4 * 144 * H * Wd, 216, 1
            dp.weight_f16 = wb.data_ptr()
        else:
            om = self.conv([mv_xhat], W["mc.offmask"], self.buf("mc.om", N, H, Wd, 216, ld=216))
            dp.input, dp.in_ld = ref_f.ptr, ref_f.ld
            dp.offset, dp.off_ld = om.ptr, om.ld
            dp.mask, dp.mask_ld, dp.mask_is_logit = om.chan(144, 72).ptr, om.ld, 1
        dp.weight_packed, dp.bias = W["mc.dcn.w"].data_ptr(), W["mc.dcn.b"].data_ptr()
        dp.out, dp.out_ld = dcn_out.ptr, dcn_out.ld
        dp.N, dp.H, dp.W, dp.C, dp.O, dp.O_pad, dp.dg = N, H, Wd, 64, 64, 64, 8
        dp.round_fp16, dp.act, dp.slope = 1, L.ACT_LRELU, 0.1
        dp.impl = self.impl
        e0 = self._prof_begin()
        L.check(self.lib.tdvc_dcn_nhwc(dp, self._st()), "dcn_nhwc")
        # algorithmic bytes: ref 256 + offsets 576 + masks 288 + out 256 B/px (SURVEY.md 8d)
        self._prof_end(e0, "dcn_tc" if tc_dcn else "dcn_nhwc", macs=N * H * Wd * 576 * 64, nbytes=N * H * Wd * 1376,
                       products=4 if tc_dcn else 0)
        self.launches += 1
        o2 = self.conv([dcn_out, ref_f], W["mc.conv"], self.buf("mc.o2", N, H, Wd, 64), **lr1)
        pred1 = self.res_stack(W, "mc.res", 3, o2, "mc", last_res2=dcn_out, out_last=self.buf("pred1", N, H, Wd, 64))
        pred = self.mcfilter(W, pred1, assign, sub_from, out2)
        if taps is not None:
            taps.update({"mcnet.om": om.clone() if tc_dcn else om.nchw(), "mcnet.dcn_act": dcn_out.nchw()})
        return pred1, pred

    def finish(self, W, rec_f, taps):
        """The reconstruction from the reconstructed features (residual x_hat + prediction): reference-based in-loop filter
        (pnet.py:213-263) with the clamp (:78) in its last convolution, then NCHW.  Returns the plan's recon buffer."""
        N, H, Wd = self.N, self.H, self.W
        recon4 = self.loopfilter(W, rec_f, taps)
        recon = self.raw("recon", (N, 3, H, Wd))
        self.call("tdvc_nhwc_to_nchw", recon4.ptr, recon4.ld, recon.data_ptr(), N, 3, H, Wd, nbytes=28 * N * H * Wd)
        return recon

    # ---------------------------------------------------------------- the closed loop: encoder and decoder of one P-frame
    def compress(self, W, tables, x_nchw, refs_nchw, cache=True, ref_keys=None, taps=None):
        """Closed-loop encoder of one P-frame (eager).  Both syntheses run on the autoregressive y_hat the strings code
        (round(y - mu) + mu, `launch_coding`), not on forward's round(y), so the reconstruction is the frame a decoder
        rebuilds.  The residual coder's input depends on the motion coder's autoregressive pass, so the two passes run one
        after the other; the host rANS of both (`coding.finish_coding`) is left to the caller and overlaps what is queued.
        tables: {"mv" | "rs": coding.CoderTables}.  Returns (the plan's recon buffer, {"mv" | "res": launch_coding handle})."""
        N, H, Wd = self.N, self.H, self.W
        self.launches = 0
        if_miss, assign, misses, keys = self._variant(refs_nchw, cache, ref_keys)
        imgs = self.buf("imgs", 2 * N, H, Wd, 3, ld=4)
        self.call("tdvc_nchw_to_nhwc", x_nchw.data_ptr(), imgs.ptr, N, 3, H, Wd, 4, nbytes=28 * N * H * Wd)
        miss_imgs = self._load_refs(refs_nchw, if_miss, misses, imgs.batch(N, N))
        self._frame_start(W, if_miss, misses, miss_imgs)
        feats = self.features(W, imgs)
        in_f, ref_f = feats.batch(0, N), feats.batch(N, N)
        estmv = self.motion_est(W, feats, imgs, None)
        handles = {}
        handles["mv"], mv_yh = self._analyse_and_code(W, tables, "mv", estmv, 0)
        mv_xhat = self.synthesis(W, "mv", mv_yh)
        resid = self.buf("resid", N, H, Wd, 64)
        pred1, pred = self.predict(W, mv_xhat, ref_f, assign, in_f, resid)
        handles["res"], rs_yh = self._analyse_and_code(W, tables, "rs", resid, 2)
        rec_f = self.synthesis(W, "rs", rs_yh, final_res=pred, out=self.buf("rec_f", N, H, Wd, 64))
        recon = self.finish(W, rec_f, None)
        if taps is not None:
            self._stage_taps(taps, mv_xhat, pred1, pred, rec_f)
        self._commit(cache, keys, assign, misses)
        return recon, handles

    def _analyse_and_code(self, W, tables, cn, x, acc_off):
        """g_a, the hyper path (as forward runs it) and the device half of coding for coder `cn`.  Returns (launch_coding
        handle, its autoregressive y_hat as an Act over the same memory)."""
        from tdvc_b200 import coding
        y, yh = self.analysis(W, cn, x)
        self._hyper_path(W, cn, y, yh, acc_off)
        h = coding.launch_coding(self, W, cn, tables[cn])
        t = h["dev"]["y_hat"]
        return h, Act(t, t.data_ptr(), y.N, y.H, y.W, 128, 128)

    def decompress(self, W, y_hat, refs_nchw, cache=True, ref_keys=None, taps=None):
        """Decoder of one P-frame from both coders' decoded y_hat ({"mv" | "rs": Act (N, H/16, W/16, 128)}) and the
        reference frames: extra_fea of refer_frames[:, -1], motion g_s, the prediction, residual g_s + prediction and the
        in-loop filter - the encoder's launches on the same shapes.  The per-GOP caches serve as in `run`.  Returns the
        plan's recon buffer."""
        N, H, Wd = self.N, self.H, self.W
        self.launches = 0
        if_miss, assign, misses, keys = self._variant(refs_nchw, cache, ref_keys)
        ref = self.buf("dec.ref", N, H, Wd, 3, ld=4)
        miss_imgs = self._load_refs(refs_nchw, if_miss, misses, ref)
        self._frame_start(W, if_miss, misses, miss_imgs)
        ref_f = self.features(W, ref, "dec.fe", "dec.ref_f")
        mv_xhat = self.synthesis(W, "mv", y_hat["mv"])
        pred1, pred = self.predict(W, mv_xhat, ref_f, assign)
        rec_f = self.synthesis(W, "rs", y_hat["rs"], final_res=pred, out=self.buf("rec_f", N, H, Wd, 64))
        recon = self.finish(W, rec_f, None)
        if taps is not None:
            self._stage_taps(taps, mv_xhat, pred1, pred, rec_f)
        self._commit(cache, keys, assign, misses)
        return recon

    def fusion_and_filter(self, W, pred1_nchw, refs_nchw, recf_nchw):
        """BASELINE config 5: the multi-frame feature fusion (reference pnet.py:266-293, 296-317) and the reference-based
        in-loop filter (:187-263) on their own.  pred1 / recf (N,64,H,W), refs (N,4,3,H,W) contiguous fp32 CUDA."""
        N, H, Wd = self.N, self.H, self.W
        self._order = 0
        self.launches = 0
        self.if_key, self.ring = None, [None, None, None]   # the cache entries are overwritten below
        ifr = self.buf("iframe", N, H, Wd, 3, ld=4)
        fr = 3 * H * Wd * 4
        imgs = [self.buf(f"mf.img{j}", N, H, Wd, 3, ld=4) for j in range(3)]
        for n in range(N):
            base = refs_nchw.data_ptr() + n * 4 * fr
            self.call("tdvc_nchw_to_nhwc", base, ifr.batch(n).ptr, 1, 3, H, Wd, 4)
            for j in range(3):
                self.call("tdvc_nchw_to_nhwc", base + (j + 1) * fr, imgs[j].batch(n).ptr, 1, 3, H, Wd, 4)
        pred1 = self.buf("pred1", N, H, Wd, 64)
        self.call("tdvc_nchw_to_nhwc", pred1_nchw.data_ptr(), pred1.ptr, N, 64, H, Wd, 64)
        rec_f = self.buf("rec_f", N, H, Wd, 64)
        self.call("tdvc_nchw_to_nhwc", recf_nchw.data_ptr(), rec_f.ptr, N, 64, H, Wd, 64)
        for j in range(3):
            self.mcfilter_front(W, imgs[j], j)
        pred = self.mcfilter(W, pred1, (0, 1, 2))
        self.loopfilter_ref(W, ifr)
        recon4 = self.loopfilter(W, rec_f, None)
        pred_out = self.raw("c5.pred", (N, 64, H, Wd))
        recon = self.raw("recon", (N, 3, H, Wd))
        self.call("tdvc_nhwc_to_nchw", pred.ptr, pred.ld, pred_out.data_ptr(), N, 64, H, Wd)
        self.call("tdvc_nhwc_to_nchw", recon4.ptr, recon4.ld, recon.data_ptr(), N, 3, H, Wd)
        return pred_out, recon

    def motion_est(self, W, feats, imgs, taps):
        N, H, Wd = self.N, self.H, self.W
        lr1 = dict(act=L.ACT_LRELU, slope=0.1)
        b = lambda nme, n, h, w, c=64: self.buf("me." + nme, n, h, w, c)
        # feature pyramid on both images at once (pnet.py:132-140)
        l2 = self.conv([feats], W["me.conv_l2_1"], b("l2a", 2 * N, H // 2, Wd // 2), stride=2, **lr1)
        l2 = self.conv([l2], W["me.conv_l2_2"], b("l2", 2 * N, H // 2, Wd // 2), **lr1)
        l3 = self.conv([l2], W["me.conv_l3_1"], b("l3a", 2 * N, H // 4, Wd // 4), stride=2, **lr1)
        l3 = self.conv([l3], W["me.conv_l3_2"], b("l3", 2 * N, H // 4, Wd // 4), **lr1)
        pyr = {1: feats, 2: l2, 3: l3}
        up = None
        for i in (3, 2, 1):  # pnet.py:146-160
            lv = f"l{i}"
            p = pyr[i]
            h, w = p.H, p.W
            o1 = self.conv([p.batch(0, N), p.batch(N, N)], W[f"me.c11.{lv}"], b(f"o1a.{lv}", N, h, w), **lr1)
            o1 = self.conv([o1], W[f"me.c11_1.{lv}"], b(f"o1.{lv}", N, h, w), **lr1)
            if i == 3:
                off = self.conv([o1], W["me.c12.l3"], b(f"off.{lv}", N, h, w), **lr1)
            else:
                off = self.conv([up, o1], W[f"me.ff.{lv}"], b(f"off.{lv}", N, h, w), **lr1)
            if i > 1:
                u = b(f"up2x.{lv}", N, 2 * h, 2 * w)
                self.call("tdvc_upsample2x", off.ptr, u.ptr, N, h, w, 64, nbytes=1280 * N * h * w, tag=f"@{h}x{w}")  # read 256 + write 4 * 256 B/px
                up = self.conv([u], W["me.upsample_conv"], b(f"up.{lv}", N, 2 * h, 2 * w))
            if taps is not None:
                taps[f"motion_est.offset_{lv}"] = off.nchw()
        flow = self.spynet(W, imgs, taps)
        offf = b("off_flow", N, H, Wd)
        self.call("tdvc_add_flow_tiled", off.ptr, flow.ptr, offf.ptr, N, H, Wd, 64, nbytes=520 * N * H * Wd)
        ff = self.conv([offf], W["me.feat_fusion_"], b("ff", N, H, Wd), csum=True)
        return self.se(ff, W["me.attn"], b("estmv", N, H, Wd), csum=self.last_csum)

    def spynet(self, W, imgs, taps):
        """reference flownet.py:82-140 with ref = input image, supp = x^(t-1) (pnet.py:162)."""
        N, H, Wd = self.N, self.H, self.W
        pyr = [imgs]
        for l in range(5):
            s = pyr[-1]
            d = self.buf(f"spy.pyr{l}", 2 * N, s.H // 2, s.W // 2, 3, ld=4)
            self.call("tdvc_avgpool2x2", s.ptr, d.ptr, 2 * N, s.H, s.W, 4, nbytes=20 * 2 * N * s.H * s.W, tag=f"@{s.H}x{s.W}")
            pyr.append(d)
        pyr = pyr[::-1]
        flow = None
        for lvl in range(6):
            im = pyr[lvl]
            h, w = im.H, im.W
            x8 = self.buf(f"spy.in{lvl}", N, h, w, 8)
            self.call("tdvc_spynet_prep", im.batch(0, N).ptr, im.batch(N, N).ptr, flow.ptr if flow is not None else None,
                      x8.ptr, N, h, w, nbytes=N * h * w * 66, tag=f"@{h}x{w}")  # ref 16 + supp 16 + coarse flow 2 + out 32 B/px
            t = self.conv([x8], W[f"spy.{lvl}.0"], self.buf(f"spy.a{lvl}", N, h, w, 32), act=L.ACT_RELU)
            t = self.conv([t], W[f"spy.{lvl}.1"], self.buf(f"spy.b{lvl}", N, h, w, 64), act=L.ACT_RELU)
            t = self.conv([t], W[f"spy.{lvl}.2"], self.buf(f"spy.c{lvl}", N, h, w, 32), act=L.ACT_RELU)
            t = self.conv([t], W[f"spy.{lvl}.3"], self.buf(f"spy.d{lvl}", N, h, w, 16), act=L.ACT_RELU)
            flow = self.conv([t], W[f"spy.{lvl}.4"], self.buf(f"spy.flow{lvl}", N, h, w, 2), res1=x8.chan(6, 2))
            if taps is not None:
                taps[f"spynet.flow{lvl}"] = flow.nchw()
        return flow

    # ---- multi-frame fusion (reference LoopFilter, pnet.py:266-293 + Bottleneck3D :296-317).  Every layer in front of the
    # temporal convolution acts on one frame at a time (Conv3d kernels (1,3,3)), so the front of a reference frame -
    # a = lrelu(conv1(conv02(lrelu(conv01 x)))) and s = spatial(lrelu(layer1.conv1 a)) - is computed once per reconstruction and
    # kept in a 3-entry ring for the three P-frames that reference it.
    def mcfilter_front(self, W, img, e):
        N, H, Wd = self.N, self.H, self.W
        lr1 = dict(act=L.ACT_LRELU, slope=0.1)
        b = lambda nme, c=64: self.buf("mf." + nme, N, H, Wd, c)
        r = self.conv([img], W["mf.conv01"], b("r01"), **lr1)
        f = self.conv([r], W["mf.conv02"], b("f02"))
        a = self.conv([f], W["mf.conv1"], b(f"a.{e}"), **lr1)
        c1 = self.conv([a], W["mf.l1.conv1"], b("c1"), **lr1)
        return self.conv([c1], W["mf.l1.spatial"], b(f"s.{e}"))

    def mcfilter(self, W, pred1, assign, sub_from=None, out2=None):
        N, H, Wd = self.N, self.H, self.W
        lr1 = dict(act=L.ACT_LRELU, slope=0.1)
        b = lambda nme, c=64: self.buf("mf." + nme, N, H, Wd, c)
        # the prediction is the 4th "frame" of the stack (pnet.py:286-288)
        a_p = self.conv([pred1], W["mf.conv1"], b("a.p"), **lr1)
        c1 = self.conv([a_p], W["mf.l1.conv1"], b("c1"), **lr1)
        s_p = self.conv([c1], W["mf.l1.spatial"], b("s.p"))
        A = [b(f"a.{e}") for e in assign] + [a_p]
        S = [b(f"s.{e}") for e in assign] + [s_p]
        # temporal (3,1,1) stride 3: one output step from frames 0..2, broadcast-added to all four (pnet.py:313-314)
        tmp = self.conv(S[:3], W["mf.l1.temporal"], b("tmp"))
        # o_t = lrelu(s_t + tmp) for the distinct frames of the stack in ONE pass (tmp is read once); duplicated references (GOP
        # warm-up, predict.py:55-60) share their entry
        keys, first = [], {}
        for t in range(4):
            k = assign[t] if t < 3 else "p"
            keys.append(k)
            first.setdefault(k, t)
        uniq = list(first.items())
        xs = (C.c_void_p * 4)(*[S[t].ptr for _, t in uniq])
        os_ = (C.c_void_p * 4)(*[b(f"o.{k}").ptr for k, _ in uniq])
        self.call("tdvc_bcast_add_lrelu_multi", xs, tmp.ptr, os_, len(uniq), N * H * Wd * 64, 0.1,
                  nbytes=(2 * len(uniq) + 1) * 256 * N * H * Wd)
        done = {k: self.conv([b(f"o.{k}")], W["mf.l1.conv3"], b(f"bo.{k}"), res1=A[t]) for k, t in uniq}
        bo = [done[k] for k in keys]
        fu = self.conv(bo, W["mf.fusion"], b("fu"), csum=True, **lr1)
        return self.se(fu, W["mf.attn"], self.buf("pred", N, H, Wd, 64), res=pred1, csum=self.last_csum, sub_from=sub_from, out2=out2)

    # ---- reference-based in-loop filter (reference FeatureFix, pnet.py:187-263)
    def _ff_geometry(self):
        H, Wd = self.H, self.W
        scale = 8 if self.training else int(H / 8)  # pnet.py:220-223
        ph, pw = H // scale, Wd // scale
        PH, PW = (ph + 3) // 3 + 1, (pw + 3) // 3 + 1
        bs = 3 * scale
        if (H + bs) // bs + 1 != PH or (Wd + bs) // bs + 1 != PW:
            raise RuntimeError(f"FeatureFix: patch grid {PH}x{PW} does not match the block grid of a {H}x{Wd} frame")
        return scale, ph, pw, PH * PW

    def _fe(self, W, pfx, x, tag):
        b = lambda nme, c=64: self.buf("lf." + nme, self.N, self.H, self.W, c)
        x1 = self.conv([x], W[pfx + ".first"], b(tag + ".x1"), act=L.ACT_LRELU, slope=0.01)
        y = self.res_stack(W, pfx + ".body", 2, x1, "lf." + tag)
        return self.conv([y], W[pfx + ".last"], b(tag + ".f"), res1=x1)

    def loopfilter_ref(self, W, ifr):
        """FeatureExtract_ref(I-frame), its pooled map and patch descriptors: once per GOP."""
        N, H, Wd = self.N, self.H, self.W
        scale, ph, pw, P = self._ff_geometry()
        f_ref = self._fe(W, "lf.fe_ref", ifr, "ref")
        p_ref = self.raw("lf.p_ref", (N, ph, pw, 64))
        self.call("tdvc_avgpool_scale", f_ref.ptr, f_ref.ld, p_ref.data_ptr(), N, H, Wd, 64, scale, nbytes=256 * N * H * Wd)
        self.call("tdvc_ff_descriptors", p_ref.data_ptr(), self.raw("lf.d_ref", (N, P, 576)).data_ptr(), N, ph, pw, 64)

    def loopfilter(self, W, rec_f, taps):
        N, H, Wd = self.N, self.H, self.W
        lr1 = dict(act=L.ACT_LRELU, slope=0.1)
        b = lambda nme, c=64: self.buf("lf." + nme, N, H, Wd, c)
        scale, ph, pw, P = self._ff_geometry()
        f_in = self._fe(W, "lf.fe_in", rec_f, "in")
        f_ref = b("ref.f")
        p_in = self.raw("lf.p_in", (N, ph, pw, 64))
        p_ref = self.raw("lf.p_ref", (N, ph, pw, 64))
        self.call("tdvc_avgpool_scale", f_in.ptr, f_in.ld, p_in.data_ptr(), N, H, Wd, 64, scale, nbytes=256 * N * H * Wd)
        d_in = self.raw("lf.d_in", (N, P, 576))
        d_ref = self.raw("lf.d_ref", (N, P, 576))
        self.call("tdvc_ff_descriptors", p_in.data_ptr(), d_in.data_ptr(), N, ph, pw, 64)
        ind = self.raw("lf.ind", (N, P), torch.int32)
        sim = self.raw("lf.sim", (N, P, P)) if taps is not None else None
        self.call("tdvc_ff_match", d_in.data_ptr(), d_ref.data_ptr(), ind.data_ptr(),
                  sim.data_ptr() if sim is not None else None, N, P, 576)
        ga, gb = b("ga"), b("gb")
        gth = b("gathered") if taps is not None else None
        cor = self.raw("lf.cor", (N, 1, H, Wd)) if taps is not None else None
        self.call("tdvc_ff_gather", f_in.ptr, f_ref.ptr, ind.data_ptr(), ga.ptr, gb.ptr,
                  gth.ptr if gth is not None else None, cor.data_ptr() if cor is not None else None, N, H, Wd, 64, scale,
                  nbytes=N * H * Wd * 1024)  # read f_in + gathered f_ref, write both gated halves
        o = self.conv([ga, gb], W["lf.featfusion"], b("o"), **lr1)
        o = self.conv([o, f_ref], W["lf.featfusion2"], b("o2"), csum=True)
        o = self.se(o, W["lf.attn"], b("o3"), act=L.ACT_LRELU, slope=0.1, csum=self.last_csum)
        o = self.res_stack(W, "lf.res", 2, o, "lf.rs", last_res2=rec_f)  # ... + feat (pnet.py:262-263)
        out = self.buf("lf.recon4", N, H, Wd, 3, ld=4)
        self.conv([o], W["lf.featdown"], out, act=L.ACT_CLAMP01)
        if taps is not None:
            taps.update({"loopfilter.f_in": f_in.nchw(), "loopfilter.f_ref": f_ref.nchw(),
                         "loopfilter.pool_in": p_in.permute(0, 3, 1, 2).contiguous(),
                         "loopfilter.pool_ref": p_ref.permute(0, 3, 1, 2).contiguous(),
                         "loopfilter.sim": sim.clone(), "loopfilter.ind": ind.clone().view(N, P, 1).long(),
                         "loopfilter.gathered": gth.nchw(), "loopfilter.cor": cor.clone()})
        return out


# =============================================================================== the module
class _AuxLoss(torch.autograd.Function):
    """EntropyBottleneck.loss() of one coder with its gradient with respect to `.quantiles` - the one backward the reference
    takes of it (`aux_loss.backward(); aux_optimizer.step()`, reference tools/train.py:147-159).  Forward value: the plan's
    `tdvc_eb_aux_loss` launch; backward: `tdvc_eb_aux_loss_grad`."""

    @staticmethod
    def forward(ctx, quantiles, value, eb_packed):
        ctx.eb = eb_packed
        return value.clone()

    @staticmethod
    def backward(ctx, grad_out):
        mats, biases, factors, _, q, target = ctx.eb
        g = torch.empty_like(q)
        go = grad_out.detach().float().reshape(1).contiguous()
        lib = L.load()
        with torch.cuda.device(q.device):
            L.check(lib.tdvc_eb_aux_loss_grad(mats.data_ptr(), biases.data_ptr(), factors.data_ptr(), q.data_ptr(),
                                              target.data_ptr(), go.data_ptr(), q.shape[0], g.data_ptr(),
                                              torch.cuda.current_stream(q.device).cuda_stream), "eb_aux_loss_grad")
        return g.view(q.shape[0], 1, 3), None, None


class _Origin:
    """Shared by a module and its nn.DataParallel replicas (replicate() copies __dict__ shallowly): lets a replica find the
    module that owns the master parameters, whose versions key the packed-weight cache."""

    def __init__(self, module):
        self.ref = weakref.ref(module)
        self.lock = threading.Lock()


class VideoCompressor(nn.Module):
    """Drop-in for reference main/model/pnet.py::VideoCompressor (constructor `:16-24`, forward `:26-83`)."""

    def __init__(self):
        super().__init__()
        self.mvCoder = _Coder(128)
        self.resCoder = _Coder(128)
        self.extra_fea = _FeaExtra(2)
        self.motion_est = _OffsetGen()
        self.mcnet = _MCNet(3)
        self.loopfilter = _FeatureFix()
        self.mcfilter = _LoopFilter()
        self._packed = {}              # device -> (key, packed weights)
        self._plans = {}               # (device, N, H, W) -> _Plan
        self._origin = _Origin(self)
        self.conv_impl = L.IMPL_AUTO   # 0 auto (tcgen05 where supported), 1 exact fp32 SIMT, 2 force tcgen05
        # "exact": fp32-class split MMA everywhere; "mixed": one fp16 MMA product in the stages behind the last quantiser of the
        # frame (residual synthesis transform, in-loop filter); "auto" (default): what the caller asks for through the reference's
        # own switch - `enabled_amp=True` (the reference then autocasts every non-coder convolution to fp16, pnet.py:28,51,75)
        # selects "mixed", `enabled_amp=False` selects "exact"
        self.precision = "auto"
        self.use_cuda_graph = False
        self.cache_features = True     # per-GOP feature caches (results are bit-identical either way)
        self.last_launches = 0

    def load_state_dict(self, *args, **kwargs):
        # weights replaced wholesale: the training path must not scale their fp16 blocks by maxima remembered from the old ones
        from tdvc_b200 import ops
        ops.forget_weight_maxima()
        return super().load_state_dict(*args, **kwargs)

    # the packed weights, plans and the replica link are runtime state: copies and pickles start without them
    def __getstate__(self):
        d = dict(self.__dict__)
        d["_packed"], d["_plans"], d["_origin"] = {}, {}, None
        return d

    def __setstate__(self, d):
        super().__setstate__(d)
        self._packed, self._plans, self._origin = {}, {}, _Origin(self)

    def __deepcopy__(self, memo):
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        new.__setstate__(copy.deepcopy(self.__getstate__(), memo))
        return new

    # -- nn.DataParallel: replicas are shallow copies made for every forward; their parameters are fresh broadcast copies.  The
    #    packed weights are therefore keyed on the ORIGINAL module's parameter versions and built from its parameters
    def _source(self):
        if getattr(self, "_is_replica", False):
            src = self._origin.ref()
            if src is not None:
                return src
        return self

    def _weights(self, dev):
        src = self._source()
        key = _param_key(src)
        with self._origin.lock:
            ent = self._packed.get(dev)
        if ent is not None and ent[0] == key:
            return ent[1]
        with torch.no_grad(), torch.cuda.device(dev):
            pk = _Packed(src, dev)
            from tdvc_b200 import tc
            tc.attach_f16(pk.c)
            tc.attach_dcn_f16(pk.c, "mc.dcn.w", 64, 8)
        with self._origin.lock:
            self._packed[dev] = (key, pk.c)
        return pk.c

    def _plan(self, N, H, W, dev):
        k = (dev, N, H, W)
        with self._origin.lock:
            p = self._plans.get(k)
            if p is None:
                p = self._plans[k] = _Plan(N, H, W, dev)
        return p

    def _check(self, a, b, c_a):
        if not a.is_cuda:
            raise RuntimeError("tdvc_b200.VideoCompressor runs on CUDA (sm_100a) only; there is no CPU fallback")
        N, C_, H, W = a.shape
        if C_ != c_a or b.shape != (N, 4, 3, H, W):
            raise RuntimeError(f"expected input (N,{c_a},H,W) and refer_frames (N,4,3,H,W), got {tuple(a.shape)} and {tuple(b.shape)}")
        if H % 64 or W % 64:
            raise RuntimeError("H and W must be multiples of 64 (pad as reference main/utils/utils.py:59-87 does)")
        if self.precision not in ("exact", "mixed", "auto"):
            raise RuntimeError(f"precision must be 'auto', 'exact' or 'mixed', not {self.precision!r}")
        return N, H, W

    def _precision(self, enabled_amp):
        return self.precision if self.precision != "auto" else ("mixed" if enabled_amp else "exact")

    def forward(self, input_image, refer_frames, enabled_amp=False, is_compress=False, taps=None, ref_keys=None):
        """Same contract as reference pnet.py:26-83.  `enabled_amp=False`: every convolution at fp32-class accuracy (the reference's
        fp32 path).  `enabled_amp=True` (the reference autocasts all non-coder convolutions to fp16): one fp16 MMA product in the
        stages behind the last quantiser only, everything in front of a quantiser stays fp32-class - more accurate than the
        reference's own AMP path and inside the parity bars against its fp32 path (DESIGN.md, precision; `self.precision`).
        ref_keys (extension, optional): four hashable identities of refer_frames[:, 0..3] from a caller that knows them (a GOP
        driver: `tdvc_b200.gop.code_gop`); the per-GOP feature caches are then keyed on them instead of on a device-side
        content hash, which saves the one host synchronisation per frame the hash costs.  Equal keys MUST mean equal content."""
        if self.training:
            if is_compress:
                raise RuntimeError("is_compress=True is served in eval() mode (the reference switches both coders to eval() "
                                   "before it codes, pnet.py:46,70)")
            if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
                return self._forward_training_autograd(input_image, refer_frames, enabled_amp=enabled_amp)
            return self._forward_training(input_image, refer_frames, taps, noise=None)
        N, H, W = self._check(input_image, refer_frames, 3)
        dev = input_image.device
        with torch.cuda.device(dev), torch.no_grad():
            x = input_image.detach().float().contiguous()
            refs = refer_frames.detach().float().contiguous()
            Wt = self._weights(dev)
            plan = self._plan(N, H, W, dev)
            plan.bind(Wt)
            plan.impl, plan.precision = self.conv_impl, self._precision(enabled_amp)
            if ref_keys is not None and len(ref_keys) != 4:
                raise RuntimeError("ref_keys: expected four identities, one per reference slice")
            recon, bpp = plan.run(Wt, x, refs, taps, graph=self.use_cuda_graph, cache=self.cache_features, ref_keys=ref_keys)
            recon, bpp = recon.clone(), bpp.clone()   # the plan's buffers are overwritten by the next frame
            if is_compress:
                self.last_coded = self._code(plan, Wt, N * H * W, taps)
            self.last_launches = plan.launches
        # reference returns (recon, bpp_res.view(-1), bpp_mv.view(-1))  (pnet.py:82-83)
        return recon, bpp[1:2], bpp[0:1]

    def _code(self, plan, Wt, num_pixels, taps=None):
        """reference pnet.py:45-49,69-73: `update(force=True)` + `compress()` of both coders on this frame's latents and the
        coded size `ac_bpp = sum(len(s[0]) for s in strings) * 8 / num_pixels`.  The reference computes ac_bpp_mv / ac_bpp_res
        and drops them (the return tuple is unchanged); here they stay readable in `self.last_coded`:
        {"mv" | "res": {"strings": [y_strings, z_strings], "shape": (h, w), "ac_bpp": float}}."""
        from tdvc_b200 import coding
        pending = []
        main = torch.cuda.current_stream(plan.dev)
        side = plan._side_stream()
        for cn, nm, stream in (("mv", "mv", main), ("rs", "res", side)):
            tabs = self._coder_tables(Wt, cn, plan.dev)
            # the two coders' autoregressive passes (one 8-16 SM cluster per image each) run side by side on two streams;
            # the host codes the motion strings while the residual pass is still running
            if stream is not main:
                stream.wait_stream(main)
            pending.append((nm, coding.launch_coding(plan, Wt, cn, tabs, stream=stream)))
        out = self._finish_coding(pending, num_pixels, taps)
        main.wait_stream(side)
        return out

    @staticmethod
    def _finish_coding(pending, num_pixels, taps=None, rows=False):
        """Host half of coding, in the order given: [(name, launch_coding handle), ...] -> `last_coded`.  rows: y as row
        streams (coding.finish_coding); ac_bpp then counts image 0's y row strings and its z string, as the reference's
        len(s[0]) counts image 0's string of each list."""
        from tdvc_b200 import coding
        out = {}
        for nm, h in pending:
            enc = coding.finish_coding(h, keep=taps is not None, rows=rows)
            hy = len(enc["strings"][0]) // len(enc["strings"][1]) if rows else 1
            enc["ac_bpp"] = (sum(len(s_) for s_ in enc["strings"][0][:hy]) + len(enc["strings"][1][0])) * 8.0 / num_pixels
            if taps is not None:
                for k in ("y_symbols", "y_indexes", "y_hat", "z_symbols"):
                    taps[f"{nm}.ac.{k}"] = enc.pop(k)
            out[nm] = enc
        return out

    def _coder_tables(self, Wt, cn, dev):
        """`update(force=True)` of coder `cn` ("mv" | "rs"), shared by the encoder and the decoder: its coding tables
        (coding.CoderTables) from the packed weights Wt, and compressai's buffers on the source module filled as update()
        leaves them.  update() recomputes the same tables from the same parameters: built once per pack."""
        from tdvc_b200 import coding
        tabs = Wt.setdefault("_tables", {})
        if cn not in tabs:
            tabs[cn] = coding.CoderTables(Wt, cn, dev)
            src = self._source()
            smod = src.mvCoder if cn == "mv" else src.resCoder
            for m, t in ((smod.entropy_bottleneck, tabs[cn].eb), (smod.gaussian_conditional, tabs[cn].gc)):
                m._quantized_cdf, m._cdf_length, m._offset = t.tensors(dev)   # compressai's buffers, as update() leaves them
            smod.gaussian_conditional.scale_table = tabs[cn].scale_table.clone()
        return tabs[cn]

    def compress(self, input_image, refer_frames, enabled_amp=False, ref_keys=None, taps=None, row_streams=False):
        """Closed-loop encoder of one P-frame: -> (recon (N,3,H,W) fp32, data: the version-2 container's bytes).
        row_streams: write a version-3 container instead, whose y strings are one rANS stream per latent row (this
        project's own format, about 12 bytes more per extra row and coder; compressai cannot read it), which `decompress`
        decodes wavefront by wavefront on the device.  The device pass, the symbols, y_hat and recon are the same.
        Unlike `forward`, both coders' syntheses run on the y_hat the strings carry (quantised relative to the predicted
        mean, round(y - mu) + mu), so `recon` is the frame `decompress(data, refer_frames)` rebuilds bit for bit; the
        prediction and the residual are computed from the decoded motion.  A GOP feeds this recon to the next frame
        (`tdvc_b200.gop.compress_gop`).  `self.last_coded` is left as `forward(..., is_compress=True)` leaves it.
        Runs eagerly (no CUDA graph) and shares the plan and the per-GOP feature caches with `forward`.
        enabled_amp / ref_keys as in `forward`; the precision mode goes into the container.  taps: also records "mv.x_hat",
        "prediction1", "prediction", "recon_feat" and each coder's "ac.*" symbols, indexes and y_hat."""
        if self.training:
            raise RuntimeError("compress is served in eval() mode (the reference switches both coders to eval() before it "
                               "codes, pnet.py:46,70)")
        N, H, W = self._check(input_image, refer_frames, 3)
        if refer_frames.device != input_image.device:
            raise RuntimeError("compress: input_image and refer_frames are on different devices")
        if ref_keys is not None and len(ref_keys) != 4:
            raise RuntimeError("ref_keys: expected four identities, one per reference slice")
        from tdvc_b200 import coding
        dev = input_image.device
        with torch.cuda.device(dev), torch.no_grad():
            x = input_image.detach().float().contiguous()
            refs = refer_frames.detach().float().contiguous()
            Wt = self._weights(dev)
            plan = self._plan(N, H, W, dev)
            plan.bind(Wt)
            plan.impl, plan.precision = self.conv_impl, self._precision(enabled_amp)
            tables = {cn: self._coder_tables(Wt, cn, dev) for cn in ("mv", "rs")}
            recon, handles = plan.compress(Wt, tables, x, refs, cache=self.cache_features, ref_keys=ref_keys, taps=taps)
            recon = recon.clone()
            # the host codes the motion strings while the residual half of the frame is still running on the device
            self.last_coded = self._finish_coding(list(handles.items()), N * H * W, taps, rows=row_streams)
        frame = {"size": (H, W), "N": N, "precision": plan.precision}
        if row_streams:
            frame["y_streams"] = "rows"
        return recon, coding.pack_frame(self.last_coded, frame=frame)

    def decompress(self, data, refer_frames, ref_keys=None, taps=None):
        """Decoder of one P-frame: a version-2 container (`compress`) and the same refer_frames (N,4,3,H,W) the encoder
        used -> recon (N,3,H,W) fp32, bit-identical to `compress`'s recon.  Two steps: both coders' latents as
        `decompress_latents` decodes them (`_decode_latents`), then the synthesis (`_synthesise`): extra_fea of
        refer_frames[:, -1], motion g_s, the prediction, residual g_s + prediction and the in-loop filter on the encoder's
        launches.  The precision mode is the container's; the per-GOP feature caches serve as in `forward` (ref_keys
        likewise).  Exactness needs the encoder's kernels on sm_100a and its `conv_impl`, which the container does not
        record: this module's own is used.
        A malformed container, or refer_frames that do not match its frame, raise RuntimeError before any device work; a
        broken string raises as in `decompress_latents`.  taps: records "mv.x_hat", "prediction1", "prediction",
        "recon_feat"."""
        from tdvc_b200 import coding
        box, rows = coding.unpack_for_decoding(data, "decompress")
        dev = self._check_refs(box["frame"], refer_frames, ref_keys, "decompress")
        return self._synthesise(self._decode_latents([(box, rows)], dev)[0], refer_frames, ref_keys, taps)

    def _check_refs(self, frame, refer_frames, ref_keys, who):
        """refer_frames must be (N,4,3,H,W) of the container's frame on this module's CUDA device, ref_keys None or four
        identities; else RuntimeError naming `who`.  -> the device."""
        (H, Wd), N = frame["size"], frame["N"]
        if not isinstance(refer_frames, torch.Tensor) or tuple(refer_frames.shape) != (N, 4, 3, H, Wd):
            got = tuple(refer_frames.shape) if isinstance(refer_frames, torch.Tensor) else type(refer_frames).__name__
            raise RuntimeError(f"{who}: refer_frames {got} do not match the container's frame (expected "
                               f"{(N, 4, 3, H, Wd)})")
        if ref_keys is not None and len(ref_keys) != 4:
            raise RuntimeError("ref_keys: expected four identities, one per reference slice")
        dev = self._decoder_device()
        if refer_frames.device != dev:
            raise RuntimeError(f"{who}: refer_frames are on {refer_frames.device}, the module on {dev}")
        return dev

    def _synthesise(self, lat, refer_frames, ref_keys=None, taps=None, who="decompress"):
        """Synthesis half of `decompress`: one container's latents (an element of `decompress_latents_many`, whose y_hat
        are wrapped as Acts, no copy) and its refer_frames -> recon (N,3,H,W), in the container's precision mode.
        refer_frames are checked here too: the launches read them through raw pointers."""
        dev = self._check_refs(lat["frame"], refer_frames, ref_keys, who)
        (H, Wd), N = lat["frame"]["size"], lat["frame"]["N"]
        with torch.cuda.device(dev), torch.no_grad():
            refs = refer_frames.detach().float().contiguous()
            Wt = self._weights(dev)
            plan = self._plan(N, H, Wd, dev)
            plan.bind(Wt)
            plan.impl, plan.precision = self.conv_impl, lat["frame"]["precision"]
            y_hat = {cn: Act(t, t.data_ptr(), *t.shape, t.shape[3])
                     for cn, t in (("mv", lat["mv"]["y_hat"]), ("rs", lat["res"]["y_hat"]))}
            recon = plan.decompress(Wt, y_hat, refs, cache=self.cache_features, ref_keys=ref_keys, taps=taps)
            return recon.clone()

    def decompress_latents(self, data):
        """Both coders' latents of one P-frame from the bytes of a version-2 container (`coding.pack_frame(net.last_coded,
        frame=...)`) and the weights alone: no reference frames and nothing the encoder left behind.  Per coder: the z strings
        are rANS-decoded on the host (compressai `EntropyBottleneck.decompress`), z_hat = symbol + median on the device, h_s
        (`_Plan.hyper_synthesis`, the encoder's own) gives the params, and `tdvc_ar_decode` decodes y with the cluster size the
        container records.  The motion coder runs on the current stream, the residual coder on the plan's side stream.
        Returns {"frame": {"size", "N", "precision"}, "mv" | "res": {"y_hat", "y_symbols", "y_indexes": (N, H/16, W/16, 128),
        "z_hat": (N, H/64, W/64, 128)}}, channels-last tensors of their own.
        The result is bit-identical to the encoder's latents only with the same kernels on sm_100a and the same `conv_impl`
        as the encoder ran with: h_s feeds every predicted mean and scale, and the container does not record conv_impl.
        A malformed container raises RuntimeError before any device work; a broken z string raises naming the coder and
        the image, a broken y string naming the latent position.  `decompress_latents_many` decodes several at once."""
        from tdvc_b200 import coding
        return self._decode_latents([coding.unpack_for_decoding(data, "decompress_latents")], self._decoder_device())[0]

    def decompress_latents_many(self, containers):
        """`decompress_latents` of T containers (version 2 or 3, in any mix) of one frame size and batch N, entropy-decoded
        as ONE batch of T * N images: their latents depend on the bytes and the weights alone, not on each other, so the z
        steps and h_s run once per coder and y one launch per coder and per (encoder cluster, y layout) group, and the
        decoder's clusters of all frames run side by side instead of one frame's 16 or 32 SMs at a time.  Returns one dict
        per container, bit-identical to `decompress_latents` of that container (h_s gives each image the bits it gives it
        alone: every convolution works on tiles of one image and picks its configuration from the layer's shape).
        Every container is checked before any device work, and all must hold the (H, W, N) of the first; a RuntimeError
        names the container index.  A broken z or y string raises naming the container, the coder and the image (for y
        the position or row) after every launch has finished; nothing of the batch is returned then.  The y tensors of a
        container are slices of its group's own tensors (no plan buffer), its z_hat a copy."""
        from tdvc_b200 import coding
        boxes = []
        for k, data in enumerate(containers):
            try:
                boxes.append(coding.unpack_for_decoding(data, "decompress_latents_many"))
            except RuntimeError as e:
                raise RuntimeError(f"container {k}: {e}") from None
        if not boxes:
            return []
        (H, Wd), N = boxes[0][0]["frame"]["size"], boxes[0][0]["frame"]["N"]
        for k, (box, _) in enumerate(boxes):
            (h, w), n = box["frame"]["size"], box["frame"]["N"]
            if (h, w, n) != (H, Wd, N):
                raise RuntimeError(f"decompress_latents_many: container {k} holds a {h}x{w} frame of N={n}, container 0 a "
                                   f"{H}x{Wd} frame of N={N} (one batch needs one frame size and batch)")
        return self._decode_latents(boxes, self._decoder_device(), named=True)

    def _decoder_device(self):
        dev = self.mvCoder.entropy_bottleneck.quantiles.device
        if dev.type != "cuda":
            raise RuntimeError("tdvc_b200.VideoCompressor runs on CUDA (sm_100a) only; there is no CPU fallback")
        return dev

    def _decode_latents(self, boxes, dev, named=False):
        """Device half of decompress_latents(_many) on checked containers [(box, rows: its y strings are row streams)] of
        one (H, W, N), decoded as one batch of T * N images on the plan of that batch (only its dec.* buffers).  Per coder,
        the batch holds the containers sorted by their (encoder cluster, y layout) group, in order inside a group, so
        that a group's params are one slice of h_s's output: the z strings of all images on the host, z_hat and h_s once,
        then one launch_decoding per group over its containers' strings.  The motion coder runs on the current stream, the
        residual coder on the side stream.  named: error messages call an image "image j of container k".
        -> per container {"frame", "mv" | "res": {"y_hat", "y_symbols", "y_indexes": slices of tensors of their own,
        "z_hat": a copy}}, both coders finished."""
        from tdvc_b200 import coding
        T = len(boxes)
        (H, Wd), N = boxes[0][0]["frame"]["size"], boxes[0][0]["frame"]["N"]
        hz, wz = H // 64, Wd // 64
        out = [{"frame": dict(box["frame"])} for box, _ in boxes]
        with torch.cuda.device(dev), torch.no_grad():
            Wt = self._weights(dev)
            plan = self._plan(T * N, H, Wd, dev)
            plan.bind(Wt)
            # h_s is fp32-class in both precision modes (only rs.g_s* and lf.* take one-product weights), so the container's
            # `precision` does not affect the latents and plan.precision is left as the last forward set it
            plan.impl = self.conv_impl
            main = torch.cuda.current_stream(dev)
            side = plan._side_stream()
            side.wait_stream(main)
            pending, z_hats = [], []
            for cn, nm, stream in (("mv", "mv", main), ("rs", "res", side)):
                tabs = self._coder_tables(Wt, cn, dev)
                group = lambda k, nm=nm: (boxes[k][0][nm]["cluster"], boxes[k][1])
                order = sorted(range(T), key=group)
                names = [f"image {j} of container {k}" if named else f"image {j}" for k in order for j in range(N)]
                z_sym = coding.decode_z_symbols(cn, [s_ for k in order for s_ in boxes[k][0][nm]["strings"][1]], tabs,
                                                hz, wz, images=names)
                # every buffer under dec.{cn}.*: the forward pass and launch_coding never read what the decoder writes
                b = lambda nme, h, w, c=128, cn=cn, **kw: plan.buf(f"dec.{cn}.{nme}", T * N, h, w, c, **kw)
                with torch.cuda.stream(stream):
                    sym_d = torch.from_numpy(z_sym).to(dev)
                    zh = b("z_hat", hz, wz)
                    coding.dequantize_z(sym_d, Wt[f"{cn}.eb"][3], zh, stream)
                    params = plan.hyper_synthesis(Wt, cn, zh, b)
                z_hats.append((nm, zh, order))
                # the motion chains are already decoding on the device while the host decodes the residual z strings
                i0 = 0
                for (cluster, rows), ks in itertools.groupby(order, key=group):
                    ks = list(ks)
                    n = len(ks) * N
                    y_strings = [s_ for k in ks for s_ in boxes[k][0][nm]["strings"][0]]
                    h = coding.launch_decoding(Wt, cn, tabs, y_strings, params.batch(i0, n), cluster, stream=stream,
                                               rows=rows)
                    if stream is not main:   # its outputs are handed to the caller's stream
                        for k_ in ("y_hat", "y_symbols", "y_indexes"):
                            h[k_].record_stream(main)
                    pending.append((nm, ks, names[i0:i0 + n], h))
                    i0 += n
            main.wait_stream(side)
            for nm, ks, images, h in pending:
                got = coding.finish_decoding(h, images=images)
                for i, k in enumerate(ks):
                    out[k][nm] = {key: v[i * N:(i + 1) * N] for key, v in got.items()}
            for nm, zh, order in z_hats:
                for i, k in enumerate(order):
                    out[k][nm]["z_hat"] = zh.t[i * N:(i + 1) * N].clone()
        return out

    def _forward_training(self, input_image, refer_frames, taps=None, noise=None):
        """`self.training` branch of reference pnet.py:26-83: uniform-noise quantisation in both coders (compressai
        quantize(.., "noise"): z + u, y + u for the synthesis / context path and a second draw for the likelihood of y),
        FeatureFix patch matching at scale 8 (pnet.py:220-221), and the 5-tuple return with the two aux losses (:80-81).
        noise: None = drawn on the device (Philox4x32-10 seeded from torch's CPU generator, so torch.manual_seed governs it), or
        {"mv.z", "mv.y", "mv.y_lik", "res.z", "res.y", "res.y_lik": (N,128,h,w) CUDA tensors} to inject given draws (tests).
        FORWARD ONLY, on the fused inference kernels (used under torch.no_grad() / for frozen models): reconstruction and bpp
        carry no autograd graph; with gradients enabled `forward` takes `_forward_training_autograd` instead.  The aux losses
        back-propagate to `.quantiles` on both paths."""
        N, H, W = self._check(input_image, refer_frames, 3)
        dev = input_image.device
        with torch.cuda.device(dev):
            with torch.no_grad():
                x = input_image.detach().float().contiguous()
                refs = refer_frames.detach().float().contiguous()
                Wt = self._weights(dev)
                plan = self._plan(N, H, W, dev)
                plan.bind(Wt)
                plan.impl, plan.precision = self.conv_impl, "exact"
                plan.training = True
                try:
                    plan.noise = self._noise(plan, noise, N, H, W)
                    recon, bpp = plan.run(Wt, x, refs, taps, graph=False, cache=False)
                finally:
                    plan.training, plan.noise = False, None
                self.last_launches = plan.launches
                recon, bpp, aux = recon.clone(), bpp.clone(), plan.aux.clone()
            mv_aux = _AuxLoss.apply(self.mvCoder.entropy_bottleneck.quantiles, aux[0], Wt["mv.eb"])
            res_aux = _AuxLoss.apply(self.resCoder.entropy_bottleneck.quantiles, aux[1], Wt["rs.eb"])
        return recon, bpp[1:2], bpp[0:1], mv_aux, res_aux

    def _forward_training_autograd(self, input_image, refer_frames, noise=None, enabled_amp=False):
        """`self.training` with gradients enabled: the same forward built from the autograd functions of `tdvc_b200.ops`
        (tdvc_b200/train_graph.py), so that the reference's training step - `rd_loss.backward()`, gradient clipping, the two
        Adam steps, `aux_loss.backward()` (tools/train.py:125-159) - runs on this module.  Returns the 5-tuple of pnet.py:80-81;
        every output carries its graph.  noise: as `_forward_training` (None: drawn on the device).  enabled_amp (the reference
        then trains with fp16 autocast products outside the coders, cfg/train.yaml `amp: True`): the weight-gradient MMAs use one
        TF32 product instead of the fp32-class three; forward and grad_input keep fp32-class accuracy either way."""
        self._check(input_image, refer_frames, 3)
        from tdvc_b200 import train_graph
        dev = input_image.device
        with torch.cuda.device(dev):
            x = input_image.float().contiguous()
            refs = refer_frames.float().contiguous()
            from tdvc_b200 import ops
            saved, ops.WGRAD_PRODUCTS = ops.WGRAD_PRODUCTS, (1 if enabled_amp else 3)
            try:
                recon, bpp_res, bpp_mv, ind = train_graph.forward(self, x, refs, noise)
            finally:
                ops.WGRAD_PRODUCTS = saved
            self.last_ind = ind
            aux = []
            lib = L.load()
            st = torch.cuda.current_stream(dev).cuda_stream
            for cd in (self.mvCoder, self.resCoder):   # EntropyBottleneck.loss() (pnet.py:35,59) and its gradient to .quantiles
                eb = pack_entropy_bottleneck(cd.entropy_bottleneck, P=lambda mod, name: getattr(mod, name).detach().float())
                val = torch.empty(1, device=dev, dtype=torch.float32)
                L.check(lib.tdvc_eb_aux_loss(eb[0].data_ptr(), eb[1].data_ptr(), eb[2].data_ptr(), eb[4].data_ptr(), eb[5].data_ptr(),
                                             eb[0].shape[0], val.data_ptr(), st), "eb_aux_loss")
                aux.append(_AuxLoss.apply(cd.entropy_bottleneck.quantiles, val[0], eb))
        return recon, bpp_res, bpp_mv, aux[0], aux[1]

    def _noise(self, plan, given, N, H, W):
        lib = L.load()
        st = torch.cuda.current_stream(plan.dev).cuda_stream
        seed = None
        out = {}
        for ci, (cn, nm) in enumerate((("mv", "mv"), ("rs", "res"))):
            for ki, (kind, sc) in enumerate((("z", 64), ("y", 16), ("y_lik", 16))):
                a = plan.buf(f"noise.{cn}.{kind}", N, H // sc, W // sc, 128)
                if given is not None:
                    t = given[f"{nm}.{kind}"]
                    if tuple(t.shape) != (N, 128, H // sc, W // sc) or not t.is_cuda:
                        raise RuntimeError(f"noise[{nm}.{kind}]: expected a CUDA tensor of shape {(N, 128, H // sc, W // sc)}")
                    t = t.detach().float().contiguous()
                    L.check(lib.tdvc_nchw_to_nhwc(t.data_ptr(), a.ptr, N, 128, H // sc, W // sc, 128, st), "nchw_to_nhwc")
                else:
                    if seed is None:
                        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
                    L.check(lib.tdvc_uniform_noise(a.ptr, N * (H // sc) * (W // sc) * 128, seed, ci * 3 + ki, st), "uniform_noise")
                out[f"{cn}.{kind}"] = a
        return out

    def fusion_and_filter(self, prediction1, refer_frames, recon_feat, enabled_amp=False):
        """BASELINE config 5 entry: `mcfilter` (reference pnet.py:53) on `prediction1` and `loopfilter` + clamp (:77-78) on
        `recon_feat`, with the 4 reference frames.  Returns (prediction (N,64,H,W), recon (N,3,H,W))."""
        N, H, W = self._check(prediction1, refer_frames, 64)
        if recon_feat.shape != prediction1.shape:
            raise RuntimeError("expected prediction1 / recon_feat (N,64,H,W) and refer_frames (N,4,3,H,W)")
        dev = prediction1.device
        with torch.cuda.device(dev), torch.no_grad():
            Wt = self._weights(dev)
            plan = self._plan(N, H, W, dev)
            plan.bind(Wt)
            plan.impl, plan.precision = self.conv_impl, self._precision(enabled_amp)
            pred, recon = plan.fusion_and_filter(Wt, prediction1.detach().float().contiguous(),
                                                 refer_frames.detach().float().contiguous(),
                                                 recon_feat.detach().float().contiguous())
            self.last_launches = plan.launches
            return pred.clone(), recon.clone()

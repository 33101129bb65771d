"""GOP evaluation driver — mirrors the reference's `validation` loop (reference tools/predict.py:43-100):
reference-frame buffer with warm-up duplication (:55-60), pad-to-64 / crop (reference
main/utils/utils.py:59-87), per-frame PSNR = 10 log10(1/MSE) (:87-88) and bpp = bpp_res + bpp_mv (:90).

Differences that do not change results: the per-frame `.cpu()` metric read-backs (one device sync per frame
per metric in the reference) become on-device accumulations (`tdvc_sq_err_sum`) read once per GOP, and GOPs
are sharded round-robin over ranks with one all-reduce of seven fp64 sums at the end (SURVEY.md 8e).
"""
import math

import torch
import torch.nn.functional as F

from tdvc_b200 import lib as L


def pad(x, p=64):
    """reference main/utils/utils.py:59-73 (zero padding, centred)."""
    h, w = x.size(2), x.size(3)
    H, W = (h + p - 1) // p * p, (w + p - 1) // p * p
    left, top = (W - w) // 2, (H - h) // 2
    if H == h and W == w:
        return x
    return F.pad(x, (left, W - w - left, top, H - h - top), mode="constant", value=0)


def crop(x, size):
    """reference main/utils/utils.py:76-87."""
    H, W = x.size(2), x.size(3)
    h, w = size
    left, top = (W - w) // 2, (H - h) // 2
    if H == h and W == w:
        return x
    return x[:, :, top:top + h, left:left + w]


def reference_window(ref_list):
    """The 4 reference frames of the next P-frame: [I, x^(t-3), x^(t-2), x^(t-1)] with the reference's
    warm-up duplication (reference tools/predict.py:55-60).  Returns (N,4,3,H,W)."""
    n = len(ref_list)
    if n == 1:
        sel = [ref_list[0], ref_list[-1], ref_list[-1], ref_list[-1]]
    elif n == 2:
        sel = [ref_list[0], ref_list[-2], ref_list[-1], ref_list[-1]]
    else:
        sel = [ref_list[0], ref_list[-3], ref_list[-2], ref_list[-1]]
    return torch.stack(sel, dim=1)


class RefBuffer:
    """The reference-frame list of one GOP (reference tools/predict.py:51-68: `ref_image` grows by one reconstruction per
    P-frame) together with a host-side identity per frame.  `window()` returns the (N,4,3,H,W) tensor the codec takes and the four
    identities of its slices; passing those to `VideoCompressor.forward(ref_keys=...)` lets the per-GOP feature caches be keyed
    without hashing the frames on the device (one host synchronisation per frame less)."""
    _serial = 0

    def __init__(self, i_frame):
        self.frames, self.ids = [i_frame], [self._new_id()]

    @classmethod
    def _new_id(cls):
        cls._serial += 1
        return cls._serial

    def push(self, recon):
        self.frames.append(recon)
        self.ids.append(self._new_id())
        if len(self.frames) > 4:   # only the I-frame and the last three reconstructions are ever referenced again
            self.frames, self.ids = [self.frames[0]] + self.frames[-3:], [self.ids[0]] + self.ids[-3:]

    def window(self):
        n = len(self.frames)
        sel = (0, n - 1, n - 1, n - 1) if n == 1 else ((0, n - 2, n - 1, n - 1) if n == 2 else (0, n - 3, n - 2, n - 1))
        return torch.stack([self.frames[i] for i in sel], dim=1), tuple(self.ids[i] for i in sel)


def sq_err_sum(a, b, acc, slot):
    """acc[slot] += sum (a-b)^2 on the device (CUDA kernel; fp64 accumulator)."""
    a, b = a.contiguous(), b.contiguous()
    lib = L.load()
    L.check(lib.tdvc_sq_err_sum(a.data_ptr(), b.data_ptr(), a.numel(), acc.data_ptr() + 8 * slot,
                                torch.cuda.current_stream(a.device).cuda_stream), "sq_err_sum")


def code_gop(net, i_frame, p_frames, enable_amp=False, keep_recon=False, with_msssim=False):
    """Code one GOP.  i_frame (1,3,h,w): the (decoded) I-frame; p_frames (T,3,h,w): the frames to code.
    Returns dict with device tensors `bpp_mv`, `bpp_res` (T,), `sse` (T,) fp64 (sum of squared error over the
    cropped frame) and `numel`; plus `recon` (list of cropped reconstructions) when keep_recon."""
    dev = p_frames.device
    T, _, h, w = p_frames.shape
    refs = RefBuffer(pad(i_frame, 64))
    keyed = "ref_keys" in getattr(getattr(net, "forward", None), "__code__", type("c", (), {"co_varnames": ()})).co_varnames
    sse = torch.zeros(T, device=dev, dtype=torch.float64)
    bmv, bres, recons, mss = [], [], [], []
    for i in range(T):
        x = pad(p_frames[i:i + 1], 64)
        window, keys = refs.window()
        if keyed:   # tdvc_b200.VideoCompressor: the identities of the reference slices key its per-GOP feature caches
            recon, bpp_res, bpp_mv = net(x, window, enable_amp, ref_keys=keys)
        else:       # any module with the reference's signature (pnet.py:26)
            recon, bpp_res, bpp_mv = net(x, window, enable_amp)
        refs.push(recon)             # padded, clamped reconstruction feeds the next frame (predict.py:68)
        rc = crop(recon, (h, w))
        sq_err_sum(rc, p_frames[i:i + 1], sse, i)
        if with_msssim:              # tools/predict.py:93-94 (the enable_amp branch of the shipped cfg/predict.yaml)
            from tdvc_b200.metrics import ms_ssim
            mss.append(ms_ssim(rc.float(), p_frames[i:i + 1], data_range=1.0))
        bmv.append(bpp_mv.reshape(-1)[0])
        bres.append(bpp_res.reshape(-1)[0])
        if keep_recon:
            recons.append(rc.clone())
    out = {"bpp_mv": torch.stack(bmv), "bpp_res": torch.stack(bres), "sse": sse, "numel": 3 * h * w}
    if with_msssim:
        out["msssim"] = torch.stack(mss)
    if keep_recon:
        out["recon"] = recons
    return out


def compress_gop(net, i_frame, p_frames, enable_amp=False, row_streams=False):
    """Closed-loop coding of one GOP with `VideoCompressor.compress`: each frame's reconstruction - the frame the decoder
    rebuilds - is the next frame's reference, so encoder and decoder never drift apart.  i_frame (1,3,h,w): the (decoded)
    I-frame; p_frames (T,3,h,w).  Frames are padded to multiples of 64 and cropped back as in `code_gop`.
    Returns (containers: one version-2 container (bytes) per P-frame, recon: the cropped reconstructions).
    row_streams: version-3 containers (`VideoCompressor.compress(..., row_streams=True)`); decompress_gop reads either."""
    T, _, h, w = p_frames.shape
    refs = RefBuffer(pad(i_frame, 64))
    containers, recons = [], []
    for i in range(T):
        window, keys = refs.window()
        recon, data = net.compress(pad(p_frames[i:i + 1], 64), window, enable_amp, ref_keys=keys, row_streams=row_streams)
        refs.push(recon)
        containers.append(data)
        recons.append(crop(recon, (h, w)))
    return containers, recons


def decompress_gop(net, i_frame, containers, size):
    """Decoder of `compress_gop`: the same I-frame (1,3,h,w), the containers in order and the frame size (h, w) ->
    the cropped reconstructions, bit-identical to the encoder's.  The latents of all frames depend on the containers and
    the weights alone, so they are entropy-decoded first, as one batch (`VideoCompressor.decompress_latents_many`); a
    broken string raises naming its container before anything is synthesised.  Then each frame's synthesis runs on its
    reference window, frame by frame (`decompress`'s second half)."""
    latents = net.decompress_latents_many(containers)
    refs = RefBuffer(pad(i_frame, 64))
    recons = []
    for lat in latents:
        window, keys = refs.window()
        recon = net._synthesise(lat, window, ref_keys=keys, who="decompress_gop")
        refs.push(recon)
        recons.append(crop(recon, size))
    return recons


def validate(dataset, net, enable_amp=True, device=None, with_msssim=True, gops=None):
    """The reference's `validation` (reference tools/predict.py:35-110) over a `tdvc_b200.data.GopDataset`: every GOP is coded
    by `code_gop`; bpp / PSNR / MS-SSIM are averaged over ALL frames, the BPG-coded I-frame of each GOP included with the bpp /
    PSNR / MS-SSIM its loader reports (:47-50), while bpp_mv / bpp_res / mse average over the P-frames only (:95-97).
    Returns (bpp, bpp_mv, bpp_res, psnr, msssim, mse) like the reference (:110).  `gops`: indices to code (a rank's shard)."""
    device = device or next(net.parameters()).device
    tot = torch.zeros(7, device=device, dtype=torch.float64)
    n_i, i_bpp, i_psnr, i_ms = 0, 0.0, 0.0, 0.0
    for g in (range(len(dataset)) if gops is None else gops):
        p_frames, i_frame, bpp_i, psnr_i, _, raw = dataset[g]
        p_frames, i_frame = p_frames.to(device), i_frame.to(device).unsqueeze(0)
        res = code_gop(net, i_frame, p_frames, enable_amp=enable_amp, with_msssim=with_msssim)
        tot += gop_stats(res)
        n_i += 1
        i_bpp += float(bpp_i)
        i_psnr += float(psnr_i)
        if with_msssim:
            from tdvc_b200.metrics import ms_ssim
            i_ms += float(ms_ssim(raw[0:1].to(device), i_frame, data_range=1.0))
    return combine_with_iframes(summarise(tot), n_i, i_bpp, i_psnr, i_ms)


def coded_rates(data):
    """Rates of one frame container (version 2 or 3) from its bytes, per padded pixel N * H * W as the reference
    normalises bpp: (bpp_mv, bpp_res, bpp_container).  bpp_mv / bpp_res: 8 x the bytes of that coder's y and z strings;
    bpp_container: 8 x every byte of the container, so that the header and the length fields count too."""
    from tdvc_b200 import coding
    box = coding.unpack_frame(data)
    (H, W), N = box["frame"]["size"], box["frame"]["N"]
    px = N * H * W
    coder = lambda nm: 8.0 * sum(len(s) for lst in box[nm]["strings"] for s in lst) / px
    return coder("mv"), coder("res"), 8.0 * len(data) / px


def validate_codec(dataset, net, decoder=None, enable_amp=True, row_streams=False, with_msssim=True, gops=None):
    """`validate` on real bitstreams: every GOP of a `tdvc_b200.data.GopDataset` (same contract and I-frame handling) is
    coded in closed loop by `compress_gop` (row_streams: version-3 containers), rates are taken from the containers'
    bytes (`coded_rates`) instead of the likelihoods, and PSNR / MS-SSIM / MSE from the frames a decoder rebuilds.
    decoder: a second module; each GOP is then also decoded by `decompress_gop` on it, its reconstructions must equal the
    encoder's (torch.equal, else RuntimeError naming GOP and P-frame) and the metrics are taken on them.  Without one, they
    are taken on the encoder's closed-loop reconstructions, which a decoder rebuilds bit for bit.
    Returns `summarise_codec` of the sums plus "stats": the sums themselves, an fp64 tensor of CODEC_STATS entries, so that
    a rank's shard (`gops=shard_gops(...)`) is combined with `reduce_stats(stats)` and `summarise_codec(stats)`."""
    from tdvc_b200.metrics import ms_ssim
    device = next(net.parameters()).device
    stats = torch.zeros(CODEC_STATS, device=device, dtype=torch.float64)
    for g in (range(len(dataset)) if gops is None else gops):
        p_frames, i_frame, bpp_i, psnr_i, _, raw = dataset[g]
        p_frames, i_frame = p_frames.to(device), i_frame.to(device).unsqueeze(0)
        T, _, h, w = p_frames.shape
        containers, recons = compress_gop(net, i_frame, p_frames, enable_amp=enable_amp, row_streams=row_streams)
        if decoder is not None:
            got = decompress_gop(decoder, i_frame.to(next(decoder.parameters()).device), containers, (h, w))
            got = [r.to(device) for r in got]
            for t, (a, b) in enumerate(zip(got, recons)):
                if not torch.equal(a, b):
                    raise RuntimeError(f"validate_codec: GOP {g}, P-frame {t}: the decoder's reconstruction differs from "
                                       "the encoder's")
            recons = got
        rates = torch.tensor([coded_rates(d) for d in containers], device=device, dtype=torch.float64)
        res = {"bpp_mv": rates[:, 0], "bpp_res": rates[:, 1], "numel": 3 * h * w,
               "sse": torch.zeros(T, device=device, dtype=torch.float64)}
        for t in range(T):
            sq_err_sum(recons[t], p_frames[t:t + 1], res["sse"], t)
        if with_msssim:
            res["msssim"] = torch.stack([ms_ssim(recons[t].float(), p_frames[t:t + 1], data_range=1.0) for t in range(T)])
        i_ms = float(ms_ssim(raw[0:1].to(device), i_frame, data_range=1.0)) if with_msssim else 0.0
        stats += torch.cat([gop_stats(res), rates[:, 2].sum().view(1),
                            torch.tensor([1.0, float(bpp_i), float(psnr_i), i_ms], device=device, dtype=torch.float64)])
    return dict(summarise_codec(stats), stats=stats)


# validate_codec's sums: gop_stats' seven [sum bpp, sum bpp_mv, sum bpp_res, sum psnr, sum msssim, sum mse, P-frames],
# then sum bpp_container, and of the I-frames [count, sum bpp, sum psnr, sum msssim] as their loader reports them
CODEC_STATS = 12


def summarise_codec(stats):
    """validate_codec's averages from its sums (over GOPs, and over ranks once reduce_stats has added them): "bpp",
    "bpp_container", "psnr" and "msssim" over the I- and P-frames as `validate` forms them (an I-frame counts with what its
    loader reports, in bpp_container as in bpp), "bpp_mv", "bpp_res" and "mse" over the P-frames; "frames" (P-frames),
    "iframes", and "p": the averages of the P-frames alone (`summarise` + "bpp_container")."""
    s = [float(v) for v in stats.tolist()]
    p = summarise(stats[:7])
    p["bpp_container"] = s[7] / max(s[6], 1.0)
    n_i = int(s[8])
    bpp, _, _, psnr, msssim, _ = combine_with_iframes(p, n_i, s[9], s[10], s[11])
    bpp_container = combine_with_iframes(dict(p, bpp=p["bpp_container"]), n_i, s[9], s[10], s[11])[0]
    return {"bpp": bpp, "bpp_mv": p["bpp_mv"], "bpp_res": p["bpp_res"], "bpp_container": bpp_container, "psnr": psnr,
            "msssim": msssim, "mse": p["mse"], "frames": p["frames"], "iframes": n_i, "p": p}


def combine_with_iframes(p_summary, n_i, sum_i_bpp, sum_i_psnr, sum_i_msssim):
    """Averages as the reference forms them (tools/predict.py:47-50, 86-110): the lists `bpps`, `psnrs`, `ssims` hold one entry per
    I-frame and per P-frame; `mvs`, `ress`, `mses` hold the P-frames only."""
    n_p = p_summary["frames"]
    n = max(n_p + n_i, 1)
    return ((p_summary["bpp"] * n_p + sum_i_bpp) / n, p_summary["bpp_mv"], p_summary["bpp_res"],
            (p_summary["psnr"] * n_p + sum_i_psnr) / n, (p_summary["msssim"] * n_p + sum_i_msssim) / n, p_summary["mse"])


def gop_stats(res):
    """Per-GOP sums in the reference's reporting units -> fp64 tensor
    [sum bpp, sum bpp_mv, sum bpp_res, sum psnr, sum msssim (0 unless code_gop(with_msssim=True)), sum mse, n_frames]."""
    mse = res["sse"] / res["numel"]
    psnr = 10.0 * torch.log10(1.0 / mse)
    bmv, bres = res["bpp_mv"].double(), res["bpp_res"].double()
    z = res["msssim"].double().sum() if "msssim" in res else torch.zeros((), device=mse.device, dtype=torch.float64)
    return torch.stack([(bmv + bres).sum(), bmv.sum(), bres.sum(), psnr.sum(), z, mse.sum(),
                        torch.tensor(float(mse.numel()), device=mse.device, dtype=torch.float64)])


def shard_gops(n_gops, rank, world):
    """GOPs are independent (each restarts from its own I-frame): rank r takes {g : g mod world == r}."""
    return [g for g in range(n_gops) if g % world == rank]


def reduce_stats(stats, group=None):
    """One all-reduce(sum) of the 7 fp64 sums over ranks (no-op without an initialised process group)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def summarise(stats):
    s = [float(v) for v in stats.tolist()]
    n = max(s[6], 1.0)
    return {"bpp": s[0] / n, "bpp_mv": s[1] / n, "bpp_res": s[2] / n, "psnr": s[3] / n, "msssim": s[4] / n, "mse": s[5] / n,
            "frames": int(s[6])}


def psnr_from_mse(mse):
    return 10.0 * math.log10(1.0 / mse)

"""CPU tests (-m "not gpu") of the host logic: C-ABI library loads and exports every symbol the header declares
(no compute calls), state_dict compatibility with the reference key set, weight packing, GOP driver semantics
(reference tools/predict.py:51-68), GOP sharding + the 7-sum all-reduce over a world_size-2 gloo group."""
import os
import re
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "tdvc_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(tdvc_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from tdvc_b200 import build, lib as L
    build.build()
    lib = L.load()
    syms = _header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/tdvc_b200.h but not exported"
        assert s in L.SIGNATURES, f"{s} has no ctypes signature"
    assert lib.tdvc_version() >= 100
    assert lib.tdvc_dcn_v2_workspace_bytes(1, 64, 64, 64, 64, 8) > 64 * 64 * (64 + 216 + 64) * 4


def test_struct_layouts_match_header():
    """ctypes mirrors of the parameter structs must have the C sizes, and the chain the encoder and the decoder of y share
    must sit at offset 0 of both (checked against a tiny C program)."""
    import ctypes
    import subprocess
    import tempfile
    from tdvc_b200 import lib as L
    structs = {"TdvcConvParams": L.ConvParams, "TdvcDcnParams": L.DcnParams, "TdvcArChain": L.ArChain,
               "TdvcArParams": L.ArParams, "TdvcArDecodeParams": L.ArDecodeParams}
    prints = "".join(f'printf("%zu\\n", sizeof({s}));' for s in structs)
    prints += 'printf("%zu\\n%zu\\n", offsetof(TdvcArParams, chain), offsetof(TdvcArDecodeParams, chain));'
    src = f'#include <stddef.h>\n#include <stdio.h>\n#include "tdvc_b200.h"\nint main(){{{prints}return 0;}}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        got = [int(v) for v in subprocess.check_output([os.path.join(d, "s")]).split()]
    assert got == [ctypes.sizeof(t) for t in structs.values()] + [0, 0]
    assert L.ArParams.chain.offset == 0 and L.ArDecodeParams.chain.offset == 0


def test_state_dict_matches_reference_key_set(oracle_model):
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor()
    osd = oracle_model.state_dict()
    assert list(net.state_dict().keys()) == list(osd.keys())
    net.load_state_dict(osd, strict=True)
    oracle_model.load_state_dict(net.state_dict(), strict=True)
    for k, v in net.state_dict().items():
        assert v.shape == osd[k].shape and torch.equal(v, osd[k]), k


def test_forward_refuses_cpu():
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()
    x, r = torch.zeros(1, 3, 64, 64), torch.zeros(1, 4, 3, 64, 64)
    with pytest.raises(RuntimeError):
        net(x, r, False)  # no CPU fallback
    with pytest.raises(RuntimeError):
        net(x, r, False, True)  # entropy coding is CUDA-only as well
    net.train()
    with pytest.raises(RuntimeError):
        net(x, r, False)  # the training-mode forward is CUDA-only as well
    with pytest.raises(RuntimeError):
        net(x, r, False, True)  # coding is served in eval() mode


def _emulate_packed_conv(xs, cw, stride=1):
    """The implicit GEMM the kernel performs, in torch: NHWC sources (stored channel counts), packed weights."""
    x = torch.cat(xs, dim=-1)  # (N,H,W,cin)
    N, Hh, Ww, cin = x.shape
    assert cin == cw.cin
    xp = F.pad(x, (0, cw.cin_pad - cin, cw.pad, cw.pad, cw.pad, cw.pad))
    Ho = (Hh + 2 * cw.pad - cw.k) // stride + 1
    Wo = (Ww + 2 * cw.pad - cw.k) // stride + 1
    out = torch.zeros(N, Ho, Wo, cw.cout_pad)
    for ky in range(cw.k):
        for kx in range(cw.k):
            patch = xp[:, ky:ky + stride * (Ho - 1) + 1:stride, kx:kx + stride * (Wo - 1) + 1:stride]
            out += patch @ cw.w[ky * cw.k + kx]
    if cw.b is not None:
        out += cw.b
    out = out[..., :cw.cout]
    if cw.shuffle == 2:
        cr = cw.cout // 4
        o = out.view(N, Ho, Wo, 2, 2, cr).permute(0, 1, 3, 2, 4, 5).reshape(N, 2 * Ho, 2 * Wo, cr)
        return o
    return out


@pytest.mark.parametrize("case", ["plain", "two_src", "image", "odd_cin", "shuffle", "stride2_1x1"])
def test_pack_conv_layouts(case):
    from tdvc_b200.model import pack_conv
    torch.manual_seed(0)
    if case == "plain":
        conv = torch.nn.Conv2d(8, 20, 3, 1, 1)
        x = torch.randn(1, 8, 6, 7)
        cw = pack_conv(conv.weight, conv.bias)
        got = _emulate_packed_conv([x.permute(0, 2, 3, 1)], cw)
        want = conv(x)
    elif case == "two_src":
        conv = torch.nn.Conv2d(16, 8, 3, 1, 1)
        a, b = torch.randn(1, 8, 5, 5), torch.randn(1, 8, 5, 5)
        cw = pack_conv(conv.weight, conv.bias, src_layout=[(8, 8), (8, 8)])
        got = _emulate_packed_conv([a.permute(0, 2, 3, 1), b.permute(0, 2, 3, 1)], cw)
        want = conv(torch.cat([a, b], 1))
    elif case == "image":
        conv = torch.nn.Conv2d(3, 16, 3, 1, 1)
        x = torch.randn(2, 3, 5, 6)
        cw = pack_conv(conv.weight, conv.bias, src_layout=[(3, 4)])
        got = _emulate_packed_conv([F.pad(x.permute(0, 2, 3, 1), (0, 1))], cw)
        want = conv(x)
    elif case == "odd_cin":
        conv = torch.nn.Conv2d(426, 341, 1)
        x = torch.randn(1, 426, 3, 3)
        cw = pack_conv(conv.weight, conv.bias, src_layout=[(426, 428)])
        assert cw.cin == 428 and cw.cin_pad == 432 and cw.cout_pad == 352 and cw.pad == 0
        got = _emulate_packed_conv([F.pad(x.permute(0, 2, 3, 1), (0, 2))], cw)
        want = conv(x)
    elif case == "shuffle":
        conv = torch.nn.Conv2d(8, 32, 3, 1, 1)
        x = torch.randn(1, 8, 4, 5)
        cw = pack_conv(conv.weight, conv.bias, shuffle=2)
        got = _emulate_packed_conv([x.permute(0, 2, 3, 1)], cw)
        want = F.pixel_shuffle(conv(x), 2)
    else:
        conv = torch.nn.Conv2d(8, 16, 1, 2)
        x = torch.randn(1, 8, 6, 8)
        cw = pack_conv(conv.weight, conv.bias, pad=0)
        got = _emulate_packed_conv([x.permute(0, 2, 3, 1)], cw, stride=2)
        want = conv(x)
    assert (got.permute(0, 3, 1, 2) - want).abs().max() < 1e-5


def test_reference_window_matches_predict_py():
    """reference tools/predict.py:55-62 builds torch.stack([...]).transpose(1,0).view(-1,4,3,H,W)."""
    from tdvc_b200 import gop as G
    fr = [torch.full((1, 3, 2, 2), float(i)) for i in range(6)]
    for n in range(1, 6):
        lst = fr[:n]
        if n == 1:
            ref = torch.stack([lst[0], lst[-1], lst[-1], lst[-1]])
        elif n == 2:
            ref = torch.stack([lst[0], lst[-2], lst[-1], lst[-1]])
        else:
            ref = torch.stack([lst[0], lst[-3], lst[-2], lst[-1]])
        want = ref.transpose(1, 0).reshape(-1, 4, 3, 2, 2)
        assert torch.equal(G.reference_window(lst), want)


def test_pad_crop_like_reference():
    from tdvc_b200 import gop as G
    x = torch.arange(2 * 3 * 70 * 130, dtype=torch.float32).view(2, 3, 70, 130)
    p = G.pad(x, 64)
    assert p.shape == (2, 3, 128, 192)
    assert torch.equal(G.crop(p, (70, 130)), x)
    assert p[:, :, :29].abs().sum() == 0 and p[:, :, :, :31].abs().sum() == 0  # (128-70)//2 = 29, (192-130)//2 = 31
    y = torch.zeros(1, 3, 64, 128)
    assert G.pad(y, 64) is y and G.crop(y, (64, 128)) is y


def test_shard_gops_partition():
    from tdvc_b200 import gop as G
    for world in (1, 2, 4, 8):
        parts = [G.shard_gops(96, r, world) for r in range(world)]
        assert sorted(sum(parts, [])) == list(range(96))
        assert len({len(p) for p in parts}) == 1


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from tdvc_b200 import gop as G
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    mine = G.shard_gops(6, rank, world)
    s = torch.zeros(7, dtype=torch.float64)
    for g in mine:  # fake per-GOP statistics: bpp = g, 11 frames each
        s += torch.tensor([11.0 * g, 4.0 * g, 7.0 * g, 11 * 30.0, 0.0, 11 * 1e-3, 11.0], dtype=torch.float64)
    G.reduce_stats(s)
    q.put((rank, s.tolist()))
    dist.destroy_process_group()


def test_stats_allreduce_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29000 + os.getpid() % 2000
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = [q.get(timeout=120) for _ in ps]
    for p in ps:
        p.join(timeout=60)
    want = [11.0 * 15, 4.0 * 15, 7.0 * 15, 6 * 11 * 30.0, 0.0, 6 * 11 * 1e-3, 66.0]
    for _, s in res:
        assert all(abs(a - b) < 1e-9 for a, b in zip(s, want))
    from tdvc_b200 import gop as G
    summ = G.summarise(torch.tensor(res[0][1], dtype=torch.float64))
    assert summ["frames"] == 66 and abs(summ["psnr"] - 30.0) < 1e-9 and abs(summ["bpp"] - 2.5) < 1e-9


def test_gop_dataset_and_iframe_averaging(tmp_path):
    """tdvc_b200.data.GopDataset lists and loads GOPs like the reference's UVGDataSet / HEVCDataSet (reference
    main/dataloader/dataset.py:16-193) and `combine_with_iframes` averages like tools/predict.py:47-50,86-110."""
    from torchvision.io import write_png
    from tdvc_b200 import data as D
    from tdvc_b200 import gop as G
    assert [D.qp_for_lambda(l) for l in (512, 1024, 2048, 4096, 64)] == [37, 32, 27, 22, 27]
    assert sorted(["im10.png", "im2.png", "im1.png"], key=D.natural_key) == ["im1.png", "im2.png", "im10.png"]
    torch.manual_seed(0)
    gop, qp = 3, 27
    frames = {}
    for seq, nfr in (("Seq10_416x240_50", 7), ("Seq2_416x240_30", 6), ("BQSquare_416x240_60", 6)):
        os.makedirs(tmp_path / "ori_img" / seq)
        os.makedirs(tmp_path / "compress_img_bpg" / seq / str(qp))
        for i in range(nfr):
            img = (torch.rand(3, 12, 20) * 255).to(torch.uint8)
            frames[(seq, i + 1)] = img
            write_png(img, str(tmp_path / "ori_img" / seq / f"im{i + 1:03d}.png"))
        for g in range(nfr // gop):
            ref = (frames[(seq, g * gop + 1)].int() + 3).clamp(0, 255).to(torch.uint8)
            write_png(ref, str(tmp_path / "compress_img_bpg" / seq / str(qp) / f"im{g * gop + 1:03d}_{qp}.png"))
            open(tmp_path / "compress_img_bpg" / seq / str(qp) / f"im{g * gop + 1:03d}_{qp}.txt", "w").write(f"{0.5 + g}\n")
    ds = D.GopDataset(str(tmp_path), 2048, gop, testfull=True)
    assert len(ds) == 2 + 2 + 2
    order = [os.path.basename(os.path.dirname(p[0])) for p in ds.input]
    assert order == ["BQSquare_416x240_60"] * 2 + ["Seq2_416x240_30"] * 2 + ["Seq10_416x240_50"] * 2   # natural order
    p_frames, i_frame, bpp_i, psnr_i, names, raw = ds[5]
    assert p_frames.shape == (2, 3, 12, 20) and raw.shape == (3, 3, 12, 20) and bpp_i == 1.5 and names[0].endswith("im004.png")
    assert torch.equal(raw[1], frames[("Seq10_416x240_50", 5)].float() / 255.0)
    want_mse = ((frames[("Seq10_416x240_50", 4)].float() / 255 - i_frame) ** 2).mean().item()
    assert abs(psnr_i - 10 * torch.log10(torch.tensor(1.0 / want_mse)).item()) < 1e-4
    hevc = D.GopDataset(str(tmp_path), 2048, gop, testfull=True, hevc_class="D")
    assert len(hevc) == 2 and all("BQSquare" in p for p in hevc.ref)
    # averaging: 2 I-frames (bpp 0.5, 1.5; psnr 30, 32) + 4 P-frames (bpp 0.1, psnr 35)
    summ = {"bpp": 0.1, "bpp_mv": 0.04, "bpp_res": 0.06, "psnr": 35.0, "msssim": 0.9, "mse": 1e-3, "frames": 4}
    bpp, mv, rs, psnr, ms, mse = G.combine_with_iframes(summ, 2, 2.0, 62.0, 1.9)
    assert abs(bpp - (0.4 + 2.0) / 6) < 1e-12 and abs(psnr - (140 + 62) / 6) < 1e-12 and abs(ms - (3.6 + 1.9) / 6) < 1e-12
    assert (mv, rs, mse) == (0.04, 0.06, 1e-3)


def test_vimeo_training_dataset(tmp_path):
    """tdvc_b200.data.VimeoDataset lists samples like the reference's training `DataSet.get_vimeo` (reference
    main/dataloader/dataset.py:210-247: references [im1, t-3, t-2, t-1] clipped at im1, short histories padded by repetition,
    plus [im1, im1, im3, im5] -> im7) and applies ONE draw of the imgauglist2 augmentation (augmentation.py:29-85) to the five
    frames of a sample."""
    from torchvision.io import write_png
    from tdvc_b200 import data as D
    torch.manual_seed(3)
    base = torch.rand(3, 40, 56)
    for d, clip in (("00002", "0010"), ("00001", "0002"), ("00001", "0010")):
        os.makedirs(tmp_path / d / clip)
        for i in range(1, 8):
            img = ((base * 0.8 + 0.02 * i) * 255).to(torch.uint8)     # frames of a clip differ by a constant
            write_png(img, str(tmp_path / d / clip / f"im{i}.png"))
    ds = D.VimeoDataset(str(tmp_path), 32, generator=torch.Generator().manual_seed(5))
    assert len(ds) == 3 * 7
    rel = lambda p: os.path.relpath(p, tmp_path)
    assert [rel(p) for p in ds.image_input_list[:7]] == [f"00001/0002/im{t}.png" for t in (2, 3, 4, 5, 6, 7, 7)]
    want = {0: (1, 1, 1, 1), 1: (1, 1, 2, 2), 2: (1, 1, 2, 3), 3: (1, 2, 3, 4), 4: (1, 3, 4, 5), 5: (1, 4, 5, 6), 6: (1, 1, 3, 5)}
    for k, ids in want.items():
        assert [rel(p) for p in ds.image_ref_list[k]] == [f"00001/0002/im{i}.png" for i in ids]
    assert rel(ds.image_input_list[7]) == "00001/0010/im2.png" and rel(ds.image_input_list[14]) == "00002/0010/im2.png"
    seen_crop = seen_resize = False
    for k in range(21):
        x, refs = ds[k]
        assert x.shape == (3, 32, 32) and refs.shape == (4, 3, 32, 32) and x.dtype == torch.float32
        assert 0.0 <= float(x.min()) and float(x.max()) <= 1.0
        # one draw for all five frames: geometry and photometric change are shared, so slots holding the same source frame agree
        ids = want[k % 7]
        for a in range(4):
            for b in range(a + 1, 4):
                if ids[a] == ids[b]:
                    assert torch.equal(refs[a], refs[b])
    # the crop branch returns source pixels unchanged up to flips / photometric change; check it is reachable, and the resize too
    g = torch.Generator().manual_seed(0)
    ds2 = D.VimeoDataset(str(tmp_path), 32, generator=g)
    fr = torch.rand(5, 3, 40, 56)
    for _ in range(40):
        out = ds2.augment(fr)
        assert out.shape == (5, 3, 32, 32)
        vals = set(torch.round(fr * 255).flatten().tolist())
        if set(torch.round(out * 255).flatten().tolist()) <= vals and torch.isin(out, fr).all():
            seen_crop = True
        else:
            seen_resize = True
    assert seen_crop and seen_resize
    with pytest.raises(RuntimeError):
        for _ in range(40):
            D.VimeoDataset(str(tmp_path), 64, generator=g).augment(fr)
    loader = torch.utils.data.DataLoader(ds, batch_size=4, shuffle=False, num_workers=0)
    xb, rb = next(iter(loader))
    assert xb.shape == (4, 3, 32, 32) and rb.shape == (4, 4, 3, 32, 32)     # forward(input_image, refer_frames) shapes (pnet.py:26)


def test_load_state_dict_forgets_remembered_weight_maxima():
    """The training path scales fp16 weight blocks by max |w| read one optimiser step late (ops._weight_max); swapping the weights
    wholesale must drop what was remembered."""
    from tdvc_b200 import ops
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor()
    ops._WMAX[12345] = ("stale",)
    net.load_state_dict(net.state_dict(), strict=True)
    assert not ops._WMAX


def test_shared_library_has_no_libcuda_dependency():
    """The library must load on a host without a driver (ADVICE r01): the driver entry point it needs is resolved at run time."""
    import subprocess
    from tdvc_b200 import lib as L
    out = subprocess.run(["readelf", "-d", L.LIB_PATH], capture_output=True, text=True).stdout
    assert "libcudart" in out and "libcuda.so" not in out

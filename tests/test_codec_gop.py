"""Decoding a GOP's latents as one batch (`VideoCompressor.decompress_latents_many`, under `gop.decompress_gop`) and
evaluating the closed-loop codec on real bitstreams (`gop.validate_codec`).

Every GPU test demands bit-identical results: the batch against decoding each container alone, h_s at batch T * N
against h_s at N, `decompress_gop` against `compress_gop`'s reconstructions.  Rates and PSNR of `validate_codec` are
checked against values computed here from the containers' bytes and the returned frames."""
import math
import os

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers: work on a copy so that the session's oracle keeps its state_dict."""
    import copy
    return copy.deepcopy(oracle_model)


def _coded(n=2, hy=1, shape=(1, 2)):
    """Both coders of a well-formed container body: n * hy y strings and n z strings of whole words."""
    s = lambda k, m: [bytes([k + i]) * 12 for i in range(m)]
    return {"mv": {"strings": [s(1, n * hy), s(2, n)], "shape": shape, "cluster": 16},
            "res": {"strings": [s(3, n * hy), s(4, n)], "shape": shape, "cluster": 8}}


FRAME = {"size": (64, 128), "N": 2, "precision": "exact"}


def _v2(**kw):
    from tdvc_b200 import coding
    return coding.pack_frame(_coded(**kw), frame=FRAME)


def _v3():
    from tdvc_b200 import coding
    return coding.pack_frame(_coded(hy=4), frame=dict(FRAME, y_streams="rows"))


# ------------------------------------------------------------------------------------------------------ CPU
def test_many_refuses_before_any_device_work(monkeypatch):
    """A list holding a container of another frame size or batch, a version-1 container, truncated bytes or y strings that
    are not whole words in position k raises RuntimeError naming container k before the weights are packed, a plan is
    built or a string is decoded; decompress_gop refuses the same way.  Versions 2 and 3 mix: such a list is refused only
    for want of a CUDA module.  An empty list decodes to an empty list."""
    from tdvc_b200 import coding, gop
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()

    def touched(*a, **k):
        raise AssertionError("device work on input that must be refused")

    monkeypatch.setattr(VideoCompressor, "_weights", touched)
    monkeypatch.setattr(VideoCompressor, "_plan", touched)
    monkeypatch.setattr(coding, "decode_z_symbols", touched)
    ragged = _coded()
    ragged["res"]["strings"][0][1] = b"\0" * 10
    cases = [([_v2(), _v2(), coding.pack_frame(_coded(shape=(2, 2)), frame=dict(FRAME, size=(128, 128)))],
              r"container 2 holds a 128x128 frame of N=2, container 0 a 64x128 frame of N=2"),
             ([_v2(), coding.pack_frame(_coded(n=1), frame=dict(FRAME, N=1))], r"container 1 holds a 64x128 frame of N=1"),
             ([_v2(), coding.pack_frame(_coded())], r"container 1: .*version-1"),
             ([_v2(), _v3(), _v2()[:-5]], r"container 2: unpack_frame"),
             ([_v3(), _v2(), _v2(), coding.pack_frame(ragged, frame=FRAME)],
              r"container 3: .*res y string of image 1 has 10 bytes"),
             ([b"TDV2"], r"container 0: unpack_frame")]
    for containers, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            net.decompress_latents_many(containers)
        with pytest.raises(RuntimeError, match=msg):
            gop.decompress_gop(net, torch.zeros(2, 3, 64, 128), containers, (64, 128))
    assert net.decompress_latents_many([]) == []
    with pytest.raises(RuntimeError, match="CUDA"):
        net.decompress_latents_many([_v2(), _v3(), _v2()])


def test_coded_rates_count_the_bytes():
    """bpp_mv / bpp_res: 8 x the bytes of that coder's y and z strings per padded pixel N * H * W; bpp_container: every
    byte of the container, for version 2 and version 3 alike."""
    from tdvc_b200 import gop
    for data, ny in ((_v2(), 2), (_v3(), 8)):
        mv, res, total = gop.coded_rates(data)
        px = 2 * 64 * 128
        assert mv == 8.0 * 12 * (ny + 2) / px and res == mv
        assert total == 8.0 * len(data) / px and total > mv + res


def test_summarise_codec_averages_like_validate():
    """From given sums: bpp, bpp_container, psnr and msssim average over the I- and P-frames (the I-frames with what their
    loader reports), bpp_mv, bpp_res and mse over the P-frames, as validate's combine_with_iframes forms them."""
    from tdvc_b200 import gop
    # two GOPs: 9 P-frames, 2 I-frames (bpp 0.5 + 0.7, PSNR 38 + 36, MS-SSIM 0.98 + 0.96)
    s = torch.tensor([9 * 0.12, 9 * 0.02, 9 * 0.10, 9 * 33.0, 9 * 0.95, 9 * 5e-4, 9.0, 9 * 0.125,
                      2.0, 1.2, 74.0, 1.94], dtype=torch.float64)
    r = gop.summarise_codec(s)
    close = lambda a, b: abs(a - b) < 1e-12
    assert r["frames"] == 9 and r["iframes"] == 2
    assert close(r["bpp"], (9 * 0.12 + 1.2) / 11) and close(r["bpp_container"], (9 * 0.125 + 1.2) / 11)
    assert close(r["psnr"], (9 * 33.0 + 74.0) / 11) and close(r["msssim"], (9 * 0.95 + 1.94) / 11)
    assert close(r["bpp_mv"], 0.02) and close(r["bpp_res"], 0.10) and close(r["mse"], 5e-4)
    p = r["p"]
    assert close(p["bpp"], 0.12) and close(p["bpp_container"], 0.125) and close(p["psnr"], 33.0) and p["frames"] == 9
    # the I+P part is validate's own averaging
    want = gop.combine_with_iframes(gop.summarise(s[:7]), 2, 1.2, 74.0, 1.94)
    assert (r["bpp"], r["bpp_mv"], r["bpp_res"], r["psnr"], r["msssim"], r["mse"]) == want
    empty = gop.summarise_codec(torch.zeros(gop.CODEC_STATS, dtype=torch.float64))
    assert empty["frames"] == 0 and empty["bpp"] == 0.0


# ------------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


def _net(oracle_model, cache=True):
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()
    net.load_state_dict(oracle_model.state_dict(), strict=True)
    net.cache_features = cache
    return net.to(DEV)


def _pair(n, hw, seed):
    from tdvc_b200 import synth
    pairs = [synth.make_frame_pair(*hw, seed=seed + 10 * i) for i in range(n)]
    return torch.cat([p[0] for p in pairs]).to(DEV), torch.cat([p[1] for p in pairs]).to(DEV)


def _assert_equal(got, want, what):
    if not torch.equal(got, want):
        d = (got != want).reshape(-1).nonzero()
        first = np.unravel_index(int(d[0]), tuple(want.shape)) if d.numel() else "shape"
        raise AssertionError(f"{what} differs at {first} ({int(d.numel())} elements, shapes {tuple(got.shape)} "
                             f"{tuple(want.shape)})")


def _containers(enc, n, hw, variants, seed):
    """One container per entry of `variants` = (motion cluster, residual cluster, row streams), each of another frame:
    the forward pass leaves the frame's latents in the plan, which are then coded with the asked cluster sizes."""
    from tdvc_b200 import coding
    W = enc._weights(torch.device(DEV))
    plan = enc._plan(n, *hw, torch.device(DEV))
    out = []
    for i, (c_mv, c_rs, rows) in enumerate(variants):
        x, refs = _pair(n, hw, seed + 100 * i)
        with torch.no_grad():
            enc(x, refs, False, is_compress=True)
        coded = {nm: coding.finish_coding(coding.launch_coding(plan, W, cn, W["_tables"][cn], cluster=cl), rows=rows)
                 for nm, cn, cl in (("mv", "mv", c_mv), ("res", "rs", c_rs))}
        assert [coded[nm]["cluster"] for nm in ("mv", "res")] == [c_mv, c_rs]
        frame = {"size": hw, "N": n, "precision": "exact"}
        if rows:
            frame["y_streams"] = "rows"
        out.append(coding.pack_frame(coded, frame=frame))
    return out


# the groups of the batch interleave: (16, 16, v2), (8, 8, v3), (16, 16, v2), (16, 8, v3), (8, 16, v2)
MIXED = [(16, 16, False), (8, 8, True), (16, 16, False), (16, 8, True), (8, 16, False)]


def _h_s_is_batch_invariant(dec, outs, n, hw, what, batch=None):
    """h_s of the concatenated z_hat (repeated to `batch` images) gives each image the bits it gives in a batch of n."""
    from tdvc_b200.model import Act
    dev = torch.device(DEV)
    W = dec._weights(dev)
    hz, wz = hw[0] // 64, hw[1] // 64
    for nm, cn in (("mv", "mv"), ("res", "rs")):
        z = torch.cat([o[nm]["z_hat"] for o in outs])
        if batch is not None:
            z = z.repeat((batch + z.shape[0] - 1) // z.shape[0], 1, 1, 1)[:batch]
        big = dec._plan(z.shape[0], *hw, dev)
        zb = big.buf(f"test.{cn}.z_hat", z.shape[0], hz, wz, 128)
        zb.t.copy_(z)
        pb = big.hyper_synthesis(W, cn, zb, lambda nme, h, w, c=128: big.buf(f"test.{cn}.{nme}", z.shape[0], h, w, c))
        small = dec._plan(n, *hw, dev)
        for i in range(0, z.shape[0], n):
            zs = small.buf(f"test.{cn}.z_hat", n, hz, wz, 128)
            zs.t.copy_(z[i:i + n])
            ps = small.hyper_synthesis(W, cn, zs, lambda nme, h, w, c=128: small.buf(f"test.{cn}.{nme}", n, h, w, c))
            _assert_equal(pb.t[i:i + n], ps.t, f"{what} {cn} h_s of images {i}..{i + n - 1} in a batch of {z.shape[0]}")


@pytest.mark.gpu
@pytest.mark.parametrize("hw,n,variants", [((64, 128), 1, MIXED), ((64, 64), 2, MIXED),
                                           ((1024, 1920), 1, [(16, 16, False), (16, 16, True), (8, 8, False)])])
def test_many_equals_one_at_a_time(oracle_model, hw, n, variants):
    """decompress_latents_many of containers of versions 2 and 3, coded with clusters of 8 and 16 (per coder, groups
    interleaved in the list), equals decompress_latents of each container alone: z_hat, symbols, indexes and y_hat of
    both coders and the frame record.  h_s at the batch's size gives each image the bits it gives at N (at 1920x1024 also
    for an 11-frame GOP's batch)."""
    enc, dec, one = _net(oracle_model), _net(oracle_model), _net(oracle_model)
    containers = _containers(enc, n, hw, variants, seed=3)
    outs = dec.decompress_latents_many(containers)
    assert len(outs) == len(containers)
    assert (torch.device(DEV), len(containers) * n, *hw) in dec._plans
    for k, (data, got) in enumerate(zip(containers, outs)):
        want = one.decompress_latents(data)
        assert got["frame"] == want["frame"]
        for nm in ("mv", "res"):
            assert set(got[nm]) == set(want[nm]) == {"y_hat", "y_symbols", "y_indexes", "z_hat"}
            for key in want[nm]:
                _assert_equal(got[nm][key], want[nm][key], f"{hw} N={n} container {k} {nm} {key}")
    _h_s_is_batch_invariant(dec, outs, n, hw, f"{hw} N={n}")
    if hw == (1024, 1920):
        _h_s_is_batch_invariant(dec, outs, n, hw, f"{hw} GOP of 11", batch=11)


@pytest.mark.gpu
@pytest.mark.parametrize("row_streams", [False, True])
def test_gop_decode_is_one_batch_and_exact(oracle_model, row_streams):
    """decompress_gop of a 6-frame GOP at 64x128 decodes the latents on one plan of batch 6 and returns compress_gop's
    reconstructions, which a frame-by-frame loop of decompress rebuilds too."""
    from tdvc_b200 import gop, synth
    frames = synth.make_gop(64, 128, gop=7, seed=8).to(DEV)
    enc, dec, ref = _net(oracle_model), _net(oracle_model, cache=False), _net(oracle_model)
    containers, recons = gop.compress_gop(enc, frames[:1], frames[1:], row_streams=row_streams)
    got = gop.decompress_gop(dec, frames[:1], containers, (64, 128))
    assert (torch.device(DEV), 6, 64, 128) in dec._plans
    refs = gop.RefBuffer(frames[:1])
    for i, data in enumerate(containers):
        window, keys = refs.window()
        one = ref.decompress(data, window, ref_keys=keys)
        refs.push(one)
        _assert_equal(one, recons[i], f"frame {i}: decompress")
        _assert_equal(got[i], recons[i], f"frame {i}: decompress_gop")


@pytest.mark.gpu
@pytest.mark.parametrize("row_streams", [False, True])
def test_damaged_container_in_a_gop(oracle_model, row_streams):
    """A truncated y string in container 2 and a truncated z string in container 1 of a 4-frame GOP raise naming the
    container, the coder and the image (for y the position or row), before anything is synthesised and without faulting
    the device; the next decompress_gop is exact."""
    from tdvc_b200 import coding, gop, synth
    frames = synth.make_gop(64, 128, gop=5, seed=9).to(DEV)
    enc, dec = _net(oracle_model), _net(oracle_model)
    containers, recons = gop.compress_gop(enc, frames[:1], frames[1:], row_streams=row_streams)

    def damaged(k, nm, which, j, fn):
        box = coding.unpack_frame(containers[k])
        frame = box.pop("frame")
        box[nm]["strings"][which][j] = fn(box[nm]["strings"][which][j])
        return containers[:k] + [coding.pack_frame(box, frame=frame)] + containers[k + 1:]

    def synthesised(*a, **k):
        raise AssertionError("a frame was synthesised before the broken string was reported")

    dec._synthesise = synthesised
    y_msg = (r"ar_decode_rows: rs y row 2 of image 0 of container 2 is truncated or corrupt at \(h=2, " if row_streams
             else r"ar_decode: the rs y string of image 0 of container 2 is truncated or corrupt at latent position \(h=")
    with pytest.raises(RuntimeError, match=y_msg):
        gop.decompress_gop(dec, frames[:1], damaged(2, "res", 0, 2 if row_streams else 0, lambda s: s[:len(s) // 8 * 4]),
                           (64, 128))
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match=r"the mv z string of image 0 of container 1 is truncated or corrupt"):
        gop.decompress_gop(dec, frames[:1], damaged(1, "mv", 1, 0, lambda s: s[:4]), (64, 128))
    torch.cuda.synchronize()
    del dec._synthesise
    got = gop.decompress_gop(dec, frames[:1], containers, (64, 128))
    for i, (a, b) in enumerate(zip(got, recons)):
        _assert_equal(a, b, f"after damaged containers: frame {i}")


def _dataset(root):
    """Two sequences laid out as the reference's datasets are (tdvc_b200/data.py): 3 GOPs of 4 frames at 176x208, the
    I-frames a brightened copy standing in for BPG with 0.75 bpp."""
    from torchvision.io import write_png
    from tdvc_b200 import data as D
    from tdvc_b200 import synth
    gop_size, qp = 4, 27
    seqs = {"a_416x240_50": synth.make_gop(176, 208, gop=8, seed=91), "b_416x240_50": synth.make_gop(176, 208, gop=4, seed=92)}
    for seq, fr in seqs.items():
        os.makedirs(root / "ori_img" / seq)
        os.makedirs(root / "compress_img_bpg" / seq / str(qp))
        for i in range(fr.shape[0]):
            write_png((fr[i] * 255).round().to(torch.uint8), str(root / "ori_img" / seq / f"im{i + 1:03d}.png"))
        for g in range(fr.shape[0] // gop_size):
            ref = ((fr[g * gop_size] * 255).round() + 2).clamp(0, 255).to(torch.uint8)
            write_png(ref, str(root / "compress_img_bpg" / seq / str(qp) / f"im{g * gop_size + 1:03d}_{qp}.png"))
            open(root / "compress_img_bpg" / seq / str(qp) / f"im{g * gop_size + 1:03d}_{qp}.txt", "w").write("0.75\n")
    ds = D.GopDataset(str(root), 2048, gop_size, testfull=True)
    assert len(ds) == 3
    return ds


@pytest.mark.gpu
def test_validate_codec_over_a_gop_dataset(oracle_model, tmp_path):
    """Rates are 8 x bytes per padded pixel of compress_gop's containers, PSNR is the mean over the returned frames with
    the I-frames' PSNR, as validate averages them; a decoder gives the same numbers; two shards' summed stats give the
    unsharded result."""
    from tdvc_b200 import coding, gop
    ds = _dataset(tmp_path)
    enc, dec, twin = _net(oracle_model), _net(oracle_model), _net(oracle_model)
    for row_streams in (False, True):
        res = gop.validate_codec(ds, enc, enable_amp=False, row_streams=row_streams)
        mv = rs = tot = psnr = 0.0
        i_bpp = i_psnr = 0.0
        for g in range(3):
            p_frames, i_frame, bpp_i, psnr_i, _, _ = ds[g]
            containers, recons = gop.compress_gop(twin, i_frame.unsqueeze(0).to(DEV), p_frames.to(DEV),
                                                  row_streams=row_streams)
            px = 192 * 256   # 176x208 padded to multiples of 64
            for data, r, x in zip(containers, recons, p_frames):
                box = coding.unpack_frame(data)
                mv += 8.0 * sum(len(s) for lst in box["mv"]["strings"] for s in lst) / px
                rs += 8.0 * sum(len(s) for lst in box["res"]["strings"] for s in lst) / px
                tot += 8.0 * len(data) / px
                psnr += 10.0 * math.log10(1.0 / (r[0].double().cpu() - x.double()).pow(2).mean().item())
            i_bpp += float(bpp_i)
            i_psnr += float(psnr_i)
        what = f"row_streams={row_streams}"
        assert res["frames"] == 9 and res["iframes"] == 3, what
        assert abs(res["bpp_mv"] - mv / 9) < 1e-12 and abs(res["bpp_res"] - rs / 9) < 1e-12, what
        assert abs(res["p"]["bpp_container"] - tot / 9) < 1e-12, what
        assert abs(res["bpp"] - (mv + rs + i_bpp) / 12) < 1e-12, what
        assert abs(res["bpp_container"] - (tot + i_bpp) / 12) < 1e-12, what
        assert abs(res["p"]["psnr"] - psnr / 9) < 1e-6 and abs(res["psnr"] - (psnr + i_psnr) / 12) < 1e-6, what
        assert 0.0 < res["msssim"] <= 1.0
        decoded = gop.validate_codec(ds, enc, decoder=dec, enable_amp=False, row_streams=row_streams)
        _assert_same_summary(decoded, res, what + " with a decoder")
    shards = [gop.validate_codec(ds, enc, enable_amp=False, gops=gop.shard_gops(3, r, 2))["stats"] for r in range(2)]
    whole = gop.validate_codec(ds, enc, enable_amp=False)
    _assert_same_summary(gop.summarise_codec(gop.reduce_stats(shards[0] + shards[1])), whole, "two shards")


def _assert_same_summary(got, want, what):
    """Equal up to the order of sums: the squared-error and MS-SSIM kernels accumulate with atomics, and shards add up in
    another order."""
    for k, v in want.items():
        if k == "stats":
            continue
        if k == "p":
            _assert_same_summary(got["p"], v, what + " (P-frames)")
        elif isinstance(v, int):
            assert got[k] == v, (what, k, got[k], v)
        else:
            assert abs(got[k] - v) <= (1e-6 if k == "msssim" else 1e-10) * max(1.0, abs(v)), (what, k, got[k], v)

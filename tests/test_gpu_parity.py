"""GPU tests (-m gpu): end-to-end parity of the CUDA P-frame forward (through VideoCompressor.forward, i.e. the
C-ABI kernels) against the oracle (restatement pinned bit-exact to the reference code) and against the committed
golden fixtures produced by the reference's own unmodified code (tests/golden, oracle/make_golden.py).

Bars (BASELINE.json north_star): reconstruction <= 1e-3 max-abs, PSNR within 0.01 dB, bpp within 0.1 % relative,
>= 99.9 % of quantised latent symbols identical.  The exact-fp32 path (conv_impl=1) and the tensor-core path
(conv_impl=0: fp16 hi/lo-split tcgen05 MMA, fp32 accumulate) are both held to the same bars.
"""
import math

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import make_golden_fullres as GF

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def net(oracle_model, dev):
    from tdvc_b200.model import VideoCompressor
    m = VideoCompressor().eval()
    m.load_state_dict(oracle_model.state_dict(), strict=True)
    return m.to(dev)


def _psnr(a, b):
    return 10.0 * math.log10(1.0 / ((a - b) ** 2).mean().item())


def _check_frame(net, oracle_model, dev, h, w, seed, impl, precision="exact"):
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(h, w, seed=seed)
    ot, gt = {}, {}
    net.conv_impl, net.precision = impl, precision
    try:
        with torch.no_grad():
            o_recon, o_bres, o_bmv = oracle_model(x, refs, False, taps=ot)
            g_recon, g_bres, g_bmv = net(x.to(dev), refs.to(dev), False, taps=gt)
    finally:
        net.precision = "auto"
    g_recon = g_recon.cpu()
    same = {}
    for c in ("mv", "res"):
        same[c + ".y"] = (ot[f"{c}.y_hat"] == gt[f"{c}.y_hat"].cpu()).float().mean().item()
        same[c + ".z"] = (ot[f"{c}.z_hat"] == gt[f"{c}.z_hat"].cpu()).float().mean().item()
    assert min(same.values()) >= 0.999, same
    # mismatches only at rounding ties: the pre-quantiser value must sit next to a half-integer
    for c in ("mv", "res"):
        bad = ot[f"{c}.y_hat"] != gt[f"{c}.y_hat"].cpu()
        if bad.any():
            frac = (ot[f"{c}.y"][bad] - torch.floor(ot[f"{c}.y"][bad]) - 0.5).abs()
            assert frac.max() < 5e-3, f"{c}: symbol mismatch away from a rounding tie ({frac.max().item()})"
    assert torch.equal(ot["loopfilter.ind"], gt["loopfilter.ind"].cpu())
    assert abs(o_bres.item() - g_bres.item()) <= 1e-3 * o_bres.item()
    assert abs(o_bmv.item() - g_bmv.item()) <= 1e-3 * o_bmv.item()
    if min(same.values()) == 1.0:
        assert (o_recon - g_recon).abs().max().item() <= 1e-3
    # PSNR of the reconstruction against the source frame: within 0.01 dB
    assert abs(_psnr(o_recon, x) - _psnr(g_recon, x)) <= 0.01
    assert g_recon.min() >= 0.0 and g_recon.max() <= 1.0
    return o_recon, g_recon, same


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("case", [(64, 64, 1), (128, 192, 2), (64, 256, 7)])
def test_pframe_forward_vs_oracle(net, oracle_model, dev, case, impl):
    _check_frame(net, oracle_model, dev, *case, impl)


def test_pframe_forward_vs_oracle_multi_tile(net, oracle_model, dev):
    """256x320: several 32- and 64-row items per column of tiles on every pyramid level (the row-phase 7x7 SPyNet layers
    walk four 64-row items), 128-channel split tiles at 1/2 scale, FeatureFix with more than one candidate block."""
    _check_frame(net, oracle_model, dev, 256, 320, 3, 0)


@pytest.mark.parametrize("case", [(64, 64, 1), (128, 192, 2), (256, 320, 3)])
def test_pframe_forward_mixed_precision_vs_oracle(net, oracle_model, dev, case):
    """`precision = "mixed"`: one fp16 MMA product (the reference's autocast arithmetic) in the stages behind the last quantiser
    of the frame - residual synthesis transform and in-loop filter - held to the SAME bars as the fp32-class path
    (budget: profiles/r02_precision_budget.txt).  The symbols of this frame cannot change (nothing in front of a quantiser
    is relaxed); reconstruction <= 1e-3, PSNR 0.01 dB, FeatureFix indices identical."""
    _, _, same = _check_frame(net, oracle_model, dev, *case, 0, precision="mixed")
    assert min(same.values()) >= 0.999


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("name", ["p64x64_s1", "p128x192_s2"])
def test_pframe_forward_vs_reference_golden(net, dev, name, impl):
    """Fixtures were produced by the reference's own code (oracle/make_golden.py); nothing from oracle/ runs here."""
    from tdvc_b200 import synth
    g = load_golden(name)
    assert abs(synth.state_checksum(net.state_dict()) - float(g["state_checksum"])) < 1e-6 * float(g["state_checksum"])
    x, refs = synth.make_frame_pair(int(g["h"]), int(g["w"]), seed=int(g["seed"]))
    taps = {}
    net.conv_impl = impl
    with torch.no_grad():
        recon, bres, bmv = net(x.to(dev), refs.to(dev), False, taps=taps)
    same = []
    for c in ("mv", "res"):
        same.append((taps[f"{c}.y_hat"].cpu().numpy().astype(np.int16) == g[f"{c}_y_hat"]).mean())
    assert min(same) >= 0.999, same
    assert (taps["loopfilter.ind"].cpu().numpy().astype(np.int32) == g["ind"]).all()
    assert abs(bres.item() - float(g["bpp_res"][0])) <= 1e-3 * float(g["bpp_res"][0])
    assert abs(bmv.item() - float(g["bpp_mv"][0])) <= 1e-3 * float(g["bpp_mv"][0])
    if min(same) == 1.0:
        assert np.abs(recon.cpu().numpy() - g["recon"]).max() <= 1e-3


@pytest.mark.parametrize("impl", [1, 0])
def test_batch_of_two_vs_oracle(net, oracle_model, dev, impl):
    """N = 2 (the reference's DataParallel / training batches, bpp aggregated over the batch: reference pnet.py:38-43,82-83):
    two different frame pairs in one call against the oracle on the same batch."""
    from tdvc_b200 import synth
    xa, ra = synth.make_frame_pair(64, 128, seed=11)
    xb, rb = synth.make_frame_pair(64, 128, seed=12)
    x, refs = torch.cat([xa, xb], 0), torch.cat([ra, rb], 0)
    ot, gt = {}, {}
    net.conv_impl = impl
    with torch.no_grad():
        o = oracle_model(x, refs, False, taps=ot)
        g = net(x.to(dev), refs.to(dev), False, taps=gt)
    net.conv_impl = 0
    for c in ("mv", "res"):
        assert (ot[f"{c}.y_hat"] == gt[f"{c}.y_hat"].cpu()).float().mean().item() >= 0.999
        assert (ot[f"{c}.z_hat"] == gt[f"{c}.z_hat"].cpu()).float().mean().item() >= 0.999
    assert torch.equal(ot["loopfilter.ind"], gt["loopfilter.ind"].cpu())
    assert (o[0] - g[0].cpu()).abs().max().item() <= 1e-3
    assert abs(o[1].item() - g[1].item()) <= 1e-3 * o[1].item() and abs(o[2].item() - g[2].item()) <= 1e-3 * o[2].item()
    # and the batch result equals the two single-frame results (recon) / their mean (bpp)
    with torch.no_grad():
        ga = net(xa.to(dev), ra.to(dev), False)
        gb = net(xb.to(dev), rb.to(dev), False)
    # (not bit-identical: the batched launches tile / reduce in a different order)
    assert (g[0][0:1] - ga[0]).abs().max().item() <= 1e-4 and (g[0][1:2] - gb[0]).abs().max().item() <= 1e-4
    assert abs(g[1].item() - 0.5 * (ga[1].item() + gb[1].item())) <= 1e-4 * g[1].item()


@pytest.mark.parametrize("impl", [1, 0])
def test_config5_fusion_and_inloop_filter_vs_oracle(net, oracle_model, dev, impl):
    """BASELINE config 5: multi-frame feature fusion + reference-based in-loop filter with 4 reference frames, fed with the
    oracle's own intermediate tensors (prediction1, recon_feat) of a synthetic frame pair."""
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(128, 192, seed=5)
    taps = {}
    with torch.no_grad():
        oracle_model(x, refs, False, taps=taps)
        pred1, recf = taps["prediction1"], taps["recon_feat"]
        want_pred = oracle_model.mcfilter(pred1, refs)
        want_recon = oracle_model.loopfilter(recf, refs).clamp(0.0, 1.0)
    net.conv_impl = impl
    got_pred, got_recon = net.fusion_and_filter(pred1.to(dev), refs.to(dev), recf.to(dev))
    net.conv_impl = 0
    assert (got_pred.cpu() - want_pred).abs().max().item() <= 1e-4 * max(1.0, want_pred.abs().max().item())
    assert (got_recon.cpu() - want_recon).abs().max().item() <= 1e-4
    assert net.last_launches > 40


def test_default_init_degenerate_case(dev):
    """Module default init (SURVEY 8d): all symbols 0, DCN offsets exactly 0 - still must agree."""
    from oracle.stats import build_oracle
    from tdvc_b200 import synth
    from tdvc_b200.model import VideoCompressor
    orc = build_oracle(conditioned=False)
    m = VideoCompressor().eval()
    m.load_state_dict(orc.state_dict(), strict=True)
    m = m.to(dev)
    x, refs = synth.make_frame_pair(64, 64, seed=3)
    with torch.no_grad():
        a = orc(x, refs, False)
        b = m(x.to(dev), refs.to(dev), False)
    assert (a[0] - b[0].cpu()).abs().max() < 1e-4
    assert abs(a[1].item() - b[1].item()) < 1e-3 * a[1].item() and abs(a[2].item() - b[2].item()) < 1e-3 * a[2].item()


def test_gop_chain_vs_oracle(net, oracle_model, dev):
    """Three chained P-frames through the GOP driver (reference tools/predict.py:51-68 semantics, incl. pad/crop
    for a frame size that is not a multiple of 64): PSNR within 0.01 dB and bpp within 0.1 % per frame."""
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    net.conv_impl = 0
    frames = synth.make_gop(56, 120, gop=4, seed=21)
    res = G.code_gop(net, frames[0:1].to(dev), frames[1:].to(dev), keep_recon=True)
    refs = [G.pad(frames[0:1], 64)]
    for i in range(3):
        x = G.pad(frames[i + 1:i + 2], 64)
        with torch.no_grad():
            recon, bres, bmv = oracle_model(x, G.reference_window(refs), False)
        refs.append(recon)
        rc = G.crop(recon, (56, 120))
        mse = ((rc - frames[i + 1:i + 2]) ** 2).mean().item()
        g_mse = res["sse"][i].item() / res["numel"]
        assert abs(10 * math.log10(1 / mse) - 10 * math.log10(1 / g_mse)) <= 0.01
        assert abs(bres.item() - res["bpp_res"][i].item()) <= 1e-3 * bres.item()
        assert abs(bmv.item() - res["bpp_mv"][i].item()) <= 1e-3 * bmv.item()
    st = G.summarise(G.gop_stats(res))
    assert st["frames"] == 3 and st["bpp"] > 0 and 5 < st["psnr"] < 60


def test_cuda_graph_equals_eager_and_is_deterministic(net, dev):
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(128, 128, seed=4)
    x, refs = x.to(dev), refs.to(dev)
    net.conv_impl = 0
    net.use_cuda_graph = False
    a = net(x, refs, False)
    b = net(x, refs, False)
    net.use_cuda_graph = True
    try:
        c = net(x, refs, False)
        d = net(x, refs, False)
    finally:
        net.use_cuda_graph = False
    for p, q, r, s in zip(a, b, c, d):
        assert torch.equal(p, q) and torch.equal(p, r) and torch.equal(p, s)
    assert net.last_launches > 200


def test_full_size_properties(net, dev):
    """1920x1024 (BASELINE config 2), where the oracle takes ~90 s: size-independent properties only -
    run-to-run bit-identical, tensor-core path vs exact-fp32 path within the parity bars, translation check of
    the in-loop filter indices' range, finite bpp."""
    from tdvc_b200 import synth
    g = synth.make_gop(1024, 1920, gop=2, seed=0).to(dev)
    x, refs = g[1:2], g[0:1].unsqueeze(1).expand(-1, 4, -1, -1, -1).contiguous()
    net.conv_impl = 0
    t0 = {}
    a = net(x, refs, False, taps=t0)
    b = net(x, refs, False)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    net.conv_impl = 1
    t1 = {}
    c = net(x, refs, False, taps=t1)
    net.conv_impl = 0
    for k in ("mv.y_hat", "res.y_hat", "mv.z_hat", "res.z_hat"):
        assert (t0[k] == t1[k]).float().mean().item() >= 0.999, k
    assert torch.equal(t0["loopfilter.ind"], t1["loopfilter.ind"])
    assert abs(a[1].item() - c[1].item()) <= 1e-3 * c[1].item() and abs(a[2].item() - c[2].item()) <= 1e-3 * c[2].item()
    assert abs(_psnr(a[0], x) - _psnr(c[0], x)) <= 0.01
    assert math.isfinite(a[1].item()) and a[1].item() > 0 and a[0].min() >= 0 and a[0].max() <= 1


# ------------------------------------------------------------------------------------------------ 1920x1024 (BASELINE configs 2, 5)
def _dilate_latent(bad, r):
    """bad: (1, C, h, w) bool at 1/16 scale -> (16h, 16w) bool mask of the pixels within r latent cells of a flipped symbol."""
    m = bad.any(1, keepdim=True).float()
    m = torch.nn.functional.max_pool2d(m, 2 * r + 1, 1, r)
    return torch.nn.functional.interpolate(m, scale_factor=16, mode="nearest")[0, 0] > 0


def _symbols_vs_golden(g, taps, net, prefix=""):
    """Fraction of identical symbols per latent + mask (1/16 scale) of the flipped y positions.  Mismatches are allowed only at
    rounding ties: a flipped motion symbol must have its pre-quantiser value next to a half-integer; a flipped residual symbol
    either sits at a tie itself or lies in the footprint (12 latent cells) of a flipped motion symbol - there the motion
    compensation, hence the residual it codes, legitimately differs."""
    same, bad_any, near_mv = {}, None, None
    for c, cn in (("mv", "mvCoder"), ("res", "resCoder")):
        yh = taps[f"{c}.y_hat"].cpu()
        bad = yh.numpy().astype(np.int16) != g[prefix + f"{c}_y_hat"].astype(np.int16)
        same[c + ".y"] = 1.0 - bad.mean()
        bad = torch.from_numpy(bad)
        if bad.any():
            y = taps[f"{c}.y"].cpu()
            tie = ((y - torch.floor(y)) - 0.5).abs()
            check = bad if near_mv is None else (bad & ~near_mv)
            if check.any():
                assert tie[check].max() < 5e-3, f"{c}: symbol mismatch away from a rounding tie ({tie[check].max().item()})"
        if c == "mv":
            near_mv = torch.nn.functional.max_pool2d(bad.any(1, keepdim=True).float(), 25, 1, 12) > 0
        bad_any = bad if bad_any is None else (bad_any | bad)
        med = getattr(net, cn).entropy_bottleneck.quantiles[:, 0, 1].detach().view(1, -1, 1, 1).cpu()
        zq = torch.round(taps[f"{c}.z_hat"].cpu() - med).numpy().astype(np.int16)
        same[c + ".z"] = (zq == g[prefix + f"{c}_z_hat_minus_med"].astype(np.int16)).mean()
    return same, bad_any


@pytest.mark.parametrize("precision", ["exact", "mixed"])
def test_fullres_pframe_vs_reference_golden(net, dev, precision):
    """BASELINE config 2's frame size against the reference's own code (tests/golden/p1024x1920_s0.npz,
    oracle/make_golden_fullres.py): 148 persistent CTAs walking dozens of items each, FeatureFix at scale 128 with 28
    patches of 384x384 blocks, 503 MB tensors, TMA box clipping at 1920 columns - all four north_star bars at full size.
    Where a symbol flipped at a rounding tie (allowed), the reconstruction is compared outside that symbol's footprint."""
    from tdvc_b200 import synth
    g = load_golden("p1024x1920_s0")
    assert abs(synth.state_checksum(net.state_dict()) - float(g["state_checksum"])) < 1e-6 * float(g["state_checksum"])
    x, refs = synth.make_frame_pair(1024, 1920, seed=0)
    chk = float(x.double().sum() + refs.double().sum())
    assert abs(chk - float(g["input_checksum"])) < 1e-7 * abs(chk), "synthetic frames differ from the fixture's"
    taps = {}
    net.conv_impl, net.precision = 0, precision
    try:
        with torch.no_grad():
            recon, bres, bmv = net(x.to(dev), refs.to(dev), False, taps=taps)
    finally:
        net.precision = "auto"
    same, bad = _symbols_vs_golden(g, taps, net)
    print("identical symbols", same, "flipped y symbols", int(bad.sum()))
    assert min(same.values()) >= 0.999, same
    assert (taps["loopfilter.ind"].cpu().numpy().astype(np.int32) == g["ind"]).all()
    assert abs(bres.item() - float(g["bpp_res"][0])) <= 1e-3 * float(g["bpp_res"][0])
    assert abs(bmv.item() - float(g["bpp_mv"][0])) <= 1e-3 * float(g["bpp_mv"][0])
    # reconstruction <= 1e-3 (on the fixture's sample of pixel positions); where a symbol flipped at a tie (a few hundred of the
    # 2 million: any two fp32 implementations differ there) the decoder legitimately differs inside that symbol's footprint:
    # every pixel above the bar must lie within 4 latent cells of a flipped symbol, and they must be rare
    want = torch.from_numpy(g["recon_q16"].astype(np.float32) / 65535.0)
    err = (GF.pixel_sample(recon.cpu(), GF.PIX_STEP) - want).abs().max(0).values
    over = err > 1e-3 + 1.0 / 65535
    print("recon max err", err.max().item(), "sampled pixels over 1e-3:", int(over.sum()), "of", over.numel())
    assert over.float().mean().item() < 1e-3 and err.max().item() < 5e-3
    if over.any():
        near = GF.sample(_dilate_latent(bad, 4), GF.PIX_STEP)
        assert bad.any() and not (over & ~near).any(), "reconstruction error above 1e-3 away from any flipped symbol"
    mse = ((recon.cpu().double() - x.double()) ** 2).mean().item()
    assert abs(10 * math.log10(1 / mse) - 10 * math.log10(1 / float(g["mse"]))) <= 0.01
    # ---- BASELINE config 5 at full size: multi-frame fusion + in-loop filter with 4 reference frames.  Stage tensors of the
    #      forward against the reference's (samples of the stride-32 grid and of the 64x64-tile means), then the standalone
    #      entry point on the same inputs, which must reproduce the forward's own prediction / reconstruction bit for bit.
    for k in GF.STAGES:
        v = taps[k].cpu()
        scale = float(g["stat_" + k][2])
        d = (GF.sample(v[:, :, ::32, ::32], GF.S32_STEP) - torch.from_numpy(g["s32_" + k])).abs()
        frac_off = (d > 1e-3 * scale).float().mean().item()
        assert frac_off < (5e-3 if bad.any() else 1e-6) and d.max().item() < 1e-2 * scale, (k, frac_off, d.max().item())
        tm = GF.sample(torch.nn.functional.avg_pool2d(v.double(), 64).float(), GF.TILE_STEP)
        assert (tm - torch.from_numpy(g["tile_" + k])).abs().max().item() <= 1e-4 * scale
    net.precision = precision
    try:
        pred, rec5 = net.fusion_and_filter(taps["prediction1"], refs.to(dev), taps["recon_feat"])
    finally:
        net.precision = "auto"
    assert torch.equal(pred, taps["prediction"]) and torch.equal(rec5, recon)


def test_enabled_amp_selects_the_precision(net, dev):
    """precision = "auto" (default): the reference's own switch decides - enabled_amp=False is the fp32-class path,
    enabled_amp=True relaxes the stages behind the last quantiser (the reference then autocasts far more, pnet.py:27,51,75)."""
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(64, 128, seed=61)
    x, refs = x.to(dev), refs.to(dev)
    net.conv_impl = 0
    res = {}
    for prec, amp in (("exact", False), ("mixed", False), ("auto", False), ("auto", True)):
        net.precision = prec
        res[(prec, amp)] = net(x, refs, amp)
    net.precision = "auto"
    assert all(torch.equal(a, b) for a, b in zip(res[("auto", False)], res[("exact", False)]))
    assert all(torch.equal(a, b) for a, b in zip(res[("auto", True)], res[("mixed", False)]))
    assert not torch.equal(res[("exact", False)][0], res[("mixed", False)][0])
    assert torch.equal(res[("exact", False)][1], res[("mixed", False)][1]) and torch.equal(res[("exact", False)][2], res[("mixed", False)][2])


@pytest.mark.parametrize("amp", [False, True])
def test_fullres_gop_chain_vs_reference_golden(net, dev, amp):
    """Six chained 1920x1024 P-frames of the GOP bench.py codes first, free running (every frame references OUR previous
    reconstructions, reference tools/predict.py:51-68), against the reference's chain: per frame bpp within 0.1 %, PSNR within
    0.01 dB, FeatureFix indices identical and >= 99.9 % of the symbols of both coders identical on EVERY frame (measured: 0.01 %
    of the motion and 0.04 % of the residual symbols differ per frame, without growth along the chain), reconstruction within
    1e-3 on >= 99.9 % of the sampled pixels."""
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    g = load_golden("chain1024x1920_s100")
    n_p = int(g["n_p"])
    frames = synth.make_gop(1024, 1920, gop=n_p + 1, seed=int(g["seed"]))
    assert abs(float(frames.double().sum()) - float(g["input_checksum"])) < 1e-7 * float(g["input_checksum"])
    frames = frames.to(dev)
    net.conv_impl, net.precision = 0, "auto"
    refs = [frames[0:1]]
    for t in range(1, n_p + 1):
        taps = {}
        x = frames[t:t + 1]
        with torch.no_grad():
            recon, bres, bmv = net(x, G.reference_window(refs), amp, taps=taps)
        refs.append(recon)
        if len(refs) > 4:
            refs = [refs[0]] + refs[-3:]
        p = f"f{t}_"
        # frame 1 sees exactly the reference's inputs: its flips must sit at rounding ties; later frames reference our own
        # reconstructions, which already differ inside the footprints of earlier flips
        same, bad = _symbols_vs_golden(g, taps, net, p) if t == 1 else _symbols_vs_golden_loose(g, taps, net, p)
        mse = ((recon.double() - x.double()) ** 2).mean().item()
        want = torch.from_numpy(g[p + "recon_s4_q16"].astype(np.float32) / 65535.0)
        d = (GF.pixel_sample(recon[:, :, ::4, ::4].cpu(), GF.S4_PIX_STEP) - want).abs()
        print(f"frame {t}: identical {same}, recon sample max err {d.max().item():.2e}, frac > 1e-3 {(d > 1e-3).float().mean().item():.2e}")
        assert min(same.values()) >= 0.999, (t, same)
        assert (taps["loopfilter.ind"].cpu().numpy().astype(np.int32) == g[p + "ind"]).all(), t
        assert abs(bres.item() - float(g[p + "bpp_res"][0])) <= 1e-3 * float(g[p + "bpp_res"][0]), t
        assert abs(bmv.item() - float(g[p + "bpp_mv"][0])) <= 1e-3 * float(g[p + "bpp_mv"][0]), t
        assert abs(10 * math.log10(1 / mse) - 10 * math.log10(1 / float(g[p + "mse"]))) <= 0.01, t
        assert (d > 1e-3).float().mean().item() < 1e-3 and d.max().item() < 5e-3, t
        tm = torch.nn.functional.avg_pool2d(recon.double(), 64).float().cpu()
        assert (tm - torch.from_numpy(g[p + "recon_tile"])).abs().max().item() <= 1e-3, t


def _symbols_vs_golden_loose(g, taps, net, prefix):
    """Later frames of a free-running chain: the inputs already differ where an earlier symbol flipped, so flips are counted
    but not required to sit at ties."""
    same = {}
    for c, cn in (("mv", "mvCoder"), ("res", "resCoder")):
        yh = GF.sample(taps[f"{c}.y_hat"].cpu().numpy().astype(np.int16), GF.Y_STEP_CHAIN)
        same[c + ".y"] = (yh == g[prefix + f"{c}_y_hat"].astype(np.int16)).mean()
        med = getattr(net, cn).entropy_bottleneck.quantiles[:, 0, 1].detach().view(1, -1, 1, 1).cpu()
        zq = torch.round(taps[f"{c}.z_hat"].cpu() - med).numpy().astype(np.int16)
        same[c + ".z"] = (zq == g[prefix + f"{c}_z_hat_minus_med"].astype(np.int16)).mean()
    return same, None


# ------------------------------------------------------------------------------------------------ per-GOP feature caches
@pytest.mark.parametrize("precision", ["exact", "mixed"])
def test_feature_caches_are_bit_exact(net, dev, precision):
    """The per-GOP caches (FeatureExtract_ref of the I-frame; the frame-wise front of the multi-frame fusion per previous
    reconstruction) must not change a single bit: a 2-GOP chain coded with and without them, eagerly and through the
    per-variant CUDA graphs."""
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    net.conv_impl, net.precision = 0, precision
    gops = [synth.make_gop(128, 192, gop=6, seed=40 + i).to(dev) for i in range(2)]

    def chain(cache, graph):
        net.cache_features, net.use_cuda_graph = cache, graph
        out, hits0 = [], net._plan(1, 128, 192, dev).cache_hits
        for _ in range(2 if graph else 1):     # the second pass replays the graphs captured by the first
            out = []
            for f in gops:
                refs = [f[0:1]]
                for t in range(1, f.shape[0]):
                    with torch.no_grad():
                        r = net(f[t:t + 1], G.reference_window(refs), False)
                    refs.append(r[0])
                    if len(refs) > 4:
                        refs = [refs[0]] + refs[-3:]
                    out.append(r)
        return out, net._plan(1, 128, 192, dev).cache_hits - hits0

    try:
        base, h0 = chain(False, False)
        cached, h1 = chain(True, False)
        graphed, h2 = chain(True, True)
    finally:
        net.cache_features, net.use_cuda_graph, net.precision = True, False, "auto"
    assert h0 == 0 and h1 >= 20 and h2 > h1
    for a, b, c in zip(base, cached, graphed):
        for u, v, w in zip(a, b, c):
            assert torch.equal(u, v) and torch.equal(u, w)


def test_forward_is_stateless_in_results(net, dev):
    """Interleaving unrelated sequences (cache misses, partial hits, changed weights) gives the same bits as fresh calls."""
    from tdvc_b200 import synth
    net.conv_impl, net.precision, net.cache_features = 0, "auto", True
    xa, ra = synth.make_frame_pair(64, 128, seed=31)
    xb, rb = synth.make_frame_pair(64, 128, seed=32)
    xa, ra, xb, rb = xa.to(dev), ra.to(dev), xb.to(dev), rb.to(dev)
    net.cache_features = False
    wa, wb = net(xa, ra, False), net(xb, rb, False)
    net.cache_features = True
    rmix = torch.stack([ra[:, 0], rb[:, 2], ra[:, 2], rb[:, 3]], 1)   # shares slices with both
    net.cache_features = False
    wm = net(xb, rmix, False)
    net.cache_features = True
    for x, r, w in ((xa, ra, wa), (xb, rb, wb), (xa, ra, wa), (xb, rmix, wm), (xb, rb, wb), (xa, ra, wa)):
        got = net(x, r, False)
        assert all(torch.equal(p, q) for p, q in zip(got, w))
    # a changed parameter invalidates the caches
    with torch.no_grad():
        net.mcfilter.conv02.bias.add_(0.01)
    try:
        g1 = net(xa, ra, False)
        assert not torch.equal(g1[0], wa[0])
    finally:
        with torch.no_grad():
            net.mcfilter.conv02.bias.sub_(0.01)
    g2 = net(xa, ra, False)
    assert (g2[0] - wa[0]).abs().max().item() < 1e-5


def test_data_parallel_replicas(oracle_model, dev):
    """The module survives nn.DataParallel as reference tools/predict.py:147-152 wraps it: replicas (fresh parameter copies
    for every forward) find the packed weights of their device through the original module instead of re-packing, run
    concurrently from threads, and return the reference's gatherable (N,) bpp tensors."""
    from torch.nn.parallel import parallel_apply, replicate
    from tdvc_b200 import synth
    from tdvc_b200.model import VideoCompressor
    m = VideoCompressor().eval()
    m.load_state_dict(oracle_model.state_dict(), strict=True)
    m = m.to(dev)
    ndev = torch.cuda.device_count()
    devices = [0, 1] if ndev >= 2 else [0]
    xa, ra = synth.make_frame_pair(64, 128, seed=51)
    xb, rb = synth.make_frame_pair(64, 64, seed=52)
    with torch.no_grad():
        wa, wb = m(xa.to(dev), ra.to(dev), False), m(xb.to(dev), rb.to(dev), False)
    if ndev >= 2:
        dp = torch.nn.DataParallel(m, device_ids=devices)
        x2, r2 = torch.cat([xa, xa], 0).to(dev), torch.cat([ra, ra], 0).to(dev)
        with torch.no_grad():
            recon, bres, bmv = dp(x2, r2, False)
            recon_b, _, _ = dp(x2, r2, False)
        assert recon.shape == (2, 3, 64, 128) and bres.shape == (2,) and bmv.shape == (2,)
        assert torch.equal(recon[0:1], wa[0]) and torch.equal(recon[1:2].cpu(), wa[0].cpu()) and torch.equal(recon, recon_b)
        assert abs(bres[1].item() - wa[1].item()) < 1e-6 and len(m._packed) == 2
    # replicas of one device running concurrently on different shapes (thread-per-replica, like DataParallel.parallel_apply)
    packs = dict(m._packed)
    reps = replicate(m, [devices[0], devices[0]])
    assert all(getattr(r, "_is_replica", False) for r in reps)
    with torch.no_grad():
        outs = parallel_apply(reps, [(xa.to(dev), ra.to(dev), False), (xb.to(dev), rb.to(dev), False)], devices=[devices[0]] * 2)
    assert all(torch.equal(p, q) for p, q in zip(outs[0], wa)) and all(torch.equal(p, q) for p, q in zip(outs[1], wb))
    assert all(m._packed[k][1] is packs[k][1] for k in packs), "a replica re-packed the weights"


# ------------------------------------------------------------------------------------------------ training-mode forward (SURVEY 8f.1, slice a)
def _train_noise(N, H, W):
    """The six uniform draws of one training forward in the order the oracle makes them (mv: z, y, y for the likelihood; then
    the residual coder), with the layouts compressai uses: EntropyBottleneck draws on the (C, 1, N*h*w) view."""
    out = {}
    for c in ("mv", "res"):
        hz, wz, hy, wy = H // 64, W // 64, H // 16, W // 16
        nz = torch.empty(128, 1, N * hz * wz).uniform_(-0.5, 0.5)
        out[f"{c}.z"] = nz.view(128, N, hz, wz).permute(1, 0, 2, 3).contiguous()
        out[f"{c}.y"] = torch.empty(N, 128, hy, wy).uniform_(-0.5, 0.5)
        out[f"{c}.y_lik"] = torch.empty(N, 128, hy, wy).uniform_(-0.5, 0.5)
    return out


@pytest.mark.parametrize("case", [(1, 64, 128, 71), (2, 128, 128, 72)])
def test_training_mode_forward_vs_oracle(net, oracle_model, dev, case):
    """`net.train()`: noise quantisation with injected draws, FeatureFix at scale 8 (reference pnet.py:220-221), aux losses and
    the 5-tuple return (:80-81) against the oracle in train() mode under the same torch seed (the oracle draws its noise from
    torch's generator in a fixed order; the same draws are reproduced here and handed to the CUDA path)."""
    from tdvc_b200 import synth
    N, H, W, seed = case
    xs, rs = zip(*[synth.make_frame_pair(H, W, seed=seed + i) for i in range(N)])
    x, refs = torch.cat(xs, 0), torch.cat(rs, 0)
    oracle_model.train()
    net.train()
    try:
        torch.manual_seed(1234)
        ot = {}
        with torch.no_grad():
            want = oracle_model(x, refs, False, taps=ot)
        torch.manual_seed(1234)
        noise = {k: v.to(dev) for k, v in _train_noise(N, H, W).items()}
        gt = {}
        got = net._forward_training(x.to(dev), refs.to(dev), taps=gt, noise=noise)
    finally:
        oracle_model.eval()
        net.eval()
    assert len(got) == 5 and got[1].shape == (1,) and got[2].shape == (1,) and got[3].dim() == 0 and got[4].dim() == 0
    for c in ("mv", "res"):
        assert (ot[f"{c}.y_hat"] - gt[f"{c}.y_hat"].cpu()).abs().max().item() < 2e-3    # y + noise: continuous, no rounding
        assert (ot[f"{c}.z_hat"] - gt[f"{c}.z_hat"].cpu()).abs().max().item() < 2e-3
    assert torch.equal(ot["loopfilter.ind"], gt["loopfilter.ind"].cpu())
    assert ot["loopfilter.ind"].shape[1] == ((H // 8 + 3) // 3 + 1) * ((W // 8 + 3) // 3 + 1)      # scale 8 patch grid
    assert (want[0] - got[0].cpu()).abs().max().item() <= 1e-3
    for i in (1, 2):
        assert abs(want[i].item() - got[i].item()) <= 1e-3 * want[i].item()
    for i in (3, 4):
        assert abs(want[i].item() - got[i].item()) <= 1e-5 * max(1.0, abs(want[i].item()))


def test_training_mode_aux_loss_backward_and_own_noise(net, oracle_model, dev):
    """The aux losses back-propagate to `.quantiles` like the reference's (`aux_loss.backward()`, tools/train.py:147-159); the
    device-side Philox noise is uniform in [-0.5, 0.5), reproducible under torch.manual_seed; with gradients enabled the
    outputs carry their graph, under no_grad the fused forward-only path answers (its own noise draws)."""
    from tdvc_b200 import lib as L
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(64, 64, seed=81)
    net.train()
    oracle_model.train()
    try:
        for m in (net, oracle_model):
            for cd in (m.mvCoder, m.resCoder):
                cd.entropy_bottleneck.quantiles.grad = None
        torch.manual_seed(5)
        a = net(x.to(dev), refs.to(dev), False)
        torch.manual_seed(5)
        b = net(x.to(dev), refs.to(dev), False)
        assert all(torch.equal(p.detach(), q.detach()) for p, q in zip(a, b))
        torch.manual_seed(6)
        c = net(x.to(dev), refs.to(dev), False)
        assert not torch.equal(a[0], c[0])
        (a[3] + a[4]).backward()
        want = oracle_model.mvCoder.aux_loss() + oracle_model.resCoder.aux_loss()
        want.backward()
        for cn in ("mvCoder", "resCoder"):
            g = getattr(net, cn).entropy_bottleneck.quantiles.grad.cpu()
            w = getattr(oracle_model, cn).entropy_bottleneck.quantiles.grad
            assert (g - w).abs().max().item() <= 1e-5 * max(1.0, w.abs().max().item())
        assert a[0].requires_grad and a[1].requires_grad          # gradients enabled: the autograd path (tests/test_training_step.py)
        with torch.no_grad():                                      # no gradients wanted: the fused forward-only path
            torch.manual_seed(5)
            d = net(x.to(dev), refs.to(dev), False)
        assert not d[0].requires_grad and len(d) == 5
    finally:
        net.eval()
        oracle_model.eval()
        for m in (net, oracle_model):
            for cd in (m.mvCoder, m.resCoder):
                cd.entropy_bottleneck.quantiles.grad = None
    n = 1 << 20
    buf = torch.empty(n, device=dev)
    L.check(L.load().tdvc_uniform_noise(buf.data_ptr(), n, 12345, 7, torch.cuda.current_stream(dev).cuda_stream), "noise")
    assert buf.min().item() >= -0.5 and buf.max().item() < 0.5
    assert abs(buf.mean().item()) < 2e-3 and abs(buf.var().item() - 1.0 / 12) < 1e-3
    assert abs(torch.corrcoef(torch.stack([buf[:-1], buf[1:]]))[0, 1].item()) < 5e-3


def test_validate_over_a_gop_dataset(net, dev, tmp_path):
    """tdvc_b200.gop.validate = the reference's `validation` (tools/predict.py:35-110) over frames on disk laid out as the
    reference's datasets are (tdvc_b200/data.py): I+P averages, the P-frame part equal to coding the GOPs by hand."""
    import os
    from torchvision.io import write_png
    from tdvc_b200 import data as D
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    net.conv_impl, net.precision = 0, "auto"
    gop, qp = 4, 27
    seqs = {"a_416x240_50": synth.make_gop(176, 208, gop=8, seed=91), "b_416x240_50": synth.make_gop(176, 208, gop=4, seed=92)}
    for seq, fr in seqs.items():
        os.makedirs(tmp_path / "ori_img" / seq)
        os.makedirs(tmp_path / "compress_img_bpg" / seq / str(qp))
        for i in range(fr.shape[0]):
            write_png((fr[i] * 255).round().to(torch.uint8), str(tmp_path / "ori_img" / seq / f"im{i + 1:03d}.png"))
        for g in range(fr.shape[0] // gop):
            ref = ((fr[g * gop] * 255).round() + 2).clamp(0, 255).to(torch.uint8)
            write_png(ref, str(tmp_path / "compress_img_bpg" / seq / str(qp) / f"im{g * gop + 1:03d}_{qp}.png"))
            open(tmp_path / "compress_img_bpg" / seq / str(qp) / f"im{g * gop + 1:03d}_{qp}.txt", "w").write("0.75\n")
    ds = D.GopDataset(str(tmp_path), 2048, gop, testfull=True)
    assert len(ds) == 3
    bpp, mv, rs, psnr, ms, mse = G.validate(ds, net, enable_amp=False)
    tot = torch.zeros(7, device=dev, dtype=torch.float64)
    i_psnr = 0.0
    for g in range(3):
        p_frames, i_frame, _, ps, _, _ = ds[g]
        tot += G.gop_stats(G.code_gop(net, i_frame.unsqueeze(0).to(dev), p_frames.to(dev), with_msssim=True))
        i_psnr += ps
    summ = G.summarise(tot)
    assert summ["frames"] == 9 and abs(mv - summ["bpp_mv"]) < 1e-9 and abs(rs - summ["bpp_res"]) < 1e-9 and abs(mse - summ["mse"]) < 1e-12
    assert abs(bpp - (summ["bpp"] * 9 + 3 * 0.75) / 12) < 1e-9 and abs(psnr - (summ["psnr"] * 9 + i_psnr) / 12) < 1e-9
    assert 0.0 < ms <= 1.0 and math.isfinite(psnr)


def test_batch_of_two_graphs_and_caches(net, dev):
    """N = 2 through the per-variant CUDA graphs and the per-GOP caches (keys are per batch element): a 4-frame chain of a
    2-sequence batch equals the eager, cache-free chain bit for bit, and each sequence equals its own single-sequence chain in
    the symbols-free outputs to fp32 rounding (batched SE / bpp reductions sum in a different order)."""
    from tdvc_b200 import gop as G
    from tdvc_b200 import synth
    net.conv_impl, net.precision = 0, "auto"
    fa, fb = synth.make_gop(64, 128, gop=5, seed=71).to(dev), synth.make_gop(64, 128, gop=5, seed=72).to(dev)
    both = torch.stack([fa, fb], 1)    # (T, 2, 3, H, W)

    def chain(frames, cache, graph, amp=False):
        net.cache_features, net.use_cuda_graph = cache, graph
        refs, out = [frames[0]], []
        for t in range(1, frames.shape[0]):
            with torch.no_grad():
                r = net(frames[t], G.reference_window(refs), amp)
            refs.append(r[0])
            out.append(r)
        return out

    try:
        base = chain(both, False, False)
        fast = chain(both, True, True)
        fast2 = chain(both, True, True)     # second pass: graph replays
        single = chain(fa.unsqueeze(1), True, False)
    finally:
        net.cache_features, net.use_cuda_graph = True, False
    for a, b, c in zip(base, fast, fast2):
        assert all(torch.equal(u, v) and torch.equal(u, w) for u, v, w in zip(a, b, c))
    for a, s in zip(base, single):
        assert (a[0][0:1] - s[0]).abs().max().item() <= 1e-4

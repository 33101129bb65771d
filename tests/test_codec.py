"""The closed-loop P-frame codec: `VideoCompressor.compress` -> version-2 container -> `VideoCompressor.decompress`, and the
GOP driver on top of it (`gop.compress_gop` / `gop.decompress_gop`).

The decoder is a second module loaded from the same state_dict.  Every GPU round trip demands the encoder's reconstruction
with torch.equal.  The closed-loop reference is built here from the oracle's own modules: the oracle's `Coder.compress`
(its autoregressive y_hat) feeds g_s on the encoder side, `Coder.decompress` on the decoder side.  (The closed-loop recon
differs from `forward`'s by design - autoregressive y_hat against round(y) - so nothing here compares the two.)"""
import copy
import math

import numpy as np
import pytest
import torch

from test_coding import _first_mismatch


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers: work on a copy so that the session's oracle keeps its state_dict."""
    return copy.deepcopy(oracle_model)


# ------------------------------------------------------------------------------------ the oracle's closed loop
def oracle_compress(orc, x, refs, taps=None):
    """Closed-loop encoder over the oracle's modules: mvCoder.compress (its ar_code y_hat) -> g_s, mcnet, mcfilter,
    residual, resCoder.compress -> g_s + prediction, loopfilter, clamp.  -> (recon, {"mv" | "res": {"strings", "shape"}})."""
    ref = refs[:, -1]
    in_f, ref_f = orc.extra_fea(x), orc.extra_fea(ref)
    estmv = orc.motion_est(in_f, ref_f, x, ref)
    coded = {}

    def code(nm, coder, v):
        coder.eval()
        coder.update(force=True)
        t = {}
        enc = coder.compress(v, taps=t)
        coded[nm] = {"strings": enc["strings"], "shape": tuple(enc["shape"])}
        if taps is not None:
            taps.update({f"{nm}.ac.{k}": w for k, w in t.items()})
        return t["y_hat"]

    mv_xhat = orc.mvCoder.g_s(code("mv", orc.mvCoder, estmv.float()))
    pred = orc.mcfilter(orc.mcnet(mv_xhat, ref_f), refs)
    rec_f = pred + orc.resCoder.g_s(code("res", orc.resCoder, (in_f - pred).float()))
    return orc.loopfilter(rec_f, refs).clamp(0.0, 1.0), coded


def oracle_decompress(orc, coded, refs):
    """Decode twin of oracle_compress from the strings and the reference frames (Coder.decompress's y_hat -> g_s)."""
    def synth(coder, nm):   # g_s on a contiguous y_hat, as the encoder's: CPU convolutions of a strided view round differently
        return coder.g_s(coder.decompress(coded[nm]["strings"], coded[nm]["shape"])["y_hat"].contiguous())

    ref_f = orc.extra_fea(refs[:, -1])
    pred = orc.mcfilter(orc.mcnet(synth(orc.mvCoder, "mv"), ref_f), refs)
    return orc.loopfilter(pred + synth(orc.resCoder, "res"), refs).clamp(0.0, 1.0)


def _coded(n=2, shape=(1, 2)):
    s = lambda k: [bytes([k + i]) * 12 for i in range(n)]
    return {"mv": {"strings": [s(1), s(2)], "shape": shape, "cluster": 16},
            "res": {"strings": [s(3), s(4)], "shape": shape, "cluster": 8}}


# ------------------------------------------------------------------------------------------------------ CPU
def test_decompress_refuses_before_any_device_work(monkeypatch):
    """Malformed containers, and reference frames that do not match the container's frame (batch, height, width, slices),
    raise RuntimeError before the weights are packed, a plan is built or a string is decoded."""
    from tdvc_b200 import coding
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()

    def touched(*a, **k):
        raise AssertionError("device work on input that must be refused")

    monkeypatch.setattr(VideoCompressor, "_weights", touched)
    monkeypatch.setattr(VideoCompressor, "_plan", touched)
    monkeypatch.setattr(coding, "decode_z_symbols", touched)
    frame = {"size": (64, 128), "N": 2, "precision": "exact"}
    refs = torch.zeros(2, 4, 3, 64, 128)
    missing = _coded()
    del missing["mv"]
    one_string = _coded()
    one_string["mv"]["strings"][0] = one_string["mv"]["strings"][0][:1]
    cases = {"version 1": (coding.pack_frame(_coded()), "version-1"),
             "missing coder": (coding.pack_frame(missing, frame=frame), "no mv coder"),
             "frame size": (coding.pack_frame(_coded(shape=(1, 1)), frame=dict(frame, size=(64, 96))), "multiples of 64"),
             "hyper shape": (coding.pack_frame(_coded(shape=(2, 1)), frame=frame), "hyper-latent shape"),
             "string count": (coding.pack_frame(one_string, frame=frame), "strings"),
             "batch": (coding.pack_frame(_coded(), frame=dict(frame, N=3)), "strings")}
    for what, (blob, msg) in cases.items():
        with pytest.raises(RuntimeError, match=msg):
            net.decompress(blob, refs)
    with pytest.raises(RuntimeError, match="unpack_frame"):
        net.decompress(coding.pack_frame(_coded(), frame=frame)[:-5], refs)
    good = coding.pack_frame(_coded(), frame=frame)
    for bad in (torch.zeros(1, 4, 3, 64, 128), torch.zeros(2, 4, 3, 128, 128), torch.zeros(2, 4, 3, 64, 64),
                torch.zeros(2, 3, 3, 64, 128), torch.zeros(2, 3, 64, 128)):
        with pytest.raises(RuntimeError, match="do not match the container"):
            net.decompress(good, bad)
    with pytest.raises(RuntimeError, match="ref_keys"):
        net.decompress(good, refs, ref_keys=(1, 2, 3))
    # well-formed input on a module that is not on a CUDA device: refused too, still without device work
    with pytest.raises(RuntimeError, match="CUDA"):
        net.decompress(good, refs)


def test_oracle_closed_loop_round_trip(oracle_model):
    """The oracle's closed-loop decoder rebuilds its encoder's reconstruction exactly from the strings alone (64x64), and
    the closed loop's y_hat is the one the strings decode to."""
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(64, 64, seed=3)
    taps = {}
    with torch.no_grad():
        recon, coded = oracle_compress(oracle_model, x, refs, taps)
        got = oracle_decompress(oracle_model, coded, refs)
        mv = oracle_model.mvCoder.decompress(coded["mv"]["strings"], coded["mv"]["shape"])
    assert recon.shape == (1, 3, 64, 64) and 0.0 <= float(recon.min()) and float(recon.max()) <= 1.0
    assert torch.equal(got, recon)
    assert torch.equal(mv["y_hat"], taps["mv.ac.y_hat"])


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
        raise AssertionError(f"{what} differs at {first} ({int(d.numel())} elements, max-abs "
                             f"{(got.float() - want.float()).abs().max().item() if got.shape == want.shape else 'n/a'})")


def _assert_stages_equal(dt, et, what):
    """First stage at which the decoder's taps leave the encoder's, so that a failure names where they diverge."""
    for k in ("mv.x_hat", "prediction1", "prediction", "recon_feat"):
        _assert_equal(dt[k], et[k], f"{what}: {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("cache", [True, False])
@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2), ((1024, 1920), 0, 1)])
def test_round_trip_is_exact(oracle_model, hw, seed, n, amp, cache):
    """decompress on a module that has never coded anything returns compress's recon bit for bit; the container records
    the frame and the precision mode; last_coded is what forward(is_compress=True) leaves (the container is its packing).
    With caches on, a second decode (now hitting the caches the first one filled) is exact too."""
    from tdvc_b200 import coding
    enc, dec = _net(oracle_model, cache), _net(oracle_model, cache)
    x, refs = _pair(n, hw, seed)
    et, dt = {}, {}
    recon, data = enc.compress(x, refs, amp, taps=et)
    assert recon.shape == (n, 3, *hw) and recon.dtype == torch.float32
    box = coding.unpack_frame(data)
    assert box["frame"] == {"size": hw, "N": n, "precision": "mixed" if amp else "exact"}
    for nm in ("mv", "res"):
        lc = enc.last_coded[nm]
        assert set(lc) == {"strings", "shape", "cluster", "ac_bpp"}
        assert lc["ac_bpp"] == sum(len(s[0]) for s in lc["strings"]) * 8.0 / (n * hw[0] * hw[1])
    assert coding.pack_frame(enc.last_coded, frame=box["frame"]) == data
    got = dec.decompress(data, refs, taps=dt)
    torch.cuda.synchronize()
    _assert_stages_equal(dt, et, f"{hw} N={n} amp={amp} cache={cache}")
    _assert_equal(got, recon, f"{hw} N={n} amp={amp} cache={cache} recon")
    if cache:
        hits = dec._plan(n, *hw, torch.device(DEV)).cache_hits
        _assert_equal(dec.decompress(data, refs), recon, "second decode")
        assert dec._plan(n, *hw, torch.device(DEV)).cache_hits == hits + 4


@pytest.mark.gpu
@pytest.mark.parametrize("enc_cache,dec_cache", [(True, True), (False, False), (True, False), (False, True)])
def test_gop_round_trip(oracle_model, enc_cache, dec_cache):
    """A 6-frame GOP at 64x128 (every warm-up window of RefBuffer, then the steady state) in closed loop: decompress_gop
    equals compress_gop frame by frame, whether the caches hit on one end, on both or on neither."""
    from tdvc_b200 import gop, synth
    frames = synth.make_gop(64, 128, gop=7, seed=5).to(DEV)
    enc, dec = _net(oracle_model, enc_cache), _net(oracle_model, dec_cache)
    containers, recons = gop.compress_gop(enc, frames[0:1], frames[1:])
    assert len(containers) == len(recons) == 6
    got = gop.decompress_gop(dec, frames[0:1], containers, (64, 128))
    for i, (a, b) in enumerate(zip(got, recons)):
        _assert_equal(a, b, f"GOP frame {i}")


@pytest.mark.gpu
def test_gop_round_trip_full_size(oracle_model):
    """A 3-frame GOP at 1920x1024 (a 1080p frame padded as code_gop pads it is 1920x1088; this one needs no padding)."""
    from tdvc_b200 import gop, synth
    frames = synth.make_gop(1024, 1920, gop=4, seed=1).to(DEV)
    enc, dec = _net(oracle_model), _net(oracle_model)
    containers, recons = gop.compress_gop(enc, frames[0:1], frames[1:])
    got = gop.decompress_gop(dec, frames[0:1], containers, (1024, 1920))
    for i, (a, b) in enumerate(zip(got, recons)):
        _assert_equal(a, b, f"1920x1024 GOP frame {i}")


def _tie(v):
    return abs(abs(v - np.floor(v)) - 0.5) < 1e-3


def _coder_agrees(gt, ot, nm, i, coder):
    """Compares one coder of image i with the oracle's closed loop as test_is_compress_vs_oracle does: identical symbols
    and indexes up to the first difference, which must be a rounding tie of y - mu (or an index one apart, a scale
    within rounding of a table entry); z symbols may differ only at ties of z - median.  Returns True when nothing differs."""
    zs, ozs = gt[f"{nm}.ac.z_symbols"][i].cpu().numpy(), ot[f"{nm}.ac.z_symbols"][i].numpy()
    if not np.array_equal(zs, ozs):
        z = ot[f"{nm}.ac.z"][i].numpy() - coder.entropy_bottleneck.quantiles[:, 0, 1].detach().reshape(-1, 1, 1).numpy()
        assert all(_tie(v) for v in z[zs != ozs]), (nm, "z symbols differ away from a rounding tie")
        return False
    sy, osy = gt[f"{nm}.ac.y_symbols"][i].cpu().numpy(), ot[f"{nm}.ac.y_symbols"][i].numpy()
    ix, oix = gt[f"{nm}.ac.y_indexes"][i].cpu().numpy(), ot[f"{nm}.ac.y_indexes"][i].numpy()
    fs, fi = _first_mismatch(sy, osy), _first_mismatch(ix, oix)
    if fs is None and fi is None:
        return True
    if fs is not None and (fi is None or fs[:2] <= fi[:2]):
        r = ot[f"{nm}.ac.y"][i].permute(1, 2, 0).numpy()[fs] - (ot[f"{nm}.ac.y_hat"][i].permute(1, 2, 0).numpy()[fs] - osy[fs])
        assert _tie(r), ("first differing symbol is not at a rounding tie", nm, fs, r)
    else:
        assert abs(int(ix[fi]) - int(oix[fi])) == 1, (nm, fi)
    return False


@pytest.mark.gpu
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2)])
def test_closed_loop_vs_oracle(oracle_model, hw, seed, n):
    """compress against the oracle's closed loop.  The motion coder must agree up to its first rounding tie; where it has
    none, the residual coder (whose input follows from the motion coder's y_hat) must too.  Where neither coder of an
    image has a tie, both coders' strings are byte-identical and recon is within max-abs 1e-3 and PSNR +-0.01 dB."""
    from tdvc_b200 import synth
    pairs = [synth.make_frame_pair(*hw, seed=seed + 10 * i) for i in range(n)]
    x, refs = torch.cat([p[0] for p in pairs]), torch.cat([p[1] for p in pairs])
    ot, gt = {}, {}
    with torch.no_grad():
        o_recon, o_coded = oracle_compress(oracle_model, x, refs, ot)
    net = _net(oracle_model)
    recon, _ = net.compress(x.to(DEV), refs.to(DEV), False, taps=gt)
    recon = recon.cpu()
    clean_images = 0
    for i in range(n):
        if not _coder_agrees(gt, ot, "mv", i, oracle_model.mvCoder):
            continue
        if not _coder_agrees(gt, ot, "res", i, oracle_model.resCoder):
            continue
        clean_images += 1
        for nm in ("mv", "res"):
            for k in (0, 1):
                assert net.last_coded[nm]["strings"][k][i] == o_coded[nm]["strings"][k][i], (nm, k, i)
        err = (recon[i] - o_recon[i]).abs().max().item()
        assert err <= 1e-3, err
        psnr = lambda r: 10 * math.log10(1.0 / (r - x[i]).pow(2).mean().item())
        assert abs(psnr(recon[i]) - psnr(o_recon[i])) <= 0.01
    print(f"closed loop vs oracle {hw} N={n}: {clean_images}/{n} images without a tie")


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_codec_between_forwards_changes_nothing(oracle_model, graph):
    """compress and decompress of another frame (same references) on the same module and plan between two forwards leave
    the next forward's recon, bpp, strings and launch count as they are without them (eager, and with CUDA graphs: the
    last forward replays the graph the one before it captured)."""
    n, hw = 2, (64, 128)
    x, refs = _pair(n, hw, 7)
    x2, _ = _pair(n, hw, 8)
    runs = []
    for interleave in (False, True):
        net = _net(oracle_model)
        net.use_cuda_graph = graph
        with torch.no_grad():
            net(x, refs, False, is_compress=True)
            net(x, refs, False, is_compress=True)
            if interleave:
                c_recon, data = net.compress(x2, refs, True)
                _assert_equal(net.decompress(data, refs), c_recon, "interleaved round trip")
            recon, bpp_res, bpp_mv = net(x, refs, False, is_compress=True)
        torch.cuda.synchronize()
        runs.append((recon.clone(), bpp_res.clone(), bpp_mv.clone(), net.last_coded, net.last_launches))
    (r0, br0, bm0, c0, l0), (r1, br1, bm1, c1, l1) = runs
    _assert_equal(r1, r0, "recon")
    _assert_equal(br1, br0, "bpp_res")
    _assert_equal(bm1, bm0, "bpp_mv")
    assert l1 == l0
    for nm in ("mv", "res"):
        assert c1[nm]["strings"] == c0[nm]["strings"] and c1[nm]["cluster"] == c0[nm]["cluster"]
        assert c1[nm]["ac_bpp"] == c0[nm]["ac_bpp"]


@pytest.mark.gpu
def test_damaged_y_string(oracle_model):
    """A truncated y string makes decompress raise naming the coder, the image and the latent position, without faulting
    the device; the next decompress of the good container is still exact."""
    from tdvc_b200 import coding
    n, hw = 2, (64, 64)
    enc, dec = _net(oracle_model), _net(oracle_model)
    x, refs = _pair(n, hw, 4)
    recon, data = enc.compress(x, refs)
    box = coding.unpack_frame(data)
    frame = box.pop("frame")
    s = box["res"]["strings"][0][1]
    box["res"]["strings"][0][1] = s[:len(s) // 8 * 4]
    with pytest.raises(RuntimeError, match=r"rs y string of image 1 .*position \(h=\d+, w=\d+, c=\d+\)"):
        dec.decompress(coding.pack_frame(box, frame=frame), refs)
    torch.cuda.synchronize()
    _assert_equal(dec.decompress(data, refs), recon, "after a damaged string")

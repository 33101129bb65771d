"""Device decoding of the y latent (`tdvc_ar_decode`, csrc/ar_decode.cu): the inverse of the wavefront encoder
`tdvc_ar_code`, compressai `_decompress_ar` + the `ans` decoder on the device.

Decoding is lossless only if the decoder predicts every mean and scale index bit for bit as the encoder did, and the
encoder's fp32 summation order depends on its cluster size: every GPU test decodes strings coded with 8 and with 16 CTAs
per image and demands identical symbols, indexes and y_hat."""
import os
import subprocess

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers: work on a copy so that the session's oracle keeps its state_dict."""
    import copy
    return copy.deepcopy(oracle_model)


# ------------------------------------------------------------------------------------------------------ CPU
def test_decode_refuses_malformed_strings_on_the_host():
    """Strings that cannot be rANS output (not whole 32-bit words, shorter than the 8-byte final state), a string count that
    does not match the batch (N strings, or N * h row strings) and an unknown encoder cluster size are refused before
    anything reaches the device."""
    from tdvc_b200 import coding
    from tdvc_b200.model import Act
    t = torch.zeros(2, 4, 8, 256)
    params = Act(t, 0, 2, 4, 8, 256, 256)
    good = b"\0" * 16
    for strings, cluster in (([good, good[:6]], 16), ([good, good[:4]], 8), ([good, good + b"\0\0"], 16), ([good], 16),
                             ([good, good], 4)):
        with pytest.raises(RuntimeError):
            coding.decode_latents({}, "mv", None, strings, params, cluster)
    # row streams: N * h = 8 strings
    for strings, cluster, msg in (([good] * 7 + [good[:6]], 16, "mv y row 3 of image 1 has 6 bytes"),
                                  ([good] * 2, 16, "2 mv y row strings for 2 images of 4 rows"),
                                  ([good] * 8, 4, "cluster size 4")):
        with pytest.raises(RuntimeError, match=msg):
            coding.decode_latents({}, "mv", None, strings, params, cluster, rows=True)


def _coded():
    return {"mv": {"strings": [[b"\x01" * 12, b"\x02" * 8], [b"zz", b"y"]], "shape": (1, 2), "ac_bpp": 0.1, "cluster": 16},
            "res": {"strings": [[b"\x03" * 16, b"\x04" * 20], [b"q", b"rr"]], "shape": (1, 2), "ac_bpp": 0.2, "cluster": 8}}


def test_container_v2_round_trips_its_fields_and_v1_is_unchanged():
    """Version 2 records what a decoder needs to be exact (frame size, batch, precision mode, each coder's cluster size);
    without `frame` pack_frame writes the version-1 bytes it always wrote, and they unpack as before."""
    from tdvc_b200 import coding
    coded = _coded()
    v1 = coding.pack_frame(coded)
    plain = {k: {"strings": v["strings"], "shape": v["shape"]} for k, v in coded.items()}
    assert v1 == coding.pack_frame(plain) and v1[:4] == b"TDVC"
    assert coding.unpack_frame(v1) == plain
    for prec in ("exact", "mixed"):
        frame = {"size": (1024, 1920), "N": 2, "precision": prec}
        v2 = coding.pack_frame(coded, frame=frame)
        assert v2[:4] == b"TDV2" and len(v2) == len(v1) + 10 + 2
        back = coding.unpack_frame(v2)
        assert back.pop("frame") == frame
        assert back == {k: dict(plain[k], cluster=coded[k]["cluster"]) for k in coded}
    with pytest.raises(RuntimeError):
        coding.pack_frame(plain, frame={"size": (64, 64), "N": 1, "precision": "exact"})   # no cluster size recorded
    with pytest.raises(RuntimeError):
        coding.pack_frame(coded, frame={"size": (64, 64), "N": 1, "precision": "fp16"})


def test_truncated_or_garbled_container_raises():
    from tdvc_b200 import coding
    for frame in (None, {"size": (64, 64), "N": 2, "precision": "exact"}):
        blob = coding.pack_frame(_coded(), frame=frame)
        for cut in range(4, len(blob)):
            with pytest.raises(RuntimeError):
                coding.unpack_frame(blob[:cut])
        with pytest.raises(RuntimeError):
            coding.unpack_frame(blob + b"\0")
        with pytest.raises(RuntimeError):
            coding.unpack_frame(b"TDVX" + blob[4:])
    blob = bytearray(coding.pack_frame(_coded(), frame={"size": (64, 64), "N": 2, "precision": "exact"}))
    bad_prec = bytearray(blob)
    bad_prec[13] = 7
    bad_cluster = bytearray(blob)
    bad_cluster[19] = 12
    bad_len = bytearray(blob)
    bad_len[33] = 0xFF
    for b in (bad_prec, bad_cluster, bad_len):
        with pytest.raises(RuntimeError):
            coding.unpack_frame(bytes(b))


def test_decoder_compiles_without_spills():
    """The decode kernel keeps its state in registers (ptxas -v: no local-memory spills)."""
    from tdvc_b200 import build
    for src, kernel in (("ar_decode.cu", "ar_decode_kernel"),):
        r = subprocess.run([build.NVCC] + build.FLAGS + ["-c", os.path.join(build.CSRC, src), "-o", os.devnull],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        lines = r.stdout + r.stderr
        i = lines.index(kernel)
        props = lines[i:].split("ptxas info    : Used")[0]
        assert "0 bytes spill stores, 0 bytes spill loads" in props, props


# ------------------------------------------------------------------------------------------------------ GPU
def _net(oracle_model, dev):
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()
    net.load_state_dict(oracle_model.state_dict(), strict=True)
    return net.to(dev)


def _frame(net, n, hw, seed, dev):
    """One coded P-frame: the forward pass leaves y and the hyper-decoder output of both coders in the plan."""
    from tdvc_b200 import synth
    pairs = [synth.make_frame_pair(*hw, seed=seed + 10 * i) for i in range(n)]
    x, refs = torch.cat([p[0] for p in pairs]).to(dev), torch.cat([p[1] for p in pairs]).to(dev)
    with torch.no_grad():
        net(x, refs, False, is_compress=True)
    W = net._weights(dev)
    return W, net._plan(n, hw[0], hw[1], dev)


def _round_trip(W, plan, cn, cluster):
    from tdvc_b200 import coding
    N, hy, wy = plan.N, plan.H // 16, plan.W // 16
    tabs = W["_tables"][cn]
    enc = coding.code_latents(plan, W, cn, tabs, cluster=cluster, keep=True)
    params = plan.buf(f"{cn}.params", N, hy, wy, 256)
    dec = coding.decode_latents(W, cn, tabs, enc["strings"][0], params, cluster)
    return enc, dec, params


def _assert_lossless(enc, dec, what):
    for k in ("y_symbols", "y_indexes", "y_hat"):
        if not torch.equal(enc[k], dec[k]):
            d = (enc[k] != dec[k]).reshape(-1).nonzero()
            first = np.unravel_index(int(d[0]), tuple(enc[k].shape))
            raise AssertionError(f"{what}: {k} differs at {first} ({int(d.numel())} elements)")


@pytest.mark.gpu
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2)])
def test_ar_decode_is_lossless(oracle_model, hw, seed, n):
    dev = torch.device("cuda:0")
    net = _net(oracle_model, dev)
    W, plan = _frame(net, n, hw, seed, dev)
    for cn in ("mv", "rs"):
        for cluster in (8, 16):
            enc, dec, _ = _round_trip(W, plan, cn, cluster)
            _assert_lossless(enc, dec, f"{cn} {hw} N={n} cluster {cluster}")


@pytest.mark.gpu
def test_ar_decode_is_lossless_full_size(oracle_model):
    """1920x1024: a 64x120 latent, 7,680 dependent decode steps per coder, wavefronts of 1..40 positions, each coded as
    one chunk (waves of two and three chunks: tests/test_ar_edges.py)."""
    dev = torch.device("cuda:0")
    net = _net(oracle_model, dev)
    W, plan = _frame(net, 1, (1024, 1920), 0, dev)
    for cn in ("mv", "rs"):
        for cluster in (8, 16):
            enc, dec, _ = _round_trip(W, plan, cn, cluster)
            assert enc["y_symbols"].shape == (1, 64, 120, 128)
            _assert_lossless(enc, dec, f"{cn} 1920x1024 cluster {cluster}")


@pytest.mark.gpu
def test_ar_decode_errors_and_determinism(oracle_model):
    """A truncated string raises RuntimeError naming the coder, image and position where the stream ends; the kernel
    treats it as a normal run (no fault), and the next decode of good strings is exact.  A garbled string never faults.
    Decoding the same bytes again, also after coding unrelated frames on the same plan, gives identical results."""
    from tdvc_b200 import coding, synth
    dev = torch.device("cuda:0")
    net = _net(oracle_model, dev)
    W, plan = _frame(net, 2, (64, 64), 4, dev)
    tabs = W["_tables"]["rs"]
    enc, dec, params = _round_trip(W, plan, "rs", 16)
    good = enc["strings"][0]
    keep = {k: v.clone() for k, v in dec.items()}
    cut = len(good[1]) // 8 * 4
    with pytest.raises(RuntimeError, match=r"rs y string of image 1 .*position \(h=\d+, w=\d+, c=\d+\)"):
        coding.decode_latents(W, "rs", tabs, [good[0], good[1][:cut]], params, 16)
    torch.cuda.synchronize()
    garbled = bytearray(good[0])
    for i in range(8, len(garbled), 7):
        garbled[i] ^= 0x5A
    try:
        coding.decode_latents(W, "rs", tabs, [bytes(garbled), good[1]], params, 16)
    except RuntimeError as e:
        assert "image 0" in str(e)
    torch.cuda.synchronize()
    again = coding.decode_latents(W, "rs", tabs, good, params, 16)
    _assert_lossless(keep, again, "after errors")
    # unrelated frames through the same plan, then the same bytes with the same params
    saved = params.t.clone()
    x, refs = synth.make_frame_pair(64, 64, seed=99)
    with torch.no_grad():
        net(torch.cat([x, x]).to(dev), torch.cat([refs, refs]).to(dev), False, is_compress=True)
    params.t.copy_(saved)
    _assert_lossless(keep, coding.decode_latents(W, "rs", tabs, good, params, 16), "after other frames")


@pytest.mark.gpu
def test_recorded_cluster_decodes_the_default_strings(oracle_model):
    """forward(is_compress=True) codes with the automatic cluster size; the size actually launched is recorded in
    net.last_coded and in a version-2 container, and decoding the unpacked strings with it reproduces the encoder's
    symbols, indexes and y_hat exactly."""
    from tdvc_b200 import coding, synth
    dev = torch.device("cuda:0")
    net = _net(oracle_model, dev)
    x, refs = synth.make_frame_pair(128, 192, seed=2)
    gt = {}
    with torch.no_grad():
        net(x.to(dev), refs.to(dev), False, is_compress=True, taps=gt)
    W = net._weights(dev)
    plan = net._plan(1, 128, 192, dev)
    blob = coding.pack_frame(net.last_coded, frame={"size": (128, 192), "N": 1, "precision": "exact"})
    back = coding.unpack_frame(blob)
    assert back["frame"] == {"size": (128, 192), "N": 1, "precision": "exact"}
    for nm, cn in (("mv", "mv"), ("res", "rs")):
        assert back[nm]["cluster"] == net.last_coded[nm]["cluster"] in (8, 16)
        params = plan.buf(f"{cn}.params", 1, 8, 12, 256)
        dec = coding.decode_latents(W, cn, W["_tables"][cn], back[nm]["strings"][0], params, back[nm]["cluster"])
        enc = {k: gt[f"{nm}.ac.{k}"] for k in ("y_symbols", "y_indexes", "y_hat")}
        _assert_lossless(enc, dec, f"{nm} recorded cluster {back[nm]['cluster']}")
    # tables that are not valid CDF rows are reported as such, not as a broken stream
    tabs = W["_tables"]["rs"]
    bad = coding.CoderTables.__new__(coding.CoderTables)
    bad.gc = coding.Tables(tabs.gc.cdf, tabs.gc.length + tabs.gc.cdf.shape[1], tabs.gc.offset)
    bad.scale_table = tabs.scale_table
    with pytest.raises(RuntimeError, match="tables"):
        coding.decode_latents(W, "rs", bad, back["res"]["strings"][0], plan.buf("rs.params", 1, 8, 12, 256),
                              back["res"]["cluster"])

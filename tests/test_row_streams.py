"""Row streams (container version 3): one rANS string per latent row, coded on the host by `coding.finish_coding(...,
rows=True)` and decoded on the device by `tdvc_ar_decode_rows` - the encoder's wavefront kernel `ar_code_kernel` with a
decoding epilogue, so the rows of a wavefront decode in parallel.

The decoder predicts the encoder's means and scale indexes only with the encoder's cluster size; every kernel test decodes
strings coded with 8 and with 16 CTAs per image and demands identical symbols, indexes and y_hat."""
import copy
import os
import subprocess

import numpy as np
import pytest
import torch

from test_ar_edges import _act, _assert_same, _coder, _latents, _longest_wave, _models, _encode
from test_codec import _assert_equal, _net, _pair

DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers and a test edits weights: work on a copy."""
    return copy.deepcopy(oracle_model)


def _coded(n=2, hy=2, shape=(1, 2)):
    s = lambda k, m: [bytes([k + i]) * 12 for i in range(m)]
    return {"mv": {"strings": [s(1, n * hy), s(2, n)], "shape": shape, "cluster": 16, "y_streams": "rows"},
            "res": {"strings": [s(3, n * hy), s(4, n)], "shape": shape, "cluster": 8, "y_streams": "rows"}}


def _rows_frame(H=32, Wd=64, N=2):
    return {"size": (H, Wd), "N": N, "precision": "exact", "y_streams": "rows"}


# ------------------------------------------------------------------------------------------------------ CPU
def test_container_v3_round_trip_and_v1_v2_unchanged():
    """Version 3 is the layout of version 2 under magic TDV3; it unpacks to version 2's dict plus frame["y_streams"].
    Without y_streams, pack_frame writes the same version-1 and version-2 bytes as before, and they unpack to the same keys."""
    from tdvc_b200 import coding
    coded = _coded()
    plain = {k: {kk: v for kk, v in c.items() if kk != "y_streams"} for k, c in coded.items()}
    f2 = {"size": (32, 64), "N": 2, "precision": "mixed"}
    v2 = coding.pack_frame(plain, frame=f2)
    v3 = coding.pack_frame(coded, frame=dict(f2, y_streams="rows"))
    assert v3[:4] == b"TDV3" and v2[:4] == b"TDV2" and v3[4:] == v2[4:]
    back = coding.unpack_frame(v3)
    assert back.pop("frame") == dict(f2, y_streams="rows")
    assert back == {k: {"strings": c["strings"], "shape": c["shape"], "cluster": c["cluster"]} for k, c in coded.items()}
    b2 = coding.unpack_frame(v2)
    assert "y_streams" not in b2["frame"] and set(b2) == {"mv", "res", "frame"}
    v1 = coding.pack_frame({k: {"strings": c["strings"], "shape": c["shape"]} for k, c in coded.items()})
    assert v1[:4] == b"TDVC" and "frame" not in coding.unpack_frame(v1)
    with pytest.raises(RuntimeError):
        coding.pack_frame(coded, frame=dict(f2, y_streams="columns"))


def test_truncated_or_garbled_v3_container_raises():
    from tdvc_b200 import coding
    blob = coding.pack_frame(_coded(), frame=_rows_frame())
    for cut in range(4, len(blob)):
        with pytest.raises(RuntimeError):
            coding.unpack_frame(blob[:cut])
    with pytest.raises(RuntimeError):
        coding.unpack_frame(blob + b"\0")
    bad_cluster = bytearray(blob)
    bad_cluster[19] = 12
    with pytest.raises(RuntimeError):
        coding.unpack_frame(bytes(bad_cluster))


def test_decompress_refuses_malformed_v3_before_any_device_work(monkeypatch):
    """A version-3 container with a y row count other than N * H / 16, or row strings that are not whole 32-bit words (or
    shorter than two), is refused before the weights are packed, a plan is built or a string is decoded."""
    from tdvc_b200 import coding
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()

    def touched(*a, **k):
        raise AssertionError("device work on input that must be refused")

    monkeypatch.setattr(VideoCompressor, "_weights", touched)
    monkeypatch.setattr(VideoCompressor, "_plan", touched)
    monkeypatch.setattr(coding, "decode_z_symbols", touched)
    frame = {"size": (64, 128), "N": 2, "precision": "exact", "y_streams": "rows"}
    refs = torch.zeros(2, 4, 3, 64, 128)
    few = _coded(n=2, hy=4)
    few["mv"]["strings"][0] = few["mv"]["strings"][0][:-1]
    v2_count = _coded(n=2, hy=1)          # N strings: a version-2 y list in a version-3 container
    ragged = _coded(n=2, hy=4)
    ragged["res"]["strings"][0][5] = b"\0" * 10
    short = _coded(n=2, hy=4)
    short["mv"]["strings"][0][7] = b"\0" * 4
    for coded, msg in ((few, "strings"), (v2_count, "strings"), (ragged, "res y row 1 of image 1 has 10 bytes"),
                       (short, "mv y row 3 of image 1 has 4 bytes")):
        with pytest.raises(RuntimeError, match=msg):
            net.decompress(coding.pack_frame(coded, frame=frame), refs)
        with pytest.raises(RuntimeError, match=msg):
            net.decompress_latents(coding.pack_frame(coded, frame=frame))
    with pytest.raises(RuntimeError, match="CUDA"):   # well formed: refused only for want of a CUDA module
        net.decompress(coding.pack_frame(_coded(n=2, hy=4), frame=frame), refs)


def _random_rows(rng, tabs, n, h, w):
    """Symbols and table indexes of an (n, h, w, 128) latent: mostly in range, one in 20 an escape of 1 to 8 digits."""
    idx = rng.integers(0, tabs.length.size, size=(n, h, w, 128)).astype(np.int32)
    off, mv = tabs.offset[idx].astype(np.int64), (tabs.length[idx] - 2).astype(np.int64)
    sym = off + (rng.integers(0, 1 << 30, size=idx.shape) % np.maximum(mv, 1))
    esc = rng.random(idx.shape) < 0.05
    mag = 2 ** rng.integers(0, 31, size=idx.shape)
    sym = np.where(esc, np.where(rng.random(idx.shape) < 0.5, off + mv + mag - 1, off - mag), sym)
    return np.clip(sym, -2 ** 31, 2 ** 31 - 1).astype(np.int32), idx


def _host_decode_row(data, indexes, tabs):
    """rANS decode of one row string -> (symbols, final state x, words consumed, words in the string)."""
    w = np.frombuffer(data, dtype="<u4").astype(np.uint64)
    x, pos = int(w[0]) | (int(w[1]) << 32), 2
    L_, mask = 1 << 31, (1 << 16) - 1

    def renorm():
        nonlocal x, pos
        if x < L_:
            x = (x << 32) | int(w[pos])
            pos += 1

    def bits():
        nonlocal x
        v = x & 15
        x >>= 4
        renorm()
        return v

    out = []
    for ci in indexes:
        cdf, ln, off = tabs.cdf[ci], int(tabs.length[ci]), int(tabs.offset[ci])
        cum = x & mask
        s = int(np.searchsorted(cdf[:ln], cum, side="right")) - 1
        x = int(cdf[s + 1] - cdf[s]) * (x >> 16) + cum - int(cdf[s])
        renorm()
        if s == ln - 2:
            nb = v = bits()
            while v == 15:
                v = bits()
                nb += v
            raw = sum(bits() << (4 * j) for j in range(nb))
            val = -(raw >> 1) - 1 if raw & 1 else (raw >> 1) + s
        else:
            val = s
        out.append(val + off)
    return np.array(out, np.int64), x, pos, w.size


def test_row_streams_match_the_oracle_coder_and_end_where_they_started():
    """Every row string of finish_coding(rows=True) is byte for byte oracle/rans.py's encode_with_indexes of that row's
    symbols; the rows concatenate to the one-string-per-image symbol sequence; and decoding a row restores its symbols
    and ends in the encoder's initial state (x = 2^31) with every word consumed - the end-of-row rule of version 3."""
    from oracle import rans
    from tdvc_b200 import coding
    tabs = coding.gc_tables()
    rng = np.random.default_rng(3)
    n, h, w = 2, 3, 4
    sym, idx = _random_rows(rng, tabs, n, h, w)
    zs, zi = np.zeros((n, 128, 1, 1), np.int32), np.zeros((n, 128, 1, 1), np.int32)

    class _Done:
        def synchronize(self):
            pass

    handle = {"done": _Done(), "host": [torch.from_numpy(a) for a in (sym, idx, zs, zi)],
              "tables": type("T", (), {"gc": tabs, "eb": coding.gc_tables()})(), "N": n, "shape": (1, 1), "cluster": 16}
    enc = coding.finish_coding(handle, rows=True)
    assert enc["y_streams"] == "rows" and len(enc["strings"][0]) == n * h
    cdfs = [r.tolist() for r in tabs.cdf]
    lens, offs = tabs.length.tolist(), tabs.offset.tolist()
    digits = 0
    for i in range(n):
        for r in range(h):
            s_, x_ = sym[i, r].reshape(-1), idx[i, r].reshape(-1)
            data = enc["strings"][0][i * h + r]
            assert data == rans.encode_with_indexes(s_.tolist(), x_.tolist(), cdfs, lens, offs), (i, r)
            got, x, pos, nw = _host_decode_row(data, x_, tabs)
            assert np.array_equal(got, s_), (i, r)
            assert x == 1 << 31 and pos == nw, (i, r, x, pos, nw)
            assert np.array_equal(coding.rans_decode(data, x_, tabs), s_)
        v = sym[i].astype(np.int64) - tabs.offset[idx[i]]
        mv = tabs.length[idx[i]] - 2
        raw = np.where(v < 0, -2 * v - 1, np.where(v >= mv, 2 * (v - mv), 0))
        digits = max(digits, int(np.ceil(np.log2(raw.max() + 1) / 4)))
    assert digits == 8


def test_row_decoder_takes_the_decode_params_and_compiles_without_spills():
    """The entry points are in the header and bound in lib.py; the row decoder takes the raster decoder's struct, which
    starts with the chain (its layout: tests/test_host.py); ptxas -v of the decode instantiation of ar_code_kernel
    reports its register use."""
    import ctypes
    from tdvc_b200 import build
    from tdvc_b200 import lib as L
    hdr = open(os.path.join(build.ROOT, "include", "tdvc_b200.h")).read()
    for name in ("tdvc_ar_decode_rows_workspace_bytes", "tdvc_ar_decode_rows"):
        assert name + "(" in hdr and name in L.SIGNATURES
    assert "tdvc_ar_decode_rows(const TdvcArDecodeParams* p," in hdr
    assert L.SIGNATURES["tdvc_ar_decode_rows"][0] is ctypes.POINTER(L.ArDecodeParams)
    assert L.ArDecodeParams._fields_[0] == ("chain", L.ArChain)
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-c", os.path.join(build.CSRC, "coding.cu"), "-o", os.devnull],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout + r.stderr
    props = {}
    for dev in ("ArRowDev", "ArDev"):
        i = lines.index(f"Function properties for _ZN4tdvc14ar_code_kernelINS_{len(dev)}{dev}EEEvT_")
        props[dev] = lines[i:].split("ptxas info    : Used")[0]
    spill = lambda p: int(p.split(" bytes spill stores")[0].split()[-1])
    # the shared wavefront loop holds ~60 values across the stages at 128 registers; the decoder may spill no more than
    # the encoder does
    assert spill(props["ArRowDev"]) <= spill(props["ArDev"]), props


# ------------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def real(oracle_model):
    return _models(oracle_model)


@pytest.fixture(scope="module")
def latent_stats(real):
    from tdvc_b200 import synth
    _, net = real
    x, refs = synth.make_frame_pair(128, 192, seed=2)
    with torch.no_grad():
        net(x.to(DEV), refs.to(DEV), False)
    plan = net._plan(1, 128, 192, DEV)
    out = {}
    for cn in ("mv", "rs"):
        for nm, c in (("y", 128), ("params", 256)):
            t = plan.buf(f"{cn}.{nm}", 1, 8, 12, c).t[..., :c].reshape(-1, c).cpu()
            out[cn, nm] = (t.mean(0), t.std(0))
    return out


def _row_strings(tabs, enc):
    from tdvc_b200 import coding
    sy, ix = enc["y_symbols"].cpu().numpy(), enc["y_indexes"].cpu().numpy()
    return [coding.rans_encode(sy[i, r], ix[i, r], tabs.gc) for i in range(sy.shape[0]) for r in range(sy.shape[1])]


def _rows_lossless(W, cn, tabs, enc, params, cluster, what):
    from tdvc_b200 import coding
    rows = _row_strings(tabs, enc)
    dec = coding.decode_latents(W, cn, tabs, rows, params, cluster, rows=True)
    _assert_same(enc, dec, f"{what}: row streams decoded with cluster {cluster}")
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,lds", [(1, 1, 1, None), (1, 1, 9, None), (1, 9, 1, None), (1, 2, 2, None),
                                       (3, 3, 5, None), (1, 2, 130, (132, 260)), (1, 44, 128, None),
                                       (1, 4, 8, None), (1, 8, 12, None), (2, 4, 4, None), (1, 64, 120, None),
                                       (1, 100, 160, None)])
def test_row_decoder_equals_the_encoder(real, latent_stats, n, h, w, lds):
    """tdvc_ar_decode_rows returns tdvc_ar_code's symbols, indexes and y_hat bit for bit for encoder clusters of 8 and 16:
    the test_ar_edges shapes (one position, one row, one column, W <= 2, a batch of 3, strided rows, waves of 40 + 3), the
    latents of 64x128, 128x192, 64x64 (N = 2) and 1920x1024 frames, and a 100x160 latent (2560x1600, waves of 54)."""
    orc, net = real
    y_ld, params_ld = lds or (128, 256)
    for cn in ("mv", "rs"):
        W, tabs, _ = _coder(orc, net, cn)
        y, params = _latents(latent_stats, cn, n, h, w, seed=5 * h + w, y_ld=y_ld, params_ld=params_ld)
        for cl in (8, 16):
            _rows_lossless(W, cn, tabs, _encode(W, cn, tabs, y, params, cl), params, cl, f"{cn} {n}x{h}x{w}")
    if (h, w) == (100, 160):
        assert _longest_wave(h, w) == 54


@pytest.mark.gpu
def test_row_decoder_every_table_bin_and_escape(oracle_model, latent_stats):
    """The context-free chain of test_ar_edges: scales on, and one ulp either side of, every scale-table entry; each
    channel codes every in-range bin of its row and escapes of 1 to 8 digits.  Row streams decode bit for bit."""
    from tdvc_b200 import coding
    T = coding.scale_table().numpy()
    up, down = np.nextafter(T, np.float32(np.inf)), np.nextafter(T, np.float32(-np.inf))
    for rnd, scales in enumerate([np.concatenate([T, up]), np.concatenate([down, np.float32([0.05, 0.0, 1e6]), T[:61]])]):
        def edit(sd):
            sd["mvCoder.context_prediction.weight"].zero_()
            sd["mvCoder.entropy_parameters.4.weight"][:128].zero_()
            sd["mvCoder.entropy_parameters.4.bias"][:128] = torch.from_numpy(scales)
        orc, net = _models(oracle_model, edit)
        W, tabs, _ = _coder(orc, net, "mv")
        gc = tabs.gc
        _, params = _latents(latent_stats, "mv", 1, 60, 60, seed=100 + rnd)
        e0 = _encode(W, "mv", tabs, _act(torch.zeros(1, 60, 60, 128), 128), params, 16)
        want_idx = e0["y_indexes"].cpu().numpy()[0, 0, 0]
        mean = e0["y_hat"] - e0["y_symbols"].float()
        g = np.random.default_rng(rnd)
        tgt = np.zeros((3600, 128), np.int64)
        for c in range(128):
            i = want_idx[c]
            mv, off = int(gc.length[i]) - 2, int(gc.offset[i])
            t = np.concatenate([off + np.arange(mv), [off + mv, off - 1], 2 ** np.arange(1, 31), -2 ** np.arange(1, 31)])
            t = np.concatenate([t, off + np.arange(3600 - t.size) % mv])
            tgt[:, c] = g.permutation(t)
        y = _act(torch.zeros(1, 60, 60, 128), 128)
        y.t.copy_(mean + torch.from_numpy(tgt.reshape(1, 60, 60, 128)).float().to(DEV))
        for cl in (16, 8):
            _rows_lossless(W, "mv", tabs, _encode(W, "mv", tabs, y, params, cl), params, cl, f"round {rnd}")


@pytest.mark.gpu
@pytest.mark.parametrize("cache", [True, False])
@pytest.mark.parametrize("amp", [False, True])
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2), ((1024, 1920), 0, 1)])
def test_v3_round_trip_is_exact(oracle_model, hw, seed, n, amp, cache):
    """compress(row_streams=True) gives compress()'s recon and symbols; a second module's decompress of the version-3
    container returns that recon bit for bit, and so does its decompress of the version-2 container of the same frame.
    The version-3 container is at most 16 bytes per extra row stream longer."""
    from tdvc_b200 import coding
    x, refs = _pair(n, hw, seed)
    enc, dec = _net(oracle_model, cache), _net(oracle_model, cache)
    t2, t3 = {}, {}
    with torch.no_grad():
        r2, d2 = enc.compress(x, refs, amp, taps=t2)
        c2 = enc.last_coded
        r3, d3 = enc.compress(x, refs, amp, taps=t3, row_streams=True)
        c3 = enc.last_coded
    _assert_equal(r3, r2, "recon with row streams")
    for k in t2:
        if ".ac." in k:
            _assert_equal(t3[k], t2[k], k)
    hy = hw[0] // 16
    for nm in ("mv", "res"):
        assert c3[nm]["y_streams"] == "rows" and len(c3[nm]["strings"][0]) == n * hy
        assert c3[nm]["strings"][1] == c2[nm]["strings"][1]
        want = (sum(len(s_) for s_ in c3[nm]["strings"][0][:hy]) + len(c3[nm]["strings"][1][0])) * 8.0 / (n * hw[0] * hw[1])
        assert c3[nm]["ac_bpp"] == want
    assert d3[:4] == b"TDV3" and d2[:4] == b"TDV2"
    assert 0 < len(d3) - len(d2) <= 16 * n * (hy - 1) * 2 or (hy == 1 and len(d3) == len(d2))
    with torch.no_grad():
        _assert_equal(dec.decompress(d3, refs), r3, "decompress of version 3")
        _assert_equal(dec.decompress(d2, refs), r2, "decompress of version 2")
        lat = dec.decompress_latents(d3)
    for nm in ("mv", "res"):
        _assert_equal(lat[nm]["y_hat"], t3[f"{nm}.ac.y_hat"], f"{nm} y_hat")


@pytest.mark.gpu
def test_gop_round_trips_with_row_streams(oracle_model):
    """6-frame GOP at 64x128 and 3-frame GOP at 1920x1024 through compress_gop(row_streams=True) / decompress_gop."""
    from tdvc_b200 import gop, synth
    for (h, w), T in (((64, 128), 6), ((1024, 1920), 3)):
        frames = torch.cat([synth.make_frame_pair(h, w, seed=30 + i)[0] for i in range(T + 1)]).to(DEV)
        enc, dec = _net(oracle_model), _net(oracle_model)
        with torch.no_grad():
            containers, recons = gop.compress_gop(enc, frames[:1], frames[1:], row_streams=True)
            assert all(c[:4] == b"TDV3" for c in containers)
            back = gop.decompress_gop(dec, frames[:1], containers, (h, w))
        for i, (a, b) in enumerate(zip(back, recons)):
            _assert_equal(a, b, f"{h}x{w} frame {i}")


@pytest.mark.gpu
def test_damaged_rows_through_the_shared_launcher(oracle_model):
    """A truncated row raises naming coder, image and row; one flipped byte inside row r raises at row r (the end-of-row
    rule); in a batch of 3 the other images decode (status -1); the good container then decodes exactly."""
    from tdvc_b200 import coding
    n, hw = 3, (64, 128)
    enc, dec = _net(oracle_model), _net(oracle_model)
    x, refs = _pair(n, hw, 6)
    with torch.no_grad():
        recon, data = enc.compress(x, refs, row_streams=True)
    hy = hw[0] // 16

    def damaged(fn, nm, i, r):
        box = coding.unpack_frame(data)
        frame = box.pop("frame")
        box[nm]["strings"][0][i * hy + r] = fn(box[nm]["strings"][0][i * hy + r])
        return coding.pack_frame(box, frame=frame)

    with pytest.raises(RuntimeError, match=r"rs y row 2 of image 1 is truncated or corrupt at \(h=2, w=\d+, c=\d+\)"):
        dec.decompress(damaged(lambda s: s[:len(s) // 8 * 4], "res", 1, 2), refs)
    for r in range(hy):
        flip = lambda s: s[:len(s) // 2] + bytes([s[len(s) // 2] ^ 0x5A]) + s[len(s) // 2 + 1:]
        with pytest.raises(RuntimeError, match=rf"mv y row {r} of image 2 is truncated or corrupt at \(h={r}, "):
            dec.decompress(damaged(flip, "mv", 2, r), refs)
    # the kernel's per-image status: the other images of the batch decode
    box = coding.unpack_frame(damaged(lambda s: s[:8], "res", 0, 1))
    W = dec._weights(DEV)
    plan = dec._plan(n, *hw, DEV)
    lat = dec.decompress_latents(data)
    del lat
    params = plan.buf("dec.rs.params", n, hy, hw[1] // 16, 256)
    h = coding.launch_decoding(W, "rs", W["_tables"]["rs"], box["res"]["strings"][0], params, box["res"]["cluster"],
                               rows=True)
    h["done"].synchronize()
    status = h["status"].tolist()
    assert status[0] >= 0 and status[1] == -1 and status[2] == -1, status
    torch.cuda.synchronize()
    with torch.no_grad():
        _assert_equal(dec.decompress(data, refs), recon, "after damaged rows")


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_row_codec_between_forwards_changes_nothing(oracle_model, graph):
    """compress(row_streams=True) + decompress between two forwards leave the second forward as it is without them."""
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
                c_recon, data = net.compress(x2, refs, row_streams=True)
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
        assert c1[nm]["strings"] == c0[nm]["strings"] and c1[nm]["ac_bpp"] == c0[nm]["ac_bpp"]

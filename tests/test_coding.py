"""Real entropy coding (`is_compress=True`, reference main/model/pnet.py:45-49,69-73 -> compressai update / compress).

CPU part (-m "not gpu"): the oracle's coder round-trips and codes close to the ideal length; the library's HOST functions
(`tdvc_pmf_to_quantized_cdf`, `tdvc_rans_encode_with_indexes`, `tdvc_rans_decode_with_indexes` - compressai runs these
on the CPU too) are byte-identical to the oracle restatement (oracle/rans.py), including the bypass escape and the
bin-stealing path.  GPU part: tables, symbols and strings of the CUDA path against the oracle.
compressai is not in the reference tree: parity here is restatement-defined (DESIGN.md section 2)."""
import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers: work on a copy so that the session's oracle keeps its state_dict."""
    import copy
    return copy.deepcopy(oracle_model)


def _gc_tables(oracle_model):
    from oracle.compressai_port import get_scale_table
    gc = oracle_model.mvCoder.gaussian_conditional
    gc.update_scale_table(get_scale_table(), force=True)
    return gc


def _as_tables(m):
    from tdvc_b200 import coding
    return coding.Tables(m._quantized_cdf.numpy(), m._cdf_length.numpy(), m._offset.numpy())


def test_pmf_to_quantized_cdf_matches_oracle():
    import ctypes as C
    from oracle import rans
    from tdvc_b200 import lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(5)
    for n, kind in ((3, "flat"), (40, "peaked"), (300, "sparse"), (2000, "gauss")):
        if kind == "flat":
            p = torch.full((n,), 1.0 / n)
        elif kind == "peaked":
            p = torch.softmax(torch.randn(n, generator=g) * 6, 0)
        elif kind == "sparse":   # most bins round to zero: exercises the stealing loop
            p = torch.softmax(torch.randn(n, generator=g) * 12, 0)
        else:
            x = torch.arange(n) - n // 2
            p = torch.exp(-0.5 * (x / 3.0) ** 2)
            p = p / p.sum()
        p = p.float().contiguous()
        want = rans.pmf_to_quantized_cdf(p.tolist(), 16)
        got = np.zeros(n + 1, dtype=np.int32)
        pn = p.numpy()
        L.check(lib.tdvc_pmf_to_quantized_cdf(pn.ctypes.data_as(C.c_void_p), n, 16, got.ctypes.data_as(C.c_void_p)), "cdf")
        assert got.tolist() == want, kind
        assert got[0] == 0 and got[-1] == 65536 and (np.diff(got) > 0).all()


def test_host_rans_is_byte_identical_to_oracle(oracle_model):
    from oracle import rans
    from tdvc_b200 import coding
    gc = _gc_tables(oracle_model)
    tabs = _as_tables(gc)
    cdf, lens, offs = gc._tables()
    g = torch.Generator().manual_seed(7)
    for n in (0, 1, 5, 4096, 50000):
        idx = torch.randint(0, 64, (n,), generator=g, dtype=torch.int32)
        sym = (torch.randn(n, generator=g) * gc.scale_table[idx.long()] * 1.5).round().int()
        if n >= 4096:   # far outliers: the bypass escape with several 4-bit digits, both signs
            sym[::97] = 70000
            sym[5::131] = -123456
            sym[11::173] = -gc._offset[idx[11::173].long()]   # exactly max_value: smallest escape
        want = rans.encode_with_indexes(sym.tolist(), idx.tolist(), cdf, lens, offs)
        got = coding.rans_encode(sym.numpy(), idx.numpy(), tabs)
        assert got == want, n
        assert len(got) % 4 == 0 and len(got) >= 8
        back = coding.rans_decode(got, idx.numpy(), tabs)
        assert np.array_equal(back, sym.numpy())
        assert rans.decode_with_indexes(got, idx.tolist(), cdf, lens, offs) == sym.tolist()
        if n:
            ideal = rans.ideal_bits(sym.tolist(), idx.tolist(), cdf, lens, offs)
            assert ideal <= 8 * len(got) <= ideal + 64 + 32


def test_host_rans_rejects_bad_input(oracle_model):
    from tdvc_b200 import coding
    tabs = _as_tables(_gc_tables(oracle_model))
    with pytest.raises(RuntimeError):
        coding.rans_encode(np.zeros(4, np.int32), np.full(4, 64, np.int32), tabs)      # table index out of range
    good = coding.rans_encode(np.arange(-50, 50, dtype=np.int32), np.full(100, 20, np.int32), tabs)
    with pytest.raises(RuntimeError):
        coding.rans_decode(good[:8], np.full(100, 20, np.int32), tabs)                 # truncated stream


def test_host_rans_rejects_an_escape_outside_int32(oracle_model, monkeypatch):
    """An escape of 16 bypass digits 0xF folds to a value near 2^63: the encoder never writes one, and the host decoder
    must raise on it (as the device decoder stops on it) instead of returning a wrapped symbol."""
    from oracle import rans
    from tdvc_b200 import coding
    gc = _gc_tables(oracle_model)
    tabs = _as_tables(gc)
    cdf, lens, offs = gc._tables()
    t = 20
    mv = lens[t] - 2
    esc = [(cdf[t][mv], cdf[t][mv + 1] - cdf[t][mv], False)]
    digits = [(15, 16, True), (1, 2, True)] + [(15, 16, True)] * 16   # digit count 15 + 1, then 16 digits 0xF
    monkeypatch.setattr(rans, "_rans_symbols", lambda *a: esc + digits)
    data = rans.encode_with_indexes([0], [t], cdf, lens, offs)
    with pytest.raises(RuntimeError):
        coding.rans_decode(data, np.array([t], np.int32), tabs)


def test_oracle_compress_round_trip(oracle_model):
    """compress -> decompress restores y_hat exactly and the strings are as long as the tables say (oracle only)."""
    from oracle import rans
    from tdvc_b200 import synth
    x, refs = synth.make_frame_pair(64, 64, seed=3)
    taps = {}
    with torch.no_grad():
        plain = oracle_model(x, refs, False)
        out = oracle_model(x, refs, False, is_compress=True, taps=taps)
    for a, b in zip(plain, out):   # the reference's return value does not depend on is_compress
        assert torch.equal(a, b)
    for nm, coder in (("mv", oracle_model.mvCoder), ("res", oracle_model.resCoder)):
        enc = oracle_model.last_coded[nm]
        assert enc["shape"] == (1, 1) and len(enc["strings"]) == 2
        with torch.no_grad():
            dec = coder.decompress(enc["strings"], enc["shape"])
        assert torch.equal(dec["y_hat"], taps[f"{nm}.ac.y_hat"])
        sy, ix = taps[f"{nm}.ac.y_symbols"].reshape(-1).tolist(), taps[f"{nm}.ac.y_indexes"].reshape(-1).tolist()
        ideal = rans.ideal_bits(sy, ix, *coder.gaussian_conditional._tables())
        assert ideal <= 8 * len(enc["strings"][0][0]) <= ideal + 96
        assert enc["ac_bpp"] == (len(enc["strings"][0][0]) + len(enc["strings"][1][0])) * 8.0 / (64 * 64)
        # quantising relative to the predicted mean differs from the forward pass's round(y) by less than one step
        assert (taps[f"{nm}.ac.y_hat"] - taps[f"{nm}.y_hat"]).abs().max() <= 1.0


def test_tables_are_bit_identical_to_oracle(oracle_model):
    """update(): host pmf + host quantisation (tdvc_b200/coding.py) against the oracle's tables, bit for bit."""
    from tdvc_b200 import coding
    from tdvc_b200.model import pack_entropy_bottleneck
    for coder in (oracle_model.mvCoder, oracle_model.resCoder):
        coder.update(force=True)
        eb = coding.eb_tables(pack_entropy_bottleneck(coder.entropy_bottleneck))
        gc = coding.gc_tables()
        for ours, ref in ((eb, coder.entropy_bottleneck), (gc, coder.gaussian_conditional)):
            assert np.array_equal(ours.length, ref._cdf_length.numpy())
            assert np.array_equal(ours.offset, ref._offset.numpy())
            assert np.array_equal(ours.cdf, ref._quantized_cdf.numpy())
            for r in range(ours.cdf.shape[0]):   # every row is a strictly increasing CDF ending at 2^16
                n = ours.length[r]
                assert ours.cdf[r, 0] == 0 and ours.cdf[r, n - 1] == 65536 and (np.diff(ours.cdf[r, :n]) > 0).all()
        assert torch.equal(coding.scale_table(), coder.gaussian_conditional.scale_table)
        assert ours.cdf.shape == (64, 3133)


def test_frame_container_round_trip(oracle_model):
    """pack_frame / unpack_frame on the oracle's own strings, and the oracle decodes what comes back out."""
    from tdvc_b200 import coding, synth
    x, refs = synth.make_frame_pair(64, 64, seed=6)
    with torch.no_grad():
        oracle_model(x, refs, False, is_compress=True)
    coded = oracle_model.last_coded
    blob = coding.pack_frame(coded)
    back = coding.unpack_frame(blob)
    assert set(back) == {"mv", "res"}
    for k in coded:
        assert back[k]["strings"] == coded[k]["strings"] and back[k]["shape"] == coded[k]["shape"]
    payload = sum(len(s) for v in coded.values() for lst in v["strings"] for s in lst)
    assert len(blob) == payload + 5 + 2 * (13 + 2 * 4 + 2 * 4)
    with torch.no_grad():
        dec = oracle_model.mvCoder.decompress(back["mv"]["strings"], back["mv"]["shape"])
    assert dec["x_hat"].shape == (1, 64, 64, 64)
    with pytest.raises(RuntimeError):
        coding.unpack_frame(blob[:-3])
    with pytest.raises(RuntimeError):
        coding.unpack_frame(b"XXXX" + blob[4:])


# ------------------------------------------------------------------------------------------------------ GPU
def _build(oracle_model, dev):
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()
    net.load_state_dict(oracle_model.state_dict(), strict=True)
    return net.to(dev)


def _first_mismatch(a, b):
    """First differing element of two (H, W, C) arrays in coding (raster) order, or None."""
    d = np.nonzero((a != b).reshape(-1))[0]
    return None if d.size == 0 else np.unravel_index(d[0], a.shape)


def _check_ar_against_oracle_loop(coder, plan, cn, sy, ix, yh, strings):
    """The wavefront kernel against compressai's raster loop (oracle `ar_code`) on the SAME latents: the y and the
    hyper-decoder output the CUDA forward pass left in the plan.  Returns the fraction of identical symbols."""
    N, hy, wy = sy.shape[:3]
    y = plan.buf(f"{cn}.y", N, hy, wy, 128).t.cpu().permute(0, 3, 1, 2).contiguous()
    params = plan.buf(f"{cn}.params", N, hy, wy, 256).t.cpu().permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        o_strings, o_sy, o_ix, o_yh = coder.ar_code(y, params)
    o_sy = np.asarray(o_sy, dtype=np.int32).reshape(sy.shape)
    o_ix = np.asarray(o_ix, dtype=np.int32).reshape(ix.shape)
    same_sym, same_idx = (o_sy == sy).mean(), (o_ix == ix).mean()
    assert same_sym >= 0.999 and same_idx >= 0.999, (cn, same_sym, same_idx)
    if same_sym == 1.0 and same_idx == 1.0:
        assert np.abs(yh - o_yh.permute(0, 2, 3, 1).numpy()).max() < 1e-4
        assert strings == o_strings            # byte-identical rANS strings
    return same_sym


@pytest.mark.gpu
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2)])
def test_is_compress_vs_oracle(oracle_model, hw, seed, n):
    """Autoregressive coding feeds every quantised value back into the prediction of its successors, so ONE symbol that
    falls on the other side of a rounding tie (the two forward passes agree to ~1e-6 on y) changes the means of everything
    coded after it.  The end-to-end comparison therefore demands identity up to the first tie and checks that it IS a tie;
    the kernel itself is held to the oracle's raster loop on identical latents, where nothing may differ."""
    from tdvc_b200 import coding, synth
    dev = torch.device("cuda:0")
    net = _build(oracle_model, dev)
    pairs = [synth.make_frame_pair(*hw, seed=seed + 10 * i) for i in range(n)]
    x, refs = torch.cat([p[0] for p in pairs]), torch.cat([p[1] for p in pairs])
    ot, gt = {}, {}
    with torch.no_grad():
        oracle_model(x, refs, False, is_compress=True, taps=ot)
        plain = net(x.to(dev), refs.to(dev), False)
        got = net(x.to(dev), refs.to(dev), False, is_compress=True, taps=gt)
    for a, b in zip(plain, got):   # same return value with and without coding (reference pnet.py:80-83)
        assert torch.equal(a, b)
    W = net._weights(dev)
    plan = net._plan(n, hw[0], hw[1], dev)
    for nm, cn, coder in (("mv", "mv", oracle_model.mvCoder), ("res", "rs", oracle_model.resCoder)):
        enc, want = net.last_coded[nm], oracle_model.last_coded[nm]
        assert enc["shape"] == want["shape"]
        sy, ix = gt[f"{nm}.ac.y_symbols"].cpu().numpy(), gt[f"{nm}.ac.y_indexes"].cpu().numpy()
        yh = gt[f"{nm}.ac.y_hat"].cpu().numpy()
        osy, oix = ot[f"{nm}.ac.y_symbols"].numpy(), ot[f"{nm}.ac.y_indexes"].numpy()
        assert sy.shape == osy.shape
        zs, ozs = gt[f"{nm}.ac.z_symbols"].cpu().numpy(), ot[f"{nm}.ac.z_symbols"].numpy()
        assert (zs == ozs).mean() >= 0.999
        tabs = W["_tables"][cn]
        gc_ref, eb_ref = _as_tables(coder.gaussian_conditional), _as_tables(coder.entropy_bottleneck)
        assert np.array_equal(tabs.gc.cdf, gc_ref.cdf) and np.array_equal(tabs.eb.cdf, eb_ref.cdf)   # tables: bit-identical
        # ---- (1) the kernel against the oracle's raster loop on the same latents
        _check_ar_against_oracle_loop(coder, plan, cn, sy, ix, yh, enc["strings"][0])
        # ---- (2) end to end against the oracle's own forward pass + loop
        oy = ot[f"{nm}.ac.y"].permute(0, 2, 3, 1).numpy()
        omu = ot[f"{nm}.ac.y_hat"].permute(0, 2, 3, 1).numpy() - osy
        for i in range(n):
            zi = np.repeat(np.arange(128, dtype=np.int32), zs.shape[2] * zs.shape[3])
            # the strings decode (with the tables and indexes that coded them) to the symbols
            assert np.array_equal(coding.rans_decode(enc["strings"][0][i], ix[i], tabs.gc), sy[i].reshape(-1))
            assert np.array_equal(coding.rans_decode(enc["strings"][1][i], zi, tabs.eb), zs[i].reshape(-1))
            if np.array_equal(zs[i], ozs[i]):
                assert enc["strings"][1][i] == want["strings"][1][i]
            fs, fi = _first_mismatch(sy[i], osy[i]), _first_mismatch(ix[i], oix[i])
            if fs is None and fi is None:
                assert enc["strings"][0][i] == want["strings"][0][i]      # byte-identical
                assert np.abs(yh[i] - ot[f"{nm}.ac.y_hat"][i].permute(1, 2, 0).numpy()).max() < 1e-3
            elif fs is not None and (fi is None or fs[:2] <= fi[:2]):
                r = oy[i][fs] - omu[i][fs]
                assert abs(abs(r - np.floor(r)) - 0.5) < 1e-3, ("first differing symbol is not at a rounding tie", nm, fs, r)
            else:   # a scale within rounding of a table entry
                tbl = coding.scale_table().numpy()
                o_scale_idx = oix[i][fi]
                assert abs(int(ix[i][fi]) - int(o_scale_idx)) == 1, (nm, fi)
    # compressai's buffers as update() leaves them
    assert net.mvCoder.gaussian_conditional._quantized_cdf.shape == oracle_model.mvCoder.gaussian_conditional._quantized_cdf.shape
    assert net.resCoder.entropy_bottleneck._cdf_length.numel() == 128


@pytest.mark.gpu
def test_is_compress_full_size(oracle_model):
    """1920x1024 (BASELINE config 2 frame size, 64x120 latent, 309 wavefronts of <= 40 positions): the kernel against the
    oracle's raster loop on the same latents (7,680 positions per coder on the host), every string decodes to the symbols
    that were coded, the coded size is the ideal code length of the symbols under the tables (+ the 8-byte final state), both
    cluster sizes give the same result, and coding does not disturb the frame's results."""
    from tdvc_b200 import coding, synth
    dev = torch.device("cuda:0")
    net = _build(oracle_model, dev)
    x, refs = synth.make_frame_pair(1024, 1920, seed=0)
    x, refs = x.to(dev), refs.to(dev)
    gt = {}
    with torch.no_grad():
        plain = net(x, refs, False)
        got = net(x, refs, False, is_compress=True, taps=gt)
    for a, b in zip(plain, got):
        assert torch.equal(a, b)
    W = net._weights(dev)
    plan = net._plan(1, 1024, 1920, dev)
    for nm, cn, coder in (("mv", "mv", oracle_model.mvCoder), ("res", "rs", oracle_model.resCoder)):
        coder.update(force=True)
        enc, tabs = net.last_coded[nm], W["_tables"][cn]
        sy, ix = gt[f"{nm}.ac.y_symbols"].cpu().numpy(), gt[f"{nm}.ac.y_indexes"].cpu().numpy()
        yh = gt[f"{nm}.ac.y_hat"].cpu().numpy()
        assert sy.shape == (1, 64, 120, 128) and ix.min() >= 0 and ix.max() <= 63
        _check_ar_against_oracle_loop(coder, plan, cn, sy, ix, yh, enc["strings"][0])
        assert np.array_equal(coding.rans_decode(enc["strings"][0][0], ix[0], tabs.gc), sy[0].reshape(-1))
        fi, fs = ix.reshape(-1), sy.reshape(-1)
        v, mv = fs - tabs.gc.offset[fi], tabs.gc.length[fi] - 2
        b = np.where((v < 0) | (v >= mv), mv, v)   # out-of-range symbols escape through the last bin
        f = tabs.gc.cdf[fi, b + 1] - tabs.gc.cdf[fi, b]
        raw = np.where(v < 0, -2 * v - 1, 2 * (v - mv)).astype(np.int64)[(v < 0) | (v >= mv)]
        nb = np.where(raw > 0, np.floor(np.log2(np.maximum(raw, 1))).astype(np.int64) // 4 + 1, 0)   # 4-bit digits of the escape
        ideal_bytes = ((16 - np.log2(f.astype(np.float64))).sum() + 4 * (nb // 15 + 1 + nb).sum()) / 8
        assert ideal_bytes <= len(enc["strings"][0][0]) <= ideal_bytes + 16
        assert 0 < enc["ac_bpp"] < 4 * (got[1].item() if nm == "res" else got[2].item()) + 0.05
        # y_hat = symbol + mean stays within half a step of y
        y = plan.buf(f"{cn}.y", 1, 64, 120, 128).t
        assert (gt[f"{nm}.ac.y_hat"] - y).abs().max().item() <= 0.5 + 1e-4
        for cl in (8, 16):   # the K splits (summation order) depend on the cluster size: only exact ties may move
            other = coding.code_latents(plan, W, cn, tabs, cluster=cl, keep=True)
            assert (other["y_symbols"].cpu().numpy() == sy).mean() >= 0.999
            oi = other["y_indexes"].cpu().numpy()
            assert (oi == ix).mean() >= 0.999
            assert np.array_equal(coding.rans_decode(other["strings"][0][0], oi[0], tabs.gc),
                                  other["y_symbols"].cpu().numpy()[0].reshape(-1))

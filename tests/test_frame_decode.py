"""Decoding both coders' latents of a P-frame from a version-2 container and the weights alone
(`VideoCompressor.decompress_latents`): z strings -> symbols on the host, z_hat = symbol + median (`tdvc_eb_dequantize`),
h_s (`_Plan.hyper_synthesis`, shared with the encoder) -> params, y strings -> y on the device (`tdvc_ar_decode`).

The decoder is a second module loaded from the same state_dict: no plan, no tables, nothing the encoder left behind.  Every
GPU test demands the encoder's z_hat, params, y symbols, indexes and y_hat bit for bit."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers: work on a copy so that the session's oracle keeps its state_dict."""
    import copy
    return copy.deepcopy(oracle_model)


def _coded(n=2, shape=(1, 2)):
    s = lambda k: [bytes([k + i]) * 12 for i in range(n)]
    return {"mv": {"strings": [s(1), s(2)], "shape": shape, "cluster": 16},
            "res": {"strings": [s(3), s(4)], "shape": shape, "cluster": 8}}


# ------------------------------------------------------------------------------------------------------ CPU
def test_malformed_containers_are_refused_before_any_device_work(monkeypatch):
    """A version-1 container (no cluster sizes), a missing coder, a frame size that is not a multiple of 64, a hyper-latent
    shape that does not fit the frame, string counts that do not match the batch and y strings that are not whole 32-bit
    words (or shorter than two) raise RuntimeError before the weights are packed or a string is decoded."""
    from tdvc_b200 import coding
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()

    def touched(*a, **k):
        raise AssertionError("device work on a malformed container")

    monkeypatch.setattr(VideoCompressor, "_weights", touched)
    monkeypatch.setattr(VideoCompressor, "_plan", touched)
    monkeypatch.setattr(coding, "decode_z_symbols", touched)
    frame = {"size": (64, 128), "N": 2, "precision": "exact"}
    missing = _coded()
    del missing["res"]
    three_lists = _coded()
    three_lists["mv"]["strings"].append([b"x", b"y"])
    one_string = _coded()
    one_string["res"]["strings"][1] = one_string["res"]["strings"][1][:1]
    ragged = _coded()
    ragged["res"]["strings"][0][1] = b"\0" * 10
    short = _coded()
    short["mv"]["strings"][0][0] = b"\0" * 4
    cases = {"version 1": (coding.pack_frame(_coded()), "version-1"),
             "missing coder": (coding.pack_frame(missing, frame=frame), "no res coder"),
             "frame size": (coding.pack_frame(_coded(shape=(1, 1)), frame=dict(frame, size=(64, 96))), "multiples of 64"),
             "frame height": (coding.pack_frame(_coded(shape=(0, 2)), frame=dict(frame, size=(32, 128))), "multiples of 64"),
             "hyper shape": (coding.pack_frame(_coded(shape=(2, 1)), frame=frame), "hyper-latent shape"),
             "string lists": (coding.pack_frame(three_lists, frame=frame), "strings"),
             "string count": (coding.pack_frame(one_string, frame=frame), "strings"),
             "batch": (coding.pack_frame(_coded(), frame=dict(frame, N=3)), "strings"),
             "y words": (coding.pack_frame(ragged, frame=frame), "res y string of image 1 has 10 bytes"),
             "y too short": (coding.pack_frame(short, frame=frame), "mv y string of image 0 has 4 bytes")}
    for what, (blob, msg) in cases.items():
        with pytest.raises(RuntimeError, match=msg):
            net.decompress_latents(blob)
    # a well-formed container on a module that is not on a CUDA device: refused too, still without device work
    with pytest.raises(RuntimeError, match="CUDA"):
        net.decompress_latents(coding.pack_frame(_coded(), frame=frame))


def test_z_symbols_and_z_hat_match_the_oracle(oracle_model):
    """The host z step against the oracle's EntropyBottleneck: strings the oracle's compress() wrote from random symbols
    (in-range bins and bypass escapes on both sides) decode to the same symbols with compressai's channel-repeated indexes,
    and the oracle's decompress() gives z_hat = symbols + medians in fp32, the addition tdvc_eb_dequantize performs."""
    from tdvc_b200 import coding
    from tdvc_b200.model import pack_entropy_bottleneck
    g = torch.Generator().manual_seed(11)
    for cn, coder in (("mv", oracle_model.mvCoder), ("rs", oracle_model.resCoder)):
        eb = coder.entropy_bottleneck
        eb.update(force=True)
        packed = pack_entropy_bottleneck(eb)
        tabs = coding.CoderTables({f"{cn}.eb": packed}, cn, "cpu")
        assert np.array_equal(tabs.eb.cdf, eb._quantized_cdf.numpy())
        med = packed[3].float()
        assert torch.equal(med, eb.quantiles[:, 0, 1].detach())
        for n, hz, wz in ((1, 1, 1), (2, 2, 3), (1, 4, 5)):
            lo = torch.as_tensor(tabs.eb.offset).view(1, -1, 1, 1)
            hi = lo + torch.as_tensor(tabs.eb.length).view(1, -1, 1, 1) - 3
            u = torch.rand(n, 128, hz, wz, generator=g)
            sym = (lo + (u * (hi - lo + 1).float()).long().clamp(max=hi - lo)).int()
            flat = sym.view(-1)
            flat[::7] = (flat[::7] + 300).int()            # above the last bin: bypass escape
            flat[3::11] = (lo.view(-1)[(torch.arange(3, flat.numel(), 11) // (hz * wz)) % 128] - 5000).int()   # below
            x = sym.float() + med.view(1, -1, 1, 1)
            assert torch.equal(torch.round(x - med.view(1, -1, 1, 1)).int(), sym)   # compress() quantises back to sym
            strings = eb.compress(x)
            assert strings == [coding.rans_encode(sym[i].reshape(-1).numpy(), coding.eb_indexes(hz, wz), tabs.eb)
                               for i in range(n)]
            assert np.array_equal(coding.eb_indexes(hz, wz), eb._build_indexes((1, 128, hz, wz)).reshape(-1).numpy())
            got = coding.decode_z_symbols(cn, strings, tabs, hz, wz)
            assert got.shape == (n, 128, hz, wz) and np.array_equal(got, sym.numpy())
            z_hat = eb.decompress(strings, (hz, wz))
            assert torch.equal(z_hat, torch.from_numpy(got).float() + med.view(1, -1, 1, 1))
        with pytest.raises(RuntimeError, match=f"the {cn} z string of image 1"):
            coding.decode_z_symbols(cn, [strings[0], strings[0][:8]], tabs, 4, 5)


def test_eb_dequantize_is_declared_bound_and_exported():
    """tdvc_eb_dequantize: in the header, exported by the library, and its ctypes argument list matches the prototype
    argument for argument (pointers as void*, int as int32)."""
    from tdvc_b200 import build, lib as L
    build.build()
    lib = L.load()
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "tdvc_b200.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+tdvc_eb_dequantize\s*\(([^)]*)\)\s*;", txt)
    assert m, "tdvc_eb_dequantize is not declared in include/tdvc_b200.h"
    kinds = {"int": L.i32, "int64_t": L.i64, "float": L.f32}
    want = []
    for arg in (a.strip() for a in m.group(1).split(",")):
        typ = arg.rsplit(None, 1)[0] if "*" not in arg else "*"
        want.append(L.vp if typ == "*" else kinds[typ.replace("const", "").strip()])
    assert L.SIGNATURES["tdvc_eb_dequantize"] == want
    assert len(want) == 8
    assert hasattr(lib, "tdvc_eb_dequantize") and lib.tdvc_eb_dequantize.argtypes == want


def test_eb_dequantize_compiles_without_spills():
    from tdvc_b200 import build
    r = subprocess.run([build.NVCC] + build.FLAGS + ["-c", os.path.join(build.CSRC, "entropy.cu"), "-o", os.devnull],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout + r.stderr
    i = lines.index("eb_dequantize_kernel")
    props = lines[i:].split("ptxas info    : Used")[0]
    assert "0 bytes spill stores, 0 bytes spill loads" in props, props


# ------------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


def _net(oracle_model):
    from tdvc_b200.model import VideoCompressor
    net = VideoCompressor().eval()
    net.load_state_dict(oracle_model.state_dict(), strict=True)
    return net.to(DEV)


def _pair(n, hw, seed):
    from tdvc_b200 import synth
    pairs = [synth.make_frame_pair(*hw, seed=seed + 10 * i) for i in range(n)]
    return torch.cat([p[0] for p in pairs]).to(DEV), torch.cat([p[1] for p in pairs]).to(DEV)


def _encode(net, n, hw, seed, amp=False, precision="exact"):
    """One coded P-frame: (taps of the forward pass, its version-2 container)."""
    from tdvc_b200 import coding
    x, refs = _pair(n, hw, seed)
    gt = {}
    with torch.no_grad():
        net(x, refs, amp, is_compress=True, taps=gt)
    return gt, coding.pack_frame(net.last_coded, frame={"size": hw, "N": n, "precision": precision})


def _assert_equal(got, want, what):
    if not torch.equal(got, want):
        d = (got != want).reshape(-1).nonzero()
        first = np.unravel_index(int(d[0]), tuple(want.shape)) if d.numel() else "shape"
        raise AssertionError(f"{what} differs at {first} ({int(d.numel())} elements, shapes {tuple(got.shape)} "
                             f"{tuple(want.shape)})")


def _assert_matches_encoder(out, gt, what):
    for nm in ("mv", "res"):
        _assert_equal(out[nm]["z_hat"], gt[f"{nm}.z_hat"].permute(0, 2, 3, 1), f"{what} {nm} z_hat")
        for k in ("y_symbols", "y_indexes", "y_hat"):
            _assert_equal(out[nm][k], gt[f"{nm}.ac.{k}"], f"{what} {nm} {k}")


def _assert_same_params(enc, dec, n, hw, what):
    hy, wy = hw[0] // 16, hw[1] // 16
    for cn in ("mv", "rs"):
        want = enc._plan(n, *hw, torch.device(DEV)).buf(f"{cn}.params", n, hy, wy, 256).t
        got = dec._plan(n, *hw, torch.device(DEV)).buf(f"dec.{cn}.params", n, hy, wy, 256).t
        _assert_equal(got, want, f"{what} {cn} params")


@pytest.mark.gpu
@pytest.mark.parametrize("hw,seed,n", [((64, 128), 1, 1), ((128, 192), 2, 1), ((64, 64), 4, 2), ((1024, 1920), 0, 1)])
def test_decompress_latents_is_exact(oracle_model, hw, seed, n):
    """z_hat, the hyper-decoder output and y of both coders equal the encoder's bit for bit, decoded by a module that has
    never coded anything; the two-stream decode equals decoding the coders one after the other with decode_latents."""
    from tdvc_b200 import coding
    enc, dec = _net(oracle_model), _net(oracle_model)
    gt, blob = _encode(enc, n, hw, seed)
    assert not dec._plans and "_tables" not in dec._weights(torch.device(DEV))
    out = dec.decompress_latents(blob)
    assert out["frame"] == {"size": hw, "N": n, "precision": "exact"}
    assert out["mv"]["y_hat"].shape == (n, hw[0] // 16, hw[1] // 16, 128)
    assert out["res"]["z_hat"].shape == (n, hw[0] // 64, hw[1] // 64, 128)
    _assert_matches_encoder(out, gt, f"{hw} N={n}")
    _assert_same_params(enc, dec, n, hw, f"{hw} N={n}")
    if hw == (128, 192):
        W = dec._weights(torch.device(DEV))
        plan = dec._plan(n, *hw, torch.device(DEV))
        back = coding.unpack_frame(blob)
        for nm, cn in (("mv", "mv"), ("res", "rs")):
            params = plan.buf(f"dec.{cn}.params", n, hw[0] // 16, hw[1] // 16, 256)
            one = coding.decode_latents(W, cn, W["_tables"][cn], back[nm]["strings"][0], params, back[nm]["cluster"])
            for k in ("y_symbols", "y_indexes", "y_hat"):
                _assert_equal(out[nm][k], one[k], f"two streams vs one coder at a time: {nm} {k}")


@pytest.mark.gpu
def test_both_cluster_sizes_decode(oracle_model):
    """Strings coded with 8 and with 16 CTAs per image, packed with that size, decode losslessly."""
    from tdvc_b200 import coding
    n, hw = 2, (64, 64)
    enc, dec = _net(oracle_model), _net(oracle_model)
    _encode(enc, n, hw, 4)
    W = enc._weights(torch.device(DEV))
    plan = enc._plan(n, *hw, torch.device(DEV))
    for cluster in (8, 16):
        coded, want = {}, {}
        for nm, cn in (("mv", "mv"), ("res", "rs")):
            e = coding.code_latents(plan, W, cn, W["_tables"][cn], cluster=cluster, keep=True)
            assert e["cluster"] == cluster
            coded[nm], want[nm] = e, e
        blob = coding.pack_frame(coded, frame={"size": hw, "N": n, "precision": "exact"})
        assert all(v["cluster"] == cluster for k, v in coding.unpack_frame(blob).items() if k != "frame")
        out = dec.decompress_latents(blob)
        for nm in ("mv", "res"):
            for k in ("y_symbols", "y_indexes", "y_hat"):
                _assert_equal(out[nm][k], want[nm][k], f"cluster {cluster} {nm} {k}")


@pytest.mark.gpu
def test_mixed_container_decodes_like_exact(oracle_model):
    """The container's precision mode does not change the latents: a frame coded with enabled_amp=True ("mixed") decodes
    exactly, and to the same latents as the same strings in an "exact" container."""
    from tdvc_b200 import coding
    n, hw = 1, (128, 192)
    enc, dec = _net(oracle_model), _net(oracle_model)
    gt, blob = _encode(enc, n, hw, 2, amp=True, precision="mixed")
    assert coding.unpack_frame(blob)["frame"]["precision"] == "mixed"
    mixed = dec.decompress_latents(blob)
    _assert_matches_encoder(mixed, gt, "mixed")
    exact = dec.decompress_latents(coding.pack_frame(enc.last_coded, frame={"size": hw, "N": n, "precision": "exact"}))
    for nm in ("mv", "res"):
        for k in ("z_hat", "y_symbols", "y_indexes", "y_hat"):
            _assert_equal(mixed[nm][k], exact[nm][k], f"mixed vs exact {nm} {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_decoding_between_forwards_changes_nothing(oracle_model, graph):
    """decompress_latents on the same module and plan between two forwards leaves the next forward's recon, bpp and strings
    bit-identical to a run without it (eager, and with CUDA graphs: the third forward of the same inputs replays one)."""
    from tdvc_b200 import coding
    n, hw = 2, (64, 128)
    x, refs = _pair(n, hw, 7)
    runs = []
    for decode in (False, True):
        net = _net(oracle_model)
        net.use_cuda_graph = graph
        with torch.no_grad():
            net(x, refs, False, is_compress=True)
            blob = coding.pack_frame(net.last_coded, frame={"size": hw, "N": n, "precision": "exact"})
            net(x, refs, False, is_compress=True)
            if decode:
                out = net.decompress_latents(blob)
                assert out["mv"]["y_hat"].shape == (n, 4, 8, 128)
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
def test_damaged_strings(oracle_model):
    """A truncated z string raises naming the coder and the image; a garbled one raises or decodes to some symbols (rANS
    cannot always tell); a truncated y string raises naming its latent position.  None of them faults the device, and the
    next decode of good bytes is exact."""
    from tdvc_b200 import coding
    n, hw = 2, (64, 64)
    enc, dec = _net(oracle_model), _net(oracle_model)
    gt, blob = _encode(enc, n, hw, 4)

    def damaged(nm, which, i, fn):
        coded = coding.unpack_frame(blob)
        frame = coded.pop("frame")
        coded[nm]["strings"][which][i] = fn(coded[nm]["strings"][which][i])
        return coding.pack_frame(coded, frame=frame)

    with pytest.raises(RuntimeError, match=r"the rs z string of image 1"):
        dec.decompress_latents(damaged("res", 1, 1, lambda s: s[:len(s) - 4]))
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match=r"the mv z string of image 0"):
        dec.decompress_latents(damaged("mv", 1, 0, lambda s: s[:4]))
    torch.cuda.synchronize()

    def garble(s):
        s = bytearray(s)
        for j in range(8, len(s), 5):
            s[j] ^= 0x5A
        return bytes(s)

    try:
        dec.decompress_latents(damaged("mv", 1, 0, garble))
    except RuntimeError as e:
        assert "image 0" in str(e), str(e)
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match=r"rs y string of image 1 .*position \(h=\d+, w=\d+, c=\d+\)"):
        dec.decompress_latents(damaged("res", 0, 1, lambda s: s[:len(s) // 8 * 4]))
    torch.cuda.synchronize()
    _assert_matches_encoder(dec.decompress_latents(blob), gt, "after damaged strings")

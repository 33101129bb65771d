"""Real entropy coding of the two latents of a P-frame (`forward(..., is_compress=True)`).

Reference path: main/model/pnet.py:45-49,69-73 - `coder.eval(); coder.update(force=True); out_enc = coder.compress(x);
ac_bpp = sum(len(s[0]) for s in out_enc["strings"]) * 8.0 / num_pixels` for `mvCoder` and `resCoder` (compressai
`Cheng2020Anchor`; compressai is not in the reference tree: SURVEY.md App. A, DESIGN.md section 7, parity is defined by
oracle/compressai_port.py + oracle/rans.py).

What runs where:
* `update`: HOST code.  The tables are integer data that the two ends of a codec must reproduce bit for bit, so nothing
  in them goes through device transcendental functions: the pmf of the factorised prior (a 5-layer MLP on <= 128 x 60
  points) and of the 64 Gaussian scales is evaluated with the same fp32 host operations compressai uses for a model that
  lives on the CPU, and quantised to 16 bits by `tdvc_pmf_to_quantized_cdf` (host code in the library, as compressai's is).
  (Measured: with the pmf from expf / erfcf on the GPU a bin edge differs by one count in ~0.1 % of the bins, which then
  changes which bins the zero-probability tail steals from.)  Tables are cached per set of packed weights (the reference
  rebuilds them on every call).
* `compress`: z symbols by `tdvc_eb_symbols`; the autoregressive pass over y - compressai's per-position Python loop - by
  the wavefront kernel `tdvc_ar_code` (one launch per coder, csrc/coding.cu) on the y / hyper-decoder buffers the forward
  pass left in the plan; rANS over the symbols on the host (`tdvc_rans_encode_with_indexes`), as in compressai.
* `decode_latents`: y strings back to symbols and y_hat on the device (`tdvc_ar_decode`, csrc/ar_decode.cu), bit-identical
  to what `tdvc_ar_code` produced when told the encoder's cluster size.
"""
import ctypes as C
import math
import statistics

import numpy as np
import torch

from tdvc_b200 import lib as L

SCALES_MIN, SCALES_MAX, SCALES_LEVELS = 0.11, 256, 64   # compressai models/priors.py
TAIL_MASS = 1e-9
PRECISION = 16


def scale_table():
    """compressai `get_scale_table()` (host arithmetic there too: torch.linspace defaults to the CPU)."""
    return torch.exp(torch.linspace(math.log(SCALES_MIN), math.log(SCALES_MAX), SCALES_LEVELS))


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Tables:
    """compressai's `_quantized_cdf`, `_cdf_length`, `_offset` of one entropy model, as int32 numpy arrays."""

    def __init__(self, cdf, length, offset):
        self.cdf = np.ascontiguousarray(cdf, dtype=np.int32)
        self.length = np.ascontiguousarray(length, dtype=np.int32)
        self.offset = np.ascontiguousarray(offset, dtype=np.int32)

    def tensors(self, device):
        return (torch.from_numpy(self.cdf.copy()).to(device), torch.from_numpy(self.length.copy()).to(device),
                torch.from_numpy(self.offset.copy()).to(device))

    def on(self, device):
        """tensors(device), built once per device (read by the device decoder)."""
        cache = self.__dict__.setdefault("_on", {})
        key = str(torch.device(device))
        if key not in cache:
            cache[key] = self.tensors(device)
        return cache[key]


def _pmf_to_cdf(pmf, tail, pmf_length, max_length):
    """compressai `EntropyModel._pmf_to_cdf`: row i = quantised CDF of (pmf[i][:len_i], tail[i]), zero padded."""
    lib = L.load()
    rows = len(pmf_length)
    cdf = np.zeros((rows, max_length + 2), dtype=np.int32)
    for i in range(rows):
        n = int(pmf_length[i])
        prob = np.ascontiguousarray(np.concatenate([pmf[i, :n], tail[i:i + 1]]), dtype=np.float32)
        row = np.zeros(n + 2, dtype=np.int32)
        L.check(lib.tdvc_pmf_to_quantized_cdf(_np_ptr(prob), n + 1, PRECISION, _np_ptr(row)), "pmf_to_quantized_cdf")
        cdf[i, :n + 2] = row
    return cdf


def eb_tables(eb_packed):
    """compressai `EntropyBottleneck.update`.  eb_packed = (mats [C][33], biases [C][13], factors [C][12], medians,
    quantiles [C][3], target) of model._Packed (matrices already softplus'ed, factors tanh'ed, on the host at pack time)."""
    mats, biases, factors, _, quantiles, _ = (t.detach().cpu() for t in eb_packed)
    Cc = quantiles.shape[0]
    medians = quantiles[:, 1]
    minima = torch.clamp(torch.ceil(medians - quantiles[:, 0]).int(), min=0)
    maxima = torch.clamp(torch.ceil(quantiles[:, 2] - medians).int(), min=0)
    pmf_start = medians - minima
    pmf_length = maxima + minima + 1
    max_length = int(pmf_length.max())
    samples = torch.arange(max_length)[None, :] + pmf_start[:, None, None]   # (C, 1, L)
    widths = (1, 3, 3, 3, 3, 1)
    mo = bo = fo = 0
    layers = []
    for i in range(5):
        fi, fn = widths[i], widths[i + 1]
        m = mats[:, mo:mo + fn * fi].reshape(Cc, fn, fi)
        bb = biases[:, bo:bo + fn].reshape(Cc, fn, 1)
        f = factors[:, fo:fo + fn].reshape(Cc, fn, 1) if i < 4 else None
        layers.append((m, bb, f))
        mo, bo, fo = mo + fn * fi, bo + fn, fo + (fn if i < 4 else 0)

    def logits(v):   # compressai `_logits_cumulative`
        for m, bb, f in layers:
            v = torch.matmul(m, v) + bb
            if f is not None:
                v = v + f * torch.tanh(v)
        return v

    lower, upper = logits(samples - 0.5), logits(samples + 0.5)
    sign = -torch.sign(lower + upper)
    pmf = torch.abs(torch.sigmoid(sign * upper) - torch.sigmoid(sign * lower))[:, 0, :]
    tail = (torch.sigmoid(lower[:, 0, :1]) + torch.sigmoid(-upper[:, 0, -1:]))[:, 0]
    cdf = _pmf_to_cdf(pmf.numpy(), tail.numpy(), pmf_length.numpy(), max_length)
    return Tables(cdf, (pmf_length + 2).numpy(), (-minima).numpy())


_GC_TABLES = {}


def gc_tables(table=None):
    """compressai `GaussianConditional.update_scale_table(get_scale_table())` + `update()`: depends on nothing but the scale
    table and the tail mass, built once per process."""
    table = scale_table() if table is None else torch.as_tensor(table, dtype=torch.float32)
    key = tuple(table.tolist())
    if key in _GC_TABLES:
        return _GC_TABLES[key]
    multiplier = -statistics.NormalDist().inv_cdf(TAIL_MASS / 2)   # scipy.stats.norm.ppf in compressai
    center = torch.ceil(table * multiplier).int()
    pmf_length = 2 * center + 1
    max_length = int(pmf_length.max())
    samples = torch.abs(torch.arange(max_length).int() - center[:, None]).float()
    scale = table.unsqueeze(1).float()

    def phi(t):   # compressai `_standardized_cumulative`
        return 0.5 * torch.erfc(-(2 ** -0.5) * t)

    upper, lower = phi((0.5 - samples) / scale), phi((-0.5 - samples) / scale)
    pmf = upper - lower
    tail = (2 * lower[:, :1])[:, 0]
    cdf = _pmf_to_cdf(pmf.numpy(), tail.numpy(), pmf_length.numpy(), max_length)
    _GC_TABLES[key] = Tables(cdf, (pmf_length + 2).numpy(), (-center).numpy())
    return _GC_TABLES[key]


def rans_encode(symbols, indexes, tables):
    """int32 numpy symbols / table indexes (same length, coding order) -> bytes."""
    lib = L.load()
    symbols = np.ascontiguousarray(symbols, dtype=np.int32).reshape(-1)
    indexes = np.ascontiguousarray(indexes, dtype=np.int32).reshape(-1)
    if symbols.shape != indexes.shape:
        raise RuntimeError("rans_encode: symbols and indexes differ in length")
    cap = 8 * symbols.size + 64
    out = np.empty(cap, dtype=np.uint8)
    n = lib.tdvc_rans_encode_with_indexes(_np_ptr(symbols), _np_ptr(indexes), symbols.size, _np_ptr(tables.cdf),
                                          tables.cdf.shape[1], _np_ptr(tables.length), _np_ptr(tables.offset),
                                          tables.cdf.shape[0], _np_ptr(out), cap)
    if n < 0:
        L.check(int(n), "rans_encode_with_indexes")
    return out[:n].tobytes()


def rans_decode(data, indexes, tables):
    """Inverse of rans_encode given the same indexes -> int32 numpy symbols."""
    lib = L.load()
    indexes = np.ascontiguousarray(indexes, dtype=np.int32).reshape(-1)
    buf = np.frombuffer(data, dtype=np.uint8)
    out = np.empty(indexes.size, dtype=np.int32)
    L.check(lib.tdvc_rans_decode_with_indexes(_np_ptr(buf), buf.size, _np_ptr(indexes), indexes.size, _np_ptr(tables.cdf),
                                              tables.cdf.shape[1], _np_ptr(tables.length), _np_ptr(tables.offset),
                                              tables.cdf.shape[0], _np_ptr(out)), "rans_decode_with_indexes")
    return out


class CoderTables:
    """Tables of one coder (`update(force=True)`), built once per set of packed weights."""

    def __init__(self, W, cn, device):
        self.eb = eb_tables(W[f"{cn}.eb"])
        self.gc = gc_tables()
        self.scale_table = scale_table().to(device)


def _pinned(plan, name, like):
    key = ("pinned", name, tuple(like.shape), like.dtype)
    t = plan.bufs.get(key)
    if t is None:
        t = plan.bufs[key] = torch.empty(like.shape, dtype=like.dtype).pin_memory()
    return t


def _ar_chain(W, cn, tables, params, out, who):
    """The autoregressive chain of coder `cn` ("mv" | "rs") as tdvc_ar_code and tdvc_ar_decode both read it: its four layers,
    the scale table, the hyper-decoder output `params` (a channels-last Act (N, h, w, >= 256 channels)) and the outputs
    out = (y_hat, symbols, indexes), each (N, h, w, 128)."""
    ctx, e0, e2, e4 = W[f"{cn}.ctx"], W[f"{cn}.ep0"], W[f"{cn}.ep2"], W[f"{cn}.ep4"]
    if ctx.cin_pad != 128 or ctx.cout_pad != 256 or e0.cin_pad != 512 or e2.cin_pad < e0.cout_pad - 4 or e4.cout_pad != 256:
        raise RuntimeError(f"{who}: unexpected entropy-parameter layer shapes")
    y_hat, y_sym, y_idx = out
    return L.ArChain(params=params.ptr, params_ld=params.ld, w_ctx=ctx.w.data_ptr(), b_ctx=ctx.b.data_ptr(),
                     w1=e0.w.data_ptr(), b1=e0.b.data_ptr(), c1=e0.cout, c1_pad=e0.cout_pad,
                     w2=e2.w.data_ptr(), b2=e2.b.data_ptr(), c2=e2.cout, c2_pad=e2.cout_pad,
                     w3=e4.w.data_ptr(), b3=e4.b.data_ptr(), scale_table=tables.scale_table.data_ptr(),
                     n_scales=SCALES_LEVELS, y_hat=y_hat.data_ptr(), symbols=y_sym.data_ptr(), indexes=y_idx.data_ptr(),
                     N=params.N, H=params.H, W=params.W, C=128)


def launch_coding(plan, W, cn, tables, cluster=0, stream=None):
    """Device half of compressai `compress()` for coder `cn` ("mv" | "rs") on the latents the forward pass of `plan` just
    produced: symbols + table indexes of z and y, copied to pinned host memory on `stream`.  Returns a handle for
    finish_coding (the host half: rANS)."""
    lib = L.load()
    dev, N = plan.dev, plan.N
    stream = stream or torch.cuda.current_stream(dev)
    st = stream.cuda_stream
    hy, wy, hz, wz = plan.H // 16, plan.W // 16, plan.H // 64, plan.W // 64
    y, z = plan.buf(f"{cn}.y", N, hy, wy, 128), plan.buf(f"{cn}.z", N, hz, wz, 128)
    params = plan.buf(f"{cn}.params", N, hy, wy, 256)
    med = W[f"{cn}.eb"][3]
    # ---- z: factorised prior, NCHW symbol order
    z_sym = plan.raw(f"{cn}.ac.z_sym", (N, 128, hz, wz), torch.int32)
    z_idx = plan.raw(f"{cn}.ac.z_idx", (N, 128, hz, wz), torch.int32)
    L.check(lib.tdvc_eb_symbols(z.ptr, z.ld, med.data_ptr(), N, hz * wz, 128, z_sym.data_ptr(), z_idx.data_ptr(), st),
            "eb_symbols")
    # ---- y: autoregressive pass, (h, w, c) symbol order
    y_hat = plan.raw(f"{cn}.ac.y_hat", (N, hy, wy, 128))
    y_sym = plan.raw(f"{cn}.ac.y_sym", (N, hy, wy, 128), torch.int32)
    y_idx = plan.raw(f"{cn}.ac.y_idx", (N, hy, wy, 128), torch.int32)
    chain = _ar_chain(W, cn, tables, params, (y_hat, y_sym, y_idx), "code_latents")
    need = lib.tdvc_ar_code_workspace_bytes(N, chain.c1_pad, chain.c2_pad)
    ws = plan.raw(f"{cn}.ac.ws", ((need + 3) // 4,))
    used = C.c_int32(0)
    p = L.ArParams(chain=chain, y=y.ptr, y_ld=y.ld, cluster=cluster, cluster_used_host=C.addressof(used))
    L.check(lib.tdvc_ar_code(C.byref(p), ws.data_ptr(), need, st), "ar_code")
    plan.launches += 2
    host = []
    with torch.cuda.stream(stream):
        for nme, t in (("y_sym", y_sym), ("y_idx", y_idx), ("z_sym", z_sym), ("z_idx", z_idx)):
            h = _pinned(plan, f"{cn}.ac.{nme}", t)
            h.copy_(t, non_blocking=True)
            host.append(h)
        done = torch.cuda.Event()
        done.record(stream)
    return {"host": host, "done": done, "tables": tables, "N": N, "shape": (hz, wz), "cluster": used.value,
            "dev": {"y_symbols": y_sym, "y_indexes": y_idx, "y_hat": y_hat, "z_symbols": z_sym}}


def finish_coding(h, keep=False):
    """Host half: rANS over the symbols, one string per image (compressai codes batch items separately).
    Returns {"strings": [y_strings, z_strings], "shape": (h, w), "cluster": CTAs per image the y pass ran with (the
    summation order a decoder must reproduce)} (+ clones of the device tensors if keep)."""
    h["done"].synchronize()
    hs = [t.numpy() for t in h["host"]]
    tables = h["tables"]
    y_strings = [rans_encode(hs[0][i], hs[1][i], tables.gc) for i in range(h["N"])]
    z_strings = [rans_encode(hs[2][i], hs[3][i], tables.eb) for i in range(h["N"])]
    out = {"strings": [y_strings, z_strings], "shape": h["shape"], "cluster": h["cluster"]}
    if keep:
        out.update({k: v.clone() for k, v in h["dev"].items()})
    return out


def code_latents(plan, W, cn, tables, cluster=0, keep=False):
    return finish_coding(launch_coding(plan, W, cn, tables, cluster=cluster), keep=keep)


def launch_decoding(W, cn, tables, y_strings, params, cluster, stream=None):
    """Device decoding of the y strings of coder `cn` ("mv" | "rs"), the inverse of launch_coding's y half
    (compressai `_decompress_ar`): `tdvc_ar_decode` runs the context model and the entropy parameters position by position
    and decodes the rANS stream on the device.  params: the hyper-decoder output of the same images, a channels-last Act
    (N, h, w, >= 256 channels).  cluster: the CTAs per image `tdvc_ar_code` coded the strings with (8 or 16); the
    predictions, and so the decoded symbols, are exact only for that value.  Returns a handle for finish_decoding."""
    lib = L.load()
    N, hy, wy = params.N, params.H, params.W
    dev = params.t.device
    if cluster not in (8, 16):
        raise RuntimeError(f"decode_latents: encoder cluster size {cluster} (8 or 16)")
    if len(y_strings) != N:
        raise RuntimeError(f"decode_latents: {len(y_strings)} {cn} y strings for {N} images")
    for i, s_ in enumerate(y_strings):
        if len(s_) < 8 or len(s_) % 4:
            raise RuntimeError(f"decode_latents: {cn} y string of image {i} has {len(s_)} bytes (rANS strings are whole "
                               "32-bit words, at least two)")
    gl = tables.gc.length
    if gl.size > 64 or (gl < 2).any() or (gl > tables.gc.cdf.shape[1]).any() or int(gl.sum()) > 32768:
        raise RuntimeError("decode_latents: the Gaussian CDF tables are not valid rows for the device decoder")
    stream = stream or torch.cuda.current_stream(dev)
    words = np.frombuffer(b"".join(bytes(s_) for s_ in y_strings), dtype="<i4")
    offsets = np.cumsum([0] + [len(s_) // 4 for s_ in y_strings]).astype(np.int64)
    cdf, length, offset = tables.gc.on(dev)
    with torch.cuda.stream(stream):
        words_d = torch.from_numpy(words.copy()).to(dev)
        offsets_d = torch.from_numpy(offsets).to(dev)
        y_hat = torch.empty((N, hy, wy, 128), device=dev)
        y_sym = torch.empty((N, hy, wy, 128), device=dev, dtype=torch.int32)
        y_idx = torch.empty((N, hy, wy, 128), device=dev, dtype=torch.int32)
        status = torch.empty((N,), device=dev, dtype=torch.int64)
    p = L.ArDecodeParams(chain=_ar_chain(W, cn, tables, params, (y_hat, y_sym, y_idx), "decode_latents"),
                         words=words_d.data_ptr(), word_offsets=offsets_d.data_ptr(),
                         cdfs=cdf.data_ptr(), cdf_stride=cdf.shape[1], cdf_lengths=length.data_ptr(),
                         cdf_offsets=offset.data_ptr(), n_tables=cdf.shape[0], cdf_total=int(gl.sum()),
                         status=status.data_ptr(), cluster=cluster)
    L.check(lib.tdvc_ar_decode(C.byref(p), stream.cuda_stream), "ar_decode")
    with torch.cuda.stream(stream):
        status_h = _pinned_like(status)
        status_h.copy_(status, non_blocking=True)
        done = torch.cuda.Event()
        done.record(stream)
    # the inputs stay referenced until the decode has run
    return {"cn": cn, "done": done, "status": status_h, "keep": (words_d, offsets_d), "shape": (hy, wy),
            "y_hat": y_hat, "y_symbols": y_sym, "y_indexes": y_idx}


def _pinned_like(t):
    return torch.empty(t.shape, dtype=t.dtype).pin_memory()


def finish_decoding(h):
    """Waits for a launch_decoding and turns a failed image into RuntimeError (naming the coder, the image and the
    latent position (h, w, c) where the stream broke).  Returns {"y_hat", "y_symbols", "y_indexes"} (N, h, w, 128)."""
    h["done"].synchronize()
    wy = h["shape"][1]
    for i, st in enumerate(h["status"].tolist()):
        if st == -2:
            raise RuntimeError(f"ar_decode: the Gaussian CDF tables of the {h['cn']} coder are not valid rows (image {i})")
        if st != -1:
            pix, c = divmod(int(st), 128)
            raise RuntimeError(f"ar_decode: the {h['cn']} y string of image {i} is truncated or corrupt at latent position "
                               f"(h={pix // wy}, w={pix % wy}, c={c})")
    return {k: h[k] for k in ("y_hat", "y_symbols", "y_indexes")}


def decode_latents(W, cn, tables, y_strings, params, cluster, stream=None):
    return finish_decoding(launch_decoding(W, cn, tables, y_strings, params, cluster, stream=stream))


# ----------------------------------------------------------------------------------------------- bitstream container
_MAGIC = b"TDVC"       # version 1: strings and hyper-latent shapes only
_MAGIC_V2 = b"TDV2"    # version 2: + frame size, batch, precision mode, and each coder's autoregressive cluster size
_PRECISIONS = ("exact", "mixed")


def pack_frame(coded, frame=None):
    """`net.last_coded` of one P-frame -> bytes.  The reference only sketches a container (dead code, reference
    tools/utils/encoder.py:61-68: per string a big-endian shape header, a length and the payload); this one follows the
    sketch with 32-bit lengths (a 1920x1024 motion string is ~1 MB, beyond the sketch's uint16).
    frame=None (version 1): magic "TDVC" | >B n_coders | per coder: >4s name | >2I hyper-latent shape (h, w) | >B n_lists |
    per list: >I n_strings | per string: >I length | payload.
    frame={"size": (H, W), "N": N, "precision": "exact" | "mixed"} (version 2, what a decoder needs to reproduce the
    encoder exactly): magic "TDV2" | >2I H, W | >B N | >B precision (0 exact, 1 mixed) | >B n_coders | per coder: >4s name |
    >B cluster (CTAs per image of the autoregressive pass: its summation order) | then as version 1."""
    import struct
    if frame is None:
        out = [_MAGIC, struct.pack(">B", len(coded))]
    else:
        if frame.get("precision") not in _PRECISIONS:
            raise RuntimeError(f"pack_frame: precision must be one of {_PRECISIONS}, not {frame.get('precision')!r}")
        H, W = (int(v) for v in frame["size"])
        out = [_MAGIC_V2, struct.pack(">2IBBB", H, W, int(frame["N"]), _PRECISIONS.index(frame["precision"]), len(coded))]
    for name, enc in coded.items():
        head = struct.pack(">4s", name.encode()[:4].ljust(4))
        if frame is not None:
            if enc.get("cluster") not in (8, 16):
                raise RuntimeError(f"pack_frame: coder {name!r} has no cluster size (8 or 16)")
            head += struct.pack(">B", enc["cluster"])
        out.append(head + struct.pack(">2IB", int(enc["shape"][0]), int(enc["shape"][1]), len(enc["strings"])))
        for lst in enc["strings"]:
            out.append(struct.pack(">I", len(lst)))
            for s_ in lst:
                out.append(struct.pack(">I", len(s_)))
                out.append(bytes(s_))
    return b"".join(out)


def unpack_frame(data):
    """Inverse of pack_frame -> {name: {"strings": [[bytes, ...], ...], "shape": (h, w)}}; a version-2 container adds
    "cluster" to every coder and "frame": {"size": (H, W), "N": N, "precision": "exact" | "mixed"}.  A truncated or
    malformed container raises RuntimeError."""
    import struct
    if data[:4] not in (_MAGIC, _MAGIC_V2):
        raise RuntimeError("unpack_frame: not a tdvc_b200 frame container")
    v2 = data[:4] == _MAGIC_V2
    pos = 4
    out = {}
    try:
        if v2:
            H, W, N, prec, n = struct.unpack_from(">2IBBB", data, pos)
            pos += struct.calcsize(">2IBBB")
            if prec >= len(_PRECISIONS):
                raise RuntimeError(f"unpack_frame: unknown precision mode {prec}")
            frame = {"size": (H, W), "N": N, "precision": _PRECISIONS[prec]}
        else:
            (n,) = struct.unpack_from(">B", data, pos)
            pos += 1
        for _ in range(n):
            (name,) = struct.unpack_from(">4s", data, pos)
            pos += 4
            cluster = None
            if v2:
                (cluster,) = struct.unpack_from(">B", data, pos)
                pos += 1
                if cluster not in (8, 16):
                    raise RuntimeError(f"unpack_frame: cluster size {cluster} (8 or 16)")
            h, w, nl = struct.unpack_from(">2IB", data, pos)
            pos += struct.calcsize(">2IB")
            lists = []
            for _ in range(nl):
                (ns,) = struct.unpack_from(">I", data, pos)
                pos += 4
                strs = []
                for _ in range(ns):
                    (ln,) = struct.unpack_from(">I", data, pos)
                    pos += 4
                    if pos + ln > len(data):
                        raise RuntimeError("unpack_frame: truncated container")
                    strs.append(bytes(data[pos:pos + ln]))
                    pos += ln
                lists.append(strs)
            out[name.decode().strip()] = {"strings": lists, "shape": (h, w)}
            if v2:
                out[name.decode().strip()]["cluster"] = cluster
    except (struct.error, UnicodeDecodeError) as e:
        raise RuntimeError(f"unpack_frame: truncated or malformed container ({e})") from None
    if pos != len(data):
        raise RuntimeError("unpack_frame: trailing bytes")
    if v2:
        out["frame"] = frame
    return out

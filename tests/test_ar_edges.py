"""Edges of the y-latent entropy path that frames of the test sizes never reach: the wavefront encoder `tdvc_ar_code`
(csrc/coding.cu) and the device decoder `tdvc_ar_decode` (csrc/ar_decode.cu) on latents the tests build themselves.

* CPU: the schedule rules both kernels take from csrc/ar_common.cuh, compiled from the header itself into a host
  program: the wave / chunk walk, the chunk length the decoder re-derives, the causality of the context taps and the
  layer slices of a cluster.
* GPU: every Gaussian table and bin, escapes of 1-8 bypass digits and scales on the table entries (a context-free chain);
  degenerate, multi-chunk and strided shapes against the oracle's raster loop (oracle/compressai_port.py `ar_code`); three
  chunks per wave; batches with more clusters than the GPU holds at once and a per-image stream error; a 2560x1600 frame.

Decoding is lossless only if the decoder repeats the encoder's every mean, index and rANS step, so every decode here
must return the encoder's symbols, indexes and y_hat bit for bit."""
import copy
import ctypes as C
import subprocess

import numpy as np
import pytest
import torch

# ------------------------------------------------------------------------------------------------------ CPU
_SCHEDULE_CHECK = r"""
#include <cstdio>
#include <cstdarg>
#include <vector>
#include "ar_common.cuh"

namespace tdvc {
void set_error(const char*, ...) {}
}
using namespace tdvc;

#define FAIL(...) do { std::printf(__VA_ARGS__); std::printf("\n"); return 1; } while (0)

// every rule of the encoder's wavefront walk that the decoder must re-derive, for one latent shape
static int check_shape(int H, int W, long& multi_chunk_waves, int& longest) {
  std::vector<int> visits(H * W, 0), wave(H * W, -1);
  const int waves = W + 3 * (H - 1);
  for (int t = 0; t < waves; ++t) {
    int h_lo, h_hi;
    ar_wave_rows(t, H, W, h_lo, h_hi);
    if (h_hi - h_lo + 1 > longest) longest = h_hi - h_lo + 1;
    int chunks = 0;
    for (int hc = h_lo; hc <= h_hi; hc += AR_PCH) {   // the loop of ar_code_kernel
      const int P = ar_chunk_len(hc, h_hi);
      ++chunks;
      if (P < 1 || P > AR_PCH) FAIL("%dx%d wave %d: chunk of %d positions", H, W, t, P);
      for (int p = 0; p < P; ++p) {
        const int h = hc + p, w = t - 3 * h;
        if (h < 0 || h >= H || w < 0 || w >= W) FAIL("%dx%d wave %d: position (%d, %d) outside the latent", H, W, t, h, w);
        ++visits[h * W + w];
        wave[h * W + w] = t;
        const int Pd = ar_position_chunk_len(h, w, H, W);
        if (Pd != P) FAIL("%dx%d (%d, %d): coded in a chunk of %d, ar_position_chunk_len says %d", H, W, h, w, P, Pd);
      }
    }
    if (chunks > 1) ++multi_chunk_waves;
  }
  for (int i = 0; i < H * W; ++i)
    if (visits[i] != 1) FAIL("%dx%d (%d, %d) visited %d times", H, W, i / W, i % W, visits[i]);
  for (int h = 0; h < H; ++h)
    for (int w = 0; w < W; ++w)
      for (int ti = 0; ti < AR_TAPS; ++ti) {
        int dy, dx;
        ar_tap(ti, dy, dx);
        const int hh = h + dy, ww = w + dx;
        if (hh < 0 || hh >= H || ww < 0 || ww >= W) continue;
        if (wave[hh * W + ww] >= wave[h * W + w])
          FAIL("%dx%d (%d, %d): tap %d at (%d, %d) is not in an earlier wavefront", H, W, h, w, ti, hh, ww);
      }
  return 0;
}

// the slices of one layer over a cluster of R: each column once, in quads, at most AR_NS_MAX per CTA
static int check_layer(const TdvcArChain& a, ArLayer L, int total, int ldw, int R) {
  std::vector<int> owner(total, 0);
  for (int r = 0; r < R; ++r) {
    const ArW w = ar_layer(a, L, r, R);
    const int n = w.split ? w.split : w.ns;
    if (w.ns > AR_NS_MAX) FAIL("layer %d R=%d rank %d: %d columns", (int)L, R, r, w.ns);
    if (w.split && w.ns != 2 * w.split) FAIL("layer %d R=%d rank %d: %d columns for %d channels", (int)L, R, r, w.ns, n);
    if (w.n0 % 4 || (n % 4 && w.n0 + n != total)) FAIL("layer %d R=%d rank %d: slice [%d, +%d) not in quads", (int)L, R, r, w.n0, n);
    if (w.ldw != ldw) FAIL("layer %d: ldw %d", (int)L, w.ldw);
    for (int j = 0; j < w.ns; j += 4) {   // the last quad may reach into the padding, never past the row (ArW::col)
      const int col = w.split && j >= w.split ? AR_C + w.n0 + (j - w.split) : w.n0 + j;
      if (col + 4 > ldw) FAIL("layer %d R=%d rank %d: quad at column %d beyond the row", (int)L, R, r, col);
    }
    for (int j = 0; j < n; ++j) ++owner[w.n0 + j];
    // the encoder's warp tasks of this slice fit in the CTA for every chunk length
    for (int P = 1; P <= AR_PCH && w.ns > 0; ++P) {
      const int tasks = ((w.ns + 31) / 32) * ((P + AR_PT - 1) / AR_PT) * ar_ksplits(w.ns, P);
      if (tasks > AR_WARPS) FAIL("layer %d R=%d rank %d P=%d: %d warp tasks", (int)L, R, r, P, tasks);
    }
  }
  for (int c = 0; c < total; ++c)
    if (owner[c] != 1) FAIL("layer %d R=%d: column %d owned %d times", (int)L, R, c, owner[c]);
  return 0;
}

int main() {
  static const int Ws[] = {1,  2,  3,  4,  5,  6,  7,  8,  9,  10, 11, 12, 13, 14, 15, 16, 17, 18,
                           19, 20, 24, 31, 32, 33, 40, 41, 63, 64, 65, 97, 119, 120, 121, 122, 123, 124,
                           125, 127, 128, 129, 130, 160, 161, 191, 192, 200, 239, 240, 241, 243, 244, 245, 256, 260};
  for (int ti = 0; ti < AR_TAPS; ++ti) {   // tap ti = element ti of the 5x5 window in raster order (mask 'A')
    int dy, dx;
    ar_tap(ti, dy, dx);
    if (dy != ti / 5 - 2 || dx != ti % 5 - 2) FAIL("tap %d at (%d, %d)", ti, dy, dx);
  }
  long shapes = 0, multi = 0;
  int longest = 0;
  for (int H = 1; H <= 110; ++H)
    for (int W : Ws) {
      if (check_shape(H, W, multi, longest)) return 1;
      ++shapes;
    }
  for (int c1 : {426, 504}) {   // the model's widths and the widest ar_check_chain accepts
    const int c2 = c1 * 8 / 10;
    TdvcArChain a = {};
    a.c1 = c1;
    a.c2 = c2;
    a.c1_pad = (c1 + 7) & ~7;
    a.c2_pad = (c2 + 7) & ~7;
    for (int R : {8, 16}) {
      if (check_layer(a, AR_CTX, 2 * AR_C, 2 * AR_C, R) || check_layer(a, AR_EP0, c1, a.c1_pad, R) ||
          check_layer(a, AR_EP2, c2, a.c2_pad, R) || check_layer(a, AR_EP4, AR_C, 2 * AR_C, R))
        return 1;
    }
  }
  std::printf("shapes %ld multi_chunk_waves %ld longest_wave %d\n", shapes, multi, longest);
  return 0;
}
"""


def test_shared_schedule_rules_compiled_from_the_header(tmp_path):
    """The rules of csrc/ar_common.cuh that the encoder and the decoder both follow, checked on the header as compiled:
    for every H <= 110 and 54 widths up to 260 the encoder's wave / chunk loop visits every position exactly once,
    ar_position_chunk_len (the decoder's) returns the length of the chunk that coded the position, and the 12 context
    taps of every position lie in earlier wavefronts; ar_layer's slices cover each layer once, in quads, within
    AR_NS_MAX columns, for clusters of 8 and 16.  A rule changed for one kernel only fails here, without a GPU."""
    from tdvc_b200 import build
    src = tmp_path / "ar_schedule_check.cu"
    src.write_text(_SCHEDULE_CHECK)
    exe = tmp_path / "ar_schedule_check"
    r = subprocess.run([build.NVCC] + [f for f in build.FLAGS if f not in ("-Xptxas", "-v")] +
                       ["-I", build.CSRC, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    stats = dict(zip(*[iter(r.stdout.split())] * 2))
    assert int(stats["shapes"]) == 110 * 54
    assert int(stats["multi_chunk_waves"]) > 100000 and int(stats["longest_wave"]) > 2 * 40


# ------------------------------------------------------------------------------------------------------ GPU
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def oracle_model(oracle_model):
    """update() fills the coders' CDF buffers and test 1 edits weights: work on copies, the session's oracle stays as is."""
    return copy.deepcopy(oracle_model)


def _models(oracle_model, edit=None):
    """(oracle, net) holding one state_dict: the oracle's, changed by edit(sd), loaded into a deep copy of the oracle and
    into a VideoCompressor on cuda:0."""
    from tdvc_b200.model import VideoCompressor
    orc = copy.deepcopy(oracle_model)
    sd = {k: v.clone() for k, v in orc.state_dict().items()}
    if edit is not None:
        edit(sd)
    orc.load_state_dict(sd)
    net = VideoCompressor().eval()
    net.load_state_dict(sd, strict=True)
    return orc, net.to(DEV)


@pytest.fixture(scope="module")
def real(oracle_model):
    return _models(oracle_model)


def _coder(orc, net, cn):
    """Packed weights, tables (compressai `update(force=True)`) and the oracle coder of coder cn ("mv" | "rs")."""
    from tdvc_b200 import coding
    W = net._weights(DEV)
    coder = orc.mvCoder if cn == "mv" else orc.resCoder
    coder.update(force=True)
    return W, coding.CoderTables(W, cn, DEV), coder


@pytest.fixture(scope="module")
def latent_stats(real):
    """Per-channel mean and std of y and of the hyper-decoder output of both coders in a 128x192 forward."""
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


def _act(t, ld):
    """(N, h, w, C) -> a channels-last Act on cuda:0 with rows of ld floats; the padding holds NaN, which a kernel that
    reads past C would carry into its outputs."""
    from tdvc_b200.model import Act
    n, h, w, c = t.shape
    buf = torch.full((n, h, w, ld), float("nan"), device=DEV)
    buf[..., :c] = t.to(DEV)
    return Act(buf, buf.data_ptr(), n, h, w, c, ld)


def _latents(stats, cn, n, h, w, seed, y_ld=128, params_ld=256):
    """Seeded Gaussian y and hyper-decoder output with the per-channel statistics of a real frame; one y in 500 is an
    outlier of up to +-900, so that large y_hat values feed the predictions of later positions."""
    g = torch.Generator().manual_seed(seed)
    (ym, ys), (pm, ps) = stats[cn, "y"], stats[cn, "params"]
    y = torch.randn(n, h, w, 128, generator=g) * ys + ym
    p = torch.randn(n, h, w, 256, generator=g) * ps + pm
    k = torch.randint(0, y.numel(), (max(1, y.numel() // 500),), generator=g)
    y.view(-1)[k] = torch.rand(k.numel(), generator=g) * 1800 - 900
    return _act(y, y_ld), _act(p, params_ld)


def _encode(W, cn, tabs, y, params, cluster):
    """The y half of coding.launch_coding on the given latents: tdvc_ar_code with `cluster` CTAs per image, then the host
    rANS coder, one string per image."""
    from tdvc_b200 import coding
    from tdvc_b200 import lib as L
    lib = L.load()
    N, h, w = params.N, params.H, params.W
    out = (torch.empty((N, h, w, 128), device=DEV), torch.empty((N, h, w, 128), device=DEV, dtype=torch.int32),
           torch.empty((N, h, w, 128), device=DEV, dtype=torch.int32))
    chain = coding._ar_chain(W, cn, tabs, params, out, "ar_code")
    need = lib.tdvc_ar_code_workspace_bytes(N, chain.c1_pad, chain.c2_pad)
    ws = torch.empty(((need + 3) // 4,), device=DEV)
    used = C.c_int32(0)
    p = L.ArParams(chain=chain, y=y.ptr, y_ld=y.ld, cluster=cluster, cluster_used_host=C.addressof(used))
    L.check(lib.tdvc_ar_code(C.byref(p), ws.data_ptr(), need, torch.cuda.current_stream(DEV).cuda_stream), "ar_code")
    torch.cuda.synchronize(DEV)
    assert used.value == cluster
    y_hat, sym, idx = out
    sy, ix = sym.cpu().numpy(), idx.cpu().numpy()
    return {"y_hat": y_hat, "y_symbols": sym, "y_indexes": idx,
            "strings": [coding.rans_encode(sy[i], ix[i], tabs.gc) for i in range(N)]}


def _assert_same(enc, dec, what, keys=("y_symbols", "y_indexes", "y_hat")):
    for k in keys:
        if not torch.equal(enc[k], dec[k]):
            d = (enc[k] != dec[k]).reshape(-1).nonzero()
            first = np.unravel_index(int(d[0]), tuple(enc[k].shape))
            raise AssertionError(f"{what}: {k} differs at {first} ({int(d.numel())} elements)")


def _assert_lossless(W, cn, tabs, enc, params, cluster, what):
    from tdvc_b200 import coding
    dec = coding.decode_latents(W, cn, tabs, enc["strings"], params, cluster)
    _assert_same(enc, dec, f"{what}: decoded with cluster {cluster}")
    return dec


def _longest_wave(H, W):
    """Positions of the longest wavefront w + 3h = t of an H x W latent (ar_wave_rows)."""
    return max(min(t // 3, H - 1) - (max(0, t - W + 1) + 2) // 3 + 1 for t in range(W + 3 * (H - 1)))


def _nchw(a):
    return a.t[..., :a.C].permute(0, 3, 1, 2).cpu().contiguous()


def _off_ties(enc, y):
    """Moves y by 4e-3 towards its symbol wherever the kernel's y - mean lies within 2e-3 of a rounding tie.  The kernel's
    symbols, and so all later predictions, stay as they are; the oracle, whose means differ from the kernel's in the last
    bits, then cannot round such a position the other way and send the rest of the image down another path."""
    sym = enc["y_symbols"].float()
    r = y.t[..., :128] - (enc["y_hat"] - sym)
    near = ((r - torch.floor(r)) - 0.5).abs() < 2e-3
    y.t[..., :128] += torch.where(near, 4e-3 * torch.sign(sym - r), torch.zeros_like(r))
    return int(near.sum())


def _vs_oracle(coder, encs, y, params, what):
    """The kernel's symbols and indexes (one result per cluster size) against the oracle's raster loop (compressai
    `_compress_ar`) on the same latents; every difference is checked.  A symbol may differ only where the loop's own
    y - mean lies within 1e-4 of a rounding tie.  An index may differ only by one, where the scale lies so near the table
    entry between the two that fp32 rounding decides: the position's scale, evaluated in float64 from the loop's y_hat,
    within 1e-5 * S of that entry, S = |bias| + sum |w_i * h_i| over the scale's 341 products - the magnitude the error of
    an fp32 sum of them scales with (the rows cancel: S is tens of times the scale).  Where nothing differs the rANS
    strings are byte-identical.  Returns the number of excused elements."""
    import torch.nn.functional as F
    yc, pc = _nchw(y), _nchw(params)
    with torch.no_grad():
        o_str, o_sy, o_ix, o_yh = coder.ar_code(yc, pc)
    shape = tuple(encs[0]["y_symbols"].shape)
    o_sy, o_ix = np.asarray(o_sy, np.int32).reshape(shape), np.asarray(o_ix, np.int32).reshape(shape)
    tbl = coder.gaussian_conditional.scale_table.numpy().astype(np.float64)
    yp = F.pad(o_yh, (2, 2, 2, 2))
    mw = coder.context_prediction.weight * coder.context_prediction.mask
    c64 = {}

    def at(n, h, w):
        """(the loop's fp32 means, float64 scales, their S) of position (n, h, w): the loop's own step on its y_hat (the
        later positions it holds meet zero weights of the mask), and the same step in float64."""
        if not c64:
            c64["m"] = copy.deepcopy(coder).double()
            c64["mw"] = mw.double()
            c64["yp"], c64["pc"] = yp.double(), pc.double()
        m = c64["m"]
        with torch.no_grad():
            _, _, means = coder._ar_step(yp[n:n + 1], pc[n:n + 1], h, w, mw)
            ctx = F.conv2d(c64["yp"][n:n + 1, :, h:h + 5, w:w + 5], c64["mw"], bias=m.context_prediction.bias)
            ep = m.entropy_parameters
            x = ep[3](ep[2](ep[1](ep[0](torch.cat((c64["pc"][n:n + 1, :, h:h + 1, w:w + 1], ctx), 1)))))[0, :, 0, 0]
            terms = ep[4].weight[:128, :, 0, 0] * x
            scale = terms.sum(1) + ep[4].bias[:128]
            mag = terms.abs().sum(1) + ep[4].bias[:128].abs()
        return means[0].numpy(), scale.numpy(), mag.numpy()

    excused = 0
    for enc in encs:
        sy, ix = enc["y_symbols"].cpu().numpy(), enc["y_indexes"].cpu().numpy()
        bad_s, bad_i = np.argwhere(sy != o_sy), np.argwhere(ix != o_ix)
        for n, h, w, c in bad_s:
            r = yc[n, c, h, w].item() - float(at(n, h, w)[0][c])
            assert abs(abs(r - np.floor(r)) - 0.5) < 1e-4, (what, "symbol", (n, h, w, c), sy[n, h, w, c], o_sy[n, h, w, c], r)
        for n, h, w, c in bad_i:
            k = min(int(ix[n, h, w, c]), int(o_ix[n, h, w, c]))
            _, scale, mag = at(n, h, w)
            s64 = max(float(scale[c]), 0.11)
            assert abs(int(ix[n, h, w, c]) - int(o_ix[n, h, w, c])) == 1 and abs(s64 - tbl[k]) <= 1e-5 * mag[c], \
                (what, "index", (n, h, w, c), ix[n, h, w, c], o_ix[n, h, w, c], s64, tbl[k], mag[c])
        excused += len(bad_s) + len(bad_i)
        if not len(bad_s) and not len(bad_i):
            assert enc["strings"] == o_str, what
    return excused


# ---- 1. every table, every bin, every escape length
def _escape_digits(sym, index, tabs):
    """4-bit bypass digits of each symbol's escape (0: no escape), as tdvc_rans_encode_with_indexes writes them."""
    v = sym.astype(np.int64) - tabs.offset[index]
    mv = tabs.length[index] - 2
    raw = np.where(v < 0, -2 * v - 1, np.where(v >= mv, 2 * (v - mv), 0))
    digits = np.zeros(raw.shape, np.int64)
    while (raw > 0).any():
        digits += raw > 0
        raw >>= 4
    return digits


@pytest.mark.gpu
def test_every_table_bin_and_escape(oracle_model, latent_stats):
    """A context-free chain (the context model's weight and the scale rows of entropy_parameters.4 zeroed): each scale is
    exactly its bias, and the means depend on the hyper-decoder output only.  The biases put the 128 channels on every
    scale-table entry, one ulp above and below each, below the 0.11 floor, at 0 and at 1e6, so that every one of the 64
    Gaussian rows is coded, the 3,133-entry rows included.  One pass gives the means; y = mean + target then makes each
    channel code every in-range bin of its row, the smallest escape on both sides and escapes of +-2^k (k = 1..30: one to
    eight bypass digits).  The indexes must be compressai's build_indexes, the symbols the targets (above 2^22, where
    mean + target is not exact in fp32, the oracle loop's), the string the oracle's, and the device decoder must return
    everything bit for bit for encoder clusters of 8 and 16."""
    from oracle import rans
    from tdvc_b200 import coding
    T = coding.scale_table().numpy()
    up, down = np.nextafter(T, np.float32(np.inf)), np.nextafter(T, np.float32(-np.inf))
    rounds = [np.concatenate([T, up]), np.concatenate([down, np.float32([0.05, 0.0, 1e6]), T[:61]])]
    seen_idx, max_digits = set(), 0
    for rnd, scales in enumerate(rounds):
        def edit(sd):
            sd["mvCoder.context_prediction.weight"].zero_()
            sd["mvCoder.entropy_parameters.4.weight"][:128].zero_()
            sd["mvCoder.entropy_parameters.4.bias"][:128] = torch.from_numpy(scales)
        orc, net = _models(oracle_model, edit)
        W, tabs, coder = _coder(orc, net, "mv")
        gc = tabs.gc
        _, params = _latents(latent_stats, "mv", 1, 60, 60, seed=100 + rnd)
        want_idx = coder.gaussian_conditional.build_indexes(torch.from_numpy(scales)[None]).numpy()[0]
        e0 = _encode(W, "mv", tabs, _act(torch.zeros(1, 60, 60, 128), 128), params, 16)
        assert (e0["y_indexes"].cpu().numpy() == want_idx).all(), rnd
        mean = e0["y_hat"] - e0["y_symbols"].float()   # exact: y = 0 leaves |y_hat| <= 0.5
        # targets per channel: every in-range symbol of its row, max_value and -1 (the smallest escapes), +-2^k
        g = np.random.default_rng(rnd)
        tgt = np.zeros((3600, 128), np.int64)
        for c in range(128):
            i = want_idx[c]
            mv, off = int(gc.length[i]) - 2, int(gc.offset[i])
            t = np.concatenate([off + np.arange(mv), [off + mv, off - 1], 2 ** np.arange(1, 31), -2 ** np.arange(1, 31)])
            t = np.concatenate([t, off + np.arange(3600 - t.size) % mv])
            tgt[:, c] = g.permutation(t)
        tgt = tgt.reshape(1, 60, 60, 128)
        y = _act(torch.zeros(1, 60, 60, 128), 128)
        y.t.copy_(mean + torch.from_numpy(tgt).float().to(DEV))
        encs = {cl: _encode(W, "mv", tabs, y, params, cl) for cl in (16, 8)}
        exact = np.abs(tgt) < 2 ** 22
        for cl, enc in encs.items():
            sy, ix = enc["y_symbols"].cpu().numpy(), enc["y_indexes"].cpu().numpy()
            assert (ix == want_idx).all(), (rnd, cl)
            assert (sy[exact] == tgt[exact]).all(), (rnd, cl)
            assert np.array_equal(coding.rans_decode(enc["strings"][0], ix[0], gc), sy[0].reshape(-1)), (rnd, cl)
            _assert_lossless(W, "mv", tabs, enc, params, cl, f"round {rnd}")
            seen_idx |= set(np.unique(ix).tolist())
            max_digits = max(max_digits, int(_escape_digits(sy, ix, gc).max()))
        if _vs_oracle(coder, list(encs.values()), y, params, f"round {rnd}"):   # a tie at 2^22: the string by itself
            for cl, enc in encs.items():
                sy, ix = enc["y_symbols"].cpu().numpy(), enc["y_indexes"].cpu().numpy()
                cdf, lens, offs = coder.gaussian_conditional._tables()
                assert enc["strings"][0] == rans.encode_with_indexes(sy[0].reshape(-1).tolist(), ix[0].reshape(-1).tolist(),
                                                                     cdf, lens, offs), (rnd, cl)
    assert seen_idx == set(range(64)) and max_digits == 8


# ---- 2. shapes against the oracle's raster loop
@pytest.mark.gpu
@pytest.mark.parametrize("n,h,w,lds", [(1, 1, 1, None), (1, 1, 9, None), (1, 9, 1, None), (1, 2, 2, None),
                                       (3, 3, 5, None), (1, 5, 3, None), (1, 2, 130, (132, 260)), (1, 44, 128, None)])
def test_shapes_against_the_oracle_loop(real, latent_stats, n, h, w, lds):
    """Latents of one position, one row, one column, W <= 2 (no (h - 1, w + 2) neighbour), a batch of 3, strided y and
    hyper-decoder rows, and 44x128 (waves of 43 positions: a chunk of 40 and one of 3), coded with the real weights:
    symbols and indexes against the oracle's raster loop, lossless decoding for clusters of 8 and 16.  At 44x128, strings
    coded with 16 CTAs and decoded as if coded with 8 must not come back bit for bit: the lossless check sees the
    summation order at that shape."""
    from tdvc_b200 import coding
    orc, net = real
    y_ld, params_ld = lds or (128, 256)
    excused = 0
    for cn in ("mv", "rs"):
        W, tabs, coder = _coder(orc, net, cn)
        y, params = _latents(latent_stats, cn, n, h, w, seed=7 * h + w, y_ld=y_ld, params_ld=params_ld)
        first = _encode(W, cn, tabs, y, params, 16)
        _off_ties(first, y)
        encs = {cl: _encode(W, cn, tabs, y, params, cl) for cl in (16, 8)}
        _assert_same(first, encs[16], f"{cn} {h}x{w} off ties", keys=("y_symbols", "y_hat"))
        excused += _vs_oracle(coder, list(encs.values()), y, params, f"{cn} {n}x{h}x{w}")
        for cl, enc in encs.items():
            assert torch.isfinite(enc["y_hat"]).all()
            _assert_lossless(W, cn, tabs, enc, params, cl, f"{cn} {n}x{h}x{w}")
        if (h, w) == (44, 128):
            assert _longest_wave(h, w) == 43
            try:
                wrong = coding.decode_latents(W, cn, tabs, encs[16]["strings"], params, 8)
                assert not torch.equal(wrong["y_hat"], encs[16]["y_hat"]), cn
            except RuntimeError:
                pass
    print(f"{n}x{h}x{w}: {excused} symbols / indexes excused as ties")


# ---- 3. three chunks per wave
@pytest.mark.gpu
def test_three_chunks_per_wave_decode(real, latent_stats):
    """84x244: waves of 82 positions, coded as chunks of 40 + 40 + 2; both coders decode losslessly for both encoder
    cluster sizes (no host oracle: its loop would take minutes here)."""
    orc, net = real
    assert _longest_wave(84, 244) == 82
    for cn in ("mv", "rs"):
        W, tabs, _ = _coder(orc, net, cn)
        y, params = _latents(latent_stats, cn, 1, 84, 244, seed=3)
        for cl in (8, 16):
            _assert_lossless(W, cn, tabs, _encode(W, cn, tabs, y, params, cl), params, cl, f"{cn} 84x244")


# ---- 4. batches and per-image errors
@pytest.mark.gpu
def test_batch_is_independent_and_errors_stay_per_image(real, latent_stats):
    """Ten distinct images in clusters of 16: more CTAs than the GPU has SMs, so clusters wait for others to finish.  Each
    image's symbols, indexes, y_hat and string from the batched encode equal those of coding it alone, and so do the
    batched decode's.  With image 6's string truncated, only image 6 reports a broken stream and the other nine decode
    exactly."""
    from tdvc_b200 import coding
    orc, net = real
    N = 10
    assert N * 16 > torch.cuda.get_device_properties(DEV).multi_processor_count
    W, tabs, _ = _coder(orc, net, "rs")
    y, params = _latents(latent_stats, "rs", N, 7, 11, seed=11)
    enc = _encode(W, "rs", tabs, y, params, 16)
    dec = _assert_lossless(W, "rs", tabs, enc, params, 16, "batch of 10")
    for i in range(N):
        one = _encode(W, "rs", tabs, y.batch(i), params.batch(i), 16)
        part = {k: enc[k][i:i + 1] for k in ("y_symbols", "y_indexes", "y_hat")}
        _assert_same(part, one, f"image {i} coded alone")
        assert one["strings"][0] == enc["strings"][i], i
        _assert_same(one, coding.decode_latents(W, "rs", tabs, one["strings"], params.batch(i), 16), f"image {i} alone")
        _assert_same(part, {k: dec[k][i:i + 1] for k in part}, f"image {i} in the batched decode")
    strings = list(enc["strings"])
    strings[6] = strings[6][:len(strings[6]) // 8 * 4]
    h = coding.launch_decoding(W, "rs", tabs, strings, params, 16)
    h["done"].synchronize()
    status = h["status"].tolist()
    assert status[6] >= 0 and all(s == -1 for i, s in enumerate(status) if i != 6), status
    for i in (i for i in range(N) if i != 6):
        _assert_same({k: enc[k][i] for k in ("y_symbols", "y_indexes", "y_hat")},
                     {k: h[k][i] for k in ("y_symbols", "y_indexes", "y_hat")}, f"image {i} beside a broken one")


# ---- 5. a real frame with multi-chunk waves
@pytest.mark.gpu
def test_2560x1600_frame_round_trip(real):
    """HEVC class A size: a 100x160 latent with waves of up to 54 positions.  forward(is_compress=True), a version-2
    container, and both coders decode losslessly with the recorded cluster size and with strings coded at the other
    size; every y string decodes on the host to the coded symbols."""
    from tdvc_b200 import coding, synth
    _, net = real
    x, refs = synth.make_frame_pair(1600, 2560, seed=5)
    gt = {}
    with torch.no_grad():
        net(x.to(DEV), refs.to(DEV), False, is_compress=True, taps=gt)
    assert _longest_wave(100, 160) == 54
    W = net._weights(DEV)
    plan = net._plan(1, 1600, 2560, DEV)
    frame = {"size": (1600, 2560), "N": 1, "precision": "exact"}
    back = coding.unpack_frame(coding.pack_frame(net.last_coded, frame=frame))
    assert back["frame"] == frame
    for nm, cn in (("mv", "mv"), ("res", "rs")):
        tabs = W["_tables"][cn]
        params = plan.buf(f"{cn}.params", 1, 100, 160, 256)
        cl = back[nm]["cluster"]
        enc = {k: gt[f"{nm}.ac.{k}"] for k in ("y_symbols", "y_indexes", "y_hat")}
        assert enc["y_symbols"].shape == (1, 100, 160, 128)
        enc["strings"] = back[nm]["strings"][0]
        other = coding.code_latents(plan, W, cn, tabs, cluster=24 - cl, keep=True)
        assert other["cluster"] == 24 - cl
        for c, e in ((cl, enc), (24 - cl, {**other, "strings": other["strings"][0]})):
            sy, ix = e["y_symbols"].cpu().numpy(), e["y_indexes"].cpu().numpy()
            assert np.array_equal(coding.rans_decode(e["strings"][0], ix[0], tabs.gc), sy[0].reshape(-1)), (nm, c)
            _assert_lossless(W, cn, tabs, e, params, c, f"{nm} 2560x1600")

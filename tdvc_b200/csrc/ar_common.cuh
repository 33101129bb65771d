// The arithmetic of the autoregressive entropy-parameter chain (context model -> ep0 -> ep2 -> ep4), shared by the encoder
// (ar_code_kernel, csrc/coding.cu) and the decoder (ar_decode_kernel, csrc/ar_decode.cu).
//
// A decoder reproduces the encoder's symbols only if it computes, at every latent position, the same scale index and the
// same mean bit for bit: one flipped index desynchronises the rANS stream for the rest of the image, one ulp in a mean
// changes y_hat and through it every later prediction.  The encoder's fp32 summation order is not a fixed function of the
// position: it splits K over KS warps, and KS depends on the number of positions P of the wavefront chunk the position is
// coded in and on the width of the column slice of the cluster CTA that owns the output channel (so on the cluster size).
// Every rule that fixes that order lives here, and both kernels call these helpers.  So do the other things the two sides
// must agree on: the layers' slicing over the cluster (ar_layer), the rANS stream format and its escape decode
// (rans_symbol, shared with the host decoder), the host checks of the chain and the cluster launch.
#pragma once
#include "common.cuh"

namespace tdvc {

constexpr int AR_THREADS = 512;
constexpr int AR_WARPS = AR_THREADS / 32;
constexpr int AR_PT = 8;        // positions per warp task (register tile)
constexpr int AR_PCH = 40;      // positions per chunk of a wavefront (1920x1024: 64x120 latent, <= 40 per wavefront)
constexpr int AR_KS_MAX = 16;   // K splits per (channel group, position group): a short wavefront still keeps every warp busy
constexpr int AR_NS_MAX = 64;   // output channels of one CTA per stage
constexpr int AR_C = 128;       // latent channels (Cheng2020Anchor N = M = 128 in both coders)
constexpr int AR_KC = 128;      // K chunk staged in shared memory (one tap of the context model)
constexpr int AR_TAPS = 12;     // live taps of the 5x5 mask 'A': the first 12 in raster order, tap 11 = (h, w - 1)

// columns [n0, n1) of `total` owned by CTA `rank` of a cluster of R (multiples of `align`)
__host__ __device__ __forceinline__ void ar_slice(int total, int align, int rank, int R, int& n0, int& n1) {
  const int q = (total + align - 1) / align;
  n0 = align * (int)((int64_t)q * rank / R);
  n1 = align * (int)((int64_t)q * (rank + 1) / R);
  if (n1 > total) n1 = total;
  if (n0 > total) n0 = total;
}

// One layer of the chain as a CTA sees it: its weight columns of Wt[K][ldw], as one or two runs of 16-byte quads:
// [n0, n0 + ns) for the first three layers; for the last one (split = number of latent channels of this CTA) the scale
// columns [n0, n0 + split) followed by the mean columns [AR_C + n0, AR_C + n0 + split), so that both parameters of a latent
// channel land in the same CTA.  n0, split and ldw are multiples of 4 (the last quad of a layer may reach into the
// zero-padded columns).
struct ArW {
  const float* Wt;
  int ldw, K, n0, ns, split;
  __device__ __forceinline__ int col(int n) const { return split && n >= split ? AR_C + n0 + (n - split) : n0 + n; }
};

// the layers of the chain: context model (the 12 live taps of mask 'A', weight row = tap * C + c), entropy_parameters[0]
// ((params | ctx) -> c1), [2] (c1 -> c2) and [4] (c2 -> (scales | means))
enum ArLayer { AR_CTX, AR_EP0, AR_EP2, AR_EP4 };

// layer L as CTA `rank` of a cluster of R sees it; called with a constant L, so that each layer stays a named value
__host__ __device__ __forceinline__ ArW ar_layer(const TdvcArChain& a, ArLayer L, int rank, int R) {
  int n0, n1;
  switch (L) {
    case AR_CTX: ar_slice(2 * AR_C, 4, rank, R, n0, n1); return {a.w_ctx, 2 * AR_C, AR_TAPS * AR_C, n0, n1 - n0, 0};
    case AR_EP0: ar_slice(a.c1, 4, rank, R, n0, n1); return {a.w1, a.c1_pad, 4 * AR_C, n0, n1 - n0, 0};
    case AR_EP2: ar_slice(a.c2, 4, rank, R, n0, n1); return {a.w2, a.c2_pad, (a.c1 + 3) & ~3, n0, n1 - n0, 0};
    default:     // AR_EP4, latent channels [n0, n1) of this CTA
      ar_slice(AR_C, 4, rank, R, n0, n1);
      return {a.w3, 2 * AR_C, (a.c2 + 3) & ~3, n0, 2 * (n1 - n0), n1 - n0};
  }
}

// number of K splits of a stage whose CTA computes `ns` output columns for P positions
__host__ __device__ __forceinline__ int ar_ksplits(int ns, int P) {
  const int NG = (ns + 31) >> 5, PG = (P + AR_PT - 1) / AR_PT;
  const int KS = AR_WARPS / (NG * PG);
  return KS < 1 ? 1 : (KS > AR_KS_MAX ? AR_KS_MAX : KS);
}

// quads [q0, q1) of a K chunk of nq quads that split ks of KS accumulates
__device__ __forceinline__ void ar_split_quads(int nq, int ks, int KS, int& q0, int& q1) {
  q0 = nq * ks / KS;
  q1 = nq * (ks + 1) / KS;
}

// quads in K chunk c of a layer of depth K
__device__ __forceinline__ int ar_chunk_quads(int K, int c) {
  const int k0 = c * AR_KC;
  return (K - k0 < AR_KC ? K - k0 : AR_KC) >> 2;
}

// one quad of a split's accumulation chain, in the order of the A operand's components
__device__ __forceinline__ float ar_fma4(float acc, float4 a, float w0, float w1, float w2, float w3) {
  acc = fmaf(a.x, w0, acc);
  acc = fmaf(a.y, w1, acc);
  acc = fmaf(a.z, w2, acc);
  acc = fmaf(a.w, w3, acc);
  return acc;
}

// sum of the KS split partials, in split order
template <class Part>
__device__ __forceinline__ float ar_reduce(int KS, Part part) {
  float v = part(0);
  for (int ks = 1; ks < KS; ++ks) v += part(ks);
  return v;
}

__device__ __forceinline__ float ar_lrelu(float v) { return v > 0.f ? v : v * 0.01f; }

// table index of a predicted scale (GaussianConditional.build_indexes after the 0.11 lower bound); table = the first
// n_cmp = n_scales - 1 entries of the scale table
__device__ __forceinline__ int ar_scale_index(float scale, const float* table, int n_cmp) {
  scale = fmaxf(scale, 0.11f);
  int ix = 0;
  for (int s = 0; s < n_cmp; ++s) ix += table[s] < scale ? 1 : 0;
  return ix;
}

// The wavefronts of the encoder: position (h, w) is coded in wavefront t = w + 3h, which holds rows [h_lo, h_hi], walked
// in chunks of <= AR_PCH positions starting at h_lo.  ar_position_chunk_len = P of the chunk that holds (h, w).
__host__ __device__ __forceinline__ void ar_wave_rows(int t, int H, int W, int& h_lo, int& h_hi) {
  h_lo = t - (W - 1);
  h_lo = h_lo <= 0 ? 0 : (h_lo + 2) / 3;
  h_hi = t / 3;
  if (h_hi > H - 1) h_hi = H - 1;
}
__host__ __device__ __forceinline__ int ar_chunk_len(int hc, int h_hi) {
  return (h_hi - hc + 1) < AR_PCH ? (h_hi - hc + 1) : AR_PCH;
}
__host__ __device__ __forceinline__ int ar_position_chunk_len(int h, int w, int H, int W) {
  int h_lo, h_hi;
  ar_wave_rows(w + 3 * h, H, W, h_lo, h_hi);
  const int hc = h_lo + (h - h_lo) / AR_PCH * AR_PCH;
  return ar_chunk_len(hc, h_hi);
}

// (dy, dx) of tap ti of the context model
__host__ __device__ __forceinline__ void ar_tap(int ti, int& dy, int& dx) {
  dy = ti < 5 ? -2 : (ti < 10 ? -1 : 0);
  dx = ti < 10 ? (ti - (ti < 5 ? 0 : 5)) - 2 : ti - 12;
}

// ---- the rANS stream (ryg_rans rans64 + compressai's bypass escape): written by tdvc_rans_encode_with_indexes, read by
// tdvc_rans_decode_with_indexes on the host and by ar_decode_kernel on the device
constexpr uint64_t RANS64_L = 1ull << 31;   // lower bound of the 64-bit state
constexpr int RANS_PRECISION = 16, RANS_BYPASS = 4;
constexpr uint32_t RANS_MAX_BYPASS = (1u << RANS_BYPASS) - 1;

// The symbol of decoded bin s of a CDF row with max_value = length - 2 and `offset`.  s == max_value is an escape: the
// digit count in unary by 15, then the digits of the folded value, least significant first; bits(v) reads the next
// RANS_BYPASS bits into v (false: the stream ended).  false: truncated stream, more than 16 digits, or a symbol outside
// int32 - none of which the encoder writes.
template <class Bits>
__host__ __device__ __forceinline__ bool rans_symbol(int s, int max_value, int32_t offset, Bits bits, int32_t& sym) {
  int64_t value = s;
  if (s == max_value) {
    uint32_t v;
    if (!bits(v)) return false;
    int n_bypass = (int)v;
    while (v == RANS_MAX_BYPASS) {
      if (n_bypass > 16 || !bits(v)) return false;
      n_bypass += (int)v;
    }
    if (n_bypass > 16) return false;
    uint64_t raw = 0;
    for (int j = 0; j < n_bypass; ++j) {
      if (!bits(v)) return false;
      raw |= (uint64_t)v << (j * RANS_BYPASS);
    }
    if ((raw >> 1) > (1ull << 32)) return false;
    value = (int64_t)(raw >> 1);
    if (raw & 1) value = -value - 1;
    else value += max_value;
  }
  value += offset;
  if (value < INT32_MIN || value > INT32_MAX) return false;
  sym = (int32_t)value;
  return true;
}

// ---- host side of tdvc_ar_code and tdvc_ar_decode

// what both entry points require of the chain
static inline int ar_check_chain(const TdvcArChain& a, const char* who) {
  TDVC_REQUIRE(a.params && a.w_ctx && a.b_ctx && a.w1 && a.b1 && a.w2 && a.b2 && a.w3 && a.b3 && a.scale_table && a.y_hat &&
                   a.symbols && a.indexes, "%s: null pointer in the chain", who);
  TDVC_REQUIRE(a.C == AR_C, "%s: C=%d (only %d latent channels)", who, a.C, AR_C);
  TDVC_REQUIRE(a.N > 0 && a.H > 0 && a.W > 0, "%s: bad shape", who);
  TDVC_REQUIRE(a.params_ld >= 2 * AR_C && a.params_ld % 4 == 0, "%s: bad leading dimension of params", who);
  // (c1 + 7) / 8 + 1 <= AR_NS_MAX: a CTA of a cluster of 8 holds its slice of c1 (c1 <= 504)
  TDVC_REQUIRE(a.c1 >= 16 && a.c2 >= 16 && a.c2 <= a.c1 && (a.c1 + 7) / 8 + 1 <= AR_NS_MAX && a.c1_pad % 4 == 0 &&
                   a.c1_pad >= ((a.c1 + 3) & ~3) && a.c2_pad % 4 == 0 && a.c2_pad >= ((a.c2 + 3) & ~3),
               "%s: hidden widths %d, %d (padded %d, %d)", who, a.c1, a.c2, a.c1_pad, a.c2_pad);
  TDVC_REQUIRE(a.n_scales >= 2 && a.n_scales <= 65, "%s: scale table of %d entries", who, a.n_scales);
  return TDVC_OK;
}

// Kernel(arg) on N clusters of R CTAs of AR_THREADS threads with `smem` bytes of dynamic shared memory (R = 16 is a
// non-portable cluster size).  With `fallback`, clusters of 16 that cannot launch become clusters of 8.  R receives the
// size launched.
template <auto Kernel, class Arg>
static inline int ar_launch_clusters(const Arg& arg, int N, int& R, bool fallback, size_t smem, cudaStream_t st,
                                     const char* who) {
  static int smem_done[kMaxDevices] = {};
  const int rc = ensure_dynamic_smem(Kernel, smem, smem_done, who);
  if (rc != TDVC_OK) return rc;
  for (;;) {
    cudaError_t e = cudaSuccess;
    if (R > 8) e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e == cudaSuccess) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)(N * R));
      cfg.blockDim = dim3(AR_THREADS);
      cfg.dynamicSmemBytes = smem;
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)R;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      e = cudaLaunchKernelEx(&cfg, Kernel, arg);
    }
    if (e == cudaSuccess) return TDVC_OK;
    (void)cudaGetLastError();
    if (!fallback || R == 8) {
      set_error("%s: launch with clusters of %d CTAs failed: %s", who, R, cudaGetErrorString(e));
      return TDVC_ECUDA;
    }
    R = 8;
  }
}

}  // namespace tdvc

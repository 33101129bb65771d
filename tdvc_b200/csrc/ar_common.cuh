// The arithmetic of the autoregressive entropy-parameter chain (context model -> ep0 -> ep2 -> ep4), shared by the encoder
// (ar_code_kernel, csrc/coding.cu) and the decoder (ar_decode_kernel, csrc/ar_decode.cu).
//
// A decoder reproduces the encoder's symbols only if it computes, at every latent position, the same scale index and the
// same mean bit for bit: one flipped index desynchronises the rANS stream for the rest of the image, one ulp in a mean
// changes y_hat and through it every later prediction.  The encoder's fp32 summation order is not a fixed function of the
// position: it splits K over KS warps, and KS depends on the number of positions P of the wavefront chunk the position is
// coded in and on the width of the column slice of the cluster CTA that owns the output channel (so on the cluster size).
// Every rule that fixes that order lives here, and both kernels call these helpers.
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

}  // namespace tdvc

// Decoding of the y latent (compressai `JointAutoregressiveHierarchicalPriors._decompress_ar` + the `ans` decoder): the
// inverse of ar_code_kernel (csrc/coding.cu).
//
// The string is in raster (h, w, c) order and position (h, w) is predicted from y_hat(h, w - 1), so decoding is H * W
// dependent steps per image: the encoder's wavefront parallelism does not exist here.  One thread-block cluster per image;
// each CTA owns a slice of the output channels of every layer and streams its weight columns from L2 (3.39 MB for the
// four layers, a 16th per CTA).  Per step: gather the 12 context taps, context model -> ep0 -> ep2 -> ep4 (each layer's
// outputs are written into every CTA's shared memory, one cluster barrier per layer), then warp 0 of CTA 0 decodes the 128
// symbols of the position from the rANS stream (Gaussian CDF rows in its shared memory, 32-ary warp search) and writes
// y_hat = symbol + mean.
//
// Bit-exactness with the encoder: every output channel is accumulated with the encoder's K splits for that channel and
// position (ar_ksplits of the encoder CTA's column count and of the wavefront chunk length), each split as the encoder's
// fmaf chain over the same K chunks and quads, the splits summed in order, then bias, LeakyReLU, the 0.11 floor and the
// index count: the helpers of ar_common.cuh, which ar_code_kernel calls too.
#include <cooperative_groups.h>
#include "ar_common.cuh"

namespace cg = cooperative_groups;

namespace tdvc {

constexpr int ARD_CDF_MAX = 32768;   // CDF entries held in shared memory (64 Gaussian rows: 27,256)
constexpr int ARD_NO_MAX = 64;       // outputs of one layer per CTA (clusters of >= 8 CTAs, c1 <= 512)
constexpr int ARD_IN_MAX = 512;      // widest layer input (ep0: params | ctx)
// Dynamic shared memory holds the CDF rows, which only CTA 0 reads.  A launch has one dynamic size for all its CTAs, and
// the reservation costs nothing: at 512 threads x 110 registers one CTA fills an SM's register file, and 128 KB + 20 KB
// of static shared memory fit beside it.
constexpr size_t ARD_SMEM = (size_t)ARD_CDF_MAX * sizeof(int32_t);

// split partials of this CTA's outputs of layer w for one position: part[ks][nl] = the encoder's fmaf chain of split ks of
// output nl; in(k) = float4 of the layer input at k .. k + 3 (shared memory)
template <class In>
__device__ __forceinline__ void ard_partials(const ArW& w, const int* ns_enc, int P, float* part, In in) {
  const int nchunks = (w.K + AR_KC - 1) / AR_KC;
  for (int i = threadIdx.x; i < AR_KS_MAX * w.ns; i += AR_THREADS) {
    const int ks = i / w.ns, nl = i - ks * w.ns;
    const int KS = ar_ksplits(ns_enc[nl], P);
    if (ks >= KS) continue;
    const float* wc = w.Wt + w.col(nl);
    float acc = 0.f;
    for (int c = 0; c < nchunks; ++c) {
      int q0, q1;
      ar_split_quads(ar_chunk_quads(w.K, c), ks, KS, q0, q1);
#pragma unroll 4
      for (int q = q0; q < q1; ++q) {
        const int k = c * AR_KC + 4 * q;
        const float* wk = wc + (int64_t)k * w.ldw;
        acc = ar_fma4(acc, in(k), __ldg(wk), __ldg(wk + w.ldw), __ldg(wk + 2 * w.ldw), __ldg(wk + 3 * w.ldw));
      }
    }
    part[ks * ARD_NO_MAX + nl] = acc;
  }
}

// the encoder's in-order sum over the splits + bias of output nl
__device__ __forceinline__ float ard_output(const ArW& w, const float* bias, const int* ns_enc, int P, const float* part, int nl) {
  const int KS = ar_ksplits(ns_enc[nl], P);
  return ar_reduce(KS, [&](int ks) { return part[ks * ARD_NO_MAX + nl]; }) + __ldg(bias + w.col(nl));
}

// outputs of this CTA (after bias and activation) into dst[w.n0 + nl] of every CTA of the cluster
template <bool LRELU>
__device__ __forceinline__ void ard_publish(cg::cluster_group& cluster, int RD, const ArW& w, const float* bias,
                                            const int* ns_enc, int P, const float* part, float* out, float* dst) {
  for (int nl = threadIdx.x; nl < w.ns; nl += AR_THREADS) {
    const float v = ard_output(w, bias, ns_enc, P, part, nl);
    out[nl] = LRELU ? ar_lrelu(v) : v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < RD * w.ns; i += AR_THREADS) {
    const int r = i / w.ns, nl = i - r * w.ns;
    cluster.map_shared_rank(dst, r)[w.n0 + nl] = out[nl];
  }
}

__global__ void __launch_bounds__(AR_THREADS, 1) ar_decode_kernel(const TdvcArDecodeParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int RD = (int)cluster.num_blocks();
  const int rank = (int)cluster.block_rank();
  const int n = blockIdx.x / RD;
  const TdvcArChain& a = p.chain;
  const int H = a.H, W = a.W;
  constexpr int C = AR_C, C2 = 2 * AR_C;
  extern __shared__ __align__(16) int32_t ard_cdf[];   // [cdf_total]: the CDF rows back to back (CTA 0)
  __shared__ __align__(16) float s_taps[AR_TAPS * C];  // context-model input: the 12 causal taps of y_hat
  __shared__ __align__(16) float s_in1[2 * C2];        // ep0 input: params | ctx
  __shared__ __align__(16) float s_in2[ARD_IN_MAX];    // ep2 input (zero beyond c1)
  __shared__ __align__(16) float s_in3[ARD_IN_MAX];    // ep4 input (zero beyond c2)
  __shared__ float s_part[AR_KS_MAX * ARD_NO_MAX];
  __shared__ float s_out[ARD_NO_MAX];
  __shared__ int s_ns[4][ARD_NO_MAX];
  __shared__ float s_table[64];
  __shared__ float s_mean[C];                          // CTA 0: means and table indexes of the position
  __shared__ int s_idx[C];
  __shared__ int s_sym[C];
  __shared__ int s_row[AR_TABLES_MAX + 1], s_len[AR_TABLES_MAX], s_off[AR_TABLES_MAX];
  __shared__ int s_stop;                               // written by CTA 0 into every CTA: stop decoding this image

  const ArW wA = ar_layer(a, AR_CTX, rank, RD), wB = ar_layer(a, AR_EP0, rank, RD), wC = ar_layer(a, AR_EP2, rank, RD),
            wD = ar_layer(a, AR_EP4, rank, RD);
  // column count of the encoder CTA (of a cluster of p.cluster) that owns output j of this CTA's layer L: it fixes the
  // output's K splits
  auto encoder_ns = [&](ArLayer L, const ArW& w, int j) {
    const int ch = w.n0 + (w.split && j >= w.split ? j - w.split : j);   // ep4: the latent channel of a scale or mean
    for (int r = 0; r < p.cluster; ++r) {
      const ArW e = ar_layer(a, L, r, p.cluster);
      if (ch >= e.n0 && ch < e.n0 + (e.split ? e.split : e.ns)) return e.ns;
    }
    return 0;
  };
  for (int i = threadIdx.x; i < ARD_NO_MAX; i += AR_THREADS) {
    s_ns[AR_CTX][i] = i < wA.ns ? encoder_ns(AR_CTX, wA, i) : 0;
    s_ns[AR_EP0][i] = i < wB.ns ? encoder_ns(AR_EP0, wB, i) : 0;
    s_ns[AR_EP2][i] = i < wC.ns ? encoder_ns(AR_EP2, wC, i) : 0;
    s_ns[AR_EP4][i] = i < wD.ns ? encoder_ns(AR_EP4, wD, i) : 0;
  }
  for (int i = threadIdx.x; i < ARD_IN_MAX; i += AR_THREADS) s_in2[i] = s_in3[i] = 0.f;
  for (int i = threadIdx.x; i < a.n_scales - 1; i += AR_THREADS) s_table[i] = a.scale_table[i];
  const int n_cmp = a.n_scales - 1;

  ArdRans rs{};
  const bool coder = rank == 0 && threadIdx.x < 32;
  if (rank == 0) {
    if (threadIdx.x == 0) {
      const bool ok = ar_cdf_rows(p, s_row, s_len, s_off);
      const int64_t w0 = p.word_offsets[n], w1 = p.word_offsets[n + 1];
      s_stop = ok && w1 - w0 >= 2 ? 0 : 1;
      p.status[n] = !ok ? AR_BAD_TABLES : (s_stop ? 0 : AR_DECODED);
    }
    __syncthreads();
    if (!s_stop) {
      for (int t = 0; t < p.n_tables; ++t)
        for (int i = threadIdx.x; i < s_len[t]; i += AR_THREADS) ard_cdf[s_row[t] + i] = p.cdfs[(int64_t)t * p.cdf_stride + i];
    }
    if (coder) {
      const int64_t w0 = p.word_offsets[n];
      rs.words = p.words + w0;
      rs.nw = p.word_offsets[n + 1] - w0;
      rs.pos = 2;
      rs.win = -64;
      if (!s_stop) rs.x = (uint64_t)__ldg(rs.words) | ((uint64_t)__ldg(rs.words + 1) << 32);
    }
  }
  cluster.sync();   // every CTA has started and initialised its shared memory before the first remote access
  if (rank != 0 && threadIdx.x == 0) s_stop = *cluster.map_shared_rank(&s_stop, 0);
  __syncthreads();

  float* yhat = a.y_hat + (int64_t)n * H * W * C;
  const float* prm = a.params + (int64_t)n * H * W * a.params_ld;
  int32_t* sym = a.symbols + (int64_t)n * H * W * C;
  int32_t* idx = a.indexes + (int64_t)n * H * W * C;

  for (int pix = 0; pix < H * W && !s_stop; ++pix) {
    const int h = pix / W, w = pix - h * W;
    const int P = ar_position_chunk_len(h, w, H, W);
    for (int i = threadIdx.x; i < AR_TAPS * C; i += AR_THREADS) {
      int dy, dx;
      ar_tap(i >> 7, dy, dx);
      const int hh = h + dy, ww = w + dx;
      s_taps[i] = hh < 0 || ww < 0 || ww >= W ? 0.f : __ldcg(yhat + ((int64_t)hh * W + ww) * C + (i & 127));
    }
    for (int i = threadIdx.x; i < C2; i += AR_THREADS) s_in1[i] = __ldg(prm + (int64_t)pix * a.params_ld + i);
    __syncthreads();
    // ---- context model -> ctx half of ep0's input
    ard_partials(wA, s_ns[AR_CTX], P, s_part, [&](int k) { return *reinterpret_cast<const float4*>(s_taps + k); });
    __syncthreads();
    ard_publish<false>(cluster, RD, wA, a.b_ctx, s_ns[AR_CTX], P, s_part, s_out, s_in1 + C2);
    cluster.sync();
    // ---- ep0: (params | ctx) -> c1, LeakyReLU
    ard_partials(wB, s_ns[AR_EP0], P, s_part, [&](int k) { return *reinterpret_cast<const float4*>(s_in1 + k); });
    __syncthreads();
    ard_publish<true>(cluster, RD, wB, a.b1, s_ns[AR_EP0], P, s_part, s_out, s_in2);
    cluster.sync();
    // ---- ep2: c1 -> c2, LeakyReLU
    ard_partials(wC, s_ns[AR_EP2], P, s_part, [&](int k) { return *reinterpret_cast<const float4*>(s_in2 + k); });
    __syncthreads();
    ard_publish<true>(cluster, RD, wC, a.b2, s_ns[AR_EP2], P, s_part, s_out, s_in3);
    cluster.sync();
    // ---- ep4: c2 -> (scales | means) of this CTA's latent channels, to CTA 0
    ard_partials(wD, s_ns[AR_EP4], P, s_part, [&](int k) { return *reinterpret_cast<const float4*>(s_in3 + k); });
    __syncthreads();
    for (int j = threadIdx.x; j < wD.split; j += AR_THREADS) {
      const float scale = ard_output(wD, a.b3, s_ns[AR_EP4], P, s_part, j);
      const float mean = ard_output(wD, a.b3, s_ns[AR_EP4], P, s_part, wD.split + j);
      *cluster.map_shared_rank(&s_mean[wD.n0 + j], 0) = mean;
      *cluster.map_shared_rank(&s_idx[wD.n0 + j], 0) = ar_scale_index(scale, s_table, n_cmp);
    }
    cluster.sync();
    // ---- the 128 symbols of the position
    if (coder) {
      int bad = -1;
      for (int c = 0; c < C; ++c) {
        const int t = s_idx[c];
        const int32_t* row = ard_cdf + s_row[t];
        int32_t v;
        if (!ard_decode_symbol(rs, [&](int j) { return (uint32_t)row[j]; }, s_len[t], s_off[t], v)) {
          bad = c;
          break;
        }
        if (threadIdx.x == 0) s_sym[c] = v;
      }
      __syncwarp();
      if (bad < 0) {
        for (int c = threadIdx.x; c < C; c += 32) {
          const int64_t o = (int64_t)pix * C + c;
          sym[o] = s_sym[c];
          idx[o] = s_idx[c];
          yhat[o] = __fadd_rn((float)s_sym[c], s_mean[c]);
        }
      } else if (threadIdx.x == 0) {
        p.status[n] = (int64_t)pix * C + bad;
        for (int r = 0; r < RD; ++r) *cluster.map_shared_rank(&s_stop, r) = 1;
      }
      __threadfence();
    }
    cluster.sync();   // y_hat of this position is visible to every CTA; s_stop is final
  }
  cluster.sync();     // no CTA leaves while another may still write into its shared memory
}

}  // namespace tdvc

using namespace tdvc;

extern "C" int tdvc_ar_decode(const TdvcArDecodeParams* p, void* stream) {
  TDVC_REQUIRE(p != nullptr, "ar_decode: null params");
  const int rc = ar_check_decode(*p, ARD_CDF_MAX, "ar_decode");
  if (rc != TDVC_OK) return rc;
  // 16 CTAs per image, 8 where that cannot launch; the result does not depend on it
  int R = 16;
  return ar_launch_clusters<ar_decode_kernel>(*p, p->chain.N, R, true, ARD_SMEM, (cudaStream_t)stream, "ar_decode");
}

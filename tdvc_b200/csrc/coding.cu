// Real entropy coding of the latents (`is_compress=True`, reference main/model/pnet.py:45-49,69-73 -> compressai
// `JointAutoregressiveHierarchicalPriors.compress` / `_compress_ar`, `EntropyModel.compress`, the `ans` rANS extension).
//
// Device side: the autoregressive pass over y.  compressai walks the latent in raster order, one position per Python
// iteration (a 5x5 masked convolution over the already-coded neighbourhood, three 1x1 layers, then the position is
// quantised RELATIVE to its predicted mean and written back for its successors).  Position (h, w) needs (h-1, w+2) and
// (h, w-1) at the latest, so all positions with w + 3h = t are independent: the kernel runs the W + 3(H-1) wavefronts
// inside ONE launch, one thread-block cluster per image; the CTAs of the cluster split the output channels of each
// layer, exchange the (<= 40 positions x <= 432 channels) stage results through L2 and meet at a cluster barrier
// (4 per wavefront).  Exact fp32 FFMA: a quantised symbol must not depend on tensor-core operand rounding, every later
// position of the image is predicted from it.
//
// Host side (as in compressai, whose entropy coder runs on the CPU): pmf -> 16-bit quantised CDF, and the 64-bit rANS
// coder (ryg_rans rans64 + compressai's bypass escape) over the symbols / table indexes the device produced.
#include <cooperative_groups.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "ar_common.cuh"

namespace cg = cooperative_groups;

namespace tdvc {

constexpr int AR_NBUF = 3;      // staging depth
constexpr int AR_RED = AR_WARPS * AR_PT * 32;   // one (AR_PT positions x 32 channels) tile of partial sums per warp task
constexpr size_t AR_SMEM = (size_t)(AR_NBUF * (AR_PCH * AR_KC + AR_KC * AR_NS_MAX) + AR_RED) * sizeof(float);

struct ArDev {
  TdvcArParams a;
  float* ctx_s;   // [N][AR_PCH][2C]
  float* h1_s;    // [N][AR_PCH][c1_pad]
  float* h2_s;    // [N][AR_PCH][c2_pad]
  unsigned long long* dbg;   // developer timing (TDVC_B200_AR_DEBUG): ns per phase, summed over the wavefronts by CTA 0
};

__device__ __forceinline__ unsigned long long ar_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define AR_MARK(i)                                                  \
  do {                                                              \
    if (d.dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {  \
      const unsigned long long now_ = ar_now();                     \
      d.dbg[i] += now_ - t_last;                                    \
      t_last = now_;                                                \
    }                                                               \
  } while (0)

__device__ __forceinline__ void cp_async16_cg(float* smem, const float* g, int src_bytes) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(g), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

// weight part of chunk c of a layer -> ring slot c % AR_NBUF
__device__ __forceinline__ void ar_issue_w(const ArW& w, int c, float* sW) {
  const int k0 = c * AR_KC;
  if (k0 < w.K) {
    const int kc = w.K - k0 < AR_KC ? w.K - k0 : AR_KC;
    float* dW = sW + (c % AR_NBUF) * (AR_KC * AR_NS_MAX);
    const int nq = (w.ns + 3) >> 2;
    for (int i = threadIdx.x; i < kc * 16; i += AR_THREADS) {
      const int kk = i >> 4, q = i & 15;
      if (q < nq) cp_async16_cg(dW + kk * AR_NS_MAX + 4 * q, w.Wt + (int64_t)(k0 + kk) * w.ldw + w.col(4 * q), 16);
    }
  }
}

// A part of chunk c: rows of the previous stage's result, written by the other CTAs of the cluster: 16-byte L2 loads, never L1.
// asrc(p, k) -> address of A(p, k .. k+3) or nullptr (zero).
template <class ASrc>
__device__ __forceinline__ void ar_issue_a(const ArW& w, int c, int P, float* sA, ASrc asrc) {
  const int k0 = c * AR_KC;
  if (k0 < w.K) {
    const int kc = w.K - k0 < AR_KC ? w.K - k0 : AR_KC;
    float* dA = sA + (c % AR_NBUF) * (AR_PCH * AR_KC);
    const int nq = kc >> 2;
    for (int i = threadIdx.x; i < P * 32; i += AR_THREADS) {
      const int p = i >> 5, q = i & 31;
      if (q < nq) {
        const float* src = asrc(p, k0 + 4 * q);
        cp_async16_cg(dA + p * AR_KC + 4 * q, src != nullptr ? src : w.Wt, src != nullptr ? 16 : 0);
      }
    }
  }
}

// partial sums of out[p][n] = sum_k A(p, k) * Wt[k][col(n)], n in [n0, n0 + ns), p < P, left in red[task][p % AR_PT][n % 32]
// with task = ((n / 32) * PG + p / AR_PT) * KS + ks (ar_sum adds the KS splits in order).
// K is walked in chunks of AR_KC staged in shared memory through a 3-deep cp.async ring.  The weight parts of chunks 0 and 1
// are already in flight when the stage starts (two committed groups, issued by the caller before the cluster barrier: they
// do not depend on the previous stage).  A warp owns one (position group, channel group, K split): lanes = output channels,
// registers = AR_PT positions, the A operand is a shared-memory broadcast.
template <class ASrc>
__device__ __forceinline__ int ar_stage(const ArW& w, int P, float* sA, float* sW, float* red, ASrc asrc) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ns = w.ns, K = w.K;
  const int NG = (ns + 31) >> 5, PG = (P + AR_PT - 1) / AR_PT;
  const int KS = ar_ksplits(ns, P);
  const int tasks = NG * PG * KS;          // <= AR_WARPS: NG <= 2, PG <= 5
  const bool busy = warp < tasks;
  const int ks = warp % KS, r = warp / KS;
  const int pg = r % PG, ng = r / PG;
  const int nl = ng * 32 + lane;
  const int p0 = pg * AR_PT;
  const int nchunks = (K + AR_KC - 1) / AR_KC;

  float acc[AR_PT];
#pragma unroll
  for (int j = 0; j < AR_PT; ++j) acc[j] = 0.f;
  ar_issue_a(w, 0, P, sA, asrc);
  cp_async_commit();
  ar_issue_a(w, 1, P, sA, asrc);
  cp_async_commit();
  for (int c = 0; c < nchunks; ++c) {
    cp_async_wait<1>();
    __syncthreads();      // chunk c has landed for every thread; chunk c - 1 has been consumed by every warp
    ar_issue_a(w, c + 2, P, sA, asrc);
    ar_issue_w(w, c + 2, sW);
    cp_async_commit();
    if (busy) {
      int q0, q1;
      ar_split_quads(ar_chunk_quads(K, c), ks, KS, q0, q1);
      const float* cA = sA + (c % AR_NBUF) * (AR_PCH * AR_KC);
      const float* cW = sW + (c % AR_NBUF) * (AR_KC * AR_NS_MAX) + nl;
      const float* pA = cA + p0 * AR_KC;
      if (p0 + AR_PT <= P) {
#pragma unroll 2
        for (int q = q0; q < q1; ++q) {
          const float w0 = cW[(4 * q) * AR_NS_MAX], w1 = cW[(4 * q + 1) * AR_NS_MAX], w2 = cW[(4 * q + 2) * AR_NS_MAX],
                      w3 = cW[(4 * q + 3) * AR_NS_MAX];
#pragma unroll
          for (int j = 0; j < AR_PT; ++j) {
            const float4 a = *reinterpret_cast<const float4*>(pA + j * AR_KC + 4 * q);
            acc[j] = ar_fma4(acc[j], a, w0, w1, w2, w3);
          }
        }
      } else {
        for (int q = q0; q < q1; ++q) {
          const float w0 = cW[(4 * q) * AR_NS_MAX], w1 = cW[(4 * q + 1) * AR_NS_MAX], w2 = cW[(4 * q + 2) * AR_NS_MAX],
                      w3 = cW[(4 * q + 3) * AR_NS_MAX];
#pragma unroll
          for (int j = 0; j < AR_PT; ++j) {
            if (p0 + j < P) {
              const float4 a = *reinterpret_cast<const float4*>(pA + j * AR_KC + 4 * q);
              acc[j] = ar_fma4(acc[j], a, w0, w1, w2, w3);
            }
          }
        }
      }
    }
  }
  cp_async_wait<0>();
  if (busy) {
#pragma unroll
    for (int j = 0; j < AR_PT; ++j) red[(warp * AR_PT + j) * 32 + lane] = acc[j];
  }
  __syncthreads();        // every warp is done with the ring: the next layer's first weight chunks may be issued
  return KS;
}

// sum over the K splits of output (position p, local channel nl) of a stage that ran with P positions and KS splits
__device__ __forceinline__ float ar_sum(const float* red, int KS, int P, int p, int nl) {
  const int PG = (P + AR_PT - 1) / AR_PT;
  const float* r = red + ((((nl >> 5) * PG + p / AR_PT) * KS) * AR_PT + (p % AR_PT)) * 32 + (nl & 31);
  return ar_reduce(KS, [&](int ks) { return r[ks * AR_PT * 32]; });
}

// weight chunks 0 and 1 of the NEXT layer: issued before this layer's results are published, so that the loads fly during
// the final sums and the cluster barrier
__device__ __forceinline__ void ar_prefetch_w(const ArW& w, float* sW) {
  ar_issue_w(w, 0, sW);
  cp_async_commit();
  ar_issue_w(w, 1, sW);
  cp_async_commit();
}

__global__ void __launch_bounds__(AR_THREADS, 1) ar_code_kernel(const ArDev d) {
  cg::cluster_group cluster = cg::this_cluster();
  const int R = (int)cluster.num_blocks();
  const int rank = (int)cluster.block_rank();
  const int n = blockIdx.x / R;
  const TdvcArChain& a = d.a.chain;
  const int H = a.H, W = a.W;
  constexpr int C = AR_C, C2 = 2 * AR_C;
  extern __shared__ __align__(16) float ar_smem[];
  float* sA = ar_smem;                                   // [AR_NBUF][AR_PCH][AR_KC]
  float* sW = sA + AR_NBUF * AR_PCH * AR_KC;             // [AR_NBUF][AR_KC][AR_NS_MAX]
  float* red = sW + AR_NBUF * AR_KC * AR_NS_MAX;         // [AR_WARPS][AR_PT][32]
  __shared__ float s_table[64];
  for (int i = threadIdx.x; i < a.n_scales - 1; i += AR_THREADS) s_table[i] = a.scale_table[i];
  __syncthreads();
  const int n_cmp = a.n_scales - 1;

  float* yhat = a.y_hat + (int64_t)n * H * W * C;
  const float* y = d.a.y + (int64_t)n * H * W * d.a.y_ld;
  const float* prm = a.params + (int64_t)n * H * W * a.params_ld;
  float* ctx_s = d.ctx_s + (int64_t)n * AR_PCH * C2;
  float* h1_s = d.h1_s + (int64_t)n * AR_PCH * a.c1_pad;
  float* h2_s = d.h2_s + (int64_t)n * AR_PCH * a.c2_pad;
  int32_t* sym = a.symbols + (int64_t)n * H * W * C;
  int32_t* idx = a.indexes + (int64_t)n * H * W * C;

  const ArW wA = ar_layer(a, AR_CTX, rank, R), wB = ar_layer(a, AR_EP0, rank, R), wC = ar_layer(a, AR_EP2, rank, R),
            wD = ar_layer(a, AR_EP4, rank, R);

  ar_prefetch_w(wA, sW);
  unsigned long long t_last = d.dbg != nullptr ? ar_now() : 0ull;
  const int waves = W + 3 * (H - 1);
  for (int t = 0; t < waves; ++t) {
    int h_lo, h_hi;
    ar_wave_rows(t, H, W, h_lo, h_hi);
    for (int hc = h_lo; hc <= h_hi; hc += AR_PCH) {
      const int P = ar_chunk_len(hc, h_hi);
      // ---- context model: 12 causal taps of the 5x5 window of y_hat (zero outside the latent)
      {
        auto asrc = [&](int p, int k) -> const float* {
          const int ti = k >> 7, c = k & 127;
          int dy, dx;
          ar_tap(ti, dy, dx);
          const int hh = hc + p + dy, ww = t - 3 * (hc + p) + dx;
          if (hh < 0 || ww < 0 || ww >= W) return nullptr;
          return yhat + ((int64_t)hh * W + ww) * C + c;
        };
        const int KS = ar_stage(wA, P, sA, sW, red, asrc);
        AR_MARK(0);
        ar_prefetch_w(wB, sW);
        for (int i = threadIdx.x; i < P * wA.ns; i += AR_THREADS) {
          const int p = i / wA.ns, nl = i - p * wA.ns;
          ctx_s[p * C2 + wA.n0 + nl] = ar_sum(red, KS, P, p, nl) + __ldg(a.b_ctx + wA.n0 + nl);
        }
      }
      AR_MARK(1);
      __threadfence();
      cluster.sync();
      AR_MARK(2);
      // ---- entropy_parameters[0]: (params | ctx) -> c1, LeakyReLU(0.01)
      {
        auto asrc = [&](int p, int k) -> const float* {
          if (k < C2) {
            const int hh = hc + p, ww = t - 3 * hh;
            return prm + ((int64_t)hh * W + ww) * a.params_ld + k;
          }
          return ctx_s + p * C2 + (k - C2);
        };
        const int KS = ar_stage(wB, P, sA, sW, red, asrc);
        AR_MARK(3);
        ar_prefetch_w(wC, sW);
        for (int i = threadIdx.x; i < P * wB.ns; i += AR_THREADS) {
          const int p = i / wB.ns, nl = i - p * wB.ns;
          const float v = ar_sum(red, KS, P, p, nl) + __ldg(a.b1 + wB.n0 + nl);
          h1_s[p * a.c1_pad + wB.n0 + nl] = ar_lrelu(v);
        }
      }
      AR_MARK(4);
      __threadfence();
      cluster.sync();
      AR_MARK(5);
      // ---- entropy_parameters[2]: c1 -> c2, LeakyReLU(0.01)
      {
        auto asrc = [&](int p, int k) -> const float* { return h1_s + p * a.c1_pad + k; };
        const int KS = ar_stage(wC, P, sA, sW, red, asrc);
        AR_MARK(6);
        ar_prefetch_w(wD, sW);
        for (int i = threadIdx.x; i < P * wC.ns; i += AR_THREADS) {
          const int p = i / wC.ns, nl = i - p * wC.ns;
          const float v = ar_sum(red, KS, P, p, nl) + __ldg(a.b2 + wC.n0 + nl);
          h2_s[p * a.c2_pad + wC.n0 + nl] = ar_lrelu(v);
        }
      }
      AR_MARK(7);
      __threadfence();
      cluster.sync();
      AR_MARK(8);
      // ---- entropy_parameters[4]: c2 -> (scales | means); quantise relative to the mean, table index of the scale
      {
        auto asrc = [&](int p, int k) -> const float* { return h2_s + p * a.c2_pad + k; };
        const int KS = ar_stage(wD, P, sA, sW, red, asrc);
        AR_MARK(9);
        ar_prefetch_w(wA, sW);
        const int nch = wD.split, ch0 = wD.n0;
        for (int i = threadIdx.x; i < P * nch; i += AR_THREADS) {
          const int p = i / nch, j = i - p * nch;
          const int ch = ch0 + j;
          const float scale = ar_sum(red, KS, P, p, j) + __ldg(a.b3 + ch);
          const float mean = ar_sum(red, KS, P, p, nch + j) + __ldg(a.b3 + C + ch);
          const int hh = hc + p, ww = t - 3 * hh;
          const int64_t pix = (int64_t)hh * W + ww;
          const float q = rintf(__fsub_rn(__ldg(y + pix * d.a.y_ld + ch), mean));
          yhat[pix * C + ch] = __fadd_rn(q, mean);
          sym[pix * C + ch] = (int32_t)q;
          idx[pix * C + ch] = ar_scale_index(scale, s_table, n_cmp);
        }
      }
      AR_MARK(10);
      __threadfence();
      cluster.sync();
      AR_MARK(11);
    }
  }
  cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------------ host rANS
struct RansSym {
  uint32_t start;
  uint32_t range;   // 0 = bypass digit (value in `start`)
};

}  // namespace tdvc

using namespace tdvc;

extern "C" size_t tdvc_ar_code_workspace_bytes(int N, int c1_pad, int c2_pad) {
  if (N <= 0 || c1_pad <= 0 || c2_pad <= 0) return 0;
  return (size_t)N * AR_PCH * (size_t)(2 * AR_C + c1_pad + c2_pad) * sizeof(float);
}

extern "C" int tdvc_ar_code(const TdvcArParams* p, void* workspace, size_t workspace_bytes, void* stream) {
  TDVC_REQUIRE(p != nullptr, "ar_code: null params");
  const int rc = ar_check_chain(p->chain, "ar_code");
  if (rc != TDVC_OK) return rc;
  const TdvcArChain& a = p->chain;
  TDVC_REQUIRE(p->y && p->y_ld >= AR_C, "ar_code: bad y");
  const bool auto_r = p->cluster <= 0;   // auto: 16 CTAs per image, 8 where that cannot launch
  int R = auto_r ? 16 : p->cluster;
  TDVC_REQUIRE(R == 8 || R == 16, "ar_code: cluster size %d (8 or 16)", R);
  const size_t need = tdvc_ar_code_workspace_bytes(a.N, a.c1_pad, a.c2_pad);
  TDVC_REQUIRE(workspace != nullptr && workspace_bytes >= need, "ar_code: workspace of %zu bytes, %zu needed", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  // the padded tail of the hidden rows is read (times zero weight rows): it must hold finite numbers
  if (cudaMemsetAsync(workspace, 0, need, st) != cudaSuccess) {
    set_error("ar_code: cudaMemsetAsync failed");
    return TDVC_ECUDA;
  }
  ArDev d;
  d.a = *p;
  d.ctx_s = (float*)workspace;
  d.h1_s = d.ctx_s + (size_t)a.N * AR_PCH * 2 * AR_C;
  d.h2_s = d.h1_s + (size_t)a.N * AR_PCH * a.c1_pad;
  d.dbg = nullptr;
  static unsigned long long* dbg_buf = nullptr;
  const bool debug = getenv("TDVC_B200_AR_DEBUG") != nullptr;
  if (debug) {
    if (dbg_buf == nullptr) cudaMalloc(&dbg_buf, 16 * sizeof(unsigned long long));
    cudaMemsetAsync(dbg_buf, 0, 16 * sizeof(unsigned long long), st);
    d.dbg = dbg_buf;
  }
  const int lrc = ar_launch_clusters<ar_code_kernel>(d, a.N, R, auto_r, AR_SMEM, st, "ar_code");
  if (lrc != TDVC_OK) return lrc;
  if (p->cluster_used_host != nullptr) *p->cluster_used_host = R;
  if (debug) {
    unsigned long long h[16];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
    static const char* nm[12] = {"A chunks", "A sums", "A fence+barrier", "B chunks", "B sums", "B fence+barrier",
                                 "C chunks", "C sums", "C fence+barrier", "D chunks", "D sums", "D fence+barrier"};
    for (int i = 0; i < 12; ++i) fprintf(stderr, "ar_code[R=%d] %-16s %8.3f ms\n", R, nm[i], h[i] * 1e-6);
  }
  return TDVC_OK;
}

// compressai `pmf_to_quantized_cdf` (C++ in its `_CXX` module, always on the host): cdf has n + 1 entries.
extern "C" int tdvc_pmf_to_quantized_cdf(const float* pmf, int n, int precision, int32_t* cdf) {
  TDVC_REQUIRE(pmf && cdf && n > 0 && precision > 0 && precision <= 16, "pmf_to_quantized_cdf: bad args");
  std::vector<uint32_t> c((size_t)n + 1);
  c[0] = 0;
  uint32_t total = 0;
  for (int i = 0; i < n; ++i) {
    TDVC_REQUIRE(pmf[i] >= 0.f && pmf[i] <= 2.f, "pmf_to_quantized_cdf: pmf[%d] = %g", i, (double)pmf[i]);
    c[i + 1] = (uint32_t)roundf(pmf[i] * (float)(1 << precision));
    total += c[i + 1];
  }
  TDVC_REQUIRE(total != 0, "pmf_to_quantized_cdf: the pmf sums to zero");
  uint32_t run = 0;
  for (int i = 0; i <= n; ++i) {
    run += (uint32_t)((((uint64_t)1 << precision) * c[i]) / total);
    c[i] = run;
  }
  c[n] = 1u << precision;
  for (int i = 0; i < n; ++i) {
    if (c[i] == c[i + 1]) {
      uint32_t best_freq = ~0u;
      int best = -1;
      for (int j = 0; j < n; ++j) {
        const uint32_t f = c[j + 1] - c[j];
        if (f > 1 && f < best_freq) { best_freq = f; best = j; }
      }
      TDVC_REQUIRE(best != -1, "pmf_to_quantized_cdf: no bin to steal from");
      if (best < i) {
        for (int j = best + 1; j <= i; ++j) c[j]--;
      } else {
        for (int j = i + 1; j <= best; ++j) c[j]++;
      }
    }
  }
  for (int i = 0; i <= n; ++i) cdf[i] = (int32_t)c[i];
  return TDVC_OK;
}

static inline bool rans_tables_ok(const int32_t* cdfs, int cdf_stride, const int32_t* cdf_lengths, const int32_t* offsets,
                                  int n_tables) {
  return cdfs && cdf_lengths && offsets && n_tables > 0 && cdf_stride >= 3;
}

// compressai rans_interface.cpp `encode_with_indexes` (+ `flush`): returns the stream length in bytes, or a negative TDVC_E*.
extern "C" int64_t tdvc_rans_encode_with_indexes(const int32_t* symbols, const int32_t* indexes, int64_t n, const int32_t* cdfs,
                                                 int cdf_stride, const int32_t* cdf_lengths, const int32_t* offsets, int n_tables,
                                                 uint8_t* out, int64_t capacity) {
  if (!(symbols && indexes && n >= 0 && out && rans_tables_ok(cdfs, cdf_stride, cdf_lengths, offsets, n_tables))) {
    set_error("rans_encode: bad args");
    return TDVC_EINVAL;
  }
  std::vector<RansSym> syms;
  syms.reserve((size_t)n + 16);
  for (int64_t i = 0; i < n; ++i) {
    const int32_t ci = indexes[i];
    if (ci < 0 || ci >= n_tables) { set_error("rans_encode: table index %d at %lld", ci, (long long)i); return TDVC_EINVAL; }
    const int32_t* cdf = cdfs + (int64_t)ci * cdf_stride;
    const int32_t max_value = cdf_lengths[ci] - 2;
    if (max_value < 0 || max_value + 1 >= cdf_stride) { set_error("rans_encode: table %d has length %d", ci, cdf_lengths[ci]); return TDVC_EINVAL; }
    int64_t value = (int64_t)symbols[i] - offsets[ci];
    uint64_t raw = 0;
    if (value < 0) {
      raw = (uint64_t)(-2 * value - 1);
      value = max_value;
    } else if (value >= max_value) {
      raw = (uint64_t)(2 * (value - max_value));
      value = max_value;
    }
    const int32_t start = cdf[value], range = cdf[value + 1] - cdf[value];
    if (range <= 0 || start < 0 || start + range > (1 << RANS_PRECISION)) {
      set_error("rans_encode: empty bin %lld of table %d", (long long)value, ci);
      return TDVC_EINVAL;
    }
    syms.push_back({(uint32_t)start, (uint32_t)range});
    if (value == max_value) {
      int32_t n_bypass = 0;
      while ((raw >> (n_bypass * RANS_BYPASS)) != 0) ++n_bypass;
      uint32_t val = (uint32_t)n_bypass;
      while (val >= RANS_MAX_BYPASS) {
        syms.push_back({RANS_MAX_BYPASS, 0u});
        val -= RANS_MAX_BYPASS;
      }
      syms.push_back({val, 0u});
      for (int32_t j = 0; j < n_bypass; ++j) syms.push_back({(uint32_t)((raw >> (j * RANS_BYPASS)) & RANS_MAX_BYPASS), 0u});
    }
  }
  std::vector<uint32_t> words(syms.size() + 2);
  uint32_t* ptr = words.data() + words.size();
  uint64_t x = RANS64_L;
  for (size_t i = syms.size(); i-- > 0;) {
    const RansSym s = syms[i];
    if (s.range != 0) {
      const uint64_t x_max = ((RANS64_L >> RANS_PRECISION) << 32) * s.range;
      if (x >= x_max) { *--ptr = (uint32_t)x; x >>= 32; }
      x = ((x / s.range) << RANS_PRECISION) + (x % s.range) + s.start;
    } else {
      const uint64_t x_max = ((RANS64_L >> 16) << 32) * (uint64_t)(1u << (16 - RANS_BYPASS));
      if (x >= x_max) { *--ptr = (uint32_t)x; x >>= 32; }
      x = (x << RANS_BYPASS) | s.start;
    }
  }
  ptr -= 2;
  ptr[0] = (uint32_t)x;
  ptr[1] = (uint32_t)(x >> 32);
  const int64_t nbytes = (int64_t)(words.data() + words.size() - ptr) * 4;
  if (nbytes > capacity) { set_error("rans_encode: %lld bytes, capacity %lld", (long long)nbytes, (long long)capacity); return TDVC_EINVAL; }
  memcpy(out, ptr, (size_t)nbytes);   // little-endian host
  return nbytes;
}

// compressai rans_interface.cpp `RansDecoder::decode_with_indexes`
extern "C" int tdvc_rans_decode_with_indexes(const uint8_t* data, int64_t nbytes, const int32_t* indexes, int64_t n,
                                             const int32_t* cdfs, int cdf_stride, const int32_t* cdf_lengths,
                                             const int32_t* offsets, int n_tables, int32_t* symbols) {
  TDVC_REQUIRE(data && nbytes >= 8 && nbytes % 4 == 0 && indexes && n >= 0 && symbols &&
                   rans_tables_ok(cdfs, cdf_stride, cdf_lengths, offsets, n_tables), "rans_decode: bad args");
  const int64_t nw = nbytes / 4;
  std::vector<uint32_t> w((size_t)nw);
  memcpy(w.data(), data, (size_t)nbytes);
  int64_t pos = 2;
  uint64_t x = (uint64_t)w[0] | ((uint64_t)w[1] << 32);
  const uint64_t mask = (1ull << RANS_PRECISION) - 1;
  auto renorm = [&]() -> bool {
    if (x < RANS64_L) {
      if (pos >= nw) return false;
      x = (x << 32) | w[(size_t)pos++];
    }
    return true;
  };
  auto bits = [&](uint32_t& v) -> bool {
    v = (uint32_t)(x & RANS_MAX_BYPASS);
    x >>= RANS_BYPASS;
    return renorm();
  };
  for (int64_t i = 0; i < n; ++i) {
    const int32_t ci = indexes[i];
    TDVC_REQUIRE(ci >= 0 && ci < n_tables, "rans_decode: table index %d at %lld", ci, (long long)i);
    const int32_t* cdf = cdfs + (int64_t)ci * cdf_stride;
    const int32_t len = cdf_lengths[ci];
    const int32_t max_value = len - 2;
    TDVC_REQUIRE(max_value >= 0 && len <= cdf_stride, "rans_decode: table %d has length %d", ci, len);
    const uint32_t cum = (uint32_t)(x & mask);
    int32_t s = 0;
    while (s + 1 < len && (uint32_t)cdf[s + 1] <= cum) ++s;
    TDVC_REQUIRE(s + 1 < len, "rans_decode: corrupt stream at symbol %lld", (long long)i);
    const uint32_t start = (uint32_t)cdf[s], freq = (uint32_t)(cdf[s + 1] - cdf[s]);
    x = (uint64_t)freq * (x >> RANS_PRECISION) + (x & mask) - start;
    TDVC_REQUIRE(renorm(), "rans_decode: stream ends at symbol %lld", (long long)i);
    TDVC_REQUIRE(rans_symbol(s, max_value, offsets[ci], bits, symbols[i]),
                 "rans_decode: truncated or corrupt bypass code at symbol %lld", (long long)i);
  }
  return TDVC_OK;
}

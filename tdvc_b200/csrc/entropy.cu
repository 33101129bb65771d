// Quantise + likelihood + bits in one pass per latent (compressai EntropyBottleneck / GaussianConditional
// in eval mode, SURVEY.md App. A; the log/sum reductions of reference main/model/pnet.py:38-43,62-67).
// Memory-bound: y-path reads 12 B/element (y, scale, mean), z-path 4 B/element (+4 B z_hat write).
// Reduction: fp64 per thread -> warp shuffle -> one atomicAdd(double) per CTA.
#include "common.cuh"

namespace tdvc {

__device__ __forceinline__ void block_accumulate(double s, double* acc) {
  s = warp_sum_d(s);
  __shared__ double sh[32];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? sh[threadIdx.x] : 0.0;
    s = warp_sum_d(s);
    if (threadIdx.x == 0) atomicAdd(acc, s);
  }
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// per-channel cumulative logits: widths 1,3,3,3,3,1.  Parameters in smem, laid out [param][C].
struct EbSmem {
  const float* m;  // 33 rows
  const float* b;  // 13 rows
  const float* f;  // 12 rows
  int C;
};

__device__ __forceinline__ float eb_logits(const EbSmem& s, int c, float v) {
  const int C = s.C;
  float h[3], g[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    float t = s.m[j * C + c] * v + s.b[j * C + c];
    h[j] = t + s.f[j * C + c] * tanhf(t);
  }
#pragma unroll
  for (int l = 0; l < 3; ++l) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const float* mr = s.m + (3 + l * 9 + i * 3) * C + c;
      float t = mr[0] * h[0] + mr[C] * h[1] + mr[2 * C] * h[2] + s.b[(3 + l * 3 + i) * C + c];
      g[i] = t + s.f[(3 + l * 3 + i) * C + c] * tanhf(t);
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) h[i] = g[i];
  }
  const float* mr = s.m + 30 * C + c;
  return mr[0] * h[0] + mr[C] * h[1] + mr[2 * C] * h[2] + s.b[12 * C + c];
}

// noise != nullptr: training-mode quantisation, z_hat = z + noise (compressai quantize(.., "noise"): the medians are not used)
__global__ void eb_bits_kernel(const float* __restrict__ z, const float* __restrict__ noise, float* __restrict__ z_hat,
                               const float* __restrict__ mats, const float* __restrict__ biases, const float* __restrict__ factors,
                               const float* __restrict__ medians, int64_t total, int C, double* acc) {
  extern __shared__ float sh[];
  float* sm = sh;                // [33][C]
  float* sb = sh + 33 * C;       // [13][C]
  float* sf = sb + 13 * C;       // [12][C]
  float* smed = sf + 12 * C;     // [C]
  for (int i = threadIdx.x; i < 33 * C; i += blockDim.x) sm[(i % 33) * C + i / 33] = mats[i];
  for (int i = threadIdx.x; i < 13 * C; i += blockDim.x) sb[(i % 13) * C + i / 13] = biases[i];
  for (int i = threadIdx.x; i < 12 * C; i += blockDim.x) sf[(i % 12) * C + i / 12] = factors[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) smed[i] = medians[i];
  __syncthreads();
  EbSmem s{sm, sb, sf, C};
  double sum = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % C);
    const float med = smed[c];
    const float q = noise != nullptr ? __fadd_rn(z[i], noise[i]) : __fadd_rn(rintf(__fsub_rn(z[i], med)), med);
    z_hat[i] = q;
    const float lower = eb_logits(s, c, q - 0.5f);
    const float upper = eb_logits(s, c, q + 0.5f);
    const float t = lower + upper;
    const float sign = t > 0.f ? -1.f : (t < 0.f ? 1.f : 0.f);
    float p = fabsf(sigmoidf_(sign * upper) - sigmoidf_(sign * lower));
    p = fmaxf(p, 1e-9f);
    sum += (double)logf(p);
  }
  block_accumulate(sum, acc);
}

// noise != nullptr: training mode, the likelihood is evaluated at y + noise instead of the dequantised value
__global__ void gc_bits_kernel(const float* __restrict__ y, const float* __restrict__ noise, const float* __restrict__ params,
                               int params_ld, int64_t total, int C, double* acc) {
  double sum = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const float kc = -0.70710678118654752440f;  // -(2 ** -0.5)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t p = i / C;
    const int c = (int)(i - p * C);
    const float yv = __ldg(y + i);
    const float scale = __ldg(params + p * params_ld + c);
    const float mean = __ldg(params + p * params_ld + C + c);
    const float out = noise != nullptr ? __fadd_rn(yv, __ldg(noise + i))
                                       : __fadd_rn(rintf(__fsub_rn(yv, mean)), mean);  // dequantised value
    const float v = fabsf(__fsub_rn(out, mean));
    const float sc = fmaxf(scale, 0.11f);
    const float upper = 0.5f * erfcf(kc * __fdiv_rn(__fsub_rn(0.5f, v), sc));
    const float lower = 0.5f * erfcf(kc * __fdiv_rn(__fsub_rn(-0.5f, v), sc));
    float lik = fmaxf(upper - lower, 1e-9f);
    sum += (double)logf(lik);
  }
  block_accumulate(sum, acc);
}

// EntropyBottleneck.loss(): sum_c sum_k |logits_cumulative(quantiles[c][k]) - target[k]|  (compressai entropy_models.py;
// reference pnet.py:35,59 `aux_loss()`).  One block; fixed-order tree: deterministic.
__global__ void eb_aux_loss_kernel(const float* __restrict__ mats, const float* __restrict__ biases,
                                   const float* __restrict__ factors, const float* __restrict__ quantiles,
                                   const float* __restrict__ target, int C, float* __restrict__ out) {
  extern __shared__ float sh[];
  float* sm = sh;
  float* sb = sh + 33 * C;
  float* sf = sb + 13 * C;
  float* red = sf + 12 * C;   // [blockDim.x]
  for (int i = threadIdx.x; i < 33 * C; i += blockDim.x) sm[(i % 33) * C + i / 33] = mats[i];
  for (int i = threadIdx.x; i < 13 * C; i += blockDim.x) sb[(i % 13) * C + i / 13] = biases[i];
  for (int i = threadIdx.x; i < 12 * C; i += blockDim.x) sf[(i % 12) * C + i / 12] = factors[i];
  __syncthreads();
  EbSmem s{sm, sb, sf, C};
  float t = 0.f;
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) {
    const int c = i / 3, k = i - 3 * c;
    t += fabsf(eb_logits(s, c, quantiles[i]) - target[k]);
  }
  red[threadIdx.x] = t;
  __syncthreads();
  for (int st = blockDim.x >> 1; st > 0; st >>= 1) {
    if (threadIdx.x < st) red[threadIdx.x] += red[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = red[0];
}

// d loss / d quantiles of eb_aux_loss (the only gradient the reference takes of it: `aux_loss.backward()` steps the aux
// optimiser on `.quantiles`, reference tools/train.py:101-113,147-159; compressai evaluates the logits with the matrices,
// biases and factors detached).  grad_q[c][k] = grad_out * sign(logits - target) * d logits / d q, one thread per (c, k).
__global__ void eb_aux_loss_grad_kernel(const float* __restrict__ mats, const float* __restrict__ biases,
                                        const float* __restrict__ factors, const float* __restrict__ quantiles,
                                        const float* __restrict__ target, const float* __restrict__ grad_out, int C,
                                        float* __restrict__ grad_q) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 3 * C) return;
  const int c = i / 3, k = i - 3 * c;
  const float* m = mats + c * 33;
  const float* b = biases + c * 13;
  const float* f = factors + c * 12;
  // forward value h and derivative d of every layer, widths 1,3,3,3,3,1
  float h[3], d[3], g[3], e[3];
  const float v = quantiles[i];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float t = m[j] * v + b[j];
    const float th = tanhf(t);
    h[j] = t + f[j] * th;
    d[j] = m[j] * (1.f + f[j] * (1.f - th * th));
  }
#pragma unroll
  for (int l = 0; l < 3; ++l) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const float* mr = m + 3 + l * 9 + r * 3;
      const float t = mr[0] * h[0] + mr[1] * h[1] + mr[2] * h[2] + b[3 + l * 3 + r];
      const float dt = mr[0] * d[0] + mr[1] * d[1] + mr[2] * d[2];
      const float th = tanhf(t);
      const float fr = f[3 + l * 3 + r];
      g[r] = t + fr * th;
      e[r] = dt * (1.f + fr * (1.f - th * th));
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) { h[r] = g[r]; d[r] = e[r]; }
  }
  const float* mr = m + 30;
  const float logit = mr[0] * h[0] + mr[1] * h[1] + mr[2] * h[2] + b[12];
  const float dlogit = mr[0] * d[0] + mr[1] * d[1] + mr[2] * d[2];
  const float diff = logit - target[k];
  const float sgn = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
  grad_q[i] = grad_out[0] * sgn * dlogit;
}

// Philox4x32-10 (Salmon et al. 2011), counter = element index / 4, key = seed: uniform noise in [-0.5, 0.5) for the
// training-mode quantisers (compressai quantize(.., "noise") draws torch.empty_like(x).uniform_(-0.5, 0.5)).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
// seed_dev != nullptr: the seed is read from device memory (a replayed CUDA graph draws fresh noise when a captured operation
// advances that word between replays)
__global__ void uniform_noise_kernel(float* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream_id,
                                     const uint64_t* __restrict__ seed_dev) {
  if (seed_dev != nullptr) seed = *seed_dev;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q * 4 < n; q += stride) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)stream_id, (uint32_t)(stream_id >> 32)),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < n) out[q * 4 + j] = (float)(v[j] >> 8) * (1.0f / 16777216.0f) - 0.5f;   // 24 random bits: exact in fp32
  }
}

// ---- real entropy coding: the "symbols" quantiser of z (compressai EntropyBottleneck.compress; reached from reference
// pnet.py:45-49,69-73 `compress()`).
// eb_symbols: z NHWC -> int32 symbols round(z - median) in NCHW order (the order compressai's EntropyBottleneck.compress
// flattens them in), indexes[i] = channel.
__global__ void eb_symbols_kernel(const float* __restrict__ z, int ld, const float* __restrict__ medians, int N, int HW, int C,
                                  int32_t* __restrict__ symbols, int32_t* __restrict__ indexes) {
  const int64_t total = (int64_t)N * C * HW;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int p = (int)(i % HW);
    const int c = (int)((i / HW) % C);
    const int n = (int)(i / ((int64_t)HW * C));
    const float v = __ldg(z + ((int64_t)n * HW + p) * ld + c);
    symbols[i] = __float2int_rn(__fsub_rn(v, medians[c]));
    indexes[i] = c;
  }
}

// eb_dequantize: the decoder's inverse of eb_symbols (compressai EntropyBottleneck.decompress -> dequantize): int32 symbols in
// NCHW order -> z_hat NHWC = symbol + median.  eb_bits_kernel writes the encoder's z_hat as __fadd_rn(rintf(z - med), med);
// rintf(z - med) is the float of the symbol, so this is the same fp32 addition on the same operands, bit for bit.
// One thread per output element in NHWC order: the writes are coalesced, the reads stride by HW (z is H/64 x W/64, small).
__global__ void eb_dequantize_kernel(const int32_t* __restrict__ symbols, const float* __restrict__ medians, int N, int HW,
                                     int C, float* __restrict__ z_hat, int ld) {
  const int64_t total = (int64_t)N * HW * C;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int c = (int)(i % C);
    const int64_t np = i / C;   // n * HW + p
    const int p = (int)(np % HW);
    const int n = (int)(np / HW);
    const int32_t s = __ldg(symbols + ((int64_t)n * C + c) * HW + p);
    z_hat[np * ld + c] = __fadd_rn((float)s, __ldg(medians + c));
  }
}

// ---- backward of the two likelihood-to-bits reductions in training (noise) mode (SURVEY.md 8f row 1; the reference takes these
// gradients from autograd through compressai's entropy models, tools/train.py:132-145).  S = sum ln max(p, 1e-9); `gS` is
// d loss / d S (device scalar).  compressai's LowerBound passes a gradient where the input is above the bound OR the gradient
// is negative (both the 1e-9 likelihood bound and the 0.11 scale bound).
//
// gc_bits_backward: p = Phi((0.5 - v) / s) - Phi((-0.5 - v) / s), v = |y + noise - mean|, s = max(scale, 0.11):
//   g_y (ld = C), g_params (ld = params_ld: d/d scale at channel c, d/d mean at C + c).  Element-wise.
__global__ void gc_bits_backward_kernel(const float* __restrict__ y, const float* __restrict__ noise, const float* __restrict__ params,
                                        int params_ld, const float* __restrict__ gS, float* __restrict__ g_y,
                                        float* __restrict__ g_params, int64_t total, int C) {
  const float g = __ldg(gS);
  const float kc = -0.70710678118654752440f, inv_sqrt_2pi = 0.39894228040143267794f;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int64_t px = i / C;
    const int c = (int)(i - px * C);
    const float scale = __ldg(params + px * params_ld + c), mean = __ldg(params + px * params_ld + C + c);
    const float d = __fsub_rn(__fadd_rn(__ldg(y + i), __ldg(noise + i)), mean);
    const float v = fabsf(d), sgn = d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f);
    const float sc = fmaxf(scale, 0.11f);
    const float u = (0.5f - v) / sc, l = (-0.5f - v) / sc;
    const float p_raw = 0.5f * erfcf(kc * u) - 0.5f * erfcf(kc * l);
    float g_p = g / fmaxf(p_raw, 1e-9f);
    if (!(p_raw >= 1e-9f || g_p < 0.f)) g_p = 0.f;
    const float g_u = g_p * inv_sqrt_2pi * expf(-0.5f * u * u), g_l = -g_p * inv_sqrt_2pi * expf(-0.5f * l * l);
    const float g_v = -(g_u + g_l) / sc;
    float g_s = -(g_u * u + g_l * l) / sc;
    if (!(scale >= 0.11f || g_s < 0.f)) g_s = 0.f;
    const float g_d = g_v * sgn;
    g_y[i] = g_d;
    g_params[px * params_ld + c] = g_s;
    g_params[px * params_ld + C + c] = -g_d;
  }
}

// eb_bits_backward: p = |sigmoid(s U) - sigmoid(s L)|, L / U = cumulative logits at z~ -+ 1/2, s = -sign(L + U) (a constant of
// the graph).  One CTA per channel: its threads walk the channel's elements, back-propagate both logits through the 5-layer
// MLP (widths 1,3,3,3,3,1) and keep the 58 parameter gradients of the channel in registers; a fixed-order block reduction
// makes them deterministic.  Gradients are with respect to the TRANSFORMED parameters the kernels read (softplus(matrix),
// bias, tanh(factor)); the caller chains through softplus / tanh.
struct EbTape {
  float v;          // input
  float h[4][3];    // layer outputs h_0..h_3
  float th[4][3];   // tanh(t_i)
};
__device__ __forceinline__ float eb_forward_tape(const float* m, const float* b, const float* f, float v, EbTape& tp) {
  tp.v = v;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float t = m[r] * v + b[r];
    tp.th[0][r] = tanhf(t);
    tp.h[0][r] = t + f[r] * tp.th[0][r];
  }
#pragma unroll
  for (int l = 1; l < 4; ++l) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const float* mr = m + 3 + (l - 1) * 9 + r * 3;
      const float t = mr[0] * tp.h[l - 1][0] + mr[1] * tp.h[l - 1][1] + mr[2] * tp.h[l - 1][2] + b[3 * l + r];
      tp.th[l][r] = tanhf(t);
      tp.h[l][r] = t + f[3 * l + r] * tp.th[l][r];
    }
  }
  return m[30] * tp.h[3][0] + m[31] * tp.h[3][1] + m[32] * tp.h[3][2] + b[12];
}
// accumulates into gm[33], gb[13], gf[12]; returns d logit / d v times g
__device__ __forceinline__ float eb_backward_tape(const float* m, const float* f, const EbTape& tp, float g, float* gm, float* gb,
                                                  float* gf) {
  float gh[3];
  gb[12] += g;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    gm[30 + j] += g * tp.h[3][j];
    gh[j] = g * m[30 + j];
  }
#pragma unroll
  for (int l = 3; l >= 1; --l) {
    float gt[3], gprev[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      gf[3 * l + r] += gh[r] * tp.th[l][r];
      gt[r] = gh[r] * (1.f + f[3 * l + r] * (1.f - tp.th[l][r] * tp.th[l][r]));
      gb[3 * l + r] += gt[r];
      const float* mr = m + 3 + (l - 1) * 9 + r * 3;
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        gm[3 + (l - 1) * 9 + r * 3 + j] += gt[r] * tp.h[l - 1][j];
        gprev[j] += gt[r] * mr[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) gh[j] = gprev[j];
  }
  float gv = 0.f;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    gf[r] += gh[r] * tp.th[0][r];
    const float gt = gh[r] * (1.f + f[r] * (1.f - tp.th[0][r] * tp.th[0][r]));
    gb[r] += gt;
    gm[r] += gt * tp.v;
    gv += gt * m[r];
  }
  return gv;
}

__global__ void __launch_bounds__(256) eb_bits_backward_kernel(const float* __restrict__ z_tilde, const float* __restrict__ mats,
                                                               const float* __restrict__ biases, const float* __restrict__ factors,
                                                               const float* __restrict__ gS, float* __restrict__ g_z,
                                                               float* __restrict__ g_mats, float* __restrict__ g_biases,
                                                               float* __restrict__ g_factors, int64_t npix, int C) {
  const int c = blockIdx.x;
  float m[33], b[13], f[12];
#pragma unroll
  for (int i = 0; i < 33; ++i) m[i] = mats[c * 33 + i];
#pragma unroll
  for (int i = 0; i < 13; ++i) b[i] = biases[c * 13 + i];
#pragma unroll
  for (int i = 0; i < 12; ++i) f[i] = factors[c * 12 + i];
  float acc[58];
#pragma unroll
  for (int i = 0; i < 58; ++i) acc[i] = 0.f;
  const float g = __ldg(gS);
  for (int64_t px = threadIdx.x; px < npix; px += blockDim.x) {
    const float q = z_tilde[px * C + c];
    EbTape tl, tu;
    const float lo = eb_forward_tape(m, b, f, q - 0.5f, tl), up = eb_forward_tape(m, b, f, q + 0.5f, tu);
    const float t = lo + up;
    const float s = t > 0.f ? -1.f : (t < 0.f ? 1.f : 0.f);
    const float a = sigmoidf_(s * up), bb = sigmoidf_(s * lo);
    const float diff = a - bb, p_raw = fabsf(diff);
    float g_p = g / fmaxf(p_raw, 1e-9f);
    if (!(p_raw >= 1e-9f || g_p < 0.f)) g_p = 0.f;
    const float g_diff = g_p * (diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f));
    const float g_up = g_diff * a * (1.f - a) * s, g_lo = -g_diff * bb * (1.f - bb) * s;
    float gz = eb_backward_tape(m, f, tu, g_up, acc, acc + 33, acc + 46);
    gz += eb_backward_tape(m, f, tl, g_lo, acc, acc + 33, acc + 46);
    g_z[px * C + c] = gz;
  }
  __shared__ float sh[8];
#pragma unroll 1
  for (int i = 0; i < 58; ++i) {
    float v = warp_sum(acc[i]);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tsum = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tsum += sh[w];
      if (i < 33) g_mats[c * 33 + i] = tsum;
      else if (i < 46) g_biases[c * 13 + (i - 33)] = tsum;
      else g_factors[c * 12 + (i - 46)] = tsum;
    }
    __syncthreads();
  }
}

}  // namespace tdvc

using namespace tdvc;

extern "C" int tdvc_eb_bits(const float* z, float* z_hat, const float* mats, const float* biases, const float* factors,
                            const float* medians, int64_t npix, int C, double* acc, void* stream) {
  TDVC_REQUIRE(z && z_hat && mats && biases && factors && medians && acc && npix > 0 && C > 0, "eb_bits: bad args");
  const size_t smem = (size_t)(33 + 13 + 12 + 1) * C * sizeof(float);
  TDVC_REQUIRE(smem <= 48 * 1024, "eb_bits: C=%d too large", C);
  const int64_t total = npix * C;
  int grid = cdiv(total, 256);
  if (grid > kNumSMs * 4) grid = kNumSMs * 4;
  eb_bits_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(z, nullptr, z_hat, mats, biases, factors, medians, total, C, acc);
  TDVC_CHECK_LAUNCH("eb_bits");
  return TDVC_OK;
}

extern "C" int tdvc_eb_bits_noise(const float* z, const float* noise, float* z_tilde, const float* mats, const float* biases,
                                  const float* factors, int64_t npix, int C, double* acc, void* stream) {
  TDVC_REQUIRE(z && noise && z_tilde && mats && biases && factors && acc && npix > 0 && C > 0, "eb_bits_noise: bad args");
  const size_t smem = (size_t)(33 + 13 + 12 + 1) * C * sizeof(float);
  TDVC_REQUIRE(smem <= 48 * 1024, "eb_bits_noise: C=%d too large", C);
  const int64_t total = npix * C;
  int grid = cdiv(total, 256);
  if (grid > kNumSMs * 4) grid = kNumSMs * 4;
  eb_bits_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(z, noise, z_tilde, mats, biases, factors, biases /* unused */, total, C, acc);
  TDVC_CHECK_LAUNCH("eb_bits_noise");
  return TDVC_OK;
}

extern "C" int tdvc_eb_aux_loss(const float* mats, const float* biases, const float* factors, const float* quantiles,
                                const float* target3, int C, float* out, void* stream) {
  TDVC_REQUIRE(mats && biases && factors && quantiles && target3 && out && C > 0, "eb_aux_loss: bad args");
  const size_t smem = (size_t)((33 + 13 + 12) * C + 256) * sizeof(float);
  TDVC_REQUIRE(smem <= 48 * 1024, "eb_aux_loss: C=%d too large", C);
  eb_aux_loss_kernel<<<1, 256, smem, (cudaStream_t)stream>>>(mats, biases, factors, quantiles, target3, C, out);
  TDVC_CHECK_LAUNCH("eb_aux_loss");
  return TDVC_OK;
}

extern "C" int tdvc_eb_aux_loss_grad(const float* mats, const float* biases, const float* factors, const float* quantiles,
                                     const float* target3, const float* grad_out, int C, float* grad_quantiles, void* stream) {
  TDVC_REQUIRE(mats && biases && factors && quantiles && target3 && grad_out && grad_quantiles && C > 0, "eb_aux_loss_grad: bad args");
  eb_aux_loss_grad_kernel<<<cdiv(3 * C, 128), 128, 0, (cudaStream_t)stream>>>(mats, biases, factors, quantiles, target3, grad_out, C,
                                                                              grad_quantiles);
  TDVC_CHECK_LAUNCH("eb_aux_loss_grad");
  return TDVC_OK;
}

extern "C" int tdvc_uniform_noise(float* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream) {
  TDVC_REQUIRE(out && n >= 0, "uniform_noise: bad args");
  if (n == 0) return TDVC_OK;
  int grid = cdiv(n / 4 + 1, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  uniform_noise_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, n, seed, stream_id, nullptr);
  TDVC_CHECK_LAUNCH("uniform_noise");
  return TDVC_OK;
}

extern "C" int tdvc_uniform_noise_dev(float* out, int64_t n, const uint64_t* seed_dev, uint64_t stream_id, void* stream) {
  TDVC_REQUIRE(out && seed_dev && n >= 0, "uniform_noise_dev: bad args");
  if (n == 0) return TDVC_OK;
  int grid = cdiv(n / 4 + 1, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  uniform_noise_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, n, 0, stream_id, seed_dev);
  TDVC_CHECK_LAUNCH("uniform_noise_dev");
  return TDVC_OK;
}

extern "C" int tdvc_gc_bits(const float* y, const float* params, int params_ld, int64_t npix, int C, double* acc, void* stream) {
  TDVC_REQUIRE(y && params && acc && npix > 0 && C > 0 && params_ld >= 2 * C, "gc_bits: bad args");
  const int64_t total = npix * C;
  int grid = cdiv(total, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  gc_bits_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(y, nullptr, params, params_ld, total, C, acc);
  TDVC_CHECK_LAUNCH("gc_bits");
  return TDVC_OK;
}

extern "C" int tdvc_gc_bits_noise(const float* y, const float* noise, const float* params, int params_ld, int64_t npix, int C,
                                  double* acc, void* stream) {
  TDVC_REQUIRE(y && noise && params && acc && npix > 0 && C > 0 && params_ld >= 2 * C, "gc_bits_noise: bad args");
  const int64_t total = npix * C;
  int grid = cdiv(total, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  gc_bits_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(y, noise, params, params_ld, total, C, acc);
  TDVC_CHECK_LAUNCH("gc_bits_noise");
  return TDVC_OK;
}

extern "C" int tdvc_eb_symbols(const float* z, int ld, const float* medians, int N, int HW, int C, int32_t* symbols,
                               int32_t* indexes, void* stream) {
  TDVC_REQUIRE(z && medians && symbols && indexes && N > 0 && HW > 0 && C > 0 && ld >= C, "eb_symbols: bad args");
  int grid = cdiv((int64_t)N * HW * C, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  eb_symbols_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(z, ld, medians, N, HW, C, symbols, indexes);
  TDVC_CHECK_LAUNCH("eb_symbols");
  return TDVC_OK;
}

extern "C" int tdvc_eb_dequantize(const int32_t* symbols, const float* medians, int N, int HW, int C, float* z_hat, int ld,
                                  void* stream) {
  TDVC_REQUIRE(symbols && medians && z_hat && N > 0 && HW > 0 && C > 0 && ld >= C, "eb_dequantize: bad args");
  int grid = cdiv((int64_t)N * HW * C, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  eb_dequantize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(symbols, medians, N, HW, C, z_hat, ld);
  TDVC_CHECK_LAUNCH("eb_dequantize");
  return TDVC_OK;
}

extern "C" int tdvc_gc_bits_backward(const float* y, const float* noise, const float* params, int params_ld, const float* grad_sum,
                                     float* grad_y, float* grad_params, int64_t npix, int C, void* stream) {
  TDVC_REQUIRE(y && noise && params && grad_sum && grad_y && grad_params && npix > 0 && C > 0 && params_ld >= 2 * C,
               "gc_bits_backward: bad args");
  const int64_t total = npix * C;
  int grid = cdiv(total, 256);
  if (grid > kNumSMs * 8) grid = kNumSMs * 8;
  gc_bits_backward_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(y, noise, params, params_ld, grad_sum, grad_y, grad_params, total, C);
  TDVC_CHECK_LAUNCH("gc_bits_backward");
  return TDVC_OK;
}

extern "C" int tdvc_eb_bits_backward(const float* z_tilde, const float* mats, const float* biases, const float* factors,
                                     const float* grad_sum, float* grad_z, float* grad_mats, float* grad_biases,
                                     float* grad_factors, int64_t npix, int C, void* stream) {
  TDVC_REQUIRE(z_tilde && mats && biases && factors && grad_sum && grad_z && grad_mats && grad_biases && grad_factors &&
                   npix > 0 && C > 0, "eb_bits_backward: bad args");
  eb_bits_backward_kernel<<<C, 256, 0, (cudaStream_t)stream>>>(z_tilde, mats, biases, factors, grad_sum, grad_z, grad_mats,
                                                               grad_biases, grad_factors, npix, C);
  TDVC_CHECK_LAUNCH("eb_bits_backward");
  return TDVC_OK;
}

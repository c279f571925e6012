// Stem: Conv1d(1->C0, k7, s2, p3) + grouped BatchNorm + ReLU + Max/AvgPool1d(3,2,1), fused.
//
// The 7-tap, single-input-channel convolution is far too thin for an MMA (K = 7), and its output
// (N,112,C0) is the largest activation of the whole network.  So it is never materialised: a CTA owns one
// BatchNorm group x 16 output channels, keeps the group's input (group x 224 fp32, zero-padded by 8 on both
// sides: 19 KB for a 20-breath sequence) in shared memory and recomputes the convolution where needed:
//   forward : mean from the 7 tap-input sums (channel independent), sweep 1 centred variance,
//             sweep 2 conv+BN+ReLU+pool -> (N,56,C0)
//   backward: from x, the saved statistics and d(pool out) only -- pool arg-max, ReLU mask, BN backward
//             and the weight gradient are all recomputed; there is no gradient w.r.t. the input.
// Every sweep walks RUNS of 28 consecutive conv outputs (= 14 pool outputs) of one breath with the 7-tap
// input window held in registers: two new inputs (one 8-byte shared-memory load, a broadcast within the
// 16 channel threads) and 7 FMAs per conv output -- the kernels are FMA-bound, not LDS-bound.
// HBM traffic: x once per channel slab (L2-resident after the first), the pooled output once.
// thread layout: 256 threads = 16 channels x 16 row lanes.
//
// Groups that do not fit in shared memory (a FLAT batch is one BatchNorm group: ResNet.forward(x), DenseNet.forward(x),
// CNNRegressor with more than ~220 breaths) are processed in CHUNKS of 64 breaths by the same device code:
//   forward : STATS pass -- every chunk CTA writes its (count, mean, centred M2) per channel; APPLY pass -- every chunk CTA
//             Chan-merges the records of its group (fixed order) and runs sweep 2 on its chunk;
//   backward: PARTIAL pass -- every chunk CTA writes its input moments and its per-channel S1, S2, G_t sums; a small combine
//             kernel adds the chunks of a group in order and applies the analytic BatchNorm / weight-gradient formula.
//             The moments and G_t are sums of x - s, with s the mean of the group's first breath when the input has a DC
//             offset (read by every chunk CTA, so their partial sums still add): with raw sums the formula cancels digits.
// The caller provides the workspace for the chunk records (stem_workspace_bytes).
//
// The second half of the file is stage 1 of the two-convolution stem (double_conv_first), see stem_alt_fwd_kernel.
#include "common.cuh"

namespace dards {

constexpr int STEM_THREADS = 256;
constexpr int STEM_CS = 16;                          // channels per CTA
constexpr int STEM_LANES = STEM_THREADS / STEM_CS;   // 16 row lanes
constexpr int STEM_L = 224, STEM_LC = 112, STEM_LP = 56, STEM_K = 7;
constexpr int STEM_PAD = 8;                          // zero floats before and after every breath in smem
constexpr int STEM_BS = STEM_L + 2 * STEM_PAD;       // 240: smem breath stride (even -> 8-byte aligned pairs)
constexpr int STEM_RUN = 28;                         // conv outputs per run; 4 runs per breath
constexpr int STEM_FUSED_GROUP = 226;                // largest group of the one-kernel path: 226 * 240 * 4 B = 212 KB of dynamic smem
constexpr int STEM_CHUNK = 64;                       // breaths per CTA on the chunked path
enum { STEM_FUSED = 0, STEM_STATS = 1, STEM_APPLY = 2, STEM_EVAL = 3 };

// 16-byte asynchronous global -> shared copy (L2-only caching: the data is read once)
__device__ __forceinline__ void stem_cp_async16(const void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void stem_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// group input -> zero-padded shared copy
__device__ __forceinline__ void stem_load_group(const float* __restrict__ xg, float* xs, int group) {
  for (int i = threadIdx.x; i < group * STEM_BS; i += STEM_THREADS) {
    const int b = i / STEM_BS, p = i % STEM_BS - STEM_PAD;
    xs[i] = (p >= 0 && p < STEM_L) ? xg[b * STEM_L + p] : 0.f;
  }
}

// sum `v` over the 16 row lanes (threads with the same channel); every thread gets the total
__device__ __forceinline__ float stem_lane_sum(float v, float* red, int c, int rl) {
  __syncthreads();
  red[rl * STEM_CS + c] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < STEM_LANES; ++r) s += red[r * STEM_CS + c];
  return s;
}

__device__ __forceinline__ float stem_dot7(const float (&w)[STEM_K], float x0, float x1, float x2, float x3, float x4,
                                           float x5, float x6) {
  float y = w[0] * x0;
  y = fmaf(w[1], x1, y);
  y = fmaf(w[2], x2, y);
  y = fmaf(w[3], x3, y);
  y = fmaf(w[4], x4, y);
  y = fmaf(w[5], x5, y);
  y = fmaf(w[6], x6, y);
  return y;
}

// X_t = sum over all conv positions of the t-th tap input (channel independent) -> xt[0..6], all threads
__device__ __forceinline__ void stem_tap_sums(const float* xs, int group, float* red /* 8*7 */, float* xt) {
  float acc[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) acc[t] = 0.f;
  const int n_conv = group * STEM_LC;
  for (int i = threadIdx.x; i < n_conv; i += STEM_THREADS) {
    const float* xb = xs + (i / STEM_LC) * STEM_BS + STEM_PAD + 2 * (i % STEM_LC) - 3;
#pragma unroll
    for (int t = 0; t < STEM_K; ++t) acc[t] += xb[t];
  }
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) acc[t] = warp_sum(acc[t]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int t = 0; t < STEM_K; ++t) red[warp * STEM_K + t] = acc[t];
  }
  __syncthreads();
  if (threadIdx.x < STEM_K) {
    float s = 0.f;
    for (int wv = 0; wv < STEM_THREADS / 32; ++wv) s += red[wv * STEM_K + threadIdx.x];
    xt[threadIdx.x] = s;
  }
  __syncthreads();
}

// MODE: STEM_FUSED (one CTA = one whole group), STEM_STATS / STEM_APPLY (one CTA = one chunk of a group; see the header),
// STEM_EVAL (one CTA = one chunk of breaths; eval-mode BatchNorm: `gamma` / `beta` carry the per-channel scale / shift)
template <typename T, int MODE>
__global__ void __launch_bounds__(STEM_THREADS)
    stem_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ gamma,
                    const float* __restrict__ beta, T* __restrict__ out, float* __restrict__ save_mean,
                    float* __restrict__ save_rstd, float* __restrict__ part, int group, int chunk, int n_chunks, int c0,
                    int out_stride, float eps, int pool) {
  extern __shared__ __align__(16) float xs[];
  __shared__ float red[STEM_THREADS];
  __shared__ float xt[STEM_K];
  const int g = blockIdx.x / n_chunks, k = blockIdx.x % n_chunks;  // fused: n_chunks = 1, chunk = group
  const int b0 = k * chunk;
  const int nb = min(chunk, group - b0);                            // breaths of this CTA
  const size_t breath0 = (size_t)g * group + b0;
  const int c = threadIdx.x % STEM_CS, rl = threadIdx.x / STEM_CS;
  const int ch = blockIdx.y * STEM_CS + c;  // c0 is a multiple of 16
  stem_load_group(x + breath0 * STEM_L, xs, nb);
  __syncthreads();
  float wr[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) wr[t] = w[ch * STEM_K + t];

  const int n_runs = nb * (STEM_LC / STEM_RUN);
  float sc, sh;
  if (MODE == STEM_EVAL) {
    sc = gamma[ch];
    sh = beta[ch];
  } else {
    float mean, var;
    if (MODE != STEM_APPLY) {
      const float inv_n = 1.f / (float)(nb * STEM_LC);
      stem_tap_sums(xs, nb, red, xt);
      mean = 0.f;
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) mean = fmaf(wr[t], xt[t], mean);
      mean *= inv_n;
      // ---- sweep 1: centred sum of squares ----------------------------------------------------------------
      float q = 0.f;
      for (int run = rl; run < n_runs; run += STEM_LANES) {
        const float* xb = xs + (run >> 2) * STEM_BS + STEM_PAD + 2 * (run & 3) * STEM_RUN - 3;
        float x0 = xb[0], x1 = xb[1], x2 = xb[2], x3 = xb[3], x4 = xb[4], x5 = xb[5], x6 = xb[6];
#pragma unroll
        for (int j = 0; j < STEM_RUN; ++j) {
          const float d = stem_dot7(wr, x0, x1, x2, x3, x4, x5, x6) - mean;
          q = fmaf(d, d, q);
          const float2 nx = *reinterpret_cast<const float2*>(xb + 7 + 2 * j);  // absolute index is even
          x0 = x2; x1 = x3; x2 = x4; x3 = x5; x4 = x6; x5 = nx.x; x6 = nx.y;
        }
      }
      const float m2 = stem_lane_sum(q, red, c, rl);
      if (MODE == STEM_STATS) {
        if (rl == 0) {
          float* r = part + (size_t)blockIdx.x * 3 * c0 + ch;
          r[0] = (float)(nb * STEM_LC);
          r[c0] = mean;
          r[2 * c0] = m2;
        }
        return;
      }
      var = m2 * inv_n + eps;
    } else {
      // Chan merge of the group's chunk records, in chunk order (every CTA of the group computes the same numbers)
      float n = 0.f, m2 = 0.f;
      mean = 0.f;
      for (int kk = 0; kk < n_chunks; ++kk) {
        const float* r = part + (size_t)(g * n_chunks + kk) * 3 * c0 + ch;
        const float ne = r[0], me = r[c0], qe = r[2 * c0];
        const float nn = n + ne, d = me - mean;
        mean += d * (ne / nn);
        m2 += qe + d * d * (n * ne / nn);
        n = nn;
      }
      var = m2 / n + eps;
    }
    float rstd = rsqrtf(var);
    rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);
    if (rl == 0 && k == 0) {
      save_mean[(size_t)g * c0 + ch] = mean;
      save_rstd[(size_t)g * c0 + ch] = rstd;
    }
    sc = rstd * gamma[ch];
    sh = beta[ch] - mean * sc;
  }

  // ---- sweep 2: conv + BN + ReLU + pool; run = 14 pool outputs = conv positions 2*lp0-1 .. 2*lp0+27 ----------
  for (int run = rl; run < n_runs; run += STEM_LANES) {
    const int b = run >> 2, lp0 = (run & 3) * (STEM_RUN / 2);
    const float* xb = xs + b * STEM_BS + STEM_PAD + 2 * (2 * lp0 - 1) - 3;
    float x0 = xb[0], x1 = xb[1], x2 = xb[2], x3 = xb[3], x4 = xb[4], x5 = xb[5], x6 = xb[6];
    // ReLU output >= 0, so 0 is the identity of the max as well as of the (count_include_pad) sum
    float zl = lp0 == 0 ? 0.f : fmaxf(fmaf(stem_dot7(wr, x0, x1, x2, x3, x4, x5, x6), sc, sh), 0.f);
    T* op = out + ((breath0 + b) * STEM_LP + lp0) * out_stride + ch;
#pragma unroll
    for (int j = 0; j < STEM_RUN / 2; ++j) {
      float2 nx = *reinterpret_cast<const float2*>(xb + 7 + 4 * j);
      x0 = x2; x1 = x3; x2 = x4; x3 = x5; x4 = x6; x5 = nx.x; x6 = nx.y;
      const float zm = fmaxf(fmaf(stem_dot7(wr, x0, x1, x2, x3, x4, x5, x6), sc, sh), 0.f);
      nx = *reinterpret_cast<const float2*>(xb + 9 + 4 * j);
      x0 = x2; x1 = x3; x2 = x4; x3 = x5; x4 = x6; x5 = nx.x; x6 = nx.y;
      const float zr = fmaxf(fmaf(stem_dot7(wr, x0, x1, x2, x3, x4, x5, x6), sc, sh), 0.f);
      const float o = pool == 0 ? fmaxf(fmaxf(zl, zm), zr) : (zl + zm + zr) * (1.f / 3.f);
      Elem<T>::st(op + (size_t)j * out_stride, o);
      zl = zr;
    }
  }
}

// number of distinct entries of the symmetric 7x7 autocorrelation matrix
constexpr int STEM_NR = STEM_K * (STEM_K + 1) / 2;  // 28
__device__ __forceinline__ int stem_r_index(int a, int b) {  // a <= b
  return a * STEM_K - a * (a - 1) / 2 + (b - a);
}

// s, the shift of the backward's input moments (xb: the group's first breath): that breath's mean when it exceeds the
// breath's spread (mean^2 > var), else 0.  Below that ratio the raw sums lose less than a digit, and s = 0 leaves the
// arithmetic exactly that of the unshifted sums (x - 0 = x, mean - 0 * sum w = mean), so centred data such as z-scored
// flow computes what it always computed.  Every CTA that needs s (the chunk CTAs of a group and the combine kernel) runs
// this same sequence -- seven warp sums of 32 samples, added in order, products rounded on their own -- so they agree bit
// for bit.  All threads of the block call it; red: 16 floats of shared memory no other code touches until the next barrier.
__device__ __forceinline__ float stem_group_shift(const float* __restrict__ xb, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int vw = warp; vw < STEM_L / 32; vw += blockDim.x >> 5) {
    const float v = xb[vw * 32 + lane];
    const float s1 = warp_sum(v), s2 = warp_sum(__fmul_rn(v, v));
    if (lane == 0) {
      red[vw] = s1;
      red[8 + vw] = s2;
    }
  }
  __syncthreads();
  float s1 = 0.f, s2 = 0.f;
  for (int vw = 0; vw < STEM_L / 32; ++vw) {
    s1 += red[vw];
    s2 += red[8 + vw];
  }
  const float m = __fmul_rn(s1, 1.f / (float)STEM_L);
  const float var = __fsub_rn(__fmul_rn(s2, 1.f / (float)STEM_L), __fmul_rn(m, m));
  return __fmul_rn(m, m) > var ? m : 0.f;
}

// H_t / rstd = sum_a w_a R'[a][t] - mean_s X'_t, with xr = X' (7) then R' (28), sums of x - s, and mean_s = mean - s sum_a w_a
// the mean of the convolution of x - s
__device__ __forceinline__ float stem_h_over_rstd(const float (&w)[STEM_K], const float* xr, int t, float mean_s) {
  float wr_r = 0.f;
#pragma unroll
  for (int a = 0; a < STEM_K; ++a) {
    const int lo = a < t ? a : t, hi = a < t ? t : a;
    wr_r = fmaf(w[a], xr[STEM_K + stem_r_index(lo, hi)], wr_r);
  }
  return wr_r - mean_s * xr[t];
}

__device__ __forceinline__ float stem_shifted_mean(const float (&w)[STEM_K], float mean, float shift) {
  float wsum = 0.f;
#pragma unroll
  for (int a = 0; a < STEM_K; ++a) wsum += w[a];
  return fmaf(-shift, wsum, mean);
}

// STAGE: the CTA's slice of dout (group x 56 rows x 16 channels) is brought into shared memory with cp.async while the
// input moments are computed, and sweep B reads it from there.  With the gradient loaded from global memory inside the
// sweep the kernel spent most of its time waiting on those loads (ncu: long-scoreboard stalls 5.9 per issue, issue
// slots 47 % busy).  Groups too large for the extra 35 KB per 20 breaths use the direct path.
// PARTIAL: one CTA = one chunk of a group; the moments and the per-channel sums go to the workspace instead of through
// section C (stem_bwd_combine_kernel finishes the group).
// FROZEN (the STEM_FROZEN backward of a network in train() whose BatchNorm is in eval()): constant statistics; one CTA = one
// chunk of breaths (n_chunks chunks of a single "group" of all breaths).  `gamma` / `beta` carry the per-channel scale / shift
// that dards_stem_eval_fwd applied, `save_mean` / `save_rstd` the running_mean and 1/sqrt(running_var + eps).  The pre-pool
// values are recomputed with exactly STEM_EVAL's arithmetic, fmaxf(fmaf(stem_dot7(..), scale, shift), 0), so the max-pool
// arg-max is the forward's.  No input moments are needed: dy = scale * g, so dW_t = scale * G_t; the chunk's S1 (dbeta),
// S2 (dgamma) and scale * G_t (dW) are written as partials, row blockIdx.x, for the batched row reduction.
template <typename T, bool STAGE, bool PARTIAL, bool FROZEN = false>
__global__ void __launch_bounds__(STEM_THREADS)
    stem_bwd_kernel(const T* __restrict__ dout, const float* __restrict__ x, const float* __restrict__ w,
                    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ save_mean,
                    const float* __restrict__ save_rstd, float* __restrict__ dw_part, float* __restrict__ dgamma_part,
                    float* __restrict__ dbeta_part, float* __restrict__ mom_part, float* __restrict__ ch_part, int group_all,
                    int chunk, int n_chunks, int c0, int dout_stride, int pool) {
  extern __shared__ __align__(16) float xs[];
  __shared__ float red[STEM_THREADS * 9];
  __shared__ float xr[STEM_K + STEM_NR];  // X_t (7) then R (28)
  const int g = blockIdx.x / n_chunks, kc = blockIdx.x % n_chunks;  // fused: n_chunks = 1, chunk = group
  const int b0 = kc * chunk;
  const int group = min(chunk, group_all - b0);                      // breaths of this CTA
  const size_t breath0 = (size_t)g * group_all + b0;
  const int tid = threadIdx.x;
  const int c = tid % STEM_CS, rl = tid / STEM_CS;
  const int ch = blockIdx.y * STEM_CS + c;
  T* ds = reinterpret_cast<T*>(xs + (size_t)group * STEM_BS);  // [group*56][16] staged dout slice (STAGE only)
  if (STAGE) {
    constexpr int EPC = 16 / (int)sizeof(T);           // elements per 16-byte chunk
    constexpr int CPR = STEM_CS / EPC;                 // chunks per row: 2 (bf16) or 4 (fp32)
    const T* src = dout + breath0 * STEM_LP * dout_stride + blockIdx.y * STEM_CS;
    const int n_vec = group * STEM_LP * CPR;
    for (int q = tid; q < n_vec; q += STEM_THREADS) {
      const int row = q / CPR, part = q % CPR;
      stem_cp_async16(ds + row * STEM_CS + part * EPC, src + (size_t)row * dout_stride + part * EPC);
    }
  }
  // the shift s of the moments, from the group's first breath in global memory (red's tail is free until section B)
  const float shift = FROZEN ? 0.f : stem_group_shift(x + (size_t)g * group_all * STEM_L, red + STEM_THREADS * 8);
  stem_load_group(x + breath0 * STEM_L, xs, group);
  __syncthreads();
  const int n_conv = group * STEM_LC;

  // ---- A. channel-independent input moments about s: X'_t = sum (xin_t - s), R'[a][b] = sum (xin_a - s)(xin_b - s) --
  if (!FROZEN) {
    float acc[STEM_K + STEM_NR];
#pragma unroll
    for (int i = 0; i < STEM_K + STEM_NR; ++i) acc[i] = 0.f;
    for (int i = tid; i < n_conv; i += STEM_THREADS) {
      const float* xb = xs + (i / STEM_LC) * STEM_BS + STEM_PAD + 2 * (i % STEM_LC) - 3;
      float xin[STEM_K];
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) xin[t] = xb[t] - shift;
      int k = STEM_K;
#pragma unroll
      for (int a = 0; a < STEM_K; ++a) {
        acc[a] += xin[a];
#pragma unroll
        for (int b = a; b < STEM_K; ++b) {
          acc[k] = fmaf(xin[a], xin[b], acc[k]);
          ++k;
        }
      }
    }
    // block reduce: warp shuffle, then 8 warps through smem
#pragma unroll
    for (int i = 0; i < STEM_K + STEM_NR; ++i) acc[i] = warp_sum(acc[i]);
    const int warp = tid >> 5, lane = tid & 31;
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < STEM_K + STEM_NR; ++i) red[warp * (STEM_K + STEM_NR) + i] = acc[i];
    }
    __syncthreads();
    if (tid < STEM_K + STEM_NR) {
      float s = 0.f;
      for (int wv = 0; wv < STEM_THREADS / 32; ++wv) s += red[wv * (STEM_K + STEM_NR) + tid];
      xr[tid] = s;
      if (PARTIAL && blockIdx.y == 0) mom_part[(size_t)blockIdx.x * (STEM_K + STEM_NR) + tid] = s;
    }
    __syncthreads();
  }

  // ---- B. per channel: S1 = sum g, S2 = sum g*xhat, G'_t = sum g * (xin_t - s) (FROZEN: G_t = sum g * xin_t) -------
  // run = 14 pool outputs; the 11-element input window x[4lp-5 .. 4lp+5] of the three conv positions feeding
  // pool output lp (2lp-1, 2lp, 2lp+1) stays in registers and slides by 4 per pool output; xd is the same window less s.
  float wr[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) wr[t] = w[ch * STEM_K + t];
  const float mean = save_mean[(size_t)g * c0 + ch], rstd = save_rstd[(size_t)g * c0 + ch];
  const float gm = gamma[ch];
  const float sc = FROZEN ? gm : rstd * gm, sh = FROZEN ? beta[ch] : beta[ch] - mean * sc;
  float s1 = 0.f, s2 = 0.f, gt[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) gt[t] = 0.f;
  const int n_runs = group * (STEM_LC / STEM_RUN);
  if (STAGE) {
    stem_cp_async_wait_all();
    __syncthreads();  // every thread's chunks have landed
  }
  const int dp_stride = STAGE ? STEM_CS : dout_stride;
  for (int run = rl; run < n_runs; run += STEM_LANES) {
    const int b = run >> 2, lp0 = (run & 3) * (STEM_RUN / 2);
    const float* xb = xs + b * STEM_BS + STEM_PAD + 4 * lp0 - 5;  // xw[i] = xb[i + 4j]
    const T* dp_ptr = STAGE ? ds + (b * STEM_LP + lp0) * STEM_CS + c
                            : dout + ((breath0 + b) * STEM_LP + lp0) * dout_stride + ch;
    float xw[11], xd[11];
#pragma unroll
    for (int i = 0; i < 7; ++i) {
      xw[i] = xb[i];
      xd[i] = FROZEN ? xw[i] : xw[i] - shift;
    }
    float yl = stem_dot7(wr, xw[0], xw[1], xw[2], xw[3], xw[4], xw[5], xw[6]);
    bool okl = lp0 != 0;  // conv position -1 does not exist
#pragma unroll
    for (int j = 0; j < STEM_RUN / 2; ++j) {
      const float dp = Elem<T>::ld(dp_ptr + (size_t)j * dp_stride);
      const float2 n0 = *reinterpret_cast<const float2*>(xb + 7 + 4 * j);
      const float2 n1 = *reinterpret_cast<const float2*>(xb + 9 + 4 * j);
      xw[7] = n0.x; xw[8] = n0.y; xw[9] = n1.x; xw[10] = n1.y;
#pragma unroll
      for (int i = 7; i < 11; ++i) xd[i] = FROZEN ? xw[i] : xw[i] - shift;
      const float ym = stem_dot7(wr, xw[2], xw[3], xw[4], xw[5], xw[6], xw[7], xw[8]);
      const float yr = stem_dot7(wr, xw[4], xw[5], xw[6], xw[7], xw[8], xw[9], xw[10]);
      const float zl = okl ? fmaxf(fmaf(yl, sc, sh), 0.f) : 0.f;
      const float zm = fmaxf(fmaf(ym, sc, sh), 0.f);
      const float zr = fmaxf(fmaf(yr, sc, sh), 0.f);
      float gl, gmid, gr;
      if (pool == 0) {
        // first strict maximum wins (ATen max_pool semantics); a zero maximum carries no gradient (ReLU)
        const bool wl = zl > 0.f;
        const bool wm = zm > (wl ? zl : 0.f);
        const float best = wm ? zm : (wl ? zl : 0.f);
        const bool wrt = zr > best;
        gl = (wl && !wm && !wrt) ? dp : 0.f;
        gmid = (wm && !wrt) ? dp : 0.f;
        gr = wrt ? dp : 0.f;
      } else {
        const float d3 = dp * (1.f / 3.f);
        gl = zl > 0.f ? d3 : 0.f;
        gmid = zm > 0.f ? d3 : 0.f;
        gr = zr > 0.f ? d3 : 0.f;
      }
      s1 += gl + gmid + gr;
      s2 = fmaf(gl, (yl - mean) * rstd, s2);
      s2 = fmaf(gmid, (ym - mean) * rstd, s2);
      s2 = fmaf(gr, (yr - mean) * rstd, s2);
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) {
        gt[t] = fmaf(gl, xd[t], gt[t]);
        gt[t] = fmaf(gmid, xd[t + 2], gt[t]);
        gt[t] = fmaf(gr, xd[t + 4], gt[t]);
      }
      // slide by 4 inputs = 2 conv positions
#pragma unroll
      for (int i = 0; i < 7; ++i) {
        xw[i] = xw[i + 4];
        xd[i] = xd[i + 4];
      }
      yl = yr;
      okl = true;
    }
  }
  // reduce the 9 accumulators over the row lanes
  __syncthreads();
  red[tid * 9 + 0] = s1;
  red[tid * 9 + 1] = s2;
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) red[tid * 9 + 2 + t] = gt[t];
  __syncthreads();
  if (rl == 0) {
    s1 = 0.f;
    s2 = 0.f;
#pragma unroll
    for (int t = 0; t < STEM_K; ++t) gt[t] = 0.f;
    for (int r = 0; r < STEM_LANES; ++r) {
      const int o = (r * STEM_CS + c) * 9;
      s1 += red[o + 0];
      s2 += red[o + 1];
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) gt[t] += red[o + 2 + t];
    }
    if (PARTIAL) {
      float* o = ch_part + (size_t)blockIdx.x * 9 * c0 + ch;
      o[0] = s1;
      o[c0] = s2;
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) o[(size_t)(2 + t) * c0] = gt[t];
      return;
    }
    if (FROZEN) {
      const size_t o = (size_t)blockIdx.x * c0 + ch;
      dbeta_part[o] = s1;
      dgamma_part[o] = s2;
#pragma unroll
      for (int t = 0; t < STEM_K; ++t) dw_part[o * STEM_K + t] = sc * gt[t];
      return;
    }
    // ---- C. BN backward folded into the weight gradient ------------------------------------------------
    // dy = gamma*rstd*(g - S1/n - xhat*S2/n);  dW_t = sum dy*xin_t = sum dy*(xin_t - s), because sum dy = 0
    //    = gamma*rstd*(G'_t - S1/n * X'_t - S2/n * H_t),  H_t = sum xhat*(xin_t - s) = rstd*(sum_a w_a R'[a][t] - mean_s*X'_t)
    // (y - mean = sum_a w_a (xin_a - s) - mean_s, mean_s = mean - s * sum_a w_a)
    const float inv_n = 1.f / (float)n_conv;
    const float mean_s = stem_shifted_mean(wr, mean, shift);
    dbeta_part[(size_t)g * c0 + ch] = s1;
    dgamma_part[(size_t)g * c0 + ch] = s2;
#pragma unroll
    for (int t = 0; t < STEM_K; ++t) {
      const float h = rstd * stem_h_over_rstd(wr, xr, t, mean_s);
      dw_part[((size_t)g * c0 + ch) * STEM_K + t] = sc * (gt[t] - s1 * inv_n * xr[t] - s2 * inv_n * h);
    }
  }
}

// chunked backward, second pass: thread = channel of one group; adds the chunk partials (sums about the group's shift s) in
// order and applies section C
__global__ void __launch_bounds__(128)
    stem_bwd_combine_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ gamma,
                            const float* __restrict__ save_mean, const float* __restrict__ save_rstd,
                            const float* __restrict__ mom_part, const float* __restrict__ ch_part, float* __restrict__ dw_part,
                            float* __restrict__ dgamma_part, float* __restrict__ dbeta_part, int group, int n_chunks, int c0) {
  __shared__ float xr[STEM_K + STEM_NR];
  __shared__ float shift_red[16];
  const int g = blockIdx.x;
  const float shift = stem_group_shift(x + (size_t)g * group * STEM_L, shift_red);  // the partial CTAs' s
  if (threadIdx.x < STEM_K + STEM_NR) {
    float s = 0.f;
    for (int k = 0; k < n_chunks; ++k) s += mom_part[(size_t)(g * n_chunks + k) * (STEM_K + STEM_NR) + threadIdx.x];
    xr[threadIdx.x] = s;
  }
  __syncthreads();
  const int ch = blockIdx.y * 128 + threadIdx.x;
  if (ch >= c0) return;
  float s1 = 0.f, s2 = 0.f, gt[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) gt[t] = 0.f;
  for (int k = 0; k < n_chunks; ++k) {
    const float* o = ch_part + (size_t)(g * n_chunks + k) * 9 * c0 + ch;
    s1 += o[0];
    s2 += o[c0];
#pragma unroll
    for (int t = 0; t < STEM_K; ++t) gt[t] += o[(size_t)(2 + t) * c0];
  }
  float wr[STEM_K];
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) wr[t] = w[ch * STEM_K + t];
  const float mean = save_mean[(size_t)g * c0 + ch], rstd = save_rstd[(size_t)g * c0 + ch];
  const float sc = rstd * gamma[ch];
  const float inv_n = 1.f / (float)(group * STEM_LC);
  const float mean_s = stem_shifted_mean(wr, mean, shift);
  dbeta_part[(size_t)g * c0 + ch] = s1;
  dgamma_part[(size_t)g * c0 + ch] = s2;
#pragma unroll
  for (int t = 0; t < STEM_K; ++t) {
    const float h = rstd * stem_h_over_rstd(wr, xr, t, mean_s);
    dw_part[((size_t)g * c0 + ch) * STEM_K + t] = sc * (gt[t] - s1 * inv_n * xr[t] - s2 * inv_n * h);
  }
}

static bool stem_c0_ok(int c0) { return c0 > 0 && c0 % STEM_CS == 0; }

template <typename K>
static int stem_smem_optin(K kernel, size_t smem, size_t* granted) {
  if (smem <= *granted) return DARDS_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) {
    set_error("stem: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
    return DARDS_ERR_CUDA;
  }
  *granted = smem;
  return DARDS_OK;
}

static int stem_n_chunks(int group) { return group <= STEM_FUSED_GROUP ? 1 : ceil_div(group, STEM_CHUNK); }

// bytes of workspace the chunked path needs (0: the group fits the one-kernel path).  backward: 0 | 1
long long stem_workspace_bytes(int n_groups, int group, int c0, int backward) {
  const int nc = stem_n_chunks(group);
  if (nc == 1 || n_groups <= 0 || c0 <= 0) return 0;
  const long long recs = (long long)n_groups * nc;
  return (backward ? recs * (9LL * c0 + STEM_K + STEM_NR) : recs * 3LL * c0) * (long long)sizeof(float);
}

int launch_stem_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out, float* save_mean,
                    float* save_rstd, int n_groups, int group, int c0, int out_stride, float eps, int pool, void* workspace,
                    long long workspace_bytes, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  DARDS_CHECK_ARG(group > 0, "stem: BatchNorm group must be at least 1 breath (got %d)", group);
  if (n_groups == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem: grid too large");
  const int nc = stem_n_chunks(group);
  if (nc == 1) {
    const size_t smem = (size_t)group * STEM_BS * sizeof(float);
    dim3 grid(n_groups, c0 / STEM_CS);
    static size_t granted[2] = {44 * 1024, 44 * 1024};  // 1 KB of static smem on top
    DARDS_DISPATCH_DTYPE(dtype, {
      int rc = stem_smem_optin(stem_fwd_kernel<T, STEM_FUSED>, smem, &granted[dtype == DARDS_BF16 ? 1 : 0]);
      if (rc) return rc;
      stem_fwd_kernel<T, STEM_FUSED><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                      save_rstd, nullptr, group, group, 1, c0, out_stride,
                                                                      eps, pool);
    })
    DARDS_CHECK_LAUNCH("stem_fwd");
    return DARDS_OK;
  }
  const long long need = stem_workspace_bytes(n_groups, group, c0, 0);
  DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need,
                  "stem_fwd: a BatchNorm group of %d breaths runs in chunks and needs %lld bytes of workspace (got %lld)", group,
                  need, workspace_bytes);
  DARDS_CHECK_ARG((long long)n_groups * nc <= 0x7fffffffLL, "stem: grid too large");
  float* part = static_cast<float*>(workspace);
  const size_t smem = (size_t)STEM_CHUNK * STEM_BS * sizeof(float);
  dim3 grid((unsigned)(n_groups * nc), c0 / STEM_CS);
  static size_t granted[4] = {44 * 1024, 44 * 1024, 44 * 1024, 44 * 1024};
  DARDS_DISPATCH_DTYPE(dtype, {
    const int slot = dtype == DARDS_BF16 ? 1 : 0;
    int rc = stem_smem_optin(stem_fwd_kernel<T, STEM_STATS>, smem, &granted[slot]);
    if (rc) return rc;
    rc = stem_smem_optin(stem_fwd_kernel<T, STEM_APPLY>, smem, &granted[2 + slot]);
    if (rc) return rc;
    stem_fwd_kernel<T, STEM_STATS><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                    save_rstd, part, group, STEM_CHUNK, nc, c0, out_stride,
                                                                    eps, pool);
    DARDS_CHECK_LAUNCH("stem_fwd (chunk statistics)");
    stem_fwd_kernel<T, STEM_APPLY><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                    save_rstd, part, group, STEM_CHUNK, nc, c0, out_stride,
                                                                    eps, pool);
  })
  DARDS_CHECK_LAUNCH("stem_fwd (chunk apply)");
  return DARDS_OK;
}

int launch_stem_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out, int n_breaths,
                         int c0, int out_stride, int pool, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  if (n_breaths == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem: grid too large");
  const int nc = ceil_div(n_breaths, STEM_CHUNK);
  const size_t smem = (size_t)STEM_CHUNK * STEM_BS * sizeof(float);
  dim3 grid((unsigned)nc, c0 / STEM_CS);
  static size_t granted[2] = {44 * 1024, 44 * 1024};
  DARDS_DISPATCH_DTYPE(dtype, {
    int rc = stem_smem_optin(stem_fwd_kernel<T, STEM_EVAL>, smem, &granted[dtype == DARDS_BF16 ? 1 : 0]);
    if (rc) return rc;
    stem_fwd_kernel<T, STEM_EVAL><<<grid, STEM_THREADS, smem, st>>>(x, w, scale, shift, static_cast<T*>(out), nullptr, nullptr,
                                                                   nullptr, n_breaths, STEM_CHUNK, nc, c0, out_stride, 0.f,
                                                                   pool);
  })
  DARDS_CHECK_LAUNCH("stem_eval_fwd");
  return DARDS_OK;
}

template <typename T>
struct StemBwdArgs {
  const T* dout;
  const float *x, *w, *gamma, *beta, *save_mean, *save_rstd;
  float *dw_part, *dgamma_part, *dbeta_part, *mom_part, *ch_part;
  int group, chunk, n_chunks, c0, dout_stride, pool;
};

template <typename T, bool STAGE, bool PARTIAL, bool FROZEN = false>
static int stem_bwd_run(const StemBwdArgs<T>& a, dim3 grid, size_t smem, cudaStream_t st) {
  static size_t granted = 36 * 1024;  // 9.4 KB of static smem on top
  int rc = stem_smem_optin(stem_bwd_kernel<T, STAGE, PARTIAL, FROZEN>, smem, &granted);
  if (rc) return rc;
  stem_bwd_kernel<T, STAGE, PARTIAL, FROZEN><<<grid, STEM_THREADS, smem, st>>>(a.dout, a.x, a.w, a.gamma, a.beta, a.save_mean,
                                                                      a.save_rstd, a.dw_part, a.dgamma_part, a.dbeta_part,
                                                                      a.mom_part, a.ch_part, a.group, a.chunk, a.n_chunks,
                                                                      a.c0, a.dout_stride, a.pool);
  return DARDS_OK;
}

int launch_stem_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* beta,
                    const float* save_mean, const float* save_rstd, float* dw_part, float* dgamma_part,
                    float* dbeta_part, int n_groups, int group, int c0, int dout_stride, int pool, void* workspace,
                    long long workspace_bytes, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  DARDS_CHECK_ARG(group > 0, "stem: BatchNorm group must be at least 1 breath (got %d)", group);
  if (n_groups == 0) return DARDS_OK;
  const int nc = stem_n_chunks(group);
  const int chunk = nc == 1 ? group : STEM_CHUNK;
  float* mom_part = nullptr;
  float* ch_part = nullptr;
  if (nc > 1) {
    const long long need = stem_workspace_bytes(n_groups, group, c0, 1);
    DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need,
                    "stem_bwd: a BatchNorm group of %d breaths runs in chunks and needs %lld bytes of workspace (got %lld)",
                    group, need, workspace_bytes);
    DARDS_CHECK_ARG((long long)n_groups * nc <= 0x7fffffffLL, "stem: grid too large");
    ch_part = static_cast<float*>(workspace);
    mom_part = ch_part + (size_t)n_groups * nc * 9 * c0;
  }
  const size_t smem_x = (size_t)chunk * STEM_BS * sizeof(float);
  dim3 grid((unsigned)(n_groups * nc), c0 / STEM_CS);
  int rc = DARDS_OK;
  DARDS_DISPATCH_DTYPE(dtype, {
    // staged gradient slice: 16-byte aligned rows, and room for it next to the input (3 CTAs per SM at group 20)
    const size_t smem_d = (size_t)chunk * STEM_LP * STEM_CS * sizeof(T);
    const bool stage = (dout_stride * sizeof(T)) % 16 == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0 &&
                       smem_x + smem_d <= 200 * 1024;
    const size_t smem = smem_x + (stage ? smem_d : 0);
    const StemBwdArgs<T> a = {static_cast<const T*>(dout), x, w, gamma, beta, save_mean, save_rstd, dw_part, dgamma_part,
                              dbeta_part, mom_part, ch_part, group, chunk, nc, c0, dout_stride, pool};
    if (nc > 1) rc = stage ? stem_bwd_run<T, true, true>(a, grid, smem, st) : stem_bwd_run<T, false, true>(a, grid, smem, st);
    else rc = stage ? stem_bwd_run<T, true, false>(a, grid, smem, st) : stem_bwd_run<T, false, false>(a, grid, smem, st);
  })
  if (rc) return rc;
  DARDS_CHECK_LAUNCH("stem_bwd");
  if (nc > 1) {
    dim3 cgrid(n_groups, ceil_div(c0, 128));
    stem_bwd_combine_kernel<<<cgrid, 128, 0, st>>>(x, w, gamma, save_mean, save_rstd, mom_part, ch_part, dw_part, dgamma_part,
                                                   dbeta_part, group, nc, c0);
    DARDS_CHECK_LAUNCH("stem_bwd (chunk combine)");
  }
  return DARDS_OK;
}

int stem_frozen_chunks(int n_breaths) { return n_breaths > 0 ? ceil_div(n_breaths, STEM_CHUNK) : 0; }

int launch_stem_frozen_bwd(const void* dout, const float* x, const float* w, const float* scale, const float* shift,
                           const float* running_mean, const float* rstd, float* dw_part, float* dgamma_part,
                           float* dbeta_part, int n_breaths, int c0, int dout_stride, int pool, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  if (n_breaths == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem: grid too large");
  const int nc = stem_frozen_chunks(n_breaths);
  const size_t smem_x = (size_t)STEM_CHUNK * STEM_BS * sizeof(float);
  dim3 grid((unsigned)nc, c0 / STEM_CS);
  int rc = DARDS_OK;
  DARDS_DISPATCH_DTYPE(dtype, {
    const size_t smem_d = (size_t)STEM_CHUNK * STEM_LP * STEM_CS * sizeof(T);
    const bool stage = (dout_stride * sizeof(T)) % 16 == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0 &&
                       smem_x + smem_d <= 200 * 1024;
    const size_t smem = smem_x + (stage ? smem_d : 0);
    const StemBwdArgs<T> a = {static_cast<const T*>(dout), x, w, scale, shift, running_mean, rstd, dw_part, dgamma_part,
                              dbeta_part, nullptr, nullptr, n_breaths, STEM_CHUNK, nc, c0, dout_stride, pool};
    rc = stage ? stem_bwd_run<T, true, false, true>(a, grid, smem, st) : stem_bwd_run<T, false, false, true>(a, grid, smem, st);
  })
  if (rc) return rc;
  DARDS_CHECK_LAUNCH("stem_frozen_bwd");
  return DARDS_OK;
}


// ==== stage 1 of the two-convolution stem (ResNet double_conv_first=True, resnet.py:145-147) ===========================
// a0 = bn1(conv1_alt(x)): Conv1d(1->C0, k3, s1, p1) + grouped BatchNorm, no ReLU, no pool; x (N,224) fp32 -> a0 (N,224,C0)
// channels-last in the plan dtype.  a0 is materialised: the following Conv1d(C0->C0, k7, s2, p3) runs on the generic
// convolution kernels, and it zero-pads a0 (the BatchNorm output), so the two convolutions do not fold into one.
// Same CTA layout, chunking and Chan merge as the stem above (group x 16 channels per CTA, x staged in shared memory);
// every sweep walks runs of 32 positions with the 3-tap window in registers.
constexpr int S1_K = 3;
constexpr int S1_RUN = 32;                      // positions per run: 7 runs per breath
constexpr int S1_RUNS = STEM_L / S1_RUN;
constexpr int S1_NR = S1_K * (S1_K + 1) / 2;    // distinct entries of the 3x3 autocorrelation matrix: 6
constexpr int S1_NM = S1_K + S1_NR;             // input moments: X_t (3) then R (6)
constexpr int S1_NC = 2 + S1_K;                 // per-channel backward sums: S1, S2, G_t (3)

__device__ __forceinline__ int s1_r_index(int a, int b) { return a * S1_K - a * (a - 1) / 2 + (b - a); }  // a <= b

// MODE: STEM_FUSED / STEM_STATS / STEM_APPLY / STEM_EVAL, as stem_fwd_kernel
template <typename T, int MODE>
__global__ void __launch_bounds__(STEM_THREADS)
    stem_alt_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ gamma,
                        const float* __restrict__ beta, T* __restrict__ out, float* __restrict__ save_mean,
                        float* __restrict__ save_rstd, float* __restrict__ part, int group, int chunk, int n_chunks, int c0,
                        int out_stride, float eps) {
  extern __shared__ __align__(16) float xs[];
  __shared__ float red[STEM_THREADS];
  __shared__ float xt[S1_K];
  const int g = blockIdx.x / n_chunks, k = blockIdx.x % n_chunks;
  const int b0 = k * chunk;
  const int nb = min(chunk, group - b0);
  const size_t breath0 = (size_t)g * group + b0;
  const int c = threadIdx.x % STEM_CS, rl = threadIdx.x / STEM_CS;
  const int ch = blockIdx.y * STEM_CS + c;
  stem_load_group(x + breath0 * STEM_L, xs, nb);
  __syncthreads();
  const float w0 = w[ch * S1_K], w1 = w[ch * S1_K + 1], w2 = w[ch * S1_K + 2];
  const int n_runs = nb * S1_RUNS;
  float sc, sh;
  if (MODE == STEM_EVAL) {
    sc = gamma[ch];
    sh = beta[ch];
  } else {
    float mean, var;
    if (MODE != STEM_APPLY) {
      const float inv_n = 1.f / (float)(nb * STEM_L);
      // X_t = sum over positions of x[l + t - 1] (channel independent)
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      for (int i = threadIdx.x; i < nb * STEM_L; i += STEM_THREADS) {
        const float* xb = xs + (i / STEM_L) * STEM_BS + STEM_PAD + (i % STEM_L) - 1;
        a0 += xb[0];
        a1 += xb[1];
        a2 += xb[2];
      }
      a0 = warp_sum(a0);
      a1 = warp_sum(a1);
      a2 = warp_sum(a2);
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      if (lane == 0) {
        red[warp * S1_K] = a0;
        red[warp * S1_K + 1] = a1;
        red[warp * S1_K + 2] = a2;
      }
      __syncthreads();
      if (threadIdx.x < S1_K) {
        float s = 0.f;
        for (int wv = 0; wv < STEM_THREADS / 32; ++wv) s += red[wv * S1_K + threadIdx.x];
        xt[threadIdx.x] = s;
      }
      __syncthreads();
      mean = fmaf(w0, xt[0], fmaf(w1, xt[1], w2 * xt[2])) * inv_n;
      // centred sum of squares
      float q = 0.f;
      for (int run = rl; run < n_runs; run += STEM_LANES) {
        const float* xb = xs + (run / S1_RUNS) * STEM_BS + STEM_PAD + (run % S1_RUNS) * S1_RUN - 1;
        float x0 = xb[0], x1 = xb[1];
#pragma unroll 8
        for (int j = 0; j < S1_RUN; ++j) {
          const float x2 = xb[j + 2];
          const float d = fmaf(w0, x0, fmaf(w1, x1, w2 * x2)) - mean;
          q = fmaf(d, d, q);
          x0 = x1;
          x1 = x2;
        }
      }
      const float m2 = stem_lane_sum(q, red, c, rl);
      if (MODE == STEM_STATS) {
        if (rl == 0) {
          float* r = part + (size_t)blockIdx.x * 3 * c0 + ch;
          r[0] = (float)(nb * STEM_L);
          r[c0] = mean;
          r[2 * c0] = m2;
        }
        return;
      }
      var = m2 * inv_n + eps;
    } else {
      float n = 0.f, m2 = 0.f;
      mean = 0.f;
      for (int kk = 0; kk < n_chunks; ++kk) {
        const float* r = part + (size_t)(g * n_chunks + kk) * 3 * c0 + ch;
        const float ne = r[0], me = r[c0], qe = r[2 * c0];
        const float nn = n + ne, d = me - mean;
        mean += d * (ne / nn);
        m2 += qe + d * d * (n * ne / nn);
        n = nn;
      }
      var = m2 / n + eps;
    }
    float rstd = rsqrtf(var);
    rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);
    if (rl == 0 && k == 0) {
      save_mean[(size_t)g * c0 + ch] = mean;
      save_rstd[(size_t)g * c0 + ch] = rstd;
    }
    sc = rstd * gamma[ch];
    sh = beta[ch] - mean * sc;
  }
  for (int run = rl; run < n_runs; run += STEM_LANES) {
    const int b = run / S1_RUNS, l0 = (run % S1_RUNS) * S1_RUN;
    const float* xb = xs + b * STEM_BS + STEM_PAD + l0 - 1;
    T* op = out + ((breath0 + b) * STEM_L + l0) * out_stride + ch;
    float x0 = xb[0], x1 = xb[1];
#pragma unroll 8
    for (int j = 0; j < S1_RUN; ++j) {
      const float x2 = xb[j + 2];
      Elem<T>::st(op + (size_t)j * out_stride, fmaf(fmaf(w0, x0, fmaf(w1, x1, w2 * x2)), sc, sh));
      x0 = x1;
      x1 = x2;
    }
  }
}

// H_t / rstd = sum_a w_a R'[a][t] - mean_s X'_t (as stem_h_over_rstd, 3 taps)
__device__ __forceinline__ float s1_h_over_rstd(const float (&w)[S1_K], const float* xr, int t, float mean_s) {
  float wr_r = 0.f;
#pragma unroll
  for (int a = 0; a < S1_K; ++a) {
    const int lo = a < t ? a : t, hi = a < t ? t : a;
    wr_r = fmaf(w[a], xr[S1_K + s1_r_index(lo, hi)], wr_r);
  }
  return wr_r - mean_s * xr[t];
}

// BatchNorm backward (no ReLU) folded into the weight gradient, from the group totals: see stem_bwd_kernel section C
__device__ __forceinline__ void s1_finish(const float (&w)[S1_K], const float* xr, float s1, float s2, const float (&gt)[S1_K],
                                          float mean, float rstd, float gm, float shift, float inv_n, float* dw,
                                          float* dgamma, float* dbeta) {
  const float sc = rstd * gm;
  const float mean_s = fmaf(-shift, w[0] + w[1] + w[2], mean);
  *dbeta = s1;
  *dgamma = s2;
#pragma unroll
  for (int t = 0; t < S1_K; ++t) {
    const float h = rstd * s1_h_over_rstd(w, xr, t, mean_s);
    dw[t] = sc * (gt[t] - s1 * inv_n * xr[t] - s2 * inv_n * h);
  }
}

// dout (N,224,C0) = d a0 -> per-group partials of dW (C0 x 3), dgamma, dbeta.  The input moments and G_t are sums of
// x - s, s the group shift of stem_group_shift (the same rule and arithmetic as the stem backward).
// PARTIAL: one CTA = one chunk of a group; moments and per-channel sums go to the workspace (stem_alt_bwd_combine_kernel).
template <typename T, bool PARTIAL>
__global__ void __launch_bounds__(STEM_THREADS)
    stem_alt_bwd_kernel(const T* __restrict__ dout, const float* __restrict__ x, const float* __restrict__ w,
                        const float* __restrict__ gamma, const float* __restrict__ save_mean,
                        const float* __restrict__ save_rstd, float* __restrict__ dw_part, float* __restrict__ dgamma_part,
                        float* __restrict__ dbeta_part, float* __restrict__ mom_part, float* __restrict__ ch_part,
                        int group_all, int chunk, int n_chunks, int c0, int dout_stride) {
  extern __shared__ __align__(16) float xs[];
  __shared__ float red[STEM_THREADS * S1_NC];
  __shared__ float xr[S1_NM];
  const int g = blockIdx.x / n_chunks, kc = blockIdx.x % n_chunks;
  const int b0 = kc * chunk;
  const int group = min(chunk, group_all - b0);
  const size_t breath0 = (size_t)g * group_all + b0;
  const int tid = threadIdx.x;
  const int c = tid % STEM_CS, rl = tid / STEM_CS;
  const int ch = blockIdx.y * STEM_CS + c;
  const float shift = stem_group_shift(x + (size_t)g * group_all * STEM_L, red + STEM_THREADS * S1_NC - 16);
  stem_load_group(x + breath0 * STEM_L, xs, group);
  __syncthreads();
  const int n_pos = group * STEM_L;

  // ---- A. input moments about s: X'_t = sum (xin_t - s), R'[a][b] = sum (xin_a - s)(xin_b - s) ----------------
  {
    float acc[S1_NM];
#pragma unroll
    for (int i = 0; i < S1_NM; ++i) acc[i] = 0.f;
    for (int i = tid; i < n_pos; i += STEM_THREADS) {
      const float* xb = xs + (i / STEM_L) * STEM_BS + STEM_PAD + (i % STEM_L) - 1;
      float xin[S1_K];
#pragma unroll
      for (int t = 0; t < S1_K; ++t) xin[t] = xb[t] - shift;
      int k = S1_K;
#pragma unroll
      for (int a = 0; a < S1_K; ++a) {
        acc[a] += xin[a];
#pragma unroll
        for (int b = a; b < S1_K; ++b) {
          acc[k] = fmaf(xin[a], xin[b], acc[k]);
          ++k;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < S1_NM; ++i) acc[i] = warp_sum(acc[i]);
    const int warp = tid >> 5, lane = tid & 31;
    __syncthreads();  // the shift's scratch in red is read
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < S1_NM; ++i) red[warp * S1_NM + i] = acc[i];
    }
    __syncthreads();
    if (tid < S1_NM) {
      float s = 0.f;
      for (int wv = 0; wv < STEM_THREADS / 32; ++wv) s += red[wv * S1_NM + tid];
      xr[tid] = s;
      if (PARTIAL && blockIdx.y == 0) mom_part[(size_t)blockIdx.x * S1_NM + tid] = s;
    }
    __syncthreads();
  }

  // ---- B. per channel: S1 = sum g, S2 = sum g*xhat, G'_t = sum g * (xin_t - s) --------------------------------
  float wr[S1_K];
#pragma unroll
  for (int t = 0; t < S1_K; ++t) wr[t] = w[ch * S1_K + t];
  const float mean = save_mean[(size_t)g * c0 + ch], rstd = save_rstd[(size_t)g * c0 + ch];
  float s1 = 0.f, s2 = 0.f, gt[S1_K] = {0.f, 0.f, 0.f};
  const int n_runs = group * S1_RUNS;
  for (int run = rl; run < n_runs; run += STEM_LANES) {
    const int b = run / S1_RUNS, l0 = (run % S1_RUNS) * S1_RUN;
    const float* xb = xs + b * STEM_BS + STEM_PAD + l0 - 1;
    const T* dp = dout + ((breath0 + b) * STEM_L + l0) * dout_stride + ch;
    float x0 = xb[0], x1 = xb[1];
#pragma unroll 8
    for (int j = 0; j < S1_RUN; ++j) {
      const float x2 = xb[j + 2];
      const float gv = Elem<T>::ld(dp + (size_t)j * dout_stride);
      const float y = fmaf(wr[0], x0, fmaf(wr[1], x1, wr[2] * x2));
      s1 += gv;
      s2 = fmaf(gv, (y - mean) * rstd, s2);
      gt[0] = fmaf(gv, x0 - shift, gt[0]);
      gt[1] = fmaf(gv, x1 - shift, gt[1]);
      gt[2] = fmaf(gv, x2 - shift, gt[2]);
      x0 = x1;
      x1 = x2;
    }
  }
  __syncthreads();
  red[tid * S1_NC + 0] = s1;
  red[tid * S1_NC + 1] = s2;
#pragma unroll
  for (int t = 0; t < S1_K; ++t) red[tid * S1_NC + 2 + t] = gt[t];
  __syncthreads();
  if (rl != 0) return;
  s1 = s2 = 0.f;
#pragma unroll
  for (int t = 0; t < S1_K; ++t) gt[t] = 0.f;
  for (int r = 0; r < STEM_LANES; ++r) {
    const int o = (r * STEM_CS + c) * S1_NC;
    s1 += red[o + 0];
    s2 += red[o + 1];
#pragma unroll
    for (int t = 0; t < S1_K; ++t) gt[t] += red[o + 2 + t];
  }
  if (PARTIAL) {
    float* o = ch_part + (size_t)blockIdx.x * S1_NC * c0 + ch;
    o[0] = s1;
    o[c0] = s2;
#pragma unroll
    for (int t = 0; t < S1_K; ++t) o[(size_t)(2 + t) * c0] = gt[t];
    return;
  }
  const size_t o = (size_t)g * c0 + ch;
  s1_finish(wr, xr, s1, s2, gt, mean, rstd, gamma[ch], shift, 1.f / (float)n_pos, dw_part + o * S1_K, dgamma_part + o,
            dbeta_part + o);
}

// chunked backward, second pass: thread = channel of one group; adds the chunk partials in order, then s1_finish
__global__ void __launch_bounds__(128)
    stem_alt_bwd_combine_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ gamma,
                                const float* __restrict__ save_mean, const float* __restrict__ save_rstd,
                                const float* __restrict__ mom_part, const float* __restrict__ ch_part,
                                float* __restrict__ dw_part, float* __restrict__ dgamma_part, float* __restrict__ dbeta_part,
                                int group, int n_chunks, int c0) {
  __shared__ float xr[S1_NM];
  __shared__ float shift_red[16];
  const int g = blockIdx.x;
  const float shift = stem_group_shift(x + (size_t)g * group * STEM_L, shift_red);
  if (threadIdx.x < S1_NM) {
    float s = 0.f;
    for (int k = 0; k < n_chunks; ++k) s += mom_part[(size_t)(g * n_chunks + k) * S1_NM + threadIdx.x];
    xr[threadIdx.x] = s;
  }
  __syncthreads();
  const int ch = blockIdx.y * 128 + threadIdx.x;
  if (ch >= c0) return;
  float s1 = 0.f, s2 = 0.f, gt[S1_K] = {0.f, 0.f, 0.f};
  for (int k = 0; k < n_chunks; ++k) {
    const float* o = ch_part + (size_t)(g * n_chunks + k) * S1_NC * c0 + ch;
    s1 += o[0];
    s2 += o[c0];
#pragma unroll
    for (int t = 0; t < S1_K; ++t) gt[t] += o[(size_t)(2 + t) * c0];
  }
  float wr[S1_K];
#pragma unroll
  for (int t = 0; t < S1_K; ++t) wr[t] = w[ch * S1_K + t];
  const size_t o = (size_t)g * c0 + ch;
  s1_finish(wr, xr, s1, s2, gt, save_mean[o], save_rstd[o], gamma[ch], shift, 1.f / (float)(group * STEM_L),
            dw_part + o * S1_K, dgamma_part + o, dbeta_part + o);
}

long long stem_alt_workspace_bytes(int n_groups, int group, int c0, int backward) {
  const int nc = stem_n_chunks(group);
  if (nc == 1 || n_groups <= 0 || c0 <= 0) return 0;
  const long long recs = (long long)n_groups * nc;
  return (backward ? recs * ((long long)S1_NC * c0 + S1_NM) : recs * 3LL * c0) * (long long)sizeof(float);
}

int launch_stem_alt_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out, float* save_mean,
                        float* save_rstd, int n_groups, int group, int c0, int out_stride, float eps, void* workspace,
                        long long workspace_bytes, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem_alt: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  DARDS_CHECK_ARG(group > 0, "stem_alt: BatchNorm group must be at least 1 breath (got %d)", group);
  if (n_groups == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem_alt: grid too large");
  const int nc = stem_n_chunks(group);
  if (nc == 1) {
    const size_t smem = (size_t)group * STEM_BS * sizeof(float);
    dim3 grid(n_groups, c0 / STEM_CS);
    static size_t granted[2] = {44 * 1024, 44 * 1024};
    DARDS_DISPATCH_DTYPE(dtype, {
      int rc = stem_smem_optin(stem_alt_fwd_kernel<T, STEM_FUSED>, smem, &granted[dtype == DARDS_BF16 ? 1 : 0]);
      if (rc) return rc;
      stem_alt_fwd_kernel<T, STEM_FUSED><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                          save_rstd, nullptr, group, group, 1, c0,
                                                                          out_stride, eps);
    })
    DARDS_CHECK_LAUNCH("stem_alt_fwd");
    return DARDS_OK;
  }
  const long long need = stem_alt_workspace_bytes(n_groups, group, c0, 0);
  DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need,
                  "stem_alt_fwd: a BatchNorm group of %d breaths runs in chunks and needs %lld bytes of workspace (got %lld)",
                  group, need, workspace_bytes);
  DARDS_CHECK_ARG((long long)n_groups * nc <= 0x7fffffffLL, "stem_alt: grid too large");
  float* part = static_cast<float*>(workspace);
  const size_t smem = (size_t)STEM_CHUNK * STEM_BS * sizeof(float);
  dim3 grid((unsigned)(n_groups * nc), c0 / STEM_CS);
  static size_t granted[4] = {44 * 1024, 44 * 1024, 44 * 1024, 44 * 1024};
  DARDS_DISPATCH_DTYPE(dtype, {
    const int slot = dtype == DARDS_BF16 ? 1 : 0;
    int rc = stem_smem_optin(stem_alt_fwd_kernel<T, STEM_STATS>, smem, &granted[slot]);
    if (rc) return rc;
    rc = stem_smem_optin(stem_alt_fwd_kernel<T, STEM_APPLY>, smem, &granted[2 + slot]);
    if (rc) return rc;
    stem_alt_fwd_kernel<T, STEM_STATS><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                        save_rstd, part, group, STEM_CHUNK, nc, c0,
                                                                        out_stride, eps);
    DARDS_CHECK_LAUNCH("stem_alt_fwd (chunk statistics)");
    stem_alt_fwd_kernel<T, STEM_APPLY><<<grid, STEM_THREADS, smem, st>>>(x, w, gamma, beta, static_cast<T*>(out), save_mean,
                                                                        save_rstd, part, group, STEM_CHUNK, nc, c0,
                                                                        out_stride, eps);
  })
  DARDS_CHECK_LAUNCH("stem_alt_fwd (chunk apply)");
  return DARDS_OK;
}

int launch_stem_alt_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out,
                             int n_breaths, int c0, int out_stride, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem_alt: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  if (n_breaths == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem_alt: grid too large");
  const int nc = ceil_div(n_breaths, STEM_CHUNK);
  const size_t smem = (size_t)STEM_CHUNK * STEM_BS * sizeof(float);
  dim3 grid((unsigned)nc, c0 / STEM_CS);
  static size_t granted[2] = {44 * 1024, 44 * 1024};
  DARDS_DISPATCH_DTYPE(dtype, {
    int rc = stem_smem_optin(stem_alt_fwd_kernel<T, STEM_EVAL>, smem, &granted[dtype == DARDS_BF16 ? 1 : 0]);
    if (rc) return rc;
    stem_alt_fwd_kernel<T, STEM_EVAL><<<grid, STEM_THREADS, smem, st>>>(x, w, scale, shift, static_cast<T*>(out), nullptr,
                                                                       nullptr, nullptr, n_breaths, STEM_CHUNK, nc, c0,
                                                                       out_stride, 0.f);
  })
  DARDS_CHECK_LAUNCH("stem_alt_eval_fwd");
  return DARDS_OK;
}

int launch_stem_alt_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* save_mean,
                        const float* save_rstd, float* dw_part, float* dgamma_part, float* dbeta_part, int n_groups, int group,
                        int c0, int dout_stride, void* workspace, long long workspace_bytes, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(stem_c0_ok(c0), "stem_alt: initial planes must be a multiple of %d (got %d)", STEM_CS, c0);
  DARDS_CHECK_ARG(group > 0, "stem_alt: BatchNorm group must be at least 1 breath (got %d)", group);
  if (n_groups == 0) return DARDS_OK;
  DARDS_CHECK_ARG(c0 / STEM_CS <= 65535, "stem_alt: grid too large");
  const int nc = stem_n_chunks(group);
  const int chunk = nc == 1 ? group : STEM_CHUNK;
  float* mom_part = nullptr;
  float* ch_part = nullptr;
  if (nc > 1) {
    const long long need = stem_alt_workspace_bytes(n_groups, group, c0, 1);
    DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need,
                    "stem_alt_bwd: a BatchNorm group of %d breaths runs in chunks and needs %lld bytes of workspace (got %lld)",
                    group, need, workspace_bytes);
    DARDS_CHECK_ARG((long long)n_groups * nc <= 0x7fffffffLL, "stem_alt: grid too large");
    ch_part = static_cast<float*>(workspace);
    mom_part = ch_part + (size_t)n_groups * nc * S1_NC * c0;
  }
  const size_t smem = (size_t)chunk * STEM_BS * sizeof(float);
  dim3 grid((unsigned)(n_groups * nc), c0 / STEM_CS);
  static size_t granted[4] = {40 * 1024, 40 * 1024, 40 * 1024, 40 * 1024};  // 6 KB of static smem on top
  DARDS_DISPATCH_DTYPE(dtype, {
    const int slot = (dtype == DARDS_BF16 ? 1 : 0) + (nc > 1 ? 2 : 0);
    const T* d = static_cast<const T*>(dout);
    if (nc > 1) {
      int rc = stem_smem_optin(stem_alt_bwd_kernel<T, true>, smem, &granted[slot]);
      if (rc) return rc;
      stem_alt_bwd_kernel<T, true><<<grid, STEM_THREADS, smem, st>>>(d, x, w, gamma, save_mean, save_rstd, dw_part,
                                                                     dgamma_part, dbeta_part, mom_part, ch_part, group,
                                                                     chunk, nc, c0, dout_stride);
    } else {
      int rc = stem_smem_optin(stem_alt_bwd_kernel<T, false>, smem, &granted[slot]);
      if (rc) return rc;
      stem_alt_bwd_kernel<T, false><<<grid, STEM_THREADS, smem, st>>>(d, x, w, gamma, save_mean, save_rstd, dw_part,
                                                                      dgamma_part, dbeta_part, nullptr, nullptr, group,
                                                                      chunk, 1, c0, dout_stride);
    }
  })
  DARDS_CHECK_LAUNCH("stem_alt_bwd");
  if (nc > 1) {
    dim3 cgrid(n_groups, ceil_div(c0, 128));
    stem_alt_bwd_combine_kernel<<<cgrid, 128, 0, st>>>(x, w, gamma, save_mean, save_rstd, mom_part, ch_part, dw_part,
                                                       dgamma_part, dbeta_part, group, nc, c0);
    DARDS_CHECK_LAUNCH("stem_alt_bwd (chunk combine)");
  }
  return DARDS_OK;
}

}  // namespace dards

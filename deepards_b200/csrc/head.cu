// Pooling, dropout and the linear classification head: small bandwidth-bound kernels.
#include "common.cuh"

namespace dards {

// ---- AvgPool1d(2,2): (N,L,C) -> (N,L/2,C) --------------------------------------------------------------
template <typename T>
__global__ void avgpool2_fwd_kernel(const T* __restrict__ in, T* __restrict__ out, long long rows_out, int l_out, int c4,
                                    int in_stride, int out_stride) {
  long long total = rows_out * c4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int cq = (int)(i % c4);
    long long r = i / c4;  // n*l_out + q
    long long n = r / l_out;
    int q = (int)(r % l_out);
    const T* src = in + ((size_t)(n * 2 * l_out) + 2 * q) * in_stride + cq * 4;
    float4 a = Elem<T>::ld4(src), b = Elem<T>::ld4(src + in_stride);
    Elem<T>::st4(out + (size_t)r * out_stride + cq * 4,
                 make_float4(0.5f * (a.x + b.x), 0.5f * (a.y + b.y), 0.5f * (a.z + b.z), 0.5f * (a.w + b.w)));
  }
}

template <typename T>
__global__ void avgpool2_bwd_kernel(const T* __restrict__ dout, T* __restrict__ din, long long rows_out, int l_out,
                                    int c4, int dout_stride, int din_stride) {
  long long total = rows_out * c4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int cq = (int)(i % c4);
    long long r = i / c4;
    long long n = r / l_out;
    int q = (int)(r % l_out);
    float4 d = Elem<T>::ld4(dout + (size_t)r * dout_stride + cq * 4);
    d.x *= 0.5f; d.y *= 0.5f; d.z *= 0.5f; d.w *= 0.5f;
    T* dst = din + ((size_t)(n * 2 * l_out) + 2 * q) * din_stride + cq * 4;
    Elem<T>::st4(dst, d);
    Elem<T>::st4(dst + din_stride, d);
  }
}

// ---- AvgPool1d(L) + flatten: (N,L,C) -> feat (N,C) fp32 --------------------------------------------------
template <typename T>
__global__ void avgpool_full_fwd_kernel(const T* __restrict__ in, float* __restrict__ feat, long long n_breaths, int l,
                                        int c4, int in_stride) {
  long long total = n_breaths * c4;
  const float inv = 1.f / (float)l;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int cq = (int)(i % c4);
    long long n = i / c4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int q = 0; q < l; ++q) {
      float4 v = Elem<T>::ld4(in + ((size_t)n * l + q) * in_stride + cq * 4);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    s.x *= inv; s.y *= inv; s.z *= inv; s.w *= inv;
    *reinterpret_cast<float4*>(feat + (size_t)n * c4 * 4 + cq * 4) = s;
  }
}

template <typename T>
__global__ void avgpool_full_bwd_kernel(const float* __restrict__ dfeat, T* __restrict__ din, long long n_breaths, int l,
                                        int c4, int din_stride) {
  long long total = n_breaths * l * c4;
  const float inv = 1.f / (float)l;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int cq = (int)(i % c4);
    long long r = i / c4;  // n*l + q
    long long n = r / l;
    float4 d = *reinterpret_cast<const float4*>(dfeat + (size_t)n * c4 * 4 + cq * 4);
    d.x *= inv; d.y *= inv; d.z *= inv; d.w *= inv;
    Elem<T>::st4(din + (size_t)r * din_stride + cq * 4, d);
  }
}

// bf16, 8 channels per thread: the pooled gradient of (breath, channel vector) is read and scaled ONCE and written to
// all l positions with 16-byte stores (the generic kernel re-reads dfeat for every position and stores 8 bytes)
__global__ void avgpool_full_bwd_bf16x8_kernel(const float* __restrict__ dfeat, __nv_bfloat16* __restrict__ din,
                                               long long n_breaths, int l, int c8, int din_stride) {
  const long long total = n_breaths * c8;
  const float inv = 1.f / (float)l;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cq = (int)(i % c8);
    const long long n = i / c8;
    const float4 a = __ldg(reinterpret_cast<const float4*>(dfeat + (size_t)n * c8 * 8 + cq * 8));
    const float4 b = __ldg(reinterpret_cast<const float4*>(dfeat + (size_t)n * c8 * 8 + cq * 8 + 4));
    __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x * inv, a.y * inv), p1 = __floats2bfloat162_rn(a.z * inv, a.w * inv);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x * inv, b.y * inv), p3 = __floats2bfloat162_rn(b.z * inv, b.w * inv);
    uint4 v;
    v.x = *reinterpret_cast<uint32_t*>(&p0); v.y = *reinterpret_cast<uint32_t*>(&p1);
    v.z = *reinterpret_cast<uint32_t*>(&p2); v.w = *reinterpret_cast<uint32_t*>(&p3);
    __nv_bfloat16* dst = din + (size_t)n * l * din_stride + cq * 8;
    for (int q = 0; q < l; ++q) *reinterpret_cast<uint4*>(dst + (size_t)q * din_stride) = v;
  }
}

// ---- dropout: keep-mask is a pure function of (seed, step, GLOBAL element index) ------------------------------
// Philox4x32-10 (Salmon et al., the generator behind torch's CUDA dropout): key = seed ^ step-dependent offset, counter =
// global element index / 4; element e takes word e % 4 of its block.  "Global" = counted from the first sequence of the
// whole (all-ranks) batch: a rank adds first_sequence * rows_per_seq to its local row index, so the masks do not depend
// on how the batch is sharded (SURVEY.md 8e(iv)) and the backward regenerates them from the same three numbers.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                              uint32_t (&out)[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// VEC consecutive channels per thread (a 16-byte access when the slice allows it, else scalar); the random number of
// an element depends only on (seed, step, global row * c + channel), never on the vector width.
template <typename T, int VEC>
__global__ void dropout_kernel(T* __restrict__ x, long long n_rows, int c, int stride, float p, float scale,
                               unsigned long long seed, const unsigned long long* __restrict__ seed_off, int rows_per_seq) {
  unsigned long long row0 = 0;
  if (seed_off) {
    seed += seed_off[0] * 0x9E3779B97F4A7C15ull;
    if (rows_per_seq > 0) row0 = seed_off[1] * (unsigned long long)rows_per_seq;
  }
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const int cv = c / VEC;
  const long long total = n_rows * cv;
  const uint32_t thresh = (uint32_t)(p * 4294967296.0);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cv;
    const int cc = (int)(i % cv) * VEC;
    T* ptr = x + (size_t)r * stride + cc;
    T v[VEC];
    if (VEC > 1) *reinterpret_cast<uint4*>(v) = *reinterpret_cast<const uint4*>(ptr);
    else v[0] = *ptr;
    const unsigned long long e0 = (row0 + (unsigned long long)r) * (unsigned long long)c + (unsigned long long)cc;
    uint32_t rnd[4];
    unsigned long long blk = ~0ull;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const unsigned long long e = e0 + j;
      if ((e >> 2) != blk) {   // VEC and cc are multiples of 4 on the vector path: one Philox block per 4 elements
        blk = e >> 2;
        philox4x32_10((uint32_t)blk, (uint32_t)(blk >> 32), 0u, 0u, k0, k1, rnd);
      }
      const float f = Elem<T>::ld(&v[j]);
      Elem<T>::st(&v[j], rnd[e & 3] < thresh ? 0.f : f * scale);
    }
    if (VEC > 1) *reinterpret_cast<uint4*>(ptr) = *reinterpret_cast<const uint4*>(v);
    else *ptr = v[0];
  }
}

// ---- linear head ----------------------------------------------------------------------------------------
// logits[r][j] = bias[j] + sum_k feat[r][k] w[j][k]; one CTA per row, n_out <= 8
constexpr int LIN_THREADS = 256;
constexpr int LIN_MAX_OUT = 8;

__global__ void __launch_bounds__(LIN_THREADS) linear_fwd_kernel(const float* __restrict__ feat,
                                                                  const float* __restrict__ w,
                                                                  const float* __restrict__ bias,
                                                                  float* __restrict__ logits, int k, int n_out) {
  __shared__ float red[LIN_THREADS / 32][LIN_MAX_OUT];
  const int r = blockIdx.x;
  float acc[LIN_MAX_OUT];
#pragma unroll
  for (int j = 0; j < LIN_MAX_OUT; ++j) acc[j] = 0.f;
  const float* f = feat + (size_t)r * k;
  if ((k & 3) == 0 && ((reinterpret_cast<uintptr_t>(feat) | reinterpret_cast<uintptr_t>(w)) & 15) == 0) {
    // 16-byte loads, every load of the row independent of the others (the kernel is latency bound: one CTA per row)
    const float4* f4 = reinterpret_cast<const float4*>(f);
    const int k4 = k >> 2;
#pragma unroll 4
    for (int i = threadIdx.x; i < k4; i += LIN_THREADS) {
      const float4 v = __ldg(f4 + i);
#pragma unroll
      for (int j = 0; j < LIN_MAX_OUT; ++j)
        if (j < n_out) {
          const float4 ww = __ldg(reinterpret_cast<const float4*>(w + (size_t)j * k) + i);
          acc[j] = fmaf(v.x, ww.x, fmaf(v.y, ww.y, fmaf(v.z, ww.z, fmaf(v.w, ww.w, acc[j]))));
        }
    }
  } else {
    for (int i = threadIdx.x; i < k; i += LIN_THREADS) {
      float v = f[i];
#pragma unroll
      for (int j = 0; j < LIN_MAX_OUT; ++j)
        if (j < n_out) acc[j] = fmaf(v, w[(size_t)j * k + i], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < LIN_MAX_OUT; ++j) acc[j] = warp_sum(acc[j]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < LIN_MAX_OUT; ++j) red[warp][j] = acc[j];
  }
  __syncthreads();
  if (threadIdx.x < n_out) {
    float s = bias[threadIdx.x];
    for (int wv = 0; wv < LIN_THREADS / 32; ++wv) s += red[wv][threadIdx.x];
    logits[(size_t)r * n_out + threadIdx.x] = s;
  }
}

// dfeat[r][k] = sum_j dlogits[r][j] w[j][k]
__global__ void linear_bwd_data_kernel(const float* __restrict__ dlogits, const float* __restrict__ w,
                                       float* __restrict__ dfeat, long long rows, int k, int n_out) {
  long long total = rows * k;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i / k;
    int kk = (int)(i % k);
    float s = 0.f;
    for (int j = 0; j < n_out; ++j) s = fmaf(dlogits[r * n_out + j], w[(size_t)j * k + kk], s);
    dfeat[i] = s;
  }
}

// dw[j][k] (+)= sum_r dlogits[r][j] feat[r][k].  256 threads = 32 columns k x 8 row lanes; every thread reads its
// feat column once for all n_out outputs with 8 rows in flight; lane sums are combined in a fixed order -> deterministic.
// The bias gradient (a sum over all rows of a few values) is reduced by the whole first CTA, not by n_out threads.
constexpr int LBW_COLS = 32, LBW_LANES = 8;
__global__ void __launch_bounds__(256) linear_bwd_weight_kernel(const float* __restrict__ dlogits,
                                                                const float* __restrict__ feat, float* __restrict__ dw,
                                                                float* __restrict__ db, int rows, int k, int n_out,
                                                                int accumulate) {
  __shared__ float red[LBW_LANES][LIN_MAX_OUT][LBW_COLS];
  const int col = threadIdx.x & (LBW_COLS - 1), ln = threadIdx.x / LBW_COLS;
  const int kk = blockIdx.x * LBW_COLS + col;
  float acc[LIN_MAX_OUT];
#pragma unroll
  for (int j = 0; j < LIN_MAX_OUT; ++j) acc[j] = 0.f;
  if (kk < k) {
#pragma unroll 8
    for (int r = ln; r < rows; r += LBW_LANES) {
      const float f = feat[(size_t)r * k + kk];
#pragma unroll
      for (int j = 0; j < LIN_MAX_OUT; ++j)
        if (j < n_out) acc[j] = fmaf(dlogits[(size_t)r * n_out + j], f, acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < LIN_MAX_OUT; ++j) red[ln][j][col] = acc[j];
  __syncthreads();
  if (ln == 0 && kk < k) {
    for (int j = 0; j < n_out; ++j) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < LBW_LANES; ++q) s += red[q][j][col];
      float* o = dw + (size_t)j * k + kk;
      *o = accumulate ? *o + s : s;
    }
  }
  if (blockIdx.x == 0 && db) {
    __syncthreads();  // `red` is reused: [warp][j]
    float* wred = &red[0][0][0];
    for (int j = 0; j < n_out; ++j) {
      float s = 0.f;
      for (int r = threadIdx.x; r < rows; r += 256) s += dlogits[(size_t)r * n_out + j];
      s = warp_sum(s);
      if ((threadIdx.x & 31) == 0) wred[(threadIdx.x >> 5) * LIN_MAX_OUT + j] = s;
    }
    __syncthreads();
    if (threadIdx.x < n_out) {
      float s = 0.f;
#pragma unroll
      for (int wv = 0; wv < 8; ++wv) s += wred[wv * LIN_MAX_OUT + threadIdx.x];
      db[threadIdx.x] = accumulate ? db[threadIdx.x] + s : s;
    }
  }
}

// ---- BCEWithLogits (mean) + gradient: n is tiny (2 per sequence), one CTA ---------------------------------
__global__ void bce_with_logits_kernel(const float* __restrict__ z, const float* __restrict__ t, float* __restrict__ loss,
                                       float* __restrict__ dz, int n, float grad_scale) {
  __shared__ float red[32];
  float s = 0.f;
  const float inv_n = 1.f / (float)n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float zi = z[i], ti = t[i];
    // max(z,0) - z*t + log1p(exp(-|z|))  (the numerically stable form torch uses)
    s += fmaxf(zi, 0.f) - zi * ti + log1pf(expf(-fabsf(zi)));
    if (dz) dz[i] = grad_scale * (1.f / (1.f + expf(-zi)) - ti) * inv_n;
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    if (loss) loss[0] = tot * inv_n;
  }
}

int launch_bce(const float* z, const float* t, float* loss, float* dz, int n, float grad_scale, cudaStream_t st) {
  if (n == 0) return DARDS_OK;
  bce_with_logits_kernel<<<1, 256, 0, st>>>(z, t, loss, dz, n, grad_scale);
  DARDS_CHECK_LAUNCH("bce_with_logits");
  return DARDS_OK;
}

// ---- launchers -------------------------------------------------------------------------------------------
static int grid_for(long long total, int threads) {
  long long b = (total + threads - 1) / threads;
  if (b > 148LL * 16) b = 148LL * 16;
  if (b < 1) b = 1;
  return (int)b;
}

int launch_avgpool2(int bwd, const void* src, void* dst, int n_breaths, int l_in, int c, int src_stride, int dst_stride,
                    int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(l_in % 2 == 0 && c % 4 == 0 && src_stride % 4 == 0 && dst_stride % 4 == 0,
                  "avgpool2: L must be even, channels/strides multiples of 4");
  long long rows_out = (long long)n_breaths * (l_in / 2);
  if (rows_out == 0) return DARDS_OK;
  int blocks = grid_for(rows_out * (c / 4), 256);
  DARDS_DISPATCH_DTYPE(dtype, {
    if (!bwd)
      avgpool2_fwd_kernel<T><<<blocks, 256, 0, st>>>(static_cast<const T*>(src), static_cast<T*>(dst), rows_out,
                                                     l_in / 2, c / 4, src_stride, dst_stride);
    else
      avgpool2_bwd_kernel<T><<<blocks, 256, 0, st>>>(static_cast<const T*>(src), static_cast<T*>(dst), rows_out,
                                                     l_in / 2, c / 4, src_stride, dst_stride);
  })
  DARDS_CHECK_LAUNCH("avgpool2");
  return DARDS_OK;
}

// ---- Max/AvgPool1d(3, 2, padding 1): (N,L,C) -> (N,(L-1)/2+1,C), the first pool of the two-convolution ResNet stem ------
// Output q covers inputs 2q-1, 2q, 2q+1; index -1 (and L when L is even) is padding: -inf for max, 0 counted in the
// divisor for avg (count_include_pad).  The max backward recomputes the window's arg-max from the stored input and routes
// the gradient to its FIRST maximum (ATen's rule); each input gathers from the one or two windows that contain it, so
// there are no atomics and the result is deterministic.
__device__ __forceinline__ float pool3_pick(float v, int idx, float& best, int& arg) {
  if (v > best) {
    best = v;
    arg = idx;
  }
  return best;
}

template <typename T>
__global__ void pool3s2_fwd_kernel(const T* __restrict__ in, T* __restrict__ out, long long rows_out, int l_in, int l_out,
                                   int c4, int in_stride, int out_stride, int pool) {
  const long long total = rows_out * c4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cq = (int)(i % c4);
    const long long r = i / c4;  // n*l_out + q
    const long long n = r / l_out;
    const int q = (int)(r % l_out);
    const T* src = in + (size_t)n * l_in * in_stride + cq * 4;
    float v[3][4];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int p = 2 * q - 1 + k;
      const bool ok = p >= 0 && p < l_in;
      const float4 a = ok ? Elem<T>::ld4(src + (size_t)p * in_stride) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float pad = pool == 0 ? -INFINITY : 0.f;
      v[k][0] = ok ? a.x : pad; v[k][1] = ok ? a.y : pad; v[k][2] = ok ? a.z : pad; v[k][3] = ok ? a.w : pad;
    }
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      o[j] = pool == 0 ? fmaxf(fmaxf(v[0][j], v[1][j]), v[2][j]) : (v[0][j] + v[1][j] + v[2][j]) * (1.f / 3.f);
    Elem<T>::st4(out + (size_t)r * out_stride + cq * 4, make_float4(o[0], o[1], o[2], o[3]));
  }
}

template <typename T>
__global__ void pool3s2_bwd_kernel(const T* __restrict__ dout, const T* __restrict__ in, T* __restrict__ din,
                                   long long rows_in, int l_in, int l_out, int c4, int dout_stride, int in_stride,
                                   int din_stride, int pool) {
  const long long total = rows_in * c4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cq = (int)(i % c4);
    const long long r = i / c4;  // n*l_in + p
    const long long n = r / l_in;
    const int p = (int)(r % l_in);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    // windows q with 2q-1 <= p <= 2q+1, in increasing q
    for (int q = p / 2; q <= (p + 1) / 2; ++q) {
      if (q >= l_out || 2 * q - 1 > p) continue;
      const float4 d = Elem<T>::ld4(dout + ((size_t)n * l_out + q) * dout_stride + cq * 4);
      const float dv[4] = {d.x, d.y, d.z, d.w};
      if (pool != 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] += dv[j] * (1.f / 3.f);
        continue;
      }
      float best[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      int arg[4] = {-1, -1, -1, -1};
      for (int k = 0; k < 3; ++k) {
        const int pp = 2 * q - 1 + k;
        if (pp < 0 || pp >= l_in) continue;
        const float4 a = Elem<T>::ld4(in + ((size_t)n * l_in + pp) * in_stride + cq * 4);
        pool3_pick(a.x, pp, best[0], arg[0]);
        pool3_pick(a.y, pp, best[1], arg[1]);
        pool3_pick(a.z, pp, best[2], arg[2]);
        pool3_pick(a.w, pp, best[3], arg[3]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (arg[j] == p) acc[j] += dv[j];
    }
    Elem<T>::st4(din + (size_t)r * din_stride + cq * 4, make_float4(acc[0], acc[1], acc[2], acc[3]));
  }
}

int launch_pool3s2(int bwd, const void* dout_or_in, const void* in, void* dst, int n_breaths, int l_in, int c,
                   int src_stride, int in_stride, int dst_stride, int pool, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(l_in >= 1 && c % 4 == 0 && src_stride % 4 == 0 && in_stride % 4 == 0 && dst_stride % 4 == 0,
                  "pool3s2: channels/strides must be multiples of 4");
  const int l_out = (l_in - 1) / 2 + 1;
  const long long rows = (long long)n_breaths * (bwd ? l_in : l_out);
  if (rows == 0) return DARDS_OK;
  const int blocks = grid_for(rows * (c / 4), 256);
  DARDS_DISPATCH_DTYPE(dtype, {
    if (!bwd)
      pool3s2_fwd_kernel<T><<<blocks, 256, 0, st>>>(static_cast<const T*>(dout_or_in), static_cast<T*>(dst), rows, l_in,
                                                    l_out, c / 4, src_stride, dst_stride, pool);
    else
      pool3s2_bwd_kernel<T><<<blocks, 256, 0, st>>>(static_cast<const T*>(dout_or_in), static_cast<const T*>(in),
                                                    static_cast<T*>(dst), rows, l_in, l_out, c / 4, src_stride, in_stride,
                                                    dst_stride, pool);
  })
  DARDS_CHECK_LAUNCH("pool3s2");
  return DARDS_OK;
}

int launch_avgpool_full_fwd(const void* in, float* feat, int n_breaths, int l, int c, int in_stride, int dtype,
                            cudaStream_t st) {
  DARDS_CHECK_ARG(c % 4 == 0 && in_stride % 4 == 0, "avgpool: channels/stride must be multiples of 4");
  if (n_breaths == 0) return DARDS_OK;
  int blocks = grid_for((long long)n_breaths * (c / 4), 256);
  DARDS_DISPATCH_DTYPE(dtype, {
    avgpool_full_fwd_kernel<T><<<blocks, 256, 0, st>>>(static_cast<const T*>(in), feat, n_breaths, l, c / 4, in_stride);
  })
  DARDS_CHECK_LAUNCH("avgpool_full_fwd");
  return DARDS_OK;
}

int launch_avgpool_full_bwd(const float* dfeat, void* din, int n_breaths, int l, int c, int din_stride, int dtype,
                            cudaStream_t st) {
  DARDS_CHECK_ARG(c % 4 == 0 && din_stride % 4 == 0, "avgpool: channels/stride must be multiples of 4");
  if (n_breaths == 0) return DARDS_OK;
  if (dtype == DARDS_BF16 && c % 8 == 0 && din_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(din) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(dfeat) & 15) == 0) {
    avgpool_full_bwd_bf16x8_kernel<<<grid_for((long long)n_breaths * (c / 8), 256), 256, 0, st>>>(
        dfeat, static_cast<__nv_bfloat16*>(din), n_breaths, l, c / 8, din_stride);
    DARDS_CHECK_LAUNCH("avgpool_full_bwd");
    return DARDS_OK;
  }
  int blocks = grid_for((long long)n_breaths * l * (c / 4), 256);
  DARDS_DISPATCH_DTYPE(dtype, {
    avgpool_full_bwd_kernel<T><<<blocks, 256, 0, st>>>(dfeat, static_cast<T*>(din), n_breaths, l, c / 4, din_stride);
  })
  DARDS_CHECK_LAUNCH("avgpool_full_bwd");
  return DARDS_OK;
}

int launch_dropout(void* x, int n_rows, int c, int stride, float p, unsigned long long seed,
                   const unsigned long long* seed_off, int rows_per_seq, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(p >= 0.f && p < 1.f, "dropout: p must be in [0,1)");
  if (n_rows == 0 || p == 0.f) return DARDS_OK;
  DARDS_DISPATCH_DTYPE(dtype, {
    constexpr int VEC = 16 / (int)sizeof(T);
    const bool vec_ok = c % VEC == 0 && stride % VEC == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
    if (vec_ok)
      dropout_kernel<T, VEC><<<grid_for((long long)n_rows * (c / VEC), 256), 256, 0, st>>>(
          static_cast<T*>(x), n_rows, c, stride, p, 1.f / (1.f - p), seed, seed_off, rows_per_seq);
    else
      dropout_kernel<T, 1><<<grid_for((long long)n_rows * c, 256), 256, 0, st>>>(static_cast<T*>(x), n_rows, c, stride, p,
                                                                                 1.f / (1.f - p), seed, seed_off, rows_per_seq);
  })
  DARDS_CHECK_LAUNCH("dropout");
  return DARDS_OK;
}

int launch_linear_fwd(const float* feat, const float* w, const float* bias, float* logits, int rows, int k, int n_out,
                      cudaStream_t st) {
  DARDS_CHECK_ARG(n_out >= 1 && n_out <= LIN_MAX_OUT, "linear: n_out must be in [1,%d]", LIN_MAX_OUT);
  if (rows == 0) return DARDS_OK;
  linear_fwd_kernel<<<rows, LIN_THREADS, 0, st>>>(feat, w, bias, logits, k, n_out);
  DARDS_CHECK_LAUNCH("linear_fwd");
  return DARDS_OK;
}

int launch_linear_bwd(const float* dlogits, const float* feat, const float* w, float* dfeat, float* dw, float* db,
                      int accumulate, int rows, int k, int n_out, cudaStream_t st) {
  DARDS_CHECK_ARG(n_out >= 1 && n_out <= LIN_MAX_OUT, "linear: n_out must be in [1,%d]", LIN_MAX_OUT);
  if (dfeat && rows > 0) {
    linear_bwd_data_kernel<<<grid_for((long long)rows * k, 256), 256, 0, st>>>(dlogits, w, dfeat, rows, k, n_out);
    DARDS_CHECK_LAUNCH("linear_bwd_data");
  }
  if (dw) {
    linear_bwd_weight_kernel<<<ceil_div(k, LBW_COLS), 256, 0, st>>>(dlogits, feat, dw, db, rows, k, n_out, accumulate);
    DARDS_CHECK_LAUNCH("linear_bwd_weight");
  }
  return DARDS_OK;
}

}  // namespace dards

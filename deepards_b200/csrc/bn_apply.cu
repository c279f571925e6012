// Elementwise half of the grouped BatchNorm1d forward, for layers whose statistics were already taken in the
// convolution epilogue (conv_bn_tc.cu, PARTIAL mode): one streaming pass
//     out = [relu]( x * scale + shift  [+ res]  [+ x2 * scale2 + shift2] )
// with scale = gamma * rstd, shift = beta - mean * scale per (group, channel).  The second, optional normalised
// operand is the 1x1 downsample branch of a ResNet block (resnet.py:34-38: out += downsample(x) where downsample is
// conv1x1 -> BatchNorm), so `out = relu(bn2(y2) + bn_d(y_d))` is ONE pass instead of a BatchNorm launch per branch.
//
// GIVEN mode (dards_bn_affine_apply): the per-channel scale / shift are inputs -- BatchNorm with constant statistics
// (running statistics) -- and `gamma` / `beta` (`gamma2` / `beta2`) carry them; there is no merge, no saved statistics,
// and a "group" is any block of rows.  fp32 and bf16.
//
// Every CTA first merges the (count, mean, M2) records that the convolution tiles of its group wrote -- a fixed-order
// Chan merge, a few dozen loads per channel -- then streams its share of the group's rows: 16-byte vectors, two rows
// per thread in flight (three CTAs per SM), no shared-memory tile, no second sweep.  HBM traffic = 1 read + 1 write (+ operands).
#include "common.cuh"

namespace dards {

template <typename T>
struct GbnApplyArgs {
  const T* x;
  T* out;
  const T* res;
  const float* gamma;
  const float* beta;
  const float* part;     // [n_groups * entries][3][c]
  float* save_mean;
  float* save_rstd;
  const T* x2;
  const float* gamma2;
  const float* beta2;
  const float* part2;
  float* save_mean2;
  float* save_rstd2;
  int entries, entries2;
  int n_groups, rows, c, splits;
  int x_stride, out_stride, res_stride, x2_stride;
  float eps;
  int relu;
};

__device__ __forceinline__ void apply_unpack8(const uint4& r, float (&v)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(h[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}

// 16-byte vectors of the storage type
template <typename T> struct ApplyVec;
template <> struct ApplyVec<__nv_bfloat16> {
  static constexpr int N = 8, SHIFT = 3;
  static __device__ __forceinline__ void unpack(const uint4& r, float (&v)[8]) { apply_unpack8(r, v); }
  static __device__ __forceinline__ uint4 pack(const float (&v)[8]) {
    uint4 o;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
    return o;
  }
};
template <> struct ApplyVec<float> {
  static constexpr int N = 4, SHIFT = 2;
  static __device__ __forceinline__ void unpack(const uint4& r, float (&v)[4]) {
    v[0] = __uint_as_float(r.x); v[1] = __uint_as_float(r.y); v[2] = __uint_as_float(r.z); v[3] = __uint_as_float(r.w);
  }
  static __device__ __forceinline__ uint4 pack(const float (&v)[4]) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  }
};

// (count, mean, M2) records e = 0..entries-1 of channel ch, merged in order -> scale / shift (and the saved statistics)
__device__ __forceinline__ void merge_moments(const float* __restrict__ part, int entries, int c, int ch, float eps,
                                              float gamma, float beta, float& sc, float& sh, float& mean_o, float& rstd_o) {
  float n = 0.f, mean = 0.f, m2 = 0.f;
  constexpr int ME = 8;   // records fetched together: the loads are independent, the merge is a dependent chain
  for (int e0 = 0; e0 < entries; e0 += ME) {
    float ne[ME], me[ME], qe[ME];
#pragma unroll
    for (int u = 0; u < ME; ++u) {
      ne[u] = 0.f;
      if (e0 + u < entries) {
        const float* r = part + (size_t)(e0 + u) * 3 * c + ch;
        ne[u] = r[0];
        me[u] = r[c];
        qe[u] = r[2 * c];
      }
    }
#pragma unroll
    for (int u = 0; u < ME; ++u) {
      if (ne[u] > 0.f) {
        const float nn = n + ne[u], d = me[u] - mean;
        mean += d * (ne[u] / nn);
        m2 += qe[u] + d * d * (n * ne[u] / nn);
        n = nn;
      }
    }
  }
  const float var = fmaxf(m2 / fmaxf(n, 1.f), 0.f) + eps;
  float rstd = rsqrtf(var);
  rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);  // one Newton step: the reference divides by sqrt()
  sc = rstd * gamma;
  sh = beta - mean * sc;
  mean_o = mean;
  rstd_o = rstd;
}

template <typename T, bool GIVEN>
__global__ void __launch_bounds__(256, 3) gbn_apply_fwd_kernel(const GbnApplyArgs<T> a) {
  constexpr int V = ApplyVec<T>::N;
  extern __shared__ float s_tab[];  // scale[c], shift[c] (, scale2[c], shift2[c])
  const int g = blockIdx.x / a.splits, split = blockIdx.x % a.splits;
  const int c = a.c;
  for (int ch = threadIdx.x; ch < c; ch += 256) {
    if (GIVEN) {
      s_tab[ch] = a.gamma[ch];
      s_tab[c + ch] = a.beta[ch];
      if (a.x2) {
        s_tab[2 * c + ch] = a.gamma2[ch];
        s_tab[3 * c + ch] = a.beta2[ch];
      }
      continue;
    }
    float sc, sh, mean, rstd;
    merge_moments(a.part + (size_t)g * a.entries * 3 * c, a.entries, c, ch, a.eps, a.gamma[ch], a.beta[ch], sc, sh, mean, rstd);
    s_tab[ch] = sc;
    s_tab[c + ch] = sh;
    if (split == 0) {
      a.save_mean[(size_t)g * c + ch] = mean;
      a.save_rstd[(size_t)g * c + ch] = rstd;
    }
    if (a.x2) {
      merge_moments(a.part2 + (size_t)g * a.entries2 * 3 * c, a.entries2, c, ch, a.eps, a.gamma2[ch], a.beta2[ch], sc, sh, mean,
                    rstd);
      s_tab[2 * c + ch] = sc;
      s_tab[3 * c + ch] = sh;
      if (split == 0) {
        a.save_mean2[(size_t)g * c + ch] = mean;
        a.save_rstd2[(size_t)g * c + ch] = rstd;
      }
    }
  }
  __syncthreads();
  const int vpr = c >> ApplyVec<T>::SHIFT;                  // 16-byte vectors per row
  const int rows_split = (a.rows + a.splits - 1) / a.splits;
  const int r_lo = split * rows_split;
  const int r_hi = min(a.rows, r_lo + rows_split);
  const int n_vec = (r_hi - r_lo) * vpr;
  const size_t grow = (size_t)g * a.rows + r_lo;
  const T* xb = a.x + grow * a.x_stride;
  T* ob = a.out + grow * a.out_stride;
  const T* rb = a.res ? a.res + grow * a.res_stride : nullptr;
  const T* x2b = a.x2 ? a.x2 + grow * a.x2_stride : nullptr;
  const bool pow2 = (vpr & (vpr - 1)) == 0;
  const int shv = 31 - __clz(vpr);
  constexpr int U = 2;
  for (int i0 = threadIdx.x; i0 < n_vec; i0 += 256 * U) {
    uint4 vx[U], vr[U], v2[U];
    int row[U], vec[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * 256;
      if (pow2) {
        row[u] = i >> shv;
        vec[u] = i & (vpr - 1);
      } else {
        row[u] = i / vpr;
        vec[u] = i - row[u] * vpr;
      }
      if (i < n_vec) {
        vx[u] = *reinterpret_cast<const uint4*>(xb + (size_t)row[u] * a.x_stride + vec[u] * V);
        if (rb) vr[u] = *reinterpret_cast<const uint4*>(rb + (size_t)row[u] * a.res_stride + vec[u] * V);
        if (x2b) v2[u] = *reinterpret_cast<const uint4*>(x2b + (size_t)row[u] * a.x2_stride + vec[u] * V);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int i = i0 + u * 256;
      if (i >= n_vec) continue;
      const int c0 = vec[u] * V;
      float v[V];
      ApplyVec<T>::unpack(vx[u], v);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] = fmaf(v[j], s_tab[c0 + j], s_tab[c + c0 + j]);
      if (rb) {
        float e[V];
        ApplyVec<T>::unpack(vr[u], e);
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] += e[j];
      }
      if (x2b) {
        float e[V];
        ApplyVec<T>::unpack(v2[u], e);
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] += fmaf(e[j], s_tab[2 * c + c0 + j], s_tab[3 * c + c0 + j]);
      }
      if (a.relu) {
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] = fmaxf(v[j], 0.f);
      }
      *reinterpret_cast<uint4*>(ob + (size_t)row[u] * a.out_stride + c0) = ApplyVec<T>::pack(v);
    }
  }
}

int launch_gbn_apply_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta, const float* part,
                         int entries, float* save_mean, float* save_rstd, const void* x2, const float* gamma2,
                         const float* beta2, const float* part2, int entries2, float* save_mean2, float* save_rstd2,
                         int n_groups, int rows, int c, int x_stride, int out_stride, int res_stride, int x2_stride, float eps,
                         int relu, cudaStream_t st) {
  DARDS_CHECK_ARG(x && out && gamma && beta && part && save_mean && save_rstd && entries > 0, "gbn_apply_fwd: null pointer");
  DARDS_CHECK_ARG(!x2 || (gamma2 && beta2 && part2 && save_mean2 && save_rstd2 && entries2 > 0),
                  "gbn_apply_fwd: the second normalised operand needs its own parameters and statistics");
  DARDS_CHECK_ARG(c > 0 && c % 8 == 0 && x_stride % 8 == 0 && out_stride % 8 == 0 && (!res || res_stride % 8 == 0) &&
                      (!x2 || x2_stride % 8 == 0),
                  "gbn_apply_fwd: channels and strides must be multiples of 8");
  DARDS_CHECK_ARG(c <= 2048, "gbn_apply_fwd: at most 2048 channels");
  DARDS_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(res) |
                    reinterpret_cast<uintptr_t>(x2)) & 15) == 0,
                  "gbn_apply_fwd: tensors must be 16-byte aligned");
  DARDS_CHECK_ARG(rows > 0, "gbn_apply_fwd: empty group");
  if (n_groups == 0) return DARDS_OK;
  GbnApplyArgs<__nv_bfloat16> a;
  a.x = static_cast<const __nv_bfloat16*>(x);
  a.out = static_cast<__nv_bfloat16*>(out);
  a.res = static_cast<const __nv_bfloat16*>(res);
  a.gamma = gamma; a.beta = beta; a.part = part; a.save_mean = save_mean; a.save_rstd = save_rstd;
  a.x2 = static_cast<const __nv_bfloat16*>(x2);
  a.gamma2 = gamma2; a.beta2 = beta2; a.part2 = part2; a.save_mean2 = save_mean2; a.save_rstd2 = save_rstd2;
  a.entries = entries; a.entries2 = entries2;
  a.n_groups = n_groups; a.rows = rows; a.c = c;
  a.x_stride = x_stride; a.out_stride = out_stride; a.res_stride = res_stride; a.x2_stride = x2_stride;
  a.eps = eps; a.relu = relu ? 1 : 0;
  // ~32 KB of each tensor per CTA: enough CTAs to fill the machine several times over, few enough that the statistics
  // merge (repeated by every CTA of a group) stays small
  long long bytes = (long long)rows * c * 2;
  int splits = (int)((bytes + 32767) / 32768);
  if (splits < 1) splits = 1;
  if (splits > rows) splits = rows;
  if (splits > 64) splits = 64;
  a.splits = splits;
  const size_t smem = (size_t)(x2 ? 4 : 2) * c * sizeof(float);
  gbn_apply_fwd_kernel<__nv_bfloat16, false><<<(unsigned)((long long)n_groups * splits), 256, smem, st>>>(a);
  DARDS_CHECK_LAUNCH("gbn_apply_fwd");
  return DARDS_OK;
}

template <typename T>
static void run_bn_affine_apply(const void* y, void* out, const void* res, const float* scale, const float* shift,
                                const void* y2, const float* scale2, const float* shift2, int rows, int c, int y_stride,
                                int out_stride, int res_stride, int y2_stride, int relu, cudaStream_t st) {
  GbnApplyArgs<T> a{};
  a.x = static_cast<const T*>(y);
  a.out = static_cast<T*>(out);
  a.res = static_cast<const T*>(res);
  a.gamma = scale; a.beta = shift;
  a.x2 = static_cast<const T*>(y2);
  a.gamma2 = scale2; a.beta2 = shift2;
  a.n_groups = 1; a.rows = rows; a.c = c;
  a.x_stride = y_stride; a.out_stride = out_stride; a.res_stride = res_stride; a.x2_stride = y2_stride;
  a.relu = relu ? 1 : 0;
  // ~32 KB of each tensor per CTA; nothing is repeated per CTA but the coefficient table, so no cap beyond the row count
  const long long bytes = (long long)rows * c * (long long)sizeof(T);
  long long splits = (bytes + 32767) / 32768;
  if (splits < 1) splits = 1;
  if (splits > rows) splits = rows;
  a.splits = (int)splits;
  const size_t smem = (size_t)(y2 ? 4 : 2) * c * sizeof(float);
  gbn_apply_fwd_kernel<T, true><<<(unsigned)splits, 256, smem, st>>>(a);
}

int launch_bn_affine_apply(const void* y, void* out, const void* res, const float* scale, const float* shift, const void* y2,
                           const float* scale2, const float* shift2, int rows, int c, int y_stride, int out_stride,
                           int res_stride, int y2_stride, int relu, int dtype, cudaStream_t st) {
  const int v = dtype == DARDS_BF16 ? 8 : 4;
  DARDS_CHECK_ARG(y && out && scale && shift, "bn_affine_apply: null pointer");
  DARDS_CHECK_ARG(!y2 || (scale2 && shift2), "bn_affine_apply: the second operand needs its own scale / shift");
  DARDS_CHECK_ARG(c > 0 && c % v == 0 && y_stride % v == 0 && out_stride % v == 0 && (!res || res_stride % v == 0) &&
                      (!y2 || y2_stride % v == 0),
                  "bn_affine_apply: channels and strides must be multiples of %d", v);
  DARDS_CHECK_ARG(y_stride >= c && out_stride >= c && (!res || res_stride >= c) && (!y2 || y2_stride >= c),
                  "bn_affine_apply: row stride smaller than channel count");
  DARDS_CHECK_ARG(c <= 2048, "bn_affine_apply: at most 2048 channels");
  DARDS_CHECK_ARG(((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(res) |
                    reinterpret_cast<uintptr_t>(y2)) & 15) == 0,
                  "bn_affine_apply: tensors must be 16-byte aligned");
  DARDS_CHECK_ARG(rows >= 0, "bn_affine_apply: negative row count");
  if (rows == 0) return DARDS_OK;
  if (dtype == DARDS_BF16)
    run_bn_affine_apply<__nv_bfloat16>(y, out, res, scale, shift, y2, scale2, shift2, rows, c, y_stride, out_stride,
                                       res_stride, y2_stride, relu, st);
  else
    run_bn_affine_apply<float>(y, out, res, scale, shift, y2, scale2, shift2, rows, c, y_stride, out_stride, res_stride,
                               y2_stride, relu, st);
  DARDS_CHECK_LAUNCH("bn_affine_apply");
  return DARDS_OK;
}

}  // namespace dards

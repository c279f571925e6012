// Shared device/host helpers for the deepards_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/deepards_b200.h"

namespace dards {

void set_error(const char* fmt, ...);
void count_launch();  // every kernel launch of the library goes through DARDS_CHECK_LAUNCH

#define DARDS_CHECK_ARG(cond, ...)            \
  do {                                        \
    if (!(cond)) {                            \
      ::dards::set_error(__VA_ARGS__);        \
      return DARDS_ERR_INVALID_ARGUMENT;      \
    }                                         \
  } while (0)

#define DARDS_CHECK_LAUNCH(name)                                                   \
  do {                                                                             \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess) {                                                      \
      ::dards::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));  \
      return DARDS_ERR_CUDA;                                                       \
    }                                                                              \
    ::dards::count_launch();                                                       \
  } while (0)

// ---- element type traits: activations are fp32 or bf16, arithmetic is always fp32 ----
template <typename T> struct Elem;
template <> struct Elem<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
  static __device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
  static __device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
  static __device__ __forceinline__ float round(float v) { return v; }
};
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
    uint2 r = *reinterpret_cast<const uint2*>(p);
    __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&r.x);
    __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&r.y);
    float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
  }
  static __device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 r;
    r.x = *reinterpret_cast<uint32_t*>(&a);
    r.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = r;
  }
  // value as it will be seen by the next reader of the stored tensor
  static __device__ __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// L2 eviction-priority hints for operands that are read for the LAST time (saved forward activations in the backward
// pass): evict_first keeps them from displacing the gradients that the next kernel re-reads.  g_dbg_l2_hint: debug key 9
// (0 = plain loads).
extern int g_dbg_l2_hint;
__device__ __forceinline__ uint64_t l2_policy(bool evict_first) {
  uint64_t p;
  if (evict_first) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// Batched ("one launch for a whole table of tensors") kernels: block b serves the descriptor j with
// first_block[j] <= b < first_block[j+1].  The whole CTA looks the table up in parallel -- a thread-0 linear scan is a
// chain of up to n dependent global loads (~0.7 us each), which was most of these small kernels' run time.
template <typename D>
__device__ __forceinline__ void find_block_desc(const D* __restrict__ descs, int n, D* s_desc) {
  const int b = (int)blockIdx.x;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const int lo = descs[j].first_block;
    const int hi = j + 1 < n ? descs[j + 1].first_block : 0x7fffffff;
    if (b >= lo && b < hi) *s_desc = descs[j];  // exactly one j matches (first_block is non-decreasing)
  }
  __syncthreads();
}

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// forward / dgrad implicit GEMM of the CUDA-core path (conv_simt.cu)
struct ConvGemmArgs {
  const void* in;
  const void* w;       // [t][c_red][c_cols]
  void* out;
  const void* addend;  // may be null
  long long m_total;   // n_breaths * l_dst
  int l_src, l_dst, c_red, c_cols, src_stride, dst_stride, addend_stride;
  int ktaps, q_mul, t_mul, off, div;  // source position = (q*q_mul + t*t_mul + off) / div
  // eval-mode BatchNorm epilogue (conv_gemm_kernel<T, true> only): out = [relu](acc * scale + shift [+ addend])
  const float* scale;
  const float* shift;
  int relu;
};

#define DARDS_DISPATCH_DTYPE(dtype, ...)                                  \
  if ((dtype) == DARDS_F32) {                                             \
    using T = float;                                                      \
    __VA_ARGS__                                                           \
  } else if ((dtype) == DARDS_BF16) {                                     \
    using T = __nv_bfloat16;                                              \
    __VA_ARGS__                                                           \
  } else {                                                                \
    ::dards::set_error("unknown dtype %d", (int)(dtype));                 \
    return DARDS_ERR_INVALID_ARGUMENT;                                    \
  }

}  // namespace dards

// Grouped BatchNorm1d (+residual, +ReLU) forward/backward on channels-last activations.
//
// Bandwidth-bound kernels.  One CTA owns (one group of `rows` = group*L rows) x (VPR 16-byte vectors of channels).
// Two implementations of each direction:
//
//  * cached (the fast path): the CTA's tile is read from global memory ONCE and parked in shared memory in a
//    thread-private layout (cache[k][tid]: every thread only ever re-reads what it wrote, so there are no bank
//    conflicts and no barriers around the cache); the later sweeps (centred variance, normalise / dx) run out of
//    shared memory.  HBM/L2 traffic = the algorithmic minimum: fwd 1 read + 1 write, bwd 2 reads (+mask) + 1 write.
//    The tile shape follows the layer: every ResNet-18 stage has rows*C = const, so (rows, channels per CTA) =
//    (1120,32) (560,32) (280,64) (140,128) all give 9 rows per thread and a 72 KB tile per tensor.
//  * streaming (generic fallback for tiles that do not fit): re-reads the tile from L1/L2 for every sweep.
//
// Statistics: the cached kernels use ONE sweep of sums shifted by a sample of the data (the group's first row), which loses
// no digits in E[d^2] - E[d]^2 beyond a factor 1 + (sample - mean)^2 / var; the streaming fallback uses two sweeps (mean of
// the differences from the group's first row, then the centred sum of squares).
// Cross-group reductions (running statistics, dgamma/dbeta) are separate BATCHED kernels: one launch handles a
// whole table of BatchNorm layers (an in-kernel "last CTA reduces" variant was measured 12-19 us slower per launch:
// the gpu-scope fence of every CTA invalidates L1 and waits for its stores).
#include "common.cuh"

namespace dards {


template <typename T> struct Vec;
template <> struct Vec<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void unpack(const uint4& r, float (&v)[4]) {
    v[0] = __uint_as_float(r.x); v[1] = __uint_as_float(r.y); v[2] = __uint_as_float(r.z); v[3] = __uint_as_float(r.w);
  }
  static __device__ __forceinline__ uint4 pack(const float (&v)[4]) {
    return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  }
};
template <> struct Vec<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void unpack(const uint4& r, float (&v)[8]) {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ uint4 pack(const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 b = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&b);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
  }
};

template <typename T> __device__ __forceinline__ uint4 ld16(const T* p) { return *reinterpret_cast<const uint4*>(p); }
template <typename T> __device__ __forceinline__ void st16(T* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }

// =====================================================================================================
// cached kernels
// =====================================================================================================
// Sum v[NV] over all threads of the CTA that share the channel vector cq = tid % VPR (i.e. over the row lanes);
// every thread gets the totals of its own vector.  Warp shuffles over the row lanes inside a warp, then ONE thread
// per value adds the warps' partial sums in a fixed order (deterministic) and broadcasts through shared memory --
// this runs a few times per tile, so it must not cost every thread a loop over all warps.
template <int NV, int VPR, int THREADS>
__device__ __forceinline__ void rowlane_reduce(float (&v)[NV], float* red /* [THREADS/32 + 1][VPR*NV] */) {
  constexpr int NW = THREADS / 32, W = VPR * NV;
  static_assert(W <= THREADS, "one thread per reduced value");
#pragma unroll
  for (int off = VPR; off < 32; off <<= 1) {
#pragma unroll
    for (int j = 0; j < NV; ++j) v[j] += __shfl_xor_sync(0xffffffffu, v[j], off);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cq = threadIdx.x % VPR;
  __syncthreads();  // previous use of `red` is over
  if (lane < VPR) {
#pragma unroll
    for (int j = 0; j < NV; ++j) red[warp * W + lane * NV + j] = v[j];
  }
  __syncthreads();
  if (threadIdx.x < W) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < NW; ++w) t += red[w * W + threadIdx.x];
    red[NW * W + threadIdx.x] = t;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NV; ++j) v[j] = red[NW * W + cq * NV + j];
}

// 16-byte asynchronous global -> shared copy (LDGSTS, L2-only caching: the data is read once)
__device__ __forceinline__ void cp_async16(const void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async16_pol(const void* smem_dst, const void* gsrc, uint64_t policy) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(
                   (uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc), "l"(policy)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// The cached kernels are PERSISTENT: gridDim.x CTAs walk the (group, channel tile) list round-robin.  A tile is
// brought in with cp.async (no registers, the whole tile in flight at once); while the last sweep of tile i reads
// row k out of the cache and stores its result, it refills slot k with row k of tile i+1 -- so the loads of the next
// tile overlap the stores of the current one and an SM always has a full tile of requests outstanding.
// Row loops of the cached kernels: a thread owns rows rl, rl + LANES, ... of its channel vector.  All but the last
// iteration are full (every lane has a row), so only the tail is guarded, and every pointer advances by a constant
// per iteration -- per-row address arithmetic and bounds checks were a third of the instructions of these
// (instruction-issue bound) kernels.
template <typename F>
__device__ __forceinline__ void bn_for_rows(int kf, bool tail, F&& body) {
#pragma unroll 3
  for (int k = 0; k < kf; ++k) body();
  if (tail) body();
}

template <typename T, int VPR, int THREADS, bool HAS_RES, bool RELU>
__global__ void __launch_bounds__(THREADS)
    gbn_fwd_cached_kernel(const T* x, T* out, const T* res, const float* __restrict__ gamma, const float* __restrict__ beta,
                          float* __restrict__ save_mean, float* __restrict__ save_rstd, int n_groups, int rows, int c,
                          int x_stride, int out_stride, int res_stride, float eps, int x_last_use) {
  constexpr int V = Vec<T>::N, LANES = THREADS / VPR, CT = VPR * V;
  // x is the convolution output saved for the backward pass: after this read it is dead until then
  const uint64_t pol = l2_policy(x_last_use != 0);
  extern __shared__ uint4 cache[];  // [K][THREADS]
  __shared__ float red[(THREADS / 32 + 1) * VPR * 2 * V];
  const int rl = threadIdx.x / VPR, cq = threadIdx.x % VPR;
  const float inv_n = 1.f / (float)rows;
  const int kf = rows / LANES;                 // full iterations
  const bool tail = rl < rows - kf * LANES;    // this lane has a row in the last, partial iteration
  const int n_ct = (c + CT - 1) / CT;
  const int n_tiles = n_ct * n_groups;
  const size_t x_step = (size_t)LANES * x_stride, o_step = (size_t)LANES * out_stride, r_step = (size_t)LANES * res_stride;
  // this thread's first row (row lane rl) of its channel vector in the tile, or nullptr past the last channel
  auto tile_x = [&](int tile) -> const T* {
    const int c0 = (tile % n_ct) * CT + cq * V;
    return c0 < c ? x + ((size_t)(tile / n_ct) * rows + rl) * x_stride + c0 : nullptr;
  };
  int tile = blockIdx.x;
  if (tile < n_tiles) {
    const T* xp = tile_x(tile);
    if (xp) {
      uint4* slot = cache + threadIdx.x;
      bn_for_rows(kf, tail, [&]() { cp_async16_pol(slot, xp, pol); slot += THREADS; xp += x_step; });
    }
  }
  for (; tile < n_tiles; tile += gridDim.x) {
    const int g = tile / n_ct, c0 = (tile % n_ct) * CT + cq * V;
    const bool active = c0 < c;
    const T* xn = tile + gridDim.x < n_tiles ? tile_x(tile + gridDim.x) : nullptr;
    cp_async_wait_all();
    __syncthreads();  // row 0 (the shift) is read from another thread's slot
    // ---- sweep 1 (shared): shifted sums  sum(x - s), sum((x - s)^2)  with s = the group's first row.  One pass
    // with fp32-faithful variance: the shift is a sample of the data, so |mean - s| ~ std and the subtraction
    // E[d^2] - E[d]^2  cancels at most a digit (a plain sum of squares would lose |mean|^2/var). ----
    float acc[2 * V], shift[V];
#pragma unroll
    for (int j = 0; j < 2 * V; ++j) acc[j] = 0.f;
#pragma unroll
    for (int j = 0; j < V; ++j) shift[j] = 0.f;
    if (active) {
      Vec<T>::unpack(cache[cq], shift);  // row 0 lives in slot 0 of the thread with row lane 0
      const uint4* slot = cache + threadIdx.x;
      bn_for_rows(kf, tail, [&]() {
        float v[V];
        Vec<T>::unpack(*slot, v);
        slot += THREADS;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float d = v[j] - shift[j];
          acc[j] += d;
          acc[V + j] = fmaf(d, d, acc[V + j]);
        }
      
      });
    }
    rowlane_reduce<2 * V, VPR, THREADS>(acc, red);
    if (active) {
      float sc[V], sh[V];
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float md = acc[j] * inv_n;  // mean - shift
        const float var = fmaxf(fmaf(-md, md, acc[V + j] * inv_n), 0.f) + eps;
        const float mean = shift[j] + md;
        float rstd = rsqrtf(var);
        rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);  // one Newton step: the reference divides by sqrt()
        sc[j] = rstd * gamma[c0 + j];
        sh[j] = beta[c0 + j] - mean * sc[j];
        if (rl == 0) {
          save_mean[(size_t)g * c + c0 + j] = mean;
          save_rstd[(size_t)g * c + c0 + j] = rstd;
        }
      }
      // ---- sweep 2 (shared -> global): normalise (+residual) (+ReLU); refill the cache with the next tile ----
      const size_t row0 = (size_t)g * rows + rl;
      T* op = out + row0 * out_stride + c0;
      const T* rp = HAS_RES ? res + row0 * res_stride + c0 : nullptr;
      uint4* slot = cache + threadIdx.x;
      auto row = [&](const uint4& rr) {
        const uint4 raw = *slot;
        if (xn) {
          cp_async16_pol(slot, xn, pol);
          xn += x_step;
        }
        float v[V];
        Vec<T>::unpack(raw, v);
#pragma unroll
        for (int j = 0; j < V; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
        if (HAS_RES) {
          float e[V];
          Vec<T>::unpack(rr, e);
#pragma unroll
          for (int j = 0; j < V; ++j) v[j] += e[j];
        }
        if (RELU) {
#pragma unroll
          for (int j = 0; j < V; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        st16(op, Vec<T>::pack(v));
        op += o_step;
        slot += THREADS;
      };
      if (HAS_RES) {
        // the residual is the only global read of this sweep: keep three rows of it in flight
        int k = 0;
        for (; k + 3 <= kf; k += 3) {
          uint4 rr[3];
#pragma unroll
          for (int u = 0; u < 3; ++u) rr[u] = ld16(rp + u * r_step);
          rp += 3 * r_step;
#pragma unroll
          for (int u = 0; u < 3; ++u) row(rr[u]);
        }
        for (; k < kf; ++k) {
          const uint4 rr = ld16(rp);
          rp += r_step;
          row(rr);
        }
        if (tail) row(ld16(rp));
      } else {
        const uint4 none = make_uint4(0u, 0u, 0u, 0u);
        bn_for_rows(kf, tail, [&]() { row(none); });
      }
    } else if (xn) {
      // a thread past the last channel of THIS tile may own channels of the next one: refill only
      uint4* slot = cache + threadIdx.x;
      bn_for_rows(kf, tail, [&]() { cp_async16_pol(slot, xn, pol); slot += THREADS; xn += x_step; });
    }
  }
}

// NT = number of cached tensors: 2 (gradient, x) or 3 (+ the ReLU mask source of relu_mode 2)
// FROZEN: BatchNorm with constant statistics (nn.BatchNorm1d in eval() under a network in train(): running statistics).
// `gamma` / `beta` carry the forward's per-channel scale / shift (dards_bn_eval_coeffs_batched), `save_mean` / `save_rstd`
// the per-channel running_mean and 1/sqrt(running_var + eps); a "group" is just a tile of rows.  dx = scale * g: there
// is no mean-of-gradient term, and the per-tile sums are partials of dbeta / dgamma only.
template <typename T, int VPR, int THREADS, int RELU_MODE, bool FROZEN = false>
__global__ void __launch_bounds__(THREADS)
    gbn_bwd_cached_kernel(const T* dout, const T* x, const T* mask_src, const float* __restrict__ gamma,
                          const float* __restrict__ beta, const float* __restrict__ save_mean,
                          const float* __restrict__ save_rstd, T* dx, int accumulate_dx, T* dres,
                          float* __restrict__ dgamma_part, float* __restrict__ dbeta_part, int n_groups, int rows, int c,
                          int dout_stride, int x_stride, int mask_stride, int dx_stride, int dres_stride, int l2_hint) {
  constexpr int V = Vec<T>::N, LANES = THREADS / VPR, CT = VPR * V;
  constexpr bool USE_MASK = RELU_MODE == 2;
  // x (the saved pre-BatchNorm activation) and the ReLU mask source are read here for the last time in the step
  const uint64_t pol = l2_policy(l2_hint != 0);
  extern __shared__ uint4 cache[];  // [NT][K][THREADS]: gradient (masked in place by sweep 1), x, [mask source]
  __shared__ float red[(THREADS / 32 + 1) * VPR * 2 * V];
  const int rl = threadIdx.x / VPR, cq = threadIdx.x % VPR;
  const float inv_n = 1.f / (float)rows;
  const int kf = rows / LANES;
  const bool tail = rl < rows - kf * LANES;
  const int K = kf + (rows - kf * LANES > 0 ? 1 : 0);
  const int n_ct = (c + CT - 1) / CT;
  const int n_tiles = n_ct * n_groups;
  const size_t plane = (size_t)K * THREADS;  // uint4 slots per cached tensor
  const size_t g_step = (size_t)LANES * dout_stride, x_step = (size_t)LANES * x_stride, m_step = (size_t)LANES * mask_stride;
  auto tile_c0 = [&](int tile) { return (tile % n_ct) * CT + cq * V; };
  // per-tile pointers to this thread's first row, computed ONCE per tile (the tile -> (group, channel tile) division
  // must not sit in the per-row path)
  struct TilePtrs {
    const T* g;
    const T* x;
    const T* m;
  };
  auto tile_ptrs = [&](int tile) {
    const size_t row0 = (size_t)(tile / n_ct) * rows + rl;
    const int c0 = tile_c0(tile);
    TilePtrs tp;
    tp.g = dout + row0 * dout_stride + c0;
    tp.x = x + row0 * x_stride + c0;
    tp.m = USE_MASK ? mask_src + row0 * mask_stride + c0 : nullptr;
    return tp;
  };
  auto issue_rows = [&](TilePtrs tp) {  // the whole tile of this thread
    uint4* slot = cache + threadIdx.x;
    bn_for_rows(kf, tail, [&]() {
      cp_async16(slot, tp.g);
      cp_async16_pol(slot + plane, tp.x, pol);
      if (USE_MASK) cp_async16_pol(slot + 2 * plane, tp.m, pol);
      slot += THREADS;
      tp.g += g_step;
      tp.x += x_step;
      if (USE_MASK) tp.m += m_step;
    
      });
  };
  int tile = blockIdx.x;
  if (tile < n_tiles && tile_c0(tile) < c) issue_rows(tile_ptrs(tile));
  for (; tile < n_tiles; tile += gridDim.x) {
    const int g = tile / n_ct, c0 = tile_c0(tile);
    const bool active = c0 < c;
    const int next = tile + gridDim.x;
    const bool refill = next < n_tiles && tile_c0(next) < c;
    TilePtrs tn = refill ? tile_ptrs(next) : TilePtrs{nullptr, nullptr, nullptr};
    cp_async_wait_all();  // every thread only reads the slots it filled itself: no barrier needed
    float acc[2 * V];
#pragma unroll
    for (int j = 0; j < 2 * V; ++j) acc[j] = 0.f;
    float mean[V], rstd[V], sc[V], sh[V];
    const size_t row0 = (size_t)g * rows + rl;
    if (active) {
#pragma unroll
      for (int j = 0; j < V; ++j) {
        if (FROZEN) {
          mean[j] = save_mean[c0 + j];
          rstd[j] = save_rstd[c0 + j];
          sc[j] = gamma[c0 + j];
          sh[j] = beta[c0 + j];
        } else {
          mean[j] = save_mean[(size_t)g * c + c0 + j];
          rstd[j] = save_rstd[(size_t)g * c + c0 + j];
          sc[j] = rstd[j] * gamma[c0 + j];          // same arithmetic as the forward: y = fmaf(x, sc, sh)
          sh[j] = beta[c0 + j] - mean[j] * sc[j];
        }
      }
      // ---- sweep 1 (shared): mask the gradient in place, accumulate sum g and sum g*(x - mean) ----
      T* drp = dres ? dres + row0 * dres_stride + c0 : nullptr;
      const size_t d_step = (size_t)LANES * dres_stride;
      uint4* slot = cache + threadIdx.x;
      bn_for_rows(kf, tail, [&]() {
        float gv[V], xv[V];
        Vec<T>::unpack(*slot, gv);
        Vec<T>::unpack(*(slot + plane), xv);
        if (RELU_MODE == 1) {
#pragma unroll
          for (int j = 0; j < V; ++j)
            if (!(fmaf(xv[j], sc[j], sh[j]) > 0.f)) gv[j] = 0.f;
        } else if (RELU_MODE == 2) {
          float m[V];
          Vec<T>::unpack(*(slot + 2 * plane), m);
#pragma unroll
          for (int j = 0; j < V; ++j)
            if (!(m[j] > 0.f)) gv[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
          acc[j] += gv[j];
          acc[V + j] = fmaf(gv[j], xv[j] - mean[j], acc[V + j]);  // x rstd after the reduction
        }
        if (RELU_MODE != 0) {
          const uint4 pg = Vec<T>::pack(gv);  // exact: masking keeps or zeroes a value that already is a T
          *slot = pg;
          if (drp) st16(drp, pg);
        } else if (drp) {
          st16(drp, *slot);
        }
        if (drp) drp += d_step;
        slot += THREADS;
      
      });
    }
    rowlane_reduce<2 * V, VPR, THREADS>(acc, red);
    if (active) {
#pragma unroll
      for (int j = 0; j < V; ++j) acc[V + j] *= rstd[j];
      if (rl == 0) {
#pragma unroll
        for (int j = 0; j < V; ++j) {
          if (dbeta_part) dbeta_part[(size_t)g * c + c0 + j] = acc[j];
          if (dgamma_part) dgamma_part[(size_t)g * c + c0 + j] = acc[V + j];
        }
      }
      // dx = sc*(g - m1 - xhat*m2) = sc*g + kb*x + kc  (FROZEN: dx = sc*g).  fp32 keeps x - mean apart: with the mean
      // folded into kc, kb*x and kc cancel when |mean| >> std (~50x torch's error at |mean|/std = 1e3); a bf16 x already
      // carries 2^-9 |x| of rounding and keeps the fold
      constexpr bool XC = sizeof(T) == 4;
      float kb[V], kc[V];
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float m1 = acc[j] * inv_n, m2 = acc[V + j] * inv_n;
        kb[j] = FROZEN ? 0.f : -sc[j] * m2 * rstd[j];
        kc[j] = FROZEN ? 0.f : (XC ? -sc[j] * m1 : -sc[j] * m1 - kb[j] * mean[j]);
      }
      // ---- sweep 2 (shared -> global): dx; refill the cache with the next tile ----
      T* dxp = dx + row0 * dx_stride + c0;
      const size_t dx_step = (size_t)LANES * dx_stride;
      uint4* slot = cache + threadIdx.x;
      bn_for_rows(kf, tail, [&]() {
        uint4 ro;
        if (accumulate_dx) ro = ld16(dxp);
        const uint4 rg = *slot, rx = *(slot + plane);
        if (refill) {
          cp_async16(slot, tn.g);
          cp_async16_pol(slot + plane, tn.x, pol);
          if (USE_MASK) cp_async16_pol(slot + 2 * plane, tn.m, pol);
          tn.g += g_step;
          tn.x += x_step;
          if (USE_MASK) tn.m += m_step;
        }
        float gv[V], xv[V], o[V];
        Vec<T>::unpack(rg, gv);
        Vec<T>::unpack(rx, xv);
#pragma unroll
        for (int j = 0; j < V; ++j)
          o[j] = FROZEN ? sc[j] * gv[j] : fmaf(sc[j], gv[j], fmaf(kb[j], XC ? xv[j] - mean[j] : xv[j], kc[j]));
        if (accumulate_dx) {
          float e[V];
          Vec<T>::unpack(ro, e);
#pragma unroll
          for (int j = 0; j < V; ++j) o[j] += e[j];
        }
        st16(dxp, Vec<T>::pack(o));
        dxp += dx_step;
        slot += THREADS;
      
      });
    } else if (refill) {
      issue_rows(tn);
    }
  }
}

// =====================================================================================================
// streaming kernels (generic fallback): 256 threads = 32 row lanes x 8 channel vectors
// =====================================================================================================
constexpr int BN_THREADS = 256;
constexpr int BN_LANES = 32;
constexpr int BN_QUADS = 8;
constexpr int BN_MAXCT = BN_QUADS * 8;  // 64 channels per CTA for bf16, 32 for fp32

// reduce v[V] over the 32 row lanes; the total for channel (cq*V + j) is returned to every thread of vector cq
template <int V>
__device__ __forceinline__ void lane_reduce(float (&v)[V], float (*red)[BN_MAXCT + 1], float* bcast, int rl, int cq) {
  __syncthreads();  // protect red/bcast from the previous use
#pragma unroll
  for (int j = 0; j < V; ++j) red[rl][cq * V + j] = v[j];
  __syncthreads();
  if (threadIdx.x < BN_QUADS * V) {
    float s = 0.f;
#pragma unroll 8
    for (int r = 0; r < BN_LANES; ++r) s += red[r][threadIdx.x];
    bcast[threadIdx.x] = s;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < V; ++j) v[j] = bcast[cq * V + j];
}

template <typename T>
__global__ void __launch_bounds__(BN_THREADS)
    gbn_fwd_kernel(const T* x, T* out, const T* res, const float* __restrict__ gamma, const float* __restrict__ beta,
                   float* __restrict__ save_mean, float* __restrict__ save_rstd, int rows, int c, int x_stride,
                   int out_stride, int res_stride, float eps, int relu) {
  constexpr int V = Vec<T>::N;
  __shared__ float red[BN_LANES][BN_MAXCT + 1];
  __shared__ float bcast[BN_MAXCT];
  const int g = blockIdx.y;
  const int rl = threadIdx.x >> 3, cq = threadIdx.x & 7;
  const int c0 = blockIdx.x * (BN_QUADS * V) + cq * V;
  const bool active = c0 < c;
  const size_t row_base = (size_t)g * rows;
  const float inv_n = 1.f / (float)rows;
  const T* xp = x + row_base * x_stride + c0;

  // the mean as the group's first row plus the mean of the differences: a constant channel gets its value exactly, however
  // 1/rows rounds (with var = 0 and rstd = 1/sqrt(eps), a mean one ulp off moves the output by ~300 ulps of x)
  float s[V], x0[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s[j] = x0[j] = 0.f;
  if (active) {
    Vec<T>::unpack(ld16(xp), x0);
    for (int r = rl; r < rows; r += BN_LANES) {
      float v[V];
      Vec<T>::unpack(ld16(xp + (size_t)r * x_stride), v);
#pragma unroll
      for (int j = 0; j < V; ++j) s[j] += v[j] - x0[j];
    }
  }
  lane_reduce<V>(s, red, bcast, rl, cq);
  float mean[V];
#pragma unroll
  for (int j = 0; j < V; ++j) mean[j] = fmaf(s[j], inv_n, x0[j]);

  float q[V];
#pragma unroll
  for (int j = 0; j < V; ++j) q[j] = 0.f;
  if (active)
    for (int r = rl; r < rows; r += BN_LANES) {
      float v[V];
      Vec<T>::unpack(ld16(xp + (size_t)r * x_stride), v);
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float d = v[j] - mean[j];
        q[j] = fmaf(d, d, q[j]);
      }
    }
  lane_reduce<V>(q, red, bcast, rl, cq);
  if (!active) return;
  float sc[V], sh[V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float var = q[j] * inv_n + eps;
    float rstd = rsqrtf(var);
    rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);
    sc[j] = rstd * gamma[c0 + j];
    sh[j] = beta[c0 + j] - mean[j] * sc[j];
    if (rl == 0) {
      save_mean[(size_t)g * c + c0 + j] = mean[j];
      save_rstd[(size_t)g * c + c0 + j] = rstd;
    }
  }
  T* op = out + row_base * out_stride + c0;
  const T* rp = res ? res + row_base * res_stride + c0 : nullptr;
  for (int r = rl; r < rows; r += BN_LANES) {
    float v[V];
    Vec<T>::unpack(ld16(xp + (size_t)r * x_stride), v);
#pragma unroll
    for (int j = 0; j < V; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
    if (rp) {
      float e[V];
      Vec<T>::unpack(ld16(rp + (size_t)r * res_stride), e);
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] += e[j];
    }
    if (relu) {
#pragma unroll
      for (int j = 0; j < V; ++j) v[j] = fmaxf(v[j], 0.f);
    }
    st16(op + (size_t)r * out_stride, Vec<T>::pack(v));
  }
}

template <typename T, bool FROZEN = false>  // FROZEN: as in gbn_bwd_cached_kernel
__global__ void __launch_bounds__(BN_THREADS)
    gbn_bwd_kernel(const T* dout, const T* x, const T* mask_src, const float* __restrict__ gamma,
                   const float* __restrict__ beta, const float* __restrict__ save_mean, const float* __restrict__ save_rstd,
                   T* dx, int accumulate_dx, T* dres, float* __restrict__ dgamma_part, float* __restrict__ dbeta_part,
                   int rows, int c, int dout_stride, int x_stride, int mask_stride, int dx_stride, int dres_stride,
                   int relu_mode) {
  constexpr int V = Vec<T>::N;
  __shared__ float red[BN_LANES][BN_MAXCT + 1];
  __shared__ float bcast[BN_MAXCT];
  const int g = blockIdx.y;
  const int rl = threadIdx.x >> 3, cq = threadIdx.x & 7;
  const int c0 = blockIdx.x * (BN_QUADS * V) + cq * V;
  const bool active = c0 < c;
  const size_t row_base = (size_t)g * rows;
  const float inv_n = 1.f / (float)rows;
  const T* gp = dout + row_base * dout_stride + c0;
  const T* xp = x + row_base * x_stride + c0;
  const T* mp = relu_mode == 2 ? mask_src + row_base * mask_stride + c0 : nullptr;

  float mean[V], rstd[V], sc[V], sh[V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const size_t so = FROZEN ? 0 : (size_t)g * c;
    mean[j] = active ? save_mean[so + c0 + j] : 0.f;
    rstd[j] = active ? save_rstd[so + c0 + j] : 0.f;
    const float gm = active ? gamma[c0 + j] : 0.f, bt = active ? beta[c0 + j] : 0.f;
    sc[j] = FROZEN ? gm : rstd[j] * gm;
    sh[j] = FROZEN ? bt : bt - mean[j] * sc[j];
  }
  auto load_row = [&](int r, float (&gv)[V], float (&xv)[V]) {
    Vec<T>::unpack(ld16(gp + (size_t)r * dout_stride), gv);
    Vec<T>::unpack(ld16(xp + (size_t)r * x_stride), xv);
    if (relu_mode == 1) {
#pragma unroll
      for (int j = 0; j < V; ++j)
        if (!(fmaf(xv[j], sc[j], sh[j]) > 0.f)) gv[j] = 0.f;
    } else if (relu_mode == 2) {
      float m[V];
      Vec<T>::unpack(ld16(mp + (size_t)r * mask_stride), m);
#pragma unroll
      for (int j = 0; j < V; ++j)
        if (!(m[j] > 0.f)) gv[j] = 0.f;
    }
  };

  float s1[V], s2[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s1[j] = s2[j] = 0.f;
  if (active)
    for (int r = rl; r < rows; r += BN_LANES) {
      float gv[V], xv[V];
      load_row(r, gv, xv);
#pragma unroll
      for (int j = 0; j < V; ++j) {
        s1[j] += gv[j];
        s2[j] = fmaf(gv[j], (xv[j] - mean[j]) * rstd[j], s2[j]);
      }
    }
  lane_reduce<V>(s1, red, bcast, rl, cq);
  lane_reduce<V>(s2, red, bcast, rl, cq);
  if (!active) return;
  if (rl == 0) {
#pragma unroll
    for (int j = 0; j < V; ++j) {
      if (dbeta_part) dbeta_part[(size_t)g * c + c0 + j] = s1[j];
      if (dgamma_part) dgamma_part[(size_t)g * c + c0 + j] = s2[j];
    }
  }
  constexpr bool XC = sizeof(T) == 4;  // fp32: kb*(x - mean) - sc*m1, as in the cached kernel
  float kb[V], kc[V];
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float m1 = s1[j] * inv_n, m2 = s2[j] * inv_n;
    kb[j] = FROZEN ? 0.f : -sc[j] * m2 * rstd[j];
    kc[j] = FROZEN ? 0.f : (XC ? -sc[j] * m1 : -sc[j] * m1 - kb[j] * mean[j]);
  }
  T* dxp = dx + row_base * dx_stride + c0;
  T* drp = dres ? dres + row_base * dres_stride + c0 : nullptr;
  for (int r = rl; r < rows; r += BN_LANES) {
    float gv[V], xv[V], o[V];
    load_row(r, gv, xv);
#pragma unroll
    for (int j = 0; j < V; ++j)
      o[j] = FROZEN ? sc[j] * gv[j] : fmaf(sc[j], gv[j], fmaf(kb[j], XC ? xv[j] - mean[j] : xv[j], kc[j]));
    if (drp) st16(drp + (size_t)r * dres_stride, Vec<T>::pack(gv));
    if (accumulate_dx) {
      float e[V];
      Vec<T>::unpack(ld16(dxp + (size_t)r * dx_stride), e);
#pragma unroll
      for (int j = 0; j < V; ++j) o[j] += e[j];
    }
    st16(dxp + (size_t)r * dx_stride, Vec<T>::pack(o));
  }
}

// =====================================================================================================
// reductions over the groups
// =====================================================================================================
// One CTA (256 threads) reduces a [rows][c] fp32 table over the rows for 64 consecutive columns: threads = 16 float4
// columns x 16 row lanes; every lane keeps 8 independent 16-byte loads in flight and the lane sums are combined in a
// fixed order -> deterministic.  wfun(r) weights row r; tfun transforms a loaded value.
template <typename WF, typename TF>
__device__ __forceinline__ float4 table_reduce64(const float* __restrict__ table, int rows, int c, int col0, WF wfun,
                                                 TF tfun, float4* scratch /* 256 */) {
  const int col = threadIdx.x & 15, ln = threadIdx.x >> 4;
  const int ch = col0 + col * 4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ch < c) {  // c % 4 == 0
#pragma unroll 8
    for (int r = ln; r < rows; r += 16) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(table + (size_t)r * c + ch));
      const float w = wfun(r);
      s.x = fmaf(w, tfun(v.x), s.x); s.y = fmaf(w, tfun(v.y), s.y);
      s.z = fmaf(w, tfun(v.z), s.z); s.w = fmaf(w, tfun(v.w), s.w);
    }
  }
  __syncthreads();
  scratch[threadIdx.x] = s;
  __syncthreads();
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  if (threadIdx.x < 16) {
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 v = scratch[k * 16 + threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
  }
  return t;  // valid in threads [0, 16): columns col0 + 4*threadIdx.x .. +3
}

// out[i] (+)= sum_r part[r][i] for a whole table of tensors in one launch
__global__ void __launch_bounds__(256) reduce_rows_batched_kernel(const dards_reduce_desc* __restrict__ descs, int n) {
  __shared__ dards_reduce_desc d;
  __shared__ float4 scratch[256];
  find_block_desc(descs, n, &d);
  const int col0 = ((int)blockIdx.x - d.first_block) * 64;
  const float4 t = table_reduce64(d.part, d.rows, d.c, col0, [](int) { return 1.f; }, [](float v) { return v; }, scratch);
  const int ch = col0 + threadIdx.x * 4;
  if (threadIdx.x < 16 && ch < d.c) {
    float4* o = reinterpret_cast<float4*>(d.out + ch);
    float4 r = t;
    if (d.accumulate) {
      const float4 old = *o;
      r.x += old.x; r.y += old.y; r.z += old.z; r.w += old.w;
    }
    *o = r;
  }
}

// nn.BatchNorm1d updates its running statistics once per group IN ORDER:  r <- (1-m) r + m v_g,  g = 0..G-1.
// Closed form (SURVEY.md hard part 6):  r_G = (1-m)^G r_0 + m * sum_g (1-m)^(G-1-g) v_g  -- a weighted reduction.
// The variance is recovered from the saved rstd: var_g = 1/rstd_g^2 - eps (biased) -> unbiased.
__device__ __forceinline__ void running_update_block(const dards_running_desc& d, int col0, float eps, float4* scratch) {
  const int n_groups = d.n_groups;
  const float momentum = d.momentum;
  const float unbias = d.rows_per_group > 1 ? (float)d.rows_per_group / (float)(d.rows_per_group - 1) : 1.f;
  const float lg = log2f(1.f - momentum);
  auto wfun = [&](int g) { return momentum * exp2f(lg * (float)(n_groups - 1 - g)); };
  const float4 tm = table_reduce64(d.save_mean, n_groups, d.c, col0, wfun, [](float v) { return v; }, scratch);
  const float4 tv = table_reduce64(d.save_rstd, n_groups, d.c, col0, wfun,
                                   [&](float r) { return fmaxf(1.f / (r * r) - eps, 0.f) * unbias; }, scratch);
  const int ch = col0 + threadIdx.x * 4;
  if (threadIdx.x < 16 && ch < d.c) {
    const float decay = exp2f(lg * (float)n_groups);
    float4* pm = reinterpret_cast<float4*>(d.running_mean + ch);
    float4* pv = reinterpret_cast<float4*>(d.running_var + ch);
    float4 m = *pm, v = *pv;
    m.x = decay * m.x + tm.x; m.y = decay * m.y + tm.y; m.z = decay * m.z + tm.z; m.w = decay * m.w + tm.w;
    v.x = decay * v.x + tv.x; v.y = decay * v.y + tv.y; v.z = decay * v.z + tv.z; v.w = decay * v.w + tv.w;
    *pm = m;
    *pv = v;
  }
  if (col0 == 0 && threadIdx.x == 0 && d.num_batches_tracked) *d.num_batches_tracked += n_groups;
}

__global__ void __launch_bounds__(256) bn_running_update_batched_kernel(const dards_running_desc* __restrict__ descs, int n,
                                                                        float eps) {
  __shared__ dards_running_desc d;
  __shared__ float4 scratch[256];
  find_block_desc(descs, n, &d);
  running_update_block(d, ((int)blockIdx.x - d.first_block) * 64, eps, scratch);
}

// eval-mode BatchNorm as y*scale + shift for every layer of a network: thread = channel, 64 channels per block.
// 1/sqrt (IEEE) rather than rsqrtf: a small running_var is amplified by gamma, and ATen's eval path divides by sqrt.
__global__ void __launch_bounds__(64) bn_eval_coeffs_batched_kernel(const dards_eval_coeff_desc* __restrict__ descs, int n,
                                                                    float eps) {
  __shared__ dards_eval_coeff_desc d;
  find_block_desc(descs, n, &d);
  const int ch = ((int)blockIdx.x - d.first_block) * 64 + (int)threadIdx.x;
  if (ch < d.c) {
    const float sc = d.gamma[ch] / sqrtf(d.running_var[ch] + eps);
    d.scale[ch] = sc;
    d.shift[ch] = d.beta[ch] - d.running_mean[ch] * sc;
  }
}

__global__ void __launch_bounds__(256) bn_running_update_kernel(dards_running_desc d, float eps) {
  __shared__ float4 scratch[256];
  running_update_block(d, (int)blockIdx.x * 64, eps, scratch);
}

// single tensor: 256 threads = 32 columns x 8 row lanes (any c), fixed summation order -> deterministic
constexpr int RR_LANES = 8;
__global__ void __launch_bounds__(256) reduce_rows_kernel(const float* __restrict__ part, float* __restrict__ out,
                                                          int rows, int c, int accumulate) {
  __shared__ float red[RR_LANES][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + cl;
  float s = 0.f;
  if (i < c) {
#pragma unroll 8
    for (int r = rl; r < rows; r += RR_LANES) s += part[(size_t)r * c + i];
  }
  red[rl][cl] = s;
  __syncthreads();
  if (rl == 0 && i < c) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < RR_LANES; ++k) t += red[k][cl];
    out[i] = accumulate ? out[i] + t : t;
  }
}

// ---- host launchers ------------------------------------------------------------------------------
static int vec_of(int dtype) { return dtype == DARDS_BF16 ? 8 : 4; }

int sm_count();  // conv_tc.cu: device SM count, or the limit set by dards_set_sm_limit
static int bn_sm_count() { return sm_count(); }

// cached-kernel configurations: (threads, vectors per row) in order of preference for a given row count
struct BnCfg { int threads, vpr; };
static const BnCfg kBnCfgs[] = {{256, 16}, {256, 8}, {256, 4}, {512, 4}};
constexpr int BN_MAX_K = 9;                 // rows per thread (bounds the cache: 9 * threads * 16 B per tensor)
constexpr int BN_CACHE_LIMIT = 222 * 1024;  // dynamic shared memory we are willing to ask for (3 x 72 KB tiles fit)

int g_dbg_bn_shift = -1;  // debug key 15 = s: skip the s widest tile configurations that would fit (narrower tiles, more of them)
int g_dbg_bn_k = -1;      // debug key 16 = 1: resident CTAs per SM chosen for the fullest last wave instead of the maximum

// picks a configuration whose tile holds the whole group; -1 -> use the streaming kernels
static int bn_pick_cfg_from(int first, int rows, int c, int v, int tensors);
static int bn_pick_cfg(int rows, int c, int v, int tensors) {
  int cfg = bn_pick_cfg_from(0, rows, c, v, tensors);
  for (int s = 0; s < g_dbg_bn_shift && cfg >= 0; ++s) {
    const int narrower = bn_pick_cfg_from(cfg + 1, rows, c, v, tensors);
    if (narrower < 0) break;
    cfg = narrower;
  }
  return cfg;
}
static int bn_pick_cfg_from(int first, int rows, int c, int v, int tensors) {
  for (int i = first; i < 4; ++i) {
    const int lanes = kBnCfgs[i].threads / kBnCfgs[i].vpr;
    const int k = ceil_div(rows, lanes);
    if (k > BN_MAX_K) continue;
    if (i < 2 && kBnCfgs[i].vpr * v / 2 >= c) continue;  // tile at least twice as wide as the tensor
    if ((long long)k * kBnCfgs[i].threads * 16 * tensors > BN_CACHE_LIMIT) continue;
    return i;
  }
  return -1;
}

template <typename K>
static int bn_smem_optin(K kernel, size_t smem, size_t* granted) {
  if (smem <= *granted) return DARDS_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess)  // the tiles are sized so that several CTAs share an SM: ask for all of the shared memory
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) {
    set_error("gbn: cannot opt in to %zu bytes of shared memory: %s", smem, cudaGetErrorString(e));
    return DARDS_ERR_CUDA;
  }
  *granted = smem;
  return DARDS_OK;
}

// persistent grid: as many CTAs per SM as the tile's shared memory allows (at most 4; 2048 threads per SM)
static int bn_persistent_grid(size_t smem_dyn, size_t smem_static, int threads, int n_tiles) {
  int per_sm = (int)((227 * 1024) / (smem_dyn + smem_static + 1024));
  if (per_sm > 4) per_sm = 4;
  if (per_sm * threads > 2048) per_sm = 2048 / threads;
  if (per_sm < 1) per_sm = 1;
  if (g_dbg_bn_k == 1 && per_sm > 2) {
    // equal tiles in lock-step rounds: the last round of ceil(n_tiles / slots) is only partly filled.  Among 2..per_sm
    // resident CTAs take the count that wastes the least of it (ties: the larger count).
    int best = per_sm;
    double best_eff = 0.0;
    for (int k = per_sm; k >= 2; --k) {
      const double x = (double)n_tiles / ((double)k * bn_sm_count());
      const double eff = x / (double)(long long)(x + 0.999999);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = k; }
    }
    per_sm = best;
  }
  int grid = per_sm * bn_sm_count();
  return grid < n_tiles ? grid : n_tiles;
}

template <typename T, int VPR, int THREADS, bool HAS_RES, bool RELU>
static int run_fwd_cached_v(const void* x, void* out, const void* res, const float* gamma, const float* beta,
                            float* save_mean, float* save_rstd, int n_groups, int rows, int c, int x_stride, int out_stride,
                            int res_stride, float eps, int x_last_use, cudaStream_t st) {
  static size_t granted = 32 * 1024;
  const size_t smem = (size_t)ceil_div(rows, THREADS / VPR) * THREADS * 16;
  int rc = bn_smem_optin(gbn_fwd_cached_kernel<T, VPR, THREADS, HAS_RES, RELU>, smem, &granted);
  if (rc) return rc;
  const int n_tiles = ceil_div(c, VPR * Vec<T>::N) * n_groups;
  const int grid = bn_persistent_grid(smem, (THREADS / 32 + 1) * VPR * 2 * Vec<T>::N * 4, THREADS, n_tiles);
  gbn_fwd_cached_kernel<T, VPR, THREADS, HAS_RES, RELU><<<grid, THREADS, smem, st>>>(
      static_cast<const T*>(x), static_cast<T*>(out), static_cast<const T*>(res), gamma, beta, save_mean, save_rstd,
      n_groups, rows, c, x_stride, out_stride, res_stride, eps, x_last_use);
  return DARDS_OK;
}

template <typename T, int VPR, int THREADS>
static int run_fwd_cached(const void* x, void* out, const void* res, const float* gamma, const float* beta,
                          float* save_mean, float* save_rstd, int n_groups, int rows, int c, int x_stride, int out_stride,
                          int res_stride, float eps, int relu, int x_last_use, cudaStream_t st) {
#define BN_FWD_V(R, A)                                                                                               \
  return run_fwd_cached_v<T, VPR, THREADS, R, A>(x, out, res, gamma, beta, save_mean, save_rstd, n_groups, rows, c, \
                                                 x_stride, out_stride, res_stride, eps, x_last_use, st)
  if (res) {
    if (relu) BN_FWD_V(true, true);
    BN_FWD_V(true, false);
  }
  if (relu) BN_FWD_V(false, true);
  BN_FWD_V(false, false);
#undef BN_FWD_V
}

template <typename T, int VPR, int THREADS, int RELU_MODE, bool FROZEN>
static int run_bwd_cached_v(const void* dout, const void* x, const void* mask_src, const float* gamma, const float* beta,
                            const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx, void* dres,
                            float* dgamma_part, float* dbeta_part, int n_groups, int rows, int c, int dout_stride,
                            int x_stride, int mask_stride, int dx_stride, int dres_stride, cudaStream_t st) {
  static size_t granted = 24 * 1024;
  const size_t smem = (size_t)ceil_div(rows, THREADS / VPR) * THREADS * 16 * (RELU_MODE == 2 ? 3 : 2);
  int rc = bn_smem_optin(gbn_bwd_cached_kernel<T, VPR, THREADS, RELU_MODE, FROZEN>, smem, &granted);
  if (rc) return rc;
  const int n_tiles = ceil_div(c, VPR * Vec<T>::N) * n_groups;
  const int grid = bn_persistent_grid(smem, (THREADS / 32 + 1) * VPR * 2 * Vec<T>::N * 4, THREADS, n_tiles);
  gbn_bwd_cached_kernel<T, VPR, THREADS, RELU_MODE, FROZEN><<<grid, THREADS, smem, st>>>(
      static_cast<const T*>(dout), static_cast<const T*>(x), static_cast<const T*>(mask_src), gamma, beta, save_mean,
      save_rstd, static_cast<T*>(dx), accumulate_dx, static_cast<T*>(dres), dgamma_part, dbeta_part, n_groups, rows, c,
      dout_stride, x_stride, mask_stride, dx_stride, dres_stride, g_dbg_l2_hint != 0 ? 1 : 0);
  return DARDS_OK;
}

template <typename T, int VPR, int THREADS, bool FROZEN>
static int run_bwd_cached(const void* dout, const void* x, const void* mask_src, const float* gamma, const float* beta,
                          const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx, void* dres,
                          float* dgamma_part, float* dbeta_part, int n_groups, int rows, int c, int dout_stride,
                          int x_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode, cudaStream_t st) {
#define BN_BWD_V(M)                                                                                                     \
  return run_bwd_cached_v<T, VPR, THREADS, M, FROZEN>(dout, x, mask_src, gamma, beta, save_mean, save_rstd, dx, accumulate_dx, \
                                              dres, dgamma_part, dbeta_part, n_groups, rows, c, dout_stride, x_stride, \
                                              mask_stride, dx_stride, dres_stride, st)
  if (relu_mode == 0) BN_BWD_V(0);
  if (relu_mode == 1) BN_BWD_V(1);
  BN_BWD_V(2);
#undef BN_BWD_V
}

#define BN_DISPATCH_CFG(cfg, CALL)                                   \
  switch (cfg) {                                                     \
    case 0: { constexpr int VPR = 16, THREADS = 256; CALL; break; }  \
    case 1: { constexpr int VPR = 8, THREADS = 256; CALL; break; }   \
    case 2: { constexpr int VPR = 4, THREADS = 256; CALL; break; }   \
    default: { constexpr int VPR = 4, THREADS = 512; CALL; break; }  \
  }

int launch_gbn_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta, float* save_mean,
                   float* save_rstd, int n_groups, int rows, int c, int x_stride, int out_stride, int res_stride,
                   float eps, int relu, int dtype, cudaStream_t st) {
  const int x_last_use = ((relu & DARDS_HINT_LAST_USE) && g_dbg_l2_hint != 0) ? 1 : 0;
  relu &= 0xff;
  const int v = vec_of(dtype);
  DARDS_CHECK_ARG(c % v == 0 && x_stride % v == 0 && out_stride % v == 0 && (!res || res_stride % v == 0),
                  "gbn_fwd: channels and strides must be multiples of %d", v);
  DARDS_CHECK_ARG(rows > 0, "gbn_fwd: empty group");
  if (n_groups == 0) return DARDS_OK;
  DARDS_CHECK_ARG(n_groups <= 65535, "gbn_fwd: too many groups (%d)", n_groups);
  const int cfg = bn_pick_cfg(rows, c, v, 1);
  if (cfg >= 0) {
    int rc = DARDS_OK;
    DARDS_DISPATCH_DTYPE(dtype, {
      BN_DISPATCH_CFG(cfg, (rc = run_fwd_cached<T, VPR, THREADS>(x, out, res, gamma, beta, save_mean, save_rstd, n_groups, rows,
                                                                 c, x_stride, out_stride, res_stride, eps, relu, x_last_use, st)));
    })
    if (rc) return rc;
  } else {
    dim3 grid(ceil_div(c, BN_QUADS * v), n_groups);
    DARDS_DISPATCH_DTYPE(dtype, {
      gbn_fwd_kernel<T><<<grid, BN_THREADS, 0, st>>>(static_cast<const T*>(x), static_cast<T*>(out),
                                                     static_cast<const T*>(res), gamma, beta, save_mean, save_rstd, rows,
                                                     c, x_stride, out_stride, res_stride, eps, relu);
    })
  }
  DARDS_CHECK_LAUNCH("gbn_fwd");
  return DARDS_OK;
}

// shared by the batch-statistics backward (launch_gbn_bwd) and the constant-statistics one (launch_bn_frozen_bwd)
template <bool FROZEN>
static int run_gbn_bwd(const char* name, const void* dout, const void* x, const void* mask_src, const float* gamma,
                       const float* beta, const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx,
                       void* dres, float* dgamma_part, float* dbeta_part, int n_groups, int rows, int c, int dout_stride,
                       int x_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype,
                       cudaStream_t st) {
  const int v = vec_of(dtype);
  DARDS_CHECK_ARG(c % v == 0 && dout_stride % v == 0 && x_stride % v == 0 && dx_stride % v == 0,
                  "%s: channels and strides must be multiples of %d", name, v);
  DARDS_CHECK_ARG(relu_mode != 2 || (mask_src && mask_stride % v == 0), "%s: relu_mode 2 needs mask_src", name);
  DARDS_CHECK_ARG(!dres || dres_stride % v == 0, "%s: dres stride", name);
  if (n_groups == 0) return DARDS_OK;
  DARDS_CHECK_ARG(n_groups <= 65535, "%s: too many groups (%d)", name, n_groups);
  const int cfg = bn_pick_cfg(rows, c, v, relu_mode == 2 ? 3 : 2);
  if (cfg >= 0) {
    int rc = DARDS_OK;
    DARDS_DISPATCH_DTYPE(dtype, {
      BN_DISPATCH_CFG(cfg, (rc = run_bwd_cached<T, VPR, THREADS, FROZEN>(dout, x, mask_src, gamma, beta, save_mean, save_rstd,
                                                                         dx, accumulate_dx, dres, dgamma_part, dbeta_part,
                                                                         n_groups, rows, c, dout_stride, x_stride,
                                                                         mask_stride, dx_stride, dres_stride, relu_mode, st)));
    })
    if (rc) return rc;
  } else {
    dim3 grid(ceil_div(c, BN_QUADS * v), n_groups);
    DARDS_DISPATCH_DTYPE(dtype, {
      gbn_bwd_kernel<T, FROZEN><<<grid, BN_THREADS, 0, st>>>(
          static_cast<const T*>(dout), static_cast<const T*>(x), static_cast<const T*>(mask_src), gamma, beta, save_mean,
          save_rstd, static_cast<T*>(dx), accumulate_dx, static_cast<T*>(dres), dgamma_part, dbeta_part, rows, c,
          dout_stride, x_stride, mask_stride, dx_stride, dres_stride, relu_mode);
    })
  }
  DARDS_CHECK_LAUNCH(name);
  return DARDS_OK;
}

int launch_gbn_bwd(const void* dout, const void* x, const void* mask_src, const float* gamma, const float* beta,
                   const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx, void* dres,
                   float* dgamma_part, float* dbeta_part, int n_groups, int rows, int c, int dout_stride, int x_stride,
                   int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype, cudaStream_t st) {
  return run_gbn_bwd<false>("gbn_bwd", dout, x, mask_src, gamma, beta, save_mean, save_rstd, dx, accumulate_dx, dres,
                            dgamma_part, dbeta_part, n_groups, rows, c, dout_stride, x_stride, mask_stride, dx_stride,
                            dres_stride, relu_mode, dtype, st);
}

int launch_bn_frozen_bwd(const void* dout, const void* y, const void* mask_src, const float* scale, const float* shift,
                         const float* running_mean, const float* rstd, void* dx, int accumulate_dx, void* dres,
                         float* dgamma_part, float* dbeta_part, int n_tiles, int rows, int c, int dout_stride, int y_stride,
                         int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype, cudaStream_t st) {
  return run_gbn_bwd<true>("bn_frozen_bwd", dout, y, mask_src, scale, shift, running_mean, rstd, dx, accumulate_dx, dres,
                           dgamma_part, dbeta_part, n_tiles, rows, c, dout_stride, y_stride, mask_stride, dx_stride,
                           dres_stride, relu_mode, dtype, st);
}

int launch_reduce_rows(const float* part, float* out, int rows, int c, int accumulate, cudaStream_t st) {
  if (c == 0) return DARDS_OK;
  reduce_rows_kernel<<<ceil_div(c, 32), 256, 0, st>>>(part, out, rows, c, accumulate);
  DARDS_CHECK_LAUNCH("reduce_rows");
  return DARDS_OK;
}

int launch_reduce_rows_batched(const dards_reduce_desc* descs_dev, int n, int total_blocks, cudaStream_t st) {
  if (n == 0 || total_blocks == 0) return DARDS_OK;
  reduce_rows_batched_kernel<<<total_blocks, 256, 0, st>>>(descs_dev, n);
  DARDS_CHECK_LAUNCH("reduce_rows_batched");
  return DARDS_OK;
}

int launch_bn_running_update(const float* save_mean, const float* save_rstd, float* rm, float* rv, long long* nbt,
                             int n_groups, int rows, int c, float momentum, float eps, cudaStream_t st) {
  DARDS_CHECK_ARG(c % 4 == 0, "bn_running_update: channels must be a multiple of 4");
  dards_running_desc d;
  d.save_mean = save_mean; d.save_rstd = save_rstd; d.running_mean = rm; d.running_var = rv;
  d.num_batches_tracked = nbt; d.n_groups = n_groups; d.rows_per_group = rows; d.c = c; d.momentum = momentum;
  d.first_block = 0;
  bn_running_update_kernel<<<ceil_div(c, 64), 256, 0, st>>>(d, eps);
  DARDS_CHECK_LAUNCH("bn_running_update");
  return DARDS_OK;
}

int launch_bn_running_update_batched(const dards_running_desc* descs_dev, int n, int total_blocks, float eps,
                                     cudaStream_t st) {
  if (n == 0 || total_blocks == 0) return DARDS_OK;
  bn_running_update_batched_kernel<<<total_blocks, 256, 0, st>>>(descs_dev, n, eps);
  DARDS_CHECK_LAUNCH("bn_running_update_batched");
  return DARDS_OK;
}

int launch_bn_eval_coeffs_batched(const dards_eval_coeff_desc* descs_dev, int n, int total_blocks, float eps,
                                  cudaStream_t st) {
  if (n == 0 || total_blocks == 0) return DARDS_OK;
  bn_eval_coeffs_batched_kernel<<<total_blocks, 64, 0, st>>>(descs_dev, n, eps);
  DARDS_CHECK_LAUNCH("bn_eval_coeffs_batched");
  return DARDS_OK;
}

}  // namespace dards

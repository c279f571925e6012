// CUDA-core (FFMA, fp32 accumulate) implicit-GEMM Conv1d kernels on channels-last activations.
//
// This is the exact-fp32 path (parity <= 1e-4 vs the reference, SURVEY.md hard part 2: tcgen05 has no
// true-fp32 MMA) and the on-device checker for the tcgen05 kernels in conv_tc.cu.
//
//   forward / dgrad : one kernel, out[row, co] = sum_t sum_k in[src(row,t), k] * w[t][k][co]
//                     with src(row,t) = (q*q_mul + t*t_mul + off) / div inside the same breath
//   wgrad           : dW[t][ci][co] = sum_rows in[src(row,t), ci] * dout[row, co], split-K over rows,
//                     partials reduced in a fixed order (deterministic)
#include "common.cuh"

namespace dards {

// ------------------------------------------------------------------------------------------------
// weight packing
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, T* __restrict__ w_kio, T* __restrict__ w_koi,
                                        int c_out, int c_in, int ktaps) {
  int total = c_out * c_in * ktaps;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int t = i % ktaps;
    int ci = (i / ktaps) % c_in;
    int co = i / (ktaps * c_in);
    float v = w[i];
    if (w_kio) Elem<T>::st(w_kio + ((size_t)t * c_in + ci) * c_out + co, v);
    if (w_koi) Elem<T>::st(w_koi + ((size_t)t * c_out + co) * c_in + ci, v);
  }
}

// All convolutions of a network in ONE launch: block b serves descriptor j with first_block[j] <= b < first_block[j+1]
// and transposes one 32 (co) x 32 (ci) x ktaps tile through shared memory, so that the fp32 reads and both packed
// writes are coalesced (a per-element scatter of 2-byte stores costs a 32-byte sector each).
constexpr int PACK_TILE = 32;
constexpr int PACK_MAX_TAPS = 8;
template <typename T>
__global__ void __launch_bounds__(256) pack_conv_weights_batched_kernel(const dards_pack_desc* __restrict__ descs, int n) {
  __shared__ dards_pack_desc d;
  __shared__ float tile[PACK_TILE][PACK_TILE * PACK_MAX_TAPS + 1];
  find_block_desc(descs, n, &d);
  const int K = d.ktaps, c_in = d.c_in, c_out = d.c_out;
  const int n_co_t = (c_out + PACK_TILE - 1) / PACK_TILE;
  const int b = (int)blockIdx.x - d.first_block;
  const int co0 = (b % n_co_t) * PACK_TILE, ci0 = (b / n_co_t) * PACK_TILE;
  const int row = PACK_TILE * K;  // floats of one co row inside the tile
  for (int i = threadIdx.x; i < PACK_TILE * row; i += 256) {
    const int co_l = i / row, rem = i % row;
    const int co = co0 + co_l, ci = ci0 + rem / K;
    tile[co_l][rem] = (co < c_out && ci < c_in) ? d.w[((size_t)co * c_in + ci0) * K + rem] : 0.f;
  }
  __syncthreads();
  T* kio = static_cast<T*>(d.w_kio);
  T* koi = static_cast<T*>(d.w_koi);
  for (int i = threadIdx.x; i < PACK_TILE * PACK_TILE * K; i += 256) {
    const int a = i % PACK_TILE, bq = (i / PACK_TILE) % PACK_TILE, t = i / (PACK_TILE * PACK_TILE);
    if (koi) {  // a = ci (fastest in w_koi), bq = co
      const int ci = ci0 + a, co = co0 + bq;
      if (ci < c_in && co < c_out) Elem<T>::st(koi + ((size_t)t * c_out + co) * c_in + ci, tile[bq][a * K + t]);
    }
    if (kio) {  // a = co (fastest in w_kio), bq = ci
      const int co = co0 + a, ci = ci0 + bq;
      if (ci < c_in && co < c_out) Elem<T>::st(kio + ((size_t)t * c_in + ci) * c_out + co, tile[a][bq * K + t]);
    }
  }
}

// The inverse for the weight GRADIENTS of the accumulate-mode tcgen05 wgrad: dw[co][ci][t] = dw_t[t][co][ci] for a whole
// table of convolutions in one launch (one 32 x 32 x ktaps tile per block, through shared memory: both sides coalesced).
__global__ void __launch_bounds__(256) unpack_wgrad_batched_kernel(const dards_unpack_desc* __restrict__ descs, int n) {
  __shared__ dards_unpack_desc d;
  __shared__ float tile[PACK_TILE][PACK_TILE * PACK_MAX_TAPS + 1];
  find_block_desc(descs, n, &d);
  const int K = d.ktaps, c_in = d.c_in, c_out = d.c_out;
  const int n_co_t = (c_out + PACK_TILE - 1) / PACK_TILE;
  const int b = (int)blockIdx.x - d.first_block;
  const int co0 = (b % n_co_t) * PACK_TILE, ci0 = (b / n_co_t) * PACK_TILE;
  for (int i = threadIdx.x; i < PACK_TILE * PACK_TILE * K; i += 256) {
    const int a = i % PACK_TILE, bq = (i / PACK_TILE) % PACK_TILE, t = i / (PACK_TILE * PACK_TILE);
    const int ci = ci0 + a, co = co0 + bq;   // a = ci, fastest in dw_t
    tile[bq][a * K + t] = (ci < c_in && co < c_out) ? d.dw_t[((size_t)t * c_out + co) * c_in + ci] : 0.f;
  }
  __syncthreads();
  const int row = PACK_TILE * K;  // floats of one co row inside the tile
  for (int i = threadIdx.x; i < PACK_TILE * row; i += 256) {
    const int co_l = i / row, rem = i % row;
    const int co = co0 + co_l, ci = ci0 + rem / K;
    if (co < c_out && ci < c_in) d.dw[((size_t)co * c_in + ci0) * K + rem] = tile[co_l][rem];
  }
}

// ------------------------------------------------------------------------------------------------
// forward / dgrad implicit GEMM:  128 rows x 64 cols per CTA, BK = 16, 256 threads, 8x4 per thread
// ------------------------------------------------------------------------------------------------

constexpr int CG_BM = 128, CG_BN = 64, CG_BK = 16, CG_THREADS = 256;

// AFFINE: eval-mode BatchNorm epilogue, out = [relu](acc * scale[c] + shift[c] [+ addend]) in fp32, one rounding
template <typename T, bool AFFINE>
__global__ void __launch_bounds__(CG_THREADS, 2) conv_gemm_kernel(ConvGemmArgs a) {
  __shared__ __align__(16) float As[2][CG_BK][CG_BM + 4];
  __shared__ __align__(16) float Bs[2][CG_BK][CG_BN];

  const T* __restrict__ in = static_cast<const T*>(a.in);
  const T* __restrict__ w = static_cast<const T*>(a.w);
  const int tid = threadIdx.x;
  const long long row0 = (long long)blockIdx.x * CG_BM;
  const int col0 = blockIdx.y * CG_BN;

  // --- loader roles -----------------------------------------------------------------------------
  // A: thread -> (row = tid/2, 8 channels starting at (tid&1)*8)
  const int a_row = tid >> 1, a_k = (tid & 1) * 8;
  const long long a_grow = row0 + a_row;
  const bool a_row_ok = a_grow < a.m_total;
  const int a_n = a_row_ok ? (int)(a_grow / a.l_dst) : 0;
  const int a_q = a_row_ok ? (int)(a_grow % a.l_dst) : 0;
  // B: thread -> (k = tid/16, 4 cols at (tid%16)*4)
  const int b_k = tid >> 4, b_c = (tid & 15) * 4;
  const bool b_col_ok = (col0 + b_c) < a.c_cols;

  const int kchunks = a.c_red / CG_BK;  // c_red % 16 == 0 checked on the host
  const int steps = a.ktaps * kchunks;

  float4 ra0, ra1, rb;
  auto load_global = [&](int step) {
    const int t = step / kchunks, k0 = (step % kchunks) * CG_BK;
    ra0 = make_float4(0.f, 0.f, 0.f, 0.f);
    ra1 = ra0;
    rb = ra0;
    if (a_row_ok) {
      int pn = a_q * a.q_mul + t * a.t_mul + a.off;
      bool ok = pn >= 0;
      int p = pn;
      if (a.div > 1) {
        ok = ok && (pn % a.div == 0);
        p = pn / a.div;
      }
      if (ok && p < a.l_src) {
        const T* src = in + ((size_t)a_n * a.l_src + p) * a.src_stride + k0 + a_k;
        ra0 = Elem<T>::ld4(src);
        ra1 = Elem<T>::ld4(src + 4);
      }
    }
    if (b_col_ok) rb = Elem<T>::ld4(w + ((size_t)t * a.c_red + k0 + b_k) * a.c_cols + col0 + b_c);
  };
  auto store_smem = [&](int buf) {
    As[buf][a_k + 0][a_row] = ra0.x;
    As[buf][a_k + 1][a_row] = ra0.y;
    As[buf][a_k + 2][a_row] = ra0.z;
    As[buf][a_k + 3][a_row] = ra0.w;
    As[buf][a_k + 4][a_row] = ra1.x;
    As[buf][a_k + 5][a_row] = ra1.y;
    As[buf][a_k + 6][a_row] = ra1.z;
    As[buf][a_k + 7][a_row] = ra1.w;
    *reinterpret_cast<float4*>(&Bs[buf][b_k][b_c]) = rb;
  };

  // --- compute roles ----------------------------------------------------------------------------
  const int ty = tid >> 4, tx = tid & 15;  // rows ty*8.., cols tx*4..
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  load_global(0);
  store_smem(0);
  __syncthreads();
  for (int s = 0; s < steps; ++s) {
    const int buf = s & 1;
    if (s + 1 < steps) load_global(s + 1);
#pragma unroll
    for (int k = 0; k < CG_BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 8 + 4]);
      float4 b = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (s + 1 < steps) {
      store_smem(buf ^ 1);
      __syncthreads();
    }
  }

  // --- epilogue ---------------------------------------------------------------------------------
  T* __restrict__ out = static_cast<T*>(a.out);
  const T* __restrict__ addend = static_cast<const T*>(a.addend);
  const int c = col0 + tx * 4;
  if (c < a.c_cols) {
    float4 sc, sh;
    if (AFFINE) {
      sc = *reinterpret_cast<const float4*>(a.scale + c);
      sh = *reinterpret_cast<const float4*>(a.shift + c);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      long long r = row0 + ty * 8 + i;
      if (r < a.m_total) {
        float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (AFFINE) {
          v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
        }
        if (addend) {
          float4 e = Elem<T>::ld4(addend + (size_t)r * a.addend_stride + c);
          v.x += e.x; v.y += e.y; v.z += e.z; v.w += e.w;
        }
        if (AFFINE && a.relu) {
          v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
        }
        Elem<T>::st4(out + (size_t)r * a.dst_stride + c, v);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// wgrad: 64 (ci) x 64 (co) per CTA, BK = 16 rows of the (n,q) reduction, split-K over rows
// ------------------------------------------------------------------------------------------------
struct WgradArgs {
  const void* in;     // (N, l_in, in_stride)
  const void* dout;   // (N, l_out, dout_stride)
  float* partial;     // [splits][ktaps][c_in][c_out]
  long long m_total;  // n_breaths * l_out
  long long rows_per_split;
  int l_in, l_out, c_in, c_out, in_stride, dout_stride, ktaps, stride, pad;
};

constexpr int WG_BM = 64, WG_BN = 64, WG_BK = 16, WG_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(WG_THREADS, 2) conv_wgrad_kernel(WgradArgs a) {
  __shared__ __align__(16) float As[2][WG_BK][WG_BM];
  __shared__ __align__(16) float Bs[2][WG_BK][WG_BN];
  const T* __restrict__ in = static_cast<const T*>(a.in);
  const T* __restrict__ dout = static_cast<const T*>(a.dout);
  const int tid = threadIdx.x;
  const int tiles_co = (a.c_out + WG_BN - 1) / WG_BN;
  const int ci0 = (blockIdx.x / tiles_co) * WG_BM;
  const int co0 = (blockIdx.x % tiles_co) * WG_BN;
  const int t = blockIdx.y;
  const int split = blockIdx.z;
  const long long r_begin = (long long)split * a.rows_per_split;
  long long r_end = r_begin + a.rows_per_split;
  if (r_end > a.m_total) r_end = a.m_total;

  const int l_k = tid >> 4, l_c = (tid & 15) * 4;  // loader: row-in-chunk, 4 channels
  const bool a_ok_c = (ci0 + l_c) < a.c_in;
  const bool b_ok_c = (co0 + l_c) < a.c_out;

  float4 ra, rb;
  auto load_global = [&](long long rbase) {
    ra = make_float4(0.f, 0.f, 0.f, 0.f);
    rb = ra;
    long long r = rbase + l_k;
    if (r < r_end) {
      int n = (int)(r / a.l_out), q = (int)(r % a.l_out);
      int p = q * a.stride + t - a.pad;
      if (a_ok_c && p >= 0 && p < a.l_in) ra = Elem<T>::ld4(in + ((size_t)n * a.l_in + p) * a.in_stride + ci0 + l_c);
      if (b_ok_c) rb = Elem<T>::ld4(dout + (size_t)r * a.dout_stride + co0 + l_c);
    }
  };
  auto store_smem = [&](int buf) {
    *reinterpret_cast<float4*>(&As[buf][l_k][l_c]) = ra;
    *reinterpret_cast<float4*>(&Bs[buf][l_k][l_c]) = rb;
  };

  const int ty = tid >> 4, tx = tid & 15;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  if (r_begin < r_end) {
    load_global(r_begin);
    store_smem(0);
    __syncthreads();
    int s = 0;
    for (long long rb0 = r_begin; rb0 < r_end; rb0 += WG_BK, ++s) {
      const int buf = s & 1;
      const bool more = rb0 + WG_BK < r_end;
      if (more) load_global(rb0 + WG_BK);
#pragma unroll
      for (int k = 0; k < WG_BK; ++k) {
        float4 av = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
        float4 bv = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
        const float aa[4] = {av.x, av.y, av.z, av.w};
        const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
      }
      if (more) {
        store_smem(buf ^ 1);
        __syncthreads();
      }
    }
  }
  // partial[split][t][ci][co]
  float* __restrict__ P = a.partial + (((size_t)split * a.ktaps + t) * a.c_in) * a.c_out;
  const int co = co0 + tx * 4;
  if (co < a.c_out) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int ci = ci0 + ty * 4 + i;
      if (ci < a.c_in)
        *reinterpret_cast<float4*>(P + (size_t)ci * a.c_out + co) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
  }
}

// dw[co][ci][t] (+)= sum_s partial[s][t][ci][co]
__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits, int ktaps,
                                    int c_in, int c_out, int accumulate) {
  const int per = ktaps * c_in * c_out;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < per; i += gridDim.x * blockDim.x) {
    // i indexes [t][ci][co] so that the reads are coalesced
    int co = i % c_out, ci = (i / c_out) % c_in, t = i / (c_out * c_in);
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += partial[(size_t)k * per + i];
    size_t o = ((size_t)co * c_in + ci) * ktaps + t;
    dw[o] = accumulate ? dw[o] + s : s;
  }
}

static int wgrad_splits(long long m_total, int c_in, int c_out, int ktaps) {
  long long tiles = (long long)ceil_div(c_in, WG_BM) * ceil_div(c_out, WG_BN) * ktaps;
  long long want = (148LL * 4 + tiles - 1) / tiles;  // ~2 waves of 2 CTAs/SM
  long long max_by_rows = (m_total + 255) / 256;     // at least 256 rows per split
  if (want > max_by_rows) want = max_by_rows;
  if (want < 1) want = 1;
  if (want > 1024) want = 1024;
  return (int)want;
}

long long simt_wgrad_workspace_bytes(int n_breaths, int l_out, int c_in, int c_out, int ktaps) {
  long long m = (long long)n_breaths * l_out;
  return (long long)wgrad_splits(m, c_in, c_out, ktaps) * ktaps * c_in * c_out * (long long)sizeof(float);
}

// ------------------------------------------------------------------------------------------------
// host launchers (called from api.cu)
// ------------------------------------------------------------------------------------------------
int simt_pack_conv_weight(const float* w, void* w_kio, void* w_koi, int c_out, int c_in, int ktaps, int dtype,
                          cudaStream_t st) {
  int total = c_out * c_in * ktaps;
  int blocks = ceil_div(total, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  DARDS_DISPATCH_DTYPE(dtype, {
    pack_conv_weight_kernel<T><<<blocks, 256, 0, st>>>(w, static_cast<T*>(w_kio), static_cast<T*>(w_koi), c_out, c_in,
                                                       ktaps);
  })
  DARDS_CHECK_LAUNCH("pack_conv_weight");
  return DARDS_OK;
}

int simt_pack_conv_weights_batched(const dards_pack_desc* descs_dev, int n, int total_blocks, int dtype, cudaStream_t st) {
  if (n == 0 || total_blocks == 0) return DARDS_OK;
  DARDS_DISPATCH_DTYPE(dtype, { pack_conv_weights_batched_kernel<T><<<total_blocks, 256, 0, st>>>(descs_dev, n); })
  DARDS_CHECK_LAUNCH("pack_conv_weights_batched");
  return DARDS_OK;
}

int simt_unpack_wgrad_batched(const dards_unpack_desc* descs_dev, int n, int total_blocks, cudaStream_t st) {
  if (n == 0 || total_blocks == 0) return DARDS_OK;
  unpack_wgrad_batched_kernel<<<total_blocks, 256, 0, st>>>(descs_dev, n);
  DARDS_CHECK_LAUNCH("unpack_wgrad_batched");
  return DARDS_OK;
}

int simt_conv_gemm(const ConvGemmArgs& a, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(a.c_red % CG_BK == 0, "conv: reduction channels (%d) must be a multiple of %d", a.c_red, CG_BK);
  DARDS_CHECK_ARG(a.c_cols % 4 == 0, "conv: output channels (%d) must be a multiple of 4", a.c_cols);
  DARDS_CHECK_ARG(a.src_stride % 4 == 0 && a.dst_stride % 4 == 0 && (a.addend == nullptr || a.addend_stride % 4 == 0),
                  "conv: row strides must be multiples of 4 elements");
  if (a.m_total == 0) return DARDS_OK;
  dim3 grid(ceil_div(a.m_total, CG_BM), ceil_div(a.c_cols, CG_BN));
  DARDS_DISPATCH_DTYPE(dtype, {
    if (a.scale) conv_gemm_kernel<T, true><<<grid, CG_THREADS, 0, st>>>(a);
    else conv_gemm_kernel<T, false><<<grid, CG_THREADS, 0, st>>>(a);
  })
  DARDS_CHECK_LAUNCH("conv_gemm");
  return DARDS_OK;
}

int simt_conv_wgrad(const void* in, const void* dout, float* dw, int accumulate, void* workspace,
                    long long workspace_bytes, int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride,
                    int dout_stride, int ktaps, int stride, int pad, int dtype, cudaStream_t st) {
  DARDS_CHECK_ARG(c_in % 4 == 0 && c_out % 4 == 0, "wgrad: channels must be multiples of 4 (c_in=%d c_out=%d)", c_in,
                  c_out);
  DARDS_CHECK_ARG(in_stride % 4 == 0 && dout_stride % 4 == 0, "wgrad: row strides must be multiples of 4 elements");
  long long m = (long long)n_breaths * l_out;
  int splits = wgrad_splits(m, c_in, c_out, ktaps);
  long long need = (long long)splits * ktaps * c_in * c_out * (long long)sizeof(float);
  DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need, "wgrad: workspace too small (%lld < %lld)",
                  workspace_bytes, need);
  WgradArgs a;
  a.in = in;
  a.dout = dout;
  a.partial = static_cast<float*>(workspace);
  a.m_total = m;
  long long rps = (m + splits - 1) / splits;
  rps = (rps + WG_BK - 1) / WG_BK * WG_BK;
  a.rows_per_split = rps;
  a.l_in = l_in; a.l_out = l_out; a.c_in = c_in; a.c_out = c_out;
  a.in_stride = in_stride; a.dout_stride = dout_stride; a.ktaps = ktaps; a.stride = stride; a.pad = pad;
  dim3 grid(ceil_div(c_in, WG_BM) * ceil_div(c_out, WG_BN), ktaps, splits);
  DARDS_DISPATCH_DTYPE(dtype, { conv_wgrad_kernel<T><<<grid, WG_THREADS, 0, st>>>(a); })
  DARDS_CHECK_LAUNCH("conv_wgrad");
  int per = ktaps * c_in * c_out;
  int blocks = ceil_div(per, 256);
  wgrad_reduce_kernel<<<blocks, 256, 0, st>>>(a.partial, dw, splits, ktaps, c_in, c_out, accumulate);
  DARDS_CHECK_LAUNCH("wgrad_reduce");
  return DARDS_OK;
}

}  // namespace dards

// tcgen05 / TMEM / TMA implicit-GEMM Conv1d for sm_100a (bf16 operands, fp32 accumulation in TMEM).
//
// GEMM view (forward; dgrad is the same kernel with the roles of the channel dims swapped):
//     D[co, pos] = sum_{tap t} sum_{ci} W_t[co, ci] * X[pos shifted by t, ci]
//   A operand  = packed weights  w[t][co][ci]  -> 128(co) x 64(ci) K-major tile, SWIZZLE_128B
//   B operand  = channels-last activations     -> N_TILE(pos) x 64(ci) K-major tile, SWIZZLE_128B
//   accumulator D in TMEM: 128 lanes (output channels) x N_TILE fp32 columns (positions)
// The convolution is im2col-free: for each tap the SAME activation tensor is fetched by TMA with the
// position coordinate shifted by (t - pad); rows that fall outside [0, L) are zero-filled by the TMA
// unit, which is exactly the conv padding.  Stride-2 convolutions address the strided side through a 4-D
// view (C, 2, L/2, N) and pick the parity plane (forward: of the input; dgrad: of the output), so no strided
// gather/scatter is needed either.
// A position tile is NB whole breaths (NB*L = 224 columns for L = 56/28/14/7), so tiles never straddle a
// breath and there is no wasted MMA column.  (A wave-balanced width -- 36 x 7 = 18 x 14 = 252 columns issued as
// N = 256 MMAs, 572 tile jobs = 3.9 waves on 148 SMs instead of 640 = 4.3 -- is implemented behind debug key 8 and
// bit-identical, but measured SLOWER: 59.8 vs 50.2 us at C=512, 35.1 vs 31.8 at C=256.  The kernel is bound by the
// L2 -> SM operand stream, not by the per-CTA job count, and the wider tile lengthens every stage.)
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc/dealloc),
// warps 2..9 = epilogue: TMEM -> registers -> bf16 -> shared staging tile [pos][co] -> ONE TMA store
// (or TMA reduce-add when accumulating into the output) per tile; the TMA unit clips channels >= Cout and
// breaths >= N, so ragged edges need no branches.
// Pipelines: smem ring (full/empty mbarriers, TMA <-> MMA) and a 2-deep TMEM accumulator ring
// (tmem_full/tmem_empty, MMA <-> epilogue) so the epilogue of tile i overlaps the MMAs of tile i+1.
// The kernel is persistent: grid = min(#tiles, #SMs), static round-robin tile schedule.
#include "tc_common.cuh"

namespace dards {

int g_dbg_lbo = -1, g_dbg_version = -1, g_dbg_sbo = -1, g_dbg_base_offset_mode = -1, g_dbg_epilogue = -1, g_dbg_conv3 = -1, g_dbg_stages = -1, g_dbg_wgrad_fuse = -1, g_dbg_tile_balance = -1;
int g_dbg_l2_hint = -1;
extern int g_dbg_cb_pertap, g_dbg_cb_bstages, g_dbg_cb_wide, g_dbg_cb_share;
extern int g_dbg_bn_shift, g_dbg_bn_k;  // bn.cu
extern int g_dbg_wgrad_pair;             // wgrad_tc.cu
int g_dbg_pair = -1;         // debug key 17 = 0: wide layers stay on the single-CTA kernel instead of tc_conv_pair_kernel
int g_dbg_pair_stages = -1;  // debug key 18: its operand ring depth (default 6)
int g_dbg_shared = -1;   // debug key 10: 1 routes the wide (> 128 channel) k3/s1 layers through conv_bn_tc.cu's main loop, 2 all of them

// conv_bn_tc.cu: k3 / s1 / p1 convolution whose weight tiles are shared by two simultaneously accumulated position tiles
int tc_conv3_shared(const void* src, const void* wts, void* dst, int n_breaths, int l, int c_red, int c_cols, int src_stride,
                    int dst_stride, bool reverse_taps, bool accumulate, cudaStream_t st);
static bool shared_applicable(int l_in, int l_out, int c_red, int ktaps, int stride, int pad) {
  // opt-in: as fast as the one-load-per-tap kernel in isolation (profiles/r02_kbench_conv_shared.txt), slower inside the step
  return g_dbg_shared >= 1 && ktaps == 3 && stride == 1 && pad == 1 && l_in == l_out && (c_red > 128 || g_dbg_shared == 2);
}

constexpr int TC_EPI_WARPS = 8;
constexpr int TC_EPI_THREADS = TC_EPI_WARPS * 32;
constexpr int TC_THREADS = 64 + TC_EPI_THREADS;
constexpr int TC_MAX_STAGES = 4;
constexpr int TC_BLOCK_M = 128;          // output channels per tile (TMEM lanes)
constexpr int TC_BLOCK_K = 64;           // reduction channels per stage = one 128-byte swizzle row
constexpr int TC_MAX_N = 256;            // positions per tile (TMEM columns per accumulator)
constexpr int TC_A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;   // 16 KB
constexpr int TC_B_BYTES = TC_MAX_N * TC_BLOCK_K * 2;     // 32 KB
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int TC_STAGING_BYTES = TC_MAX_N * TC_BLOCK_M * 2;  // 64 KB: [pos][co] bf16
// shared memory: `stages` operand stages, then the staging tile (whole tile, or half of it when the epilogue stores
// the tile in two halves to make room for a 4th stage), alignment slack, barriers
static int tc_smem_bytes(int stages, int halves) {
  return stages * TC_STAGE_BYTES + TC_STAGING_BYTES / halves + 1024 + 256;
}
constexpr int TC_MAX_TAPS = 8;

struct TcConvParams {
  int n_taps;                 // taps issued by this launch
  int w_tap[TC_MAX_TAPS];     // tap coordinate in the weight map
  int in_par[TC_MAX_TAPS];    // parity-plane coordinate in the source activation map
  int in_start[TC_MAX_TAPS];  // first position coordinate in the source activation map (may be negative)
  int k_chunks;               // ceil(reduction channels / 64)
  int c_cols;                 // valid output channels
  int nb, l_tile;             // breaths per tile, positions per breath in the tile; N_TILE = nb*l_tile
  int n_breaths;
  int out_par;                // parity plane of the destination view written by this launch
  int out_l, out_mul, out_off;  // direct-store epilogue: output row = n*out_l + m*out_mul + out_off
  int out_stride;
  int accumulate;             // destination += result
  int tma_epilogue;           // 1: staging tile + TMA store; 0: direct global stores (debug fallback)
  int n_pos_tiles, n_co_tiles;
  int stages;                 // operand ring depth (3 or 4)
  int halves;                 // 1: one store per tile; 2: two stores of nb/2 breaths through a half-size staging tile
};

// Eval-mode BatchNorm in the forward epilogue (AFFINE = true instantiations): every epilogue thread owns one output
// channel, so scale / shift are two registers per tile.  The residual is read with plain loads straight from global
// memory while the accumulator chunk is in flight: in channels-last layout the 32 lanes of a warp read 64 contiguous
// bytes per position, and it keeps the staging tile and the TMA store path exactly as in the training kernels.
struct TcAffine {
  const float* scale;
  const float* shift;
  const __nv_bfloat16* res;  // nullable; (n_breaths, l, res_stride), never the output
  int res_stride, relu, n_breaths, l;
};

__device__ __forceinline__ void tc_affine_coeffs(const TcAffine& af, int co, int c_cols, float& sc, float& sh) {
  sc = co < c_cols ? af.scale[co] : 0.f;
  sh = co < c_cols ? af.shift[co] : 0.f;
}

// residual of 16 consecutive tile columns from column c0 on: column = b*lp + m (breath n0+b, position m, valid for m < l)
__device__ __forceinline__ void tc_res_ld16(const TcAffine& af, bool co_ok, int co, int n0, int lp, int c0, float (&r)[16]) {
  int b = c0 / lp, m = c0 - b * lp;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int n = n0 + b;
    r[j] = 0.f;
    if (af.res != nullptr && co_ok && n < af.n_breaths && m < af.l)
      r[j] = __bfloat162float(af.res[((size_t)n * af.l + m) * af.res_stride + co]);
    if (++m == lp) {
      m = 0;
      ++b;
    }
  }
}

__device__ __forceinline__ float tc_affine(float acc, float sc, float sh, float r, int relu) {
  const float y = fmaf(acc, sc, sh) + r;
  return relu ? fmaxf(y, 0.f) : y;
}

template <int HALVES, bool AFFINE>
__global__ void __launch_bounds__(TC_THREADS, 1)
    tc_conv_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                   const __grid_constant__ CUtensorMap tm_o, __nv_bfloat16* __restrict__ out, const TcConvParams p,
                   uint32_t desc_lbo16, uint32_t desc_sbo16, uint32_t desc_version, const TcAffine af) {
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int n_stages = p.stages;
  const uint32_t staging = smem_base + n_stages * TC_STAGE_BYTES;
  const uint32_t bar_base = staging + TC_STAGING_BYTES / HALVES;
  // barrier layout (8 bytes each): full[S], empty[S], tmem_full[2], tmem_empty[2], then the TMEM base word
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (TC_MAX_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * TC_MAX_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * TC_MAX_STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * TC_MAX_STAGES + 4);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));  // generic pointer to the aligned base
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tile = p.nb * p.l_tile;
  const int total_tiles = p.n_pos_tiles * p.n_co_tiles;
  const int k_steps = p.n_taps * p.k_chunks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_o);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), TC_EPI_WARPS);  // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);  // 2 accumulators x 256 columns
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================== TMA producer (whole warp, one elected lane issues: see elect_one) ===========
    {
      const bool issuer = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t stage_tx = TC_A_BYTES + (uint32_t)n_tile * (TC_BLOCK_K * 2);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int co_tile = tile % p.n_co_tiles, pos_tile = tile / p.n_co_tiles;
        const int co0 = co_tile * TC_BLOCK_M, n0 = pos_tile * p.nb;
        for (int ti = 0; ti < p.n_taps; ++ti) {
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait_tight(empty_bar(stage), phase ^ 1u);
            if (issuer) {
              const uint32_t sa = smem_base + stage * TC_STAGE_BYTES, sb = sa + TC_A_BYTES;
              mbar_arrive_expect_tx(full_bar(stage), stage_tx);
              tma_load_3d(sa, &tm_w, full_bar(stage), kc * TC_BLOCK_K, co0, p.w_tap[ti]);
              tma_load_4d(sb, &tm_x, full_bar(stage), kc * TC_BLOCK_K, p.in_par[ti], p.in_start[ti], n0);
            }
            if (++stage == n_stages) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    // A single warp issues everything and a dependent scalar instruction costs ~5 cycles, so the loop is kept to a
    // handful of instructions per MMA: 32-bit arithmetic on the descriptors' low words, tight waits, no per-stage
    // descriptor construction (profiles/r02_mma_issue_probe.txt: the tensor pipe itself sustains 98 % of its rate).
    {
      const bool issuer = elect_one();
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1,
      // A,B K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29)
      // N = the tile's columns rounded up to 16: accumulator column j depends on B row j only, so the surplus columns
      // (rows the TMA never wrote) cannot contaminate the real ones
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(((n_tile + 15) & ~15) >> 3) << 17) |
                             ((uint32_t)(TC_BLOCK_M >> 4) << 24);
      const uint64_t tmpl = make_sw128_desc(0, desc_lbo16, desc_sbo16, desc_version, 0);
      const uint32_t desc_hi = (uint32_t)(tmpl >> 32);
      const uint32_t a_lo0 = (uint32_t)tmpl + (smem_base >> 4);
      const uint32_t step = TC_STAGE_BYTES >> 4;
      int stage = 0;
      uint32_t phase = 0;
      uint32_t a_lo = a_lo0, fb = full_bar(0), eb = empty_bar(0);
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        mbar_wait_tight(tempty_bar(buf), acc_phase ^ 1u);  // epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)buf * TC_MAX_N;
        uint32_t acc = 0u;
        for (int ks = 0; ks < k_steps; ++ks) {
          mbar_wait_tight(fb, phase);
          tc_fence_after();
          if (issuer) {
            const uint32_t b_lo = a_lo + (TC_A_BYTES >> 4);
            // advance 16 bf16 = 32 bytes along K inside the 128-byte swizzle row: +2 in the (addr>>4) field
            umma_bf16_lo(d_tmem, a_lo, b_lo, desc_hi, idesc, acc);
            umma_bf16_lo(d_tmem, a_lo + 2, b_lo + 2, desc_hi, idesc, 1u);
            umma_bf16_lo(d_tmem, a_lo + 4, b_lo + 4, desc_hi, idesc, 1u);
            umma_bf16_lo(d_tmem, a_lo + 6, b_lo + 6, desc_hi, idesc, 1u);
            umma_commit(eb);  // frees the smem slot when these MMAs are done
          }
          acc = 1u;
          a_lo += step; fb += 8; eb += 8;
          if (++stage == n_stages) {
            stage = 0; phase ^= 1u; a_lo = a_lo0; fb = full_bar(0); eb = empty_bar(0);
          }
        }
        if (issuer) umma_commit(tfull_bar(buf));  // accumulator complete -> epilogue
      }
    }
  } else {
    // =========================== epilogue (warps 2..9) ===========================
    const int ew = warp - 2;
    const int quarter = warp & 3;  // a warp may only touch TMEM lanes [32*(warp%4), +32)
    const int half = ew >> 2;      // two warps per lane quarter: each takes half of the column chunks
    const int n_chunks = (n_tile + 15) >> 4;
    const int chunk_lo = half == 0 ? 0 : (n_chunks + 1) / 2;
    const int chunk_hi = half == 0 ? (n_chunks + 1) / 2 : n_chunks;
    const int cl = quarter * 32 + lane;  // channel within the tile
    const bool leader = (threadIdx.x == 64);
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      const int co_tile = tile % p.n_co_tiles, pos_tile = tile / p.n_co_tiles;
      const int co0 = co_tile * TC_BLOCK_M, n0 = pos_tile * p.nb;
      float a_sc = 0.f, a_sh = 0.f;
      if (AFFINE) tc_affine_coeffs(af, co0 + cl, p.c_cols, a_sc, a_sh);
      mbar_wait(tfull_bar(buf), acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)buf * TC_MAX_N;
      if (p.tma_epilogue) {
        __nv_bfloat16* stg = reinterpret_cast<__nv_bfloat16*>(smem_gen + (staging - smem_base));
        constexpr int n_halves = HALVES;
        const int cols_h = n_tile / n_halves;  // columns per store: nb/halves whole breaths
#pragma unroll
        for (int h = 0; h < n_halves; ++h) {
          // the previous TMA store must have finished reading the staging tile
          if (leader) tma_store_wait_read();
          named_bar_sync(1, TC_EPI_THREADS);
          const int col_lo = h * cols_h, col_hi = col_lo + cols_h;
          for (int ch = (col_lo >> 4) + half; (ch << 4) < col_hi; ch += 2) {
            uint32_t v[16];
            tmem_ld16(t_row + (uint32_t)(ch << 4), v);
            float r[16];
            if (AFFINE) tc_res_ld16(af, co0 + cl < p.c_cols, co0 + cl, n0, p.l_tile, ch << 4, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int col = (ch << 4) + j;
              float val = __uint_as_float(v[j]);
              if (AFFINE) val = tc_affine(val, a_sc, a_sh, r[j], af.relu);
              if (HALVES == 1 || (col >= col_lo && col < col_hi))  // a 16-column chunk may straddle the two halves
                stg[(col - col_lo) * TC_BLOCK_M + cl] = __float2bfloat16_rn(val);
            }
          }
          if (h == n_halves - 1) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(buf));  // TMEM buffer may be overwritten by the next-but-one tile
          }
          fence_proxy_async();
          named_bar_sync(1, TC_EPI_THREADS);
          if (leader) {
            const int nh = n0 + h * (p.nb / n_halves);
            if (p.accumulate) tma_reduce_add_4d(&tm_o, staging, co0, p.out_par, 0, nh);
            else tma_store_4d(&tm_o, staging, co0, p.out_par, 0, nh);
            tma_store_commit();
          }
        }
      } else {
        const int co = co0 + cl;
        const bool co_ok = co < p.c_cols;
        for (int ch = chunk_lo; ch < chunk_hi; ++ch) {
          const int c0 = ch << 4;
          uint32_t v[16];
          tmem_ld16(t_row + (uint32_t)c0, v);
          tmem_ld_wait();
          if (co_ok) {
            int b = c0 / p.l_tile, m = c0 % p.l_tile;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int n = n0 + b;
              if (n < p.n_breaths && c0 + j < n_tile) {
                const size_t idx = ((size_t)n * p.out_l + (size_t)m * p.out_mul + p.out_off) * p.out_stride + co;
                float val = __uint_as_float(v[j]);
                if (AFFINE)  // forward only: output row = n * l + m
                  val = tc_affine(val, a_sc, a_sh,
                                  af.res ? __bfloat162float(af.res[((size_t)n * af.l + m) * af.res_stride + co]) : 0.f,
                                  af.relu);
                if (p.accumulate) val += __bfloat162float(out[idx]);
                out[idx] = __float2bfloat16_rn(val);
              }
              if (++m == p.l_tile) {
                m = 0;
                ++b;
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(buf));
      }
    }
    if (p.tma_epilogue && leader) tma_store_wait_all();  // global writes complete before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ===================================================================================================
// CTA-pair variant of tc_conv_kernel<2> for the wide layers (>= 256 output channels): cta_group::2, M = 256.
// The per-tap kernel above re-fetches the activation tile for every tap and every output-channel tile, and at
// C >= 256 its operand stream (44 KB per 4 MMAs = 97 B/clk/SM) runs into the L2 -> SM limit (~12 TB/s, ncu:
// 478 MB per launch in 40 us) long before the tensor pipe is busy.  Here two CTAs of a cluster take the two
// output-channel tiles (2j, 2j+1) of the SAME position tile: each loads its own 128 x 64 weight tile and HALF of the
// activation tile (its nb/2 breaths), and the leader's tcgen05.mma.cta_group::2 reads both halves -- 30 KB per CTA
// per 4 MMAs instead of 44 KB, and a 32 KB stage leaves room for a 6-deep ring.  Each CTA's TMEM receives the 128
// accumulator lanes of its own channel tile, so the epilogue (two half-tile TMA stores) is unchanged.
// Protocol: full[s] lives in the LEADER (its producer expects the bytes of both CTAs; both CTAs' TMA loads signal it);
// empty[s] and tmem_full[b] live in both CTAs and are signalled by the leader's multicast commits; tmem_empty[b]
// lives in the leader and collects one arrive per epilogue warp of both CTAs.
// ===================================================================================================
constexpr int TP_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES / 2;  // 32 KB
constexpr int TP_MAX_STAGES = 6;
static int tp_smem_bytes(int stages) { return stages * TP_STAGE_BYTES + TC_STAGING_BYTES / 2 + 1024 + 256; }

template <bool AFFINE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
    tc_conv_pair_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                        const __grid_constant__ CUtensorMap tm_o, const TcConvParams p, uint32_t desc_lbo16,
                        uint32_t desc_sbo16, uint32_t desc_version, const TcAffine af) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int n_stages = p.stages;
  const uint32_t staging = smem_base + n_stages * TP_STAGE_BYTES;
  const uint32_t bar_base = staging + TC_STAGING_BYTES / 2;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (TP_MAX_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * TP_MAX_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * TP_MAX_STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * TP_MAX_STAGES + 4);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool lead = rank == 0;
  const int n_tile = p.nb * p.l_tile;
  const int n_co_pairs = p.n_co_tiles >> 1;
  const int total_jobs = p.n_pos_tiles * n_co_pairs;
  const int first_job = (int)(blockIdx.x >> 1), job_step = (int)(gridDim.x >> 1);
  const int k_steps = p.n_taps * p.k_chunks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_o);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 2 * TC_EPI_WARPS);  // one arrive per epilogue warp of BOTH CTAs (used in the leader only)
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_2sm(tmem_slot, 512);
    tmem_relinquish_2sm();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them remotely
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================== TMA producer (both CTAs) ===========================
    const bool issuer = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t stage_tx = TC_A_BYTES + (uint32_t)(n_tile >> 1) * (TC_BLOCK_K * 2);
    const int nb_half = p.nb >> 1;
    for (int job = first_job; job < total_jobs; job += job_step) {
      const int co_tile = 2 * (job % n_co_pairs) + (int)rank, pos_tile = job / n_co_pairs;
      const int co0 = co_tile * TC_BLOCK_M, n0 = pos_tile * p.nb + (int)rank * nb_half;
      for (int ti = 0; ti < p.n_taps; ++ti) {
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait_tight(empty_bar(stage), phase ^ 1u);
          if (issuer) {
            const uint32_t sa = smem_base + stage * TP_STAGE_BYTES, sb = sa + TC_A_BYTES;
            const uint32_t fb = full_bar(stage) & TC_PEER_MASK;  // the leader's barrier
            if (lead) mbar_arrive_expect_tx(full_bar(stage), 2u * stage_tx);
            tma_load_3d_2sm(sa, &tm_w, fb, kc * TC_BLOCK_K, co0, p.w_tap[ti]);
            tma_load_4d_2sm(sb, &tm_x, fb, kc * TC_BLOCK_K, p.in_par[ti], p.in_start[ti], n0);
          }
          if (++stage == n_stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (lead) {
      const bool issuer = elect_one();
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n_tile >> 3) << 17) |
                             ((uint32_t)((2 * TC_BLOCK_M) >> 4) << 24);
      const uint64_t tmpl = make_sw128_desc(0, desc_lbo16, desc_sbo16, desc_version, 0);
      const uint32_t desc_hi = (uint32_t)(tmpl >> 32);
      // the descriptor's 14-bit address field holds the CTA-relative address: drop the cluster-rank bits
      const uint32_t a_lo0 = (uint32_t)tmpl + ((smem_base & 0x3FFFFu) >> 4);
      const uint32_t step = TP_STAGE_BYTES >> 4;
      int stage = 0, it = 0;
      uint32_t phase = 0;
      uint32_t a_lo = a_lo0, fb = full_bar(0), eb = empty_bar(0);
      for (int job = first_job; job < total_jobs; job += job_step, ++it) {
        const int buf = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        mbar_wait_tight(tempty_bar(buf), acc_phase ^ 1u);  // both CTAs' epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)buf * TC_MAX_N;
        uint32_t acc = 0u;
        for (int ks = 0; ks < k_steps; ++ks) {
          mbar_wait_tight(fb, phase);
          tc_fence_after();
          if (issuer) {
            const uint32_t b_lo = a_lo + (TC_A_BYTES >> 4);
            umma2_bf16_lo(d_tmem, a_lo, b_lo, desc_hi, idesc, acc);
            umma2_bf16_lo(d_tmem, a_lo + 2, b_lo + 2, desc_hi, idesc, 1u);
            umma2_bf16_lo(d_tmem, a_lo + 4, b_lo + 4, desc_hi, idesc, 1u);
            umma2_bf16_lo(d_tmem, a_lo + 6, b_lo + 6, desc_hi, idesc, 1u);
            umma2_commit_mc(eb, 3u);  // frees the stage in both CTAs
          }
          acc = 1u;
          a_lo += step; fb += 8; eb += 8;
          if (++stage == n_stages) {
            stage = 0; phase ^= 1u; a_lo = a_lo0; fb = full_bar(0); eb = empty_bar(0);
          }
        }
        if (issuer) umma2_commit_mc(tfull_bar(buf), 3u);  // accumulators complete -> both epilogues
      }
    }
  } else {
    // =========================== epilogue (warps 2..9 of both CTAs): two half-tile TMA stores ===========
    const int ew = warp - 2;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    const int cl = quarter * 32 + lane;
    const bool leader = (threadIdx.x == 64);
    const int cols_h = n_tile >> 1;
    __nv_bfloat16* stg = reinterpret_cast<__nv_bfloat16*>(smem_gen + (staging - smem_base));
    int it = 0;
    for (int job = first_job; job < total_jobs; job += job_step, ++it) {
      const int buf = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      const int co_tile = 2 * (job % n_co_pairs) + (int)rank, pos_tile = job / n_co_pairs;
      const int co0 = co_tile * TC_BLOCK_M, n0 = pos_tile * p.nb;
      float a_sc = 0.f, a_sh = 0.f;
      if (AFFINE) tc_affine_coeffs(af, co0 + cl, p.c_cols, a_sc, a_sh);
      mbar_wait(tfull_bar(buf), acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)buf * TC_MAX_N;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (leader) tma_store_wait_read();
        named_bar_sync(1, TC_EPI_THREADS);
        const int col_lo = h * cols_h, col_hi = col_lo + cols_h;
        for (int ch = (col_lo >> 4) + half; (ch << 4) < col_hi; ch += 2) {
          uint32_t v[16];
          tmem_ld16(t_row + (uint32_t)(ch << 4), v);
          float r[16];
          if (AFFINE) tc_res_ld16(af, co0 + cl < p.c_cols, co0 + cl, n0, p.l_tile, ch << 4, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int col = (ch << 4) + j;
            float val = __uint_as_float(v[j]);
            if (AFFINE) val = tc_affine(val, a_sc, a_sh, r[j], af.relu);
            if (col >= col_lo && col < col_hi) stg[(col - col_lo) * TC_BLOCK_M + cl] = __float2bfloat16_rn(val);
          }
        }
        if (h == 1) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(tempty_bar(buf) & TC_PEER_MASK);
        }
        fence_proxy_async();
        named_bar_sync(1, TC_EPI_THREADS);
        if (leader) {
          const int nh = n0 + h * (p.nb >> 1);
          if (p.accumulate) tma_reduce_add_4d(&tm_o, staging, co0, p.out_par, 0, nh);
          else tma_store_4d(&tm_o, staging, co0, p.out_par, 0, nh);
          tma_store_commit();
        }
      }
    }
    if (leader) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA leaves while its partner may still signal its barriers or read its shared memory
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ===================================================================================================
// v3: 3-tap, stride-1, pad-1 convolutions (16 of ResNet-18's 20 convs, forward and dgrad) with ONE activation load
// for all three taps.
//
// The activation tile is staged WITH its halo: the TMA box is (64 ch, L+2 positions starting at -1, NB breaths), so
// breath b occupies staged rows b(L+2) .. b(L+2)+L+1 = positions -1 .. L, the out-of-range rows zero-filled by the
// TMA unit (= the conv padding).  Output column j = b(L+2) + q then needs staged row j + t for tap t: the SAME tile
// read through a shared-memory descriptor whose start is advanced by t rows (t * 128 B; the 128-byte swizzle is a
// function of the absolute shared-memory address, so a row-shifted start needs no other change).  Columns with
// q >= L straddle two breaths; they are computed and dropped (2 of every L+2 columns).
// Versus one load per tap this cuts the shared-memory fill per MMA from (A+B) to (A + B/3): an SS-mode tcgen05.mma
// already reads (M+N)*32 B per K=16 step, and TMA writes + MMA reads share the SM's 128 B/clk.
// Two rings: activation tiles (one per 64-channel chunk, 3 stages = up to 3 TILES of look-ahead on the narrow layers,
// which are load-latency bound) and weight tiles (one per chunk and tap, 3 stages).
// The epilogue is the wide kernel's: every accumulator column j goes to staging row j (the straddling columns too),
// then one TMA store per breath reads its L rows out of the staging tile.
constexpr int C3_B_STAGES = 3;
constexpr int C3_A_STAGES = 3;
constexpr int C3_EPI_WARPS = 8;
constexpr int C3_EPI_THREADS = C3_EPI_WARPS * 32;
constexpr int C3_THREADS = 64 + C3_EPI_THREADS;
constexpr int C3_MAX_ROWS = 258;                                       // staged rows read by the MMAs (N <= 256, + 2)
constexpr int C3_B_BYTES = ((C3_MAX_ROWS * 128 + 1023) / 1024) * 1024;  // 33 KB
constexpr int C3_STAGING_BYTES = 256 * 128 * 2;                        // one row per MMA column x 128 channels, bf16
constexpr int C3_SMEM_BYTES = C3_B_STAGES * C3_B_BYTES + C3_A_STAGES * TC_A_BYTES + C3_STAGING_BYTES + 1024 + 256;

struct TcConv3Params {
  int w_tap[3];   // weight tap used with a row shift of 0, 1, 2
  int k_chunks;   // ceil(reduction channels / 64)
  int nb, l;      // breaths per tile (even), positions per breath
  int n_cols;     // MMA N: nb*(l+2) - 2 rounded up to 16
  int n_pos_tiles, n_co_tiles;
  int accumulate;
  int src_evict_first;  // the activation tensor is read once by this launch and not again soon: L2 evict_first loads
  int c_cols;           // valid output channels (read by the affine epilogue)
};

template <bool AFFINE>
__global__ void __launch_bounds__(C3_THREADS, 1)
    tc_conv3_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                    const __grid_constant__ CUtensorMap tm_o, const TcConv3Params p, const TcAffine af) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_base = smem_base;
  const uint32_t a_base = b_base + C3_B_STAGES * C3_B_BYTES;
  const uint32_t staging = a_base + C3_A_STAGES * TC_A_BYTES;
  const uint32_t bar_base = staging + C3_STAGING_BYTES;
  auto fullb = [&](int s) { return bar_base + 8u * s; };
  auto emptyb = [&](int s) { return bar_base + 8u * (C3_B_STAGES + s); };
  auto fulla = [&](int s) { return bar_base + 8u * (2 * C3_B_STAGES + s); };
  auto emptya = [&](int s) { return bar_base + 8u * (2 * C3_B_STAGES + C3_A_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * C3_B_STAGES + 2 * C3_A_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * C3_B_STAGES + 2 * C3_A_STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * C3_B_STAGES + 2 * C3_A_STAGES + 4);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = p.n_pos_tiles * p.n_co_tiles;
  const int lp = p.l + 2;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_o);
    for (int s = 0; s < C3_B_STAGES; ++s) {
      mbar_init(fullb(s), 1);
      mbar_init(emptyb(s), 1);
    }
    for (int s = 0; s < C3_A_STAGES; ++s) {
      mbar_init(fulla(s), 1);
      mbar_init(emptya(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), C3_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // =========================== TMA producer (whole warp, one elected lane issues) ===========================
    {
      const bool issuer = elect_one();
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      const uint32_t b_tx = (uint32_t)(p.nb * lp) * 128u;
      const uint64_t pol_x = l2_policy(p.src_evict_first != 0);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int co0 = (tile % p.n_co_tiles) * TC_BLOCK_M, n0 = (tile / p.n_co_tiles) * p.nb;
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait_tight(emptyb(sb), phb ^ 1u);
          if (issuer) {
            mbar_arrive_expect_tx(fullb(sb), b_tx);
            tma_load_4d_pol(b_base + sb * C3_B_BYTES, &tm_x, fullb(sb), kc * TC_BLOCK_K, 0, -1, n0, pol_x);
          }
          if (++sb == C3_B_STAGES) {
            sb = 0;
            phb ^= 1u;
          }
          for (int t = 0; t < 3; ++t) {
            mbar_wait_tight(emptya(sa), pha ^ 1u);
            if (issuer) {
              mbar_arrive_expect_tx(fulla(sa), TC_A_BYTES);
              tma_load_3d(a_base + sa * TC_A_BYTES, &tm_w, fulla(sa), kc * TC_BLOCK_K, co0, p.w_tap[t]);
            }
            if (++sa == C3_A_STAGES) {
              sa = 0;
              pha ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    {
      const bool issuer = elect_one();
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.n_cols >> 3) << 17) |
                             ((uint32_t)(TC_BLOCK_M >> 4) << 24);
      const uint64_t tmpl = make_sw128_desc(0, 1, 1024 >> 4, 1, 0);
      const uint32_t desc_hi = (uint32_t)(tmpl >> 32);
      const uint32_t a_lo0 = (uint32_t)tmpl + (a_base >> 4), b_lo0 = (uint32_t)tmpl + (b_base >> 4);
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      uint32_t a_lo = a_lo0, b_lo = b_lo0, fa = fulla(0), ea = emptya(0), fb = fullb(0), eb = emptyb(0);
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        mbar_wait_tight(tempty_bar(buf), ((uint32_t)(it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)buf * TC_MAX_N;
        uint32_t acc = 0u;
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait_tight(fb, phb);
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            mbar_wait_tight(fa, pha);
            tc_fence_after();
            if (issuer) {
              // tap t: start advanced by t rows (128 B = 8 x 16 B); k: 16 bf16 = 32 B along the swizzle row
              const uint32_t bt = b_lo + (uint32_t)(8 * t);
              umma_bf16_lo(d_tmem, a_lo, bt, desc_hi, idesc, acc);
              umma_bf16_lo(d_tmem, a_lo + 2, bt + 2, desc_hi, idesc, 1u);
              umma_bf16_lo(d_tmem, a_lo + 4, bt + 4, desc_hi, idesc, 1u);
              umma_bf16_lo(d_tmem, a_lo + 6, bt + 6, desc_hi, idesc, 1u);
              umma_commit(ea);
              if (t == 2) umma_commit(eb);
            }
            acc = 1u;
            a_lo += TC_A_BYTES >> 4; fa += 8; ea += 8;
            if (++sa == C3_A_STAGES) {
              sa = 0; pha ^= 1u; a_lo = a_lo0; fa = fulla(0); ea = emptya(0);
            }
          }
          b_lo += C3_B_BYTES >> 4; fb += 8; eb += 8;
          if (++sb == C3_B_STAGES) {
            sb = 0; phb ^= 1u; b_lo = b_lo0; fb = fullb(0); eb = emptyb(0);
          }
        }
        if (issuer) umma_commit(tfull_bar(buf));
      }
    }
  } else {
    // =========================== epilogue (warps 2..9) ===========================
    const int ew = warp - 2;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, +32)
    const int sub = ew >> 2;       // the two warps of a quarter alternate over the column chunks
    const int cl = quarter * 32 + lane;
    const bool leader = (threadIdx.x == 64);
    const int n_chunks = p.n_cols >> 4;
    __nv_bfloat16* stg = reinterpret_cast<__nv_bfloat16*>(smem_gen + (staging - smem_base));
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const int co0 = (tile % p.n_co_tiles) * TC_BLOCK_M, n0 = (tile / p.n_co_tiles) * p.nb;
      float a_sc = 0.f, a_sh = 0.f;
      if (AFFINE) tc_affine_coeffs(af, co0 + cl, p.c_cols, a_sc, a_sh);
      mbar_wait(tfull_bar(buf), (uint32_t)(it >> 1) & 1u);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)buf * TC_MAX_N;
      if (leader) tma_store_wait_read();  // the previous tile's stores have finished reading the staging tile
      named_bar_sync(1, C3_EPI_THREADS);
      for (int ch = sub; ch < n_chunks; ch += 2) {
        uint32_t v[16];
        tmem_ld16(t_row + (uint32_t)(ch << 4), v);
        float r[16];
        if (AFFINE) tc_res_ld16(af, co0 + cl < p.c_cols, co0 + cl, n0, lp, ch << 4, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float val = __uint_as_float(v[j]);
          if (AFFINE) val = tc_affine(val, a_sc, a_sh, r[j], af.relu);
          stg[((ch << 4) + j) * TC_BLOCK_M + cl] = __float2bfloat16_rn(val);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(buf));  // TMEM buffer may be overwritten by the next-but-one tile
      fence_proxy_async();
      named_bar_sync(1, C3_EPI_THREADS);
      if (leader) {
        // breath b = staging rows [b*(L+2), b*(L+2) + L); the TMA unit clips channels >= Cout and breaths >= N
        for (int b = 0; b < p.nb; ++b) {
          const uint32_t src = staging + (uint32_t)(b * lp * TC_BLOCK_M * 2);
          if (p.accumulate) tma_reduce_add_4d(&tm_o, src, co0, 0, 0, n0 + b);
          else tma_store_4d(&tm_o, src, co0, 0, 0, n0 + b);
        }
        tma_store_commit();
      }
    }
    if (leader) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

static int make_map(CUtensorMap* m, CUtensorMapDataType dt, const void* base, int rank, const cuuint64_t* dims,
                    const cuuint64_t* strides_b, const cuuint32_t* box, bool swizzle128) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return DARDS_ERR_CUDA;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, dt, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_b, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d): rank %d dims [%llu %llu %llu %llu] box [%u %u %u %u]", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)dims[1], (unsigned long long)(rank > 2 ? dims[2] : 0),
              (unsigned long long)(rank > 3 ? dims[3] : 0), box[0], box[1], rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return DARDS_ERR_CUDA;
  }
  return DARDS_OK;
}

int make_bf16_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_b,
                  const cuuint32_t* box, bool swizzle128) {
  return make_map(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rank, dims, strides_b, box, swizzle128);
}

int make_f32_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_b,
                 const cuuint32_t* box, bool swizzle128) {
  return make_map(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, rank, dims, strides_b, box, swizzle128);
}

// SMs the persistent kernels size their grids for.  dards_set_sm_limit(n) (data-parallel runs) leaves a few SMs to the
// NCCL kernels that overlap the backward pass: a persistent kernel launched with one CTA per SM while NCCL holds some of
// them runs its last CTAs as a second wave.
static int g_sm_limit = 0;
int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return (g_sm_limit > 0 && g_sm_limit < n) ? g_sm_limit : n;
}
int set_sm_limit(int n) {
  g_sm_limit = n > 0 ? n : 0;
  return DARDS_OK;
}

// breaths per position tile: the largest nb with nb*l <= 256 and (nb*l) % 16 == 0
static int pick_nb(int l) {
  int best = 0;
  for (int nb = 1; nb * l <= TC_MAX_N && nb <= 256; ++nb)
    if ((nb * l) % 16 == 0) best = nb;
  return best;
}

// The same with the persistent schedule in mind: the kernel's makespan is (tile jobs per CTA) x (MMA columns per job).
// Tiles of at least half the widest width are compared (narrower ones re-fetch the weights too often); `want_even`
// keeps nb even where the long-reduction variant (4 stages, two half-tile stores) needs it.
static int pick_nb_balanced(int l, int n_breaths, int n_co_tiles, bool want_even) {
  const int widest = pick_nb(l);
  if (widest <= 0 || g_dbg_tile_balance != 1) return widest;  // opt-in: measured slower (see the header comment)
  const int sms = sm_count();
  auto cost = [&](int nb) {
    const long long jobs = (long long)ceil_div(n_breaths, nb) * n_co_tiles;
    return ((jobs + sms - 1) / sms) * (long long)((nb * l + 15) & ~15);
  };
  int best = widest;
  long long best_cost = cost(widest);
  for (int nb = (widest + 1) / 2; nb * l <= TC_MAX_N; ++nb) {
    if (want_even && (nb & 1)) continue;
    const long long c = cost(nb);
    if (c * 100 < best_cost * 96 || (nb > best && best != widest && c <= best_cost)) {  // >= 4 % better, or wider at par
      best = nb;
      best_cost = c;
    }
  }
  return best;
}

struct TcProblem {
  const void* src;     // activations read by the MMA (x for fwd, dout for dgrad)
  const void* w;       // packed weights [ktaps][c_cols][c_red]
  void* dst;
  int n_breaths;
  int l_src, src_planes;  // source length and number of parity planes of its view (forward stride)
  int l_dst, dst_planes;  // destination length and parity planes of its view (dgrad stride)
  int c_red, c_cols, src_stride, dst_stride, ktaps_total;
  TcConvParams p;
};

// dynamic shared memory opt-in, once per kernel and size
template <typename K>
static int tc_smem_optin(K kernel, int smem_bytes, int* granted, const char* what) {
  if (smem_bytes <= *granted) return DARDS_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
  if (e != cudaSuccess) {
    set_error("%s: cannot opt in to %d bytes of shared memory: %s", what, smem_bytes, cudaGetErrorString(e));
    return DARDS_ERR_CUDA;
  }
  *granted = smem_bytes;
  return DARDS_OK;
}

// af == nullptr: the training kernels; otherwise the eval-mode BatchNorm epilogue (AFFINE instantiations)
static int tc_launch(const TcProblem& q, cudaStream_t st, const TcAffine* af = nullptr) {
  DARDS_CHECK_ARG(q.c_red % 8 == 0 && q.src_stride % 8 == 0 && q.dst_stride % 8 == 0,
                  "tcgen05 conv: channels/strides must be multiples of 8");
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(q.src) & 15) == 0 && (reinterpret_cast<uintptr_t>(q.w) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(q.dst) & 15) == 0,
                  "tcgen05 conv: operands must be 16-byte aligned");
  DARDS_CHECK_ARG(q.l_src % q.src_planes == 0 && q.l_dst % q.dst_planes == 0,
                  "tcgen05 conv: length not divisible by the stride");
  if (q.n_breaths == 0) return DARDS_OK;
  TcConvParams p = q.p;
  const int n_tile = p.nb * p.l_tile;
  DARDS_CHECK_ARG(p.nb > 0 && n_tile <= TC_MAX_N && n_tile >= 8,
                  "tcgen05 conv: unsupported position tile (%d breaths x %d)", p.nb, p.l_tile);
  DARDS_CHECK_ARG(p.n_taps > 0, "tcgen05 conv: no taps");
  // Long reductions are LOAD-LATENCY bound with 3 stages (a stage is consumed in 448 cycles, a TMA load takes ~1 us:
  // measured 59 % tensor-pipe activity): give them a 4th stage, paid for by storing the tile in two halves through a
  // half-size staging buffer.  Short reductions are epilogue-bound and keep the one-store epilogue.
  const int k_steps_total = p.n_taps * ceil_div(q.c_red, TC_BLOCK_K);
  p.stages = 3;
  p.halves = 1;
  if (k_steps_total >= 12 && p.nb % 2 == 0 && (g_dbg_stages < 0 || g_dbg_stages == 4)) {
    p.stages = 4;
    p.halves = 2;
  }
  // CTA pairs (tc_conv_pair_kernel): long reductions with an even number of full output-channel tiles and a position tile
  // that splits into two halves of whole 8-row swizzle groups.  Measured (profiles/r02_kbench_conv_pair.txt): 43.9 vs
  // 48.5 us at C = 512, 27.4 vs 30.6 us at C = 256; debug key 17 = 0 keeps the single-CTA kernel.
  const bool pair = g_dbg_pair != 0 && p.halves == 2 && (g_dbg_epilogue < 0 || g_dbg_epilogue == 1) && q.c_cols % (2 * TC_BLOCK_M) == 0 && n_tile % 16 == 0 &&
                    (n_tile / 2) % 8 == 0 && q.c_red % TC_BLOCK_K == 0;
  CUtensorMap tm_w, tm_x, tm_o;
  {
    cuuint64_t dims[3] = {(cuuint64_t)q.c_red, (cuuint64_t)q.c_cols, (cuuint64_t)q.ktaps_total};
    cuuint64_t str[2] = {(cuuint64_t)q.c_red * 2, (cuuint64_t)q.c_red * q.c_cols * 2};
    cuuint32_t box[3] = {TC_BLOCK_K, TC_BLOCK_M, 1};
    int rc = make_bf16_map(&tm_w, q.w, 3, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const int planes = q.src_planes, l_plane = q.l_src / planes;
    cuuint64_t dims[4] = {(cuuint64_t)q.c_red, (cuuint64_t)planes, (cuuint64_t)l_plane, (cuuint64_t)q.n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)q.src_stride * 2, (cuuint64_t)q.src_stride * planes * 2,
                         (cuuint64_t)q.src_stride * q.l_src * 2};
    cuuint32_t box[4] = {TC_BLOCK_K, 1, (cuuint32_t)p.l_tile, (cuuint32_t)(pair ? p.nb / 2 : p.nb)};
    int rc = make_bf16_map(&tm_x, q.src, 4, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const int planes = q.dst_planes, l_plane = q.l_dst / planes;
    cuuint64_t dims[4] = {(cuuint64_t)q.c_cols, (cuuint64_t)planes, (cuuint64_t)l_plane, (cuuint64_t)q.n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)q.dst_stride * 2, (cuuint64_t)q.dst_stride * planes * 2,
                         (cuuint64_t)q.dst_stride * q.l_dst * 2};
    cuuint32_t box[4] = {TC_BLOCK_M, 1, (cuuint32_t)p.l_tile, (cuuint32_t)(p.nb / p.halves)};
    int rc = make_bf16_map(&tm_o, q.dst, 4, dims, str, box, false);
    if (rc) return rc;
  }
  p.k_chunks = ceil_div(q.c_red, TC_BLOCK_K);
  p.c_cols = q.c_cols;
  p.n_breaths = q.n_breaths;
  p.out_stride = q.dst_stride;
  p.out_l = q.l_dst;
  p.out_mul = q.dst_planes;
  p.out_off = p.out_par;
  p.tma_epilogue = g_dbg_epilogue >= 0 ? g_dbg_epilogue : 1;
  p.n_pos_tiles = ceil_div(q.n_breaths, p.nb);
  p.n_co_tiles = ceil_div(q.c_cols, TC_BLOCK_M);
  const int smem_bytes = tc_smem_bytes(p.stages, p.halves);
  const int tiles = p.n_pos_tiles * p.n_co_tiles;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  const uint32_t lbo = g_dbg_lbo >= 0 ? (uint32_t)g_dbg_lbo : 1u;
  const uint32_t sbo = g_dbg_sbo >= 0 ? (uint32_t)g_dbg_sbo : (1024u >> 4);
  const uint32_t ver = g_dbg_version >= 0 ? (uint32_t)g_dbg_version : 1u;
  const TcAffine a = af ? *af : TcAffine{};
  __nv_bfloat16* dst = static_cast<__nv_bfloat16*>(q.dst);
  if (pair) {
    p.stages = g_dbg_pair_stages > 0 && g_dbg_pair_stages <= TP_MAX_STAGES ? g_dbg_pair_stages : TP_MAX_STAGES;
    const int pair_smem = tp_smem_bytes(p.stages);
    static int pair_attr[2] = {0, 0};
    int rc = af ? tc_smem_optin(tc_conv_pair_kernel<true>, pair_smem, &pair_attr[1], "tcgen05 conv (CTA pairs)")
                : tc_smem_optin(tc_conv_pair_kernel<false>, pair_smem, &pair_attr[0], "tcgen05 conv (CTA pairs)");
    if (rc) return rc;
    // one cluster of two per TPC; clusters that do not become resident at once simply start when an earlier one ends (the
    // pairs of different clusters never wait for each other)
    int clusters = sm_count() / 2;
    if (clusters > tiles / 2) clusters = tiles / 2;
    if (af) tc_conv_pair_kernel<true><<<2 * clusters, TC_THREADS, pair_smem, st>>>(tm_w, tm_x, tm_o, p, lbo, sbo, ver, a);
    else tc_conv_pair_kernel<false><<<2 * clusters, TC_THREADS, pair_smem, st>>>(tm_w, tm_x, tm_o, p, lbo, sbo, ver, a);
    DARDS_CHECK_LAUNCH("tc_conv_pair");
    return DARDS_OK;
  }
  static int attr_smem[2][2] = {{0, 0}, {0, 0}};
  int* granted = &attr_smem[af ? 1 : 0][p.halves - 1];
  int rc;
  if (p.halves == 1) {
    rc = af ? tc_smem_optin(tc_conv_kernel<1, true>, smem_bytes, granted, "tcgen05 conv")
            : tc_smem_optin(tc_conv_kernel<1, false>, smem_bytes, granted, "tcgen05 conv");
    if (rc) return rc;
    if (af) tc_conv_kernel<1, true><<<grid, TC_THREADS, smem_bytes, st>>>(tm_w, tm_x, tm_o, dst, p, lbo, sbo, ver, a);
    else tc_conv_kernel<1, false><<<grid, TC_THREADS, smem_bytes, st>>>(tm_w, tm_x, tm_o, dst, p, lbo, sbo, ver, a);
  } else {
    rc = af ? tc_smem_optin(tc_conv_kernel<2, true>, smem_bytes, granted, "tcgen05 conv")
            : tc_smem_optin(tc_conv_kernel<2, false>, smem_bytes, granted, "tcgen05 conv");
    if (rc) return rc;
    if (af) tc_conv_kernel<2, true><<<grid, TC_THREADS, smem_bytes, st>>>(tm_w, tm_x, tm_o, dst, p, lbo, sbo, ver, a);
    else tc_conv_kernel<2, false><<<grid, TC_THREADS, smem_bytes, st>>>(tm_w, tm_x, tm_o, dst, p, lbo, sbo, ver, a);
  }
  DARDS_CHECK_LAUNCH("tc_conv");
  return DARDS_OK;
}

// v3 launch for k=3, s=1, p=1 (see tc_conv3_kernel).  `reverse_taps`: dgrad (tap s uses weight tap 2-s).
// Measured (profiles/r01_kbench_conv.txt): 21.6 vs 23.5 us at C = 64 and 22.4 vs 24.7 us at C = 128 -- the narrow layers
// are load-latency bound and gain from 3 tiles of look-ahead; at C >= 256 the one-load-per-tap kernel with its 4-stage
// ring is faster (no straddling columns: 32.0 vs 33.7 us, 50.8 vs 54.0 us).  dards_tc_debug_set(5, 0 | 1) forces it off | on.
static bool tc3_applicable(int l, int c_red, int ktaps, int stride, int pad) {
  if (g_dbg_conv3 == 0) return false;
  if (!(ktaps == 3 && stride == 1 && pad == 1 && l + 2 <= C3_MAX_ROWS && l >= 2)) return false;
  return g_dbg_conv3 == 1 || c_red <= 128;
}

static int tc3_launch(const void* src, const void* w, void* dst, int n_breaths, int l, int c_red, int c_cols,
                      int src_stride, int dst_stride, bool reverse_taps, bool accumulate, int src_last_use,
                      cudaStream_t st, const TcAffine* af = nullptr) {
  DARDS_CHECK_ARG(c_red % 8 == 0 && src_stride % 8 == 0 && dst_stride % 8 == 0,
                  "tcgen05 conv: channels/strides must be multiples of 8");
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
                  "tcgen05 conv: operands must be 16-byte aligned");
  if (n_breaths == 0) return DARDS_OK;
  TcConv3Params p{};
  const int nb = C3_MAX_ROWS / (l + 2);
  DARDS_CHECK_ARG(nb >= 1, "tcgen05 conv v3: sequence length %d too long for one tile", l);
  p.nb = nb;
  p.l = l;
  p.n_cols = ((nb * (l + 2) - 2 + 15) / 16) * 16;
  p.k_chunks = ceil_div(c_red, TC_BLOCK_K);
  p.n_pos_tiles = ceil_div(n_breaths, nb);
  p.n_co_tiles = ceil_div(c_cols, TC_BLOCK_M);
  p.c_cols = c_cols;
  p.accumulate = accumulate ? 1 : 0;
  // every activation byte is fetched once only when there is a single output-channel tile
  p.src_evict_first = (src_last_use && p.n_co_tiles == 1 && g_dbg_l2_hint != 0) ? 1 : 0;
  for (int t = 0; t < 3; ++t) p.w_tap[t] = reverse_taps ? 2 - t : t;
  CUtensorMap tm_w, tm_x, tm_o;
  {
    cuuint64_t dims[3] = {(cuuint64_t)c_red, (cuuint64_t)c_cols, 3};
    cuuint64_t str[2] = {(cuuint64_t)c_red * 2, (cuuint64_t)c_red * c_cols * 2};
    cuuint32_t box[3] = {TC_BLOCK_K, TC_BLOCK_M, 1};
    int rc = make_bf16_map(&tm_w, w, 3, dims, str, box, true);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)c_red, 1, (cuuint64_t)l, (cuuint64_t)n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)src_stride * 2, (cuuint64_t)src_stride * 2, (cuuint64_t)src_stride * l * 2};
    cuuint32_t box[4] = {TC_BLOCK_K, 1, (cuuint32_t)(l + 2), (cuuint32_t)nb};
    int rc = make_bf16_map(&tm_x, src, 4, dims, str, box, true);
    if (rc) return rc;
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)c_cols, 1, (cuuint64_t)l, (cuuint64_t)n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)dst_stride * 2, (cuuint64_t)dst_stride * 2, (cuuint64_t)dst_stride * l * 2};
    cuuint32_t box[4] = {TC_BLOCK_M, 1, (cuuint32_t)l, 1};
    int rc = make_bf16_map(&tm_o, dst, 4, dims, str, box, false);
    if (rc) return rc;
  }
  static int attr_set[2] = {0, 0};
  const int rc = af ? tc_smem_optin(tc_conv3_kernel<true>, C3_SMEM_BYTES, &attr_set[1], "tcgen05 conv v3")
                    : tc_smem_optin(tc_conv3_kernel<false>, C3_SMEM_BYTES, &attr_set[0], "tcgen05 conv v3");
  if (rc) return rc;
  const int tiles = p.n_pos_tiles * p.n_co_tiles;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  const TcAffine a = af ? *af : TcAffine{};
  if (af) tc_conv3_kernel<true><<<grid, C3_THREADS, C3_SMEM_BYTES, st>>>(tm_w, tm_x, tm_o, p, a);
  else tc_conv3_kernel<false><<<grid, C3_THREADS, C3_SMEM_BYTES, st>>>(tm_w, tm_x, tm_o, p, a);
  DARDS_CHECK_LAUNCH("tc_conv3");
  return DARDS_OK;
}

// forward; af != nullptr: eval-mode BatchNorm (+ residual, + ReLU) in the epilogue, through the same kernel selection
static int tc_conv_fwd_sel(const void* in, const void* w_koi, void* out, const void* addend, int n_breaths, int l_in,
                           int l_out, int c_in, int c_out, int in_stride, int out_stride, int addend_stride, int ktaps,
                           int stride, int pad, int src_last_use, cudaStream_t st, const TcAffine* af) {
  DARDS_CHECK_ARG(stride == 1 || stride == 2, "tcgen05 conv: stride must be 1 or 2");
  DARDS_CHECK_ARG(ktaps <= TC_MAX_TAPS, "tcgen05 conv: at most %d taps", TC_MAX_TAPS);
  if (addend != nullptr && (addend != out || addend_stride != out_stride)) {
    set_error("tcgen05 conv: the addend must be the output itself (in-place accumulation)");
    return DARDS_ERR_UNSUPPORTED;
  }
  if (af == nullptr && shared_applicable(l_in, l_out, c_in, ktaps, stride, pad)) {
    const int rc = tc_conv3_shared(in, w_koi, out, n_breaths, l_in, c_in, c_out, in_stride, out_stride, false, addend != nullptr, st);
    if (rc != DARDS_ERR_UNSUPPORTED) return rc;
  }
  if (tc3_applicable(l_in, c_in, ktaps, stride, pad) && l_in == l_out)
    return tc3_launch(in, w_koi, out, n_breaths, l_in, c_in, c_out, in_stride, out_stride, false, addend != nullptr,
                      src_last_use, st, af);
  TcProblem q{};
  q.src = in; q.w = w_koi; q.dst = out;
  q.n_breaths = n_breaths; q.l_src = l_in; q.src_planes = stride; q.l_dst = l_out; q.dst_planes = 1;
  q.c_red = c_in; q.c_cols = c_out; q.src_stride = in_stride; q.dst_stride = out_stride;
  q.ktaps_total = ktaps;
  TcConvParams& p = q.p;
  p.n_taps = ktaps;
  for (int t = 0; t < ktaps; ++t) {
    // source position = q*stride + (t - pad) = stride*(q + floor((t-pad)/stride)) + ((t-pad) mod stride)
    const int d = t - pad;
    const int fl = d >= 0 ? d / stride : -((-d + stride - 1) / stride);
    p.w_tap[t] = t;
    p.in_par[t] = d - fl * stride;
    p.in_start[t] = fl;
  }
  p.l_tile = l_out;
  p.nb = pick_nb_balanced(l_out, n_breaths, ceil_div(c_out, TC_BLOCK_M), p.n_taps * ceil_div(c_in, TC_BLOCK_K) >= 12);
  p.out_par = 0;
  p.accumulate = addend != nullptr;
  return tc_launch(q, st, af);
}

int tc_conv_fwd(const void* in, const void* w_koi, void* out, const void* addend, int n_breaths, int l_in, int l_out,
                int c_in, int c_out, int in_stride, int out_stride, int addend_stride, int ktaps, int stride, int pad,
                int src_last_use, cudaStream_t st) {
  return tc_conv_fwd_sel(in, w_koi, out, addend, n_breaths, l_in, l_out, c_in, c_out, in_stride, out_stride, addend_stride,
                         ktaps, stride, pad, src_last_use, st, nullptr);
}

int tc_conv_affine_fwd(const void* in, const void* w_koi, void* out, const void* res, const float* scale, const float* shift,
                       int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride, int out_stride, int res_stride,
                       int ktaps, int stride, int pad, int relu, int src_last_use, cudaStream_t st) {
  const TcAffine af = {scale, shift, static_cast<const __nv_bfloat16*>(res), res_stride, relu, n_breaths, l_out};
  return tc_conv_fwd_sel(in, w_koi, out, nullptr, n_breaths, l_in, l_out, c_in, c_out, in_stride, out_stride, 0, ktaps,
                         stride, pad, src_last_use, st, &af);
}

int tc_conv_dgrad(const void* dout, const void* w_kio, void* din, const void* addend, int n_breaths, int l_in, int l_out,
                  int c_in, int c_out, int dout_stride, int din_stride, int addend_stride, int ktaps, int stride, int pad,
                  int src_last_use, cudaStream_t st) {
  DARDS_CHECK_ARG(stride == 1 || stride == 2, "tcgen05 conv: stride must be 1 or 2");
  DARDS_CHECK_ARG(ktaps <= TC_MAX_TAPS, "tcgen05 conv: at most %d taps", TC_MAX_TAPS);
  DARDS_CHECK_ARG(l_in % stride == 0 && l_in / stride == l_out, "tcgen05 dgrad: needs l_in == stride * l_out");
  if (addend != nullptr && (addend != din || addend_stride != din_stride)) {
    set_error("tcgen05 dgrad: the addend must be the output itself (in-place accumulation)");
    return DARDS_ERR_UNSUPPORTED;
  }
  if (shared_applicable(l_in, l_out, c_out, ktaps, stride, pad)) {
    const int rc = tc_conv3_shared(dout, w_kio, din, n_breaths, l_in, c_out, c_in, dout_stride, din_stride, true, addend != nullptr, st);
    if (rc != DARDS_ERR_UNSUPPORTED) return rc;
  }
  if (tc3_applicable(l_in, c_out, ktaps, stride, pad))
    return tc3_launch(dout, w_kio, din, n_breaths, l_in, c_out, c_in, dout_stride, din_stride, true, addend != nullptr,
                      src_last_use, st);
  // din[p = stride*m + r] = sum over taps t with (r + pad - t) % stride == 0 of dout[m + (r+pad-t)/stride] * W_t:
  // one launch per output parity plane r; reduction over c_out.
  for (int r = 0; r < stride; ++r) {
    TcProblem q{};
    q.src = dout; q.w = w_kio; q.dst = din;
    q.n_breaths = n_breaths; q.l_src = l_out; q.src_planes = 1; q.l_dst = l_in; q.dst_planes = stride;
    q.c_red = c_out; q.c_cols = c_in; q.src_stride = dout_stride; q.dst_stride = din_stride;
    q.ktaps_total = ktaps;
    TcConvParams& p = q.p;
    p.n_taps = 0;
    for (int t = 0; t < ktaps; ++t) {
      const int d = r + pad - t;
      if (((d % stride) + stride) % stride != 0) continue;
      p.w_tap[p.n_taps] = t;
      p.in_par[p.n_taps] = 0;
      p.in_start[p.n_taps] = d >= 0 ? d / stride : -((-d) / stride);
      ++p.n_taps;
    }
    p.l_tile = l_in / stride;
    p.nb = pick_nb_balanced(p.l_tile, n_breaths, ceil_div(c_in, TC_BLOCK_M), p.n_taps * ceil_div(c_out, TC_BLOCK_K) >= 12);
    p.out_par = r;
    p.accumulate = addend != nullptr;
    if (p.n_taps == 0) {
      if (p.accumulate) continue;  // nothing to add on this parity plane
      set_error("tcgen05 dgrad: output plane %d receives no tap; call with in-place accumulation", r);
      return DARDS_ERR_UNSUPPORTED;
    }
    int rc = tc_launch(q, st);
    if (rc) return rc;
  }
  return DARDS_OK;
}

int tc_debug_set(int key, int value) {
  if (key == 0) g_dbg_lbo = value;
  else if (key == 1) g_dbg_version = value;
  else if (key == 2) g_dbg_sbo = value;
  else if (key == 3) g_dbg_base_offset_mode = value;
  else if (key == 4) g_dbg_epilogue = value;
  else if (key == 5) g_dbg_conv3 = value;
  else if (key == 6) g_dbg_stages = value;
  else if (key == 7) g_dbg_wgrad_fuse = value;
  else if (key == 8) g_dbg_tile_balance = value;
  else if (key == 9) g_dbg_l2_hint = value;
  else if (key == 10) g_dbg_shared = value;
  else if (key == 11) g_dbg_cb_pertap = value;
  else if (key == 12) g_dbg_cb_bstages = value;
  else if (key == 13) g_dbg_cb_wide = value;
  else if (key == 14) g_dbg_cb_share = value;
  else if (key == 15) g_dbg_bn_shift = value;
  else if (key == 16) g_dbg_bn_k = value;
  else if (key == 17) g_dbg_pair = value;
  else if (key == 18) g_dbg_pair_stages = value;
  else if (key == 19) g_dbg_wgrad_pair = value;
  else {
    set_error("tc_debug_set: unknown key %d", key);
    return DARDS_ERR_INVALID_ARGUMENT;
  }
  return DARDS_OK;
}

}  // namespace dards

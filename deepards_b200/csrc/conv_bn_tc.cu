// Conv1d + grouped BatchNorm1d (+ residual) (+ ReLU) in ONE tcgen05 kernel (bf16 operands, fp32 accumulation in TMEM).
//
// Replaces conv -> bn -> relu [-> += residual -> relu] of resnet.py:27-38 and conv -> norm -> relu of
// densenet.py:25-29 without the separate BatchNorm pass over the convolution output.  The same main loop with a plain
// store epilogue serves the wide (C >= 256) data-gradient convolutions.
//
// The BatchNorm statistics of a channel are sums over ALL positions of a group (= one sequence of `group` breaths),
// so the unit of work is a JOB = (whole groups, tile of 128 output channels), never a tile that straddles two groups:
//   * an epilogue thread owns ONE output channel (its TMEM lane) and sees every position of the job's accumulators:
//     sum(y) and sum(y^2) are in-thread sums over the tcgen05.ld values, taken from the fp32 accumulators (shifted by
//     a sample of the data, so E[d^2] - E[d]^2 loses no digits), before the rounding to bf16;
//   * FUSED (a group is at most three position tiles: 20 breaths x L <= 14 positions, ResNet-18 layers 3-4 / DenseNet
//     blocks 3-4): the job's accumulators are drained straight to y in global memory (bf16; the backward needs it),
//     the two epilogue threads of a channel merge their moments (Chan's formula), mean / rstd / gamma / beta become one
//     scale and shift per channel, and a second sweep re-reads the job's y -- 70 KB that this CTA has just written, an
//     L2 hit -- row-wise and writes out = relu(y * scale + shift + res) with 16-byte coalesced accesses.  No
//     BatchNorm launch, y is never re-read from HBM.  Nothing is staged in shared memory: every byte of it belongs to
//     the operand rings (the kernel is bound by the bytes it can keep in flight, see below);
//   * PARTIAL (long sequences, L >= 28: the group is several tiles of different CTAs): every tile writes its
//     (count, mean, M2) per channel; gbn_apply_fwd (bn_apply.cu) merges them in a fixed order and does the elementwise
//     normalisation in one streaming pass;
//   * PLAIN: y only (optionally accumulated into the destination with a TMA reduce-add): data gradients.
// Deterministic: no atomics, every merge has a fixed order.
//
// Main loop (A = packed weights w[t][co][ci] 128 x 64 K-major SWIZZLE_128B, B = channels-last activations, rows =
// positions, accumulator = 128 channel lanes x N position columns).  Two things keep the L2 -> SM operand stream, which
// bounds the plain wide-layer kernel (conv_tc.cu), small:
//   * the job's `nsub` sub-tiles (position tiles of nb breaths) are accumulated SIMULTANEOUSLY in nsub TMEM buffers, so
//     every weight tile is fetched once per job and feeds 4 * nsub MMAs;
//   * mode3 (k = 3, stride 1, pad 1): the activation tile is staged once per 64-channel chunk with ONE zero row
//     between consecutive breaths (TMA box (64 ch, L + 1 positions from -1, nb breaths): the out-of-range row is
//     zero-filled = the padding of both neighbours; the row after the last breath is zeroed once by the kernel) and the
//     three taps read it through descriptors advanced by 0 / 1 / 2 rows.  Column q = L of a breath sits on the zero row:
//     computed and dropped (1 of every L + 1 columns).
//   Per-tap loads (stride 2, 1x1) take the tap shift / parity plane in the TMA coordinates instead.
// The TMEM ring has 512 / n_cols buffers (3 for the 160-column tiles of L = 7 / 14).
// Measured (profiles/r02_kbench_*): with an 80 KB output staging tile in shared memory this loop ran at 45 % of the MMA
// rate although it moves half the L2 bytes of conv_tc.cu -- ~130 KB of operand buffers in flight at ~1.4 us effective TMA
// latency cap the SM at ~33 B/clk.  Hence direct stores and 8 weight stages.
#include "tc_common.cuh"

namespace dards {

constexpr int CB_EPI_WARPS = 8;
constexpr int CB_EPI_THREADS = CB_EPI_WARPS * 32;
constexpr int CB_THREADS = 64 + CB_EPI_THREADS;
// FUSED: 8 more warps do the normalisation sweep of job j while the drain warps are on job j + 1
constexpr int CB_THREADS_FUSED = CB_THREADS + CB_EPI_THREADS;
constexpr int CB_MAX_A = 8, CB_MAX_B = 8;
constexpr int CB_A_BYTES = 128 * 64 * 2;   // 16 KB weight tile
constexpr int CB_MAX_TAPS = 8;
constexpr int CB_MAX_COLS = 256;
constexpr int CB_MAX_SUB = 2;
constexpr int CB_MAX_GPJ = 2;              // groups per job
// tail of the shared memory: barriers + TMEM slot (512 B) | moments [2 jobs][2 groups][2 halves][4][128] (16 KB) |
// scale/shift [2 jobs][2 groups][2][128] (4 KB) | column -> element offset table [256] u32 (1 KB) |
// per-drain-warp transpose scratch [8 warps][16 columns][32 channels] bf16 (8 KB)
constexpr int CB_OFF_MOM = 512, CB_OFF_SCSH = CB_OFF_MOM + 16384, CB_OFF_CROW = CB_OFF_SCSH + 4096,
              CB_OFF_TR = CB_OFF_CROW + 1024, CB_TAIL_BYTES = CB_OFF_TR + 8192;
// named barriers: 2 + par "job's y and moments are ready" (drain warps arrive, apply warps wait), 4 + par "moments consumed"
// (apply warps arrive, drain warps wait before reusing the slot two jobs later), 6 apply-warp internal
constexpr int CB_SMEM_LIMIT = 227 * 1024;

enum { CB_PARTIAL = 0, CB_FUSED = 1, CB_PLAIN = 2 };
int g_dbg_cb_pertap = -1;   // debug key 11 = 1: k3/s1 convolutions with BatchNorm use one activation load per tap
int g_dbg_cb_bstages = -1;  // debug key 12: activation-ring depth of the mode3 loop (default 2 chunks)
int g_dbg_cb_wide = -1;     // debug key 13 = 1: plain convolutions use one 256-column tile per job instead of two 160-column ones
int g_dbg_cb_share = -1;    // debug key 14 = 1: the job's two sub-tiles are accumulated simultaneously (weight tiles fetched once)

struct CbParams {
  int mode3;
  int n_taps;
  int w_tap[CB_MAX_TAPS], in_par[CB_MAX_TAPS], in_start[CB_MAX_TAPS];
  int k_chunks;
  int nb, l, lp;        // breaths per sub-tile, valid positions per breath, staged rows per breath (l + 1 | l)
  int n_cols;           // MMA N (multiple of 16)
  int nsub;             // sub-tiles per job, accumulated simultaneously
  int spg;              // sub-tiles per BatchNorm group
  int n_bufs;           // TMEM accumulator ring
  int n_pos_jobs, n_co_tiles;
  int a_stages, b_stages, b_bytes;
  int nshare;           // sub-tiles accumulated simultaneously (1: one after the other)
  int c_out;
  int epi, relu, accumulate;
  int x_evict_first;
  float eps;
  const float* gamma;
  const float* beta;
  float* save_mean;
  float* save_rstd;
  float* part;          // PARTIAL: [pos job][2][3][c_out]
  __nv_bfloat16* y;      // convolution output (N, l, c_out) rows of y_stride elements; y_l = its full length,
  int y_stride, y_l;     // y_mul / y_off place position q at row q*y_mul + y_off (stride-2 data gradients)
  int y_mul, y_off;
  __nv_bfloat16* out;
  const __nv_bfloat16* res;
  int out_stride, res_stride;
};

__device__ __forceinline__ void unpack8(const uint4& r, float (&v)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(h[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  uint4 r;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  return r;
}

__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t threads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

template <int EPI, bool ACC, bool MODE3, int NSH>
__global__ void __launch_bounds__(EPI == CB_FUSED ? CB_THREADS_FUSED : CB_THREADS, 1)
    tc_conv_bn_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x,
                      const CbParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_base = smem_base;
  const uint32_t a_base = b_base + p.b_stages * p.b_bytes;
  const uint32_t bar_base = a_base + p.a_stages * CB_A_BYTES;
  auto fullb = [&](int s) { return bar_base + 8u * s; };
  auto emptyb = [&](int s) { return bar_base + 8u * (CB_MAX_B + s); };
  auto fulla = [&](int s) { return bar_base + 8u * (2 * CB_MAX_B + s); };
  auto emptya = [&](int s) { return bar_base + 8u * (2 * CB_MAX_B + CB_MAX_A + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * CB_MAX_B + 2 * CB_MAX_A + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * CB_MAX_B + 2 * CB_MAX_A + 4 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * CB_MAX_B + 2 * CB_MAX_A + 8);
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  uint8_t* tail = smem_gen + (bar_base - smem_base);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(tail + 8 * (2 * CB_MAX_B + 2 * CB_MAX_A + 8));
  float* mom = reinterpret_cast<float*>(tail + CB_OFF_MOM);      // [group][half][cnt, s, ss, shift][128]
  float* scsh = reinterpret_cast<float*>(tail + CB_OFF_SCSH);    // [group][scale, shift][128]
  // [n_cols]: accumulator column (breath b, position q) -> element offset (b*y_l + q*y_mul) * y_stride into y, ~0 for
  // the junk columns (32-bit: a tile spans at most 256 rows of at most a few thousand elements)
  uint32_t* crow = reinterpret_cast<uint32_t*>(tail + CB_OFF_CROW);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_jobs = p.n_pos_jobs * p.n_co_tiles;
  const int job_breaths = p.nb * p.nsub;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x);
    for (int s = 0; s < p.b_stages; ++s) {
      mbar_init(fullb(s), 1);
      mbar_init(emptyb(s), 1);
    }
    for (int s = 0; s < p.a_stages; ++s) {
      mbar_init(fulla(s), 1);
      mbar_init(emptya(s), 1);
    }
    for (int b = 0; b < p.n_bufs; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), CB_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (p.mode3) {
    // the zero row after the last breath of every activation stage (TMA never writes it)
    for (int i = threadIdx.x; i < p.b_stages * 8; i += blockDim.x) {
      uint4* row = reinterpret_cast<uint4*>(smem_gen + (b_base - smem_base) + (i >> 3) * p.b_bytes + p.nb * p.lp * 128);
      row[i & 7] = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_proxy_async();
  }
  if (warp >= 2 && warp < 10) {
    // accumulator column -> output row within the sub-tile, the same for every job
    const int et = threadIdx.x - 64;
    for (int c = et; c < CB_MAX_COLS; c += CB_EPI_THREADS) {
      const int b = c / p.lp, q = c - b * p.lp;
      crow[c] = (c < p.n_cols && q < p.l && b < p.nb) ? (uint32_t)(b * p.y_l + q * p.y_mul) * (uint32_t)p.y_stride : 0xFFFFFFFFu;
    }
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
      const uint32_t b_tx = (uint32_t)(p.nb * p.lp) * 128u;
      const uint64_t pol_x = l2_policy(p.x_evict_first != 0);
      auto load_b = [&](int kc, int par, int start, int n0) {
        mbar_wait(emptyb(sb), phb ^ 1u);
        if (issuer) {
          mbar_arrive_expect_tx(fullb(sb), b_tx);
          tma_load_4d_pol(b_base + sb * p.b_bytes, &tm_x, fullb(sb), kc * 64, par, start, n0, pol_x);
        }
        __syncwarp();
        if (++sb == p.b_stages) {
          sb = 0;
          phb ^= 1u;
        }
      };
      for (int job = blockIdx.x; job < total_jobs; job += gridDim.x) {
        const int co0 = (job % p.n_co_tiles) * 128;
        // the job's sub-tiles, NSH at a time
        for (int sg = 0; sg < p.nsub; sg += NSH) {
        const int nj = (job / p.n_co_tiles) * job_breaths + sg * p.nb;
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          if (MODE3) {
#pragma unroll
            for (int sub = 0; sub < NSH; ++sub) load_b(kc, 0, -1, nj + sub * p.nb);
          }
          for (int t = 0; t < p.n_taps; ++t) {
            mbar_wait(emptya(sa), pha ^ 1u);
            if (issuer) {
              mbar_arrive_expect_tx(fulla(sa), CB_A_BYTES);
              tma_load_3d(a_base + sa * CB_A_BYTES, &tm_w, fulla(sa), kc * 64, co0, p.w_tap[t]);
            }
            __syncwarp();
            if (++sa == p.a_stages) {
              sa = 0;
              pha ^= 1u;
            }
            if (!MODE3) {
#pragma unroll
              for (int sub = 0; sub < NSH; ++sub) load_b(kc, p.in_par[t], p.in_start[t], nj + sub * p.nb);
            }
          }
        }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer (whole warp, one elected lane issues) ===========================
    // The loop is the kernel's critical path: a single warp issues everything, and at ~5 cycles per dependent scalar
    // instruction anything but a handful of instructions per MMA shows up as idle tensor cycles (measured: ~80
    // instructions per group of four 80-cycle MMAs -> 43 % tensor-pipe activity).  So: mode and sub-tile count are
    // compile-time, every parameter is hoisted, descriptor arithmetic is 32-bit on the low word.
    {
      const bool issuer = elect_one();
      const int n_cols = p.n_cols, n_bufs = p.n_bufs, k_chunks = p.k_chunks, n_taps = p.n_taps;
      const int a_stages = p.a_stages, b_stages = p.b_stages;
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n_cols >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      const uint64_t tmpl = make_sw128_desc(0, 1, 1024 >> 4, 1, 0);
      const uint32_t desc_hi = (uint32_t)(tmpl >> 32);
      const uint32_t a_lo0 = (uint32_t)tmpl + (a_base >> 4), b_lo0 = (uint32_t)tmpl + (b_base >> 4);
      const uint32_t a_step = CB_A_BYTES >> 4, b_step = (uint32_t)p.b_bytes >> 4;
      int sa = 0, sb = 0;
      uint32_t pha = 0, phb = 0;
      uint32_t a_lo = a_lo0, b_lo = b_lo0;   // low descriptor words of stage sa / sb
      uint32_t fa = fulla(0), ea = emptya(0), fb = fullb(0), eb = emptyb(0);
      int buf = 0;        // TMEM ring position of the job's first accumulator
      uint32_t bph = 0;   // its phase
      const int groups_per_job = p.nsub / NSH;
      for (int job = blockIdx.x; job < total_jobs; job += gridDim.x) {
      for (int sg = 0; sg < groups_per_job; ++sg) {
        uint32_t d_tmem[NSH];
        uint32_t tfull[NSH];
#pragma unroll
        for (int sub = 0; sub < NSH; ++sub) {
          mbar_wait_tight(tempty_bar(buf), bph ^ 1u);  // the epilogue has drained it
          d_tmem[sub] = tmem_base + (uint32_t)(buf * n_cols);
          tfull[sub] = tfull_bar(buf);
          if (++buf == n_bufs) {
            buf = 0;
            bph ^= 1u;
          }
        }
        tc_fence_after();
        uint32_t acc = 0u;
        // both rings hold a multiple of NSH activation stages (cb_plan), so the NSH tiles of a chunk / tap are
        // consecutive stages that never wrap in between: one wrap test per group
        for (int kc = 0; kc < k_chunks; ++kc) {
          uint32_t bl0 = 0, eb0 = 0;
          if (MODE3) {
            // the chunk's NSH activation tiles stay until its three taps are done
#pragma unroll
            for (int sub = 0; sub < NSH; ++sub) mbar_wait_tight(fb + 8u * sub, phb);
            bl0 = b_lo;
            eb0 = eb;
            b_lo += NSH * b_step; fb += 8 * NSH; eb += 8 * NSH; sb += NSH;
            if (sb == b_stages) {
              sb = 0; phb ^= 1u; b_lo = b_lo0; fb = fullb(0); eb = emptyb(0);
            }
          }
          for (int t = 0; t < n_taps; ++t) {
            mbar_wait_tight(fa, pha);
            if (!MODE3) {
#pragma unroll
              for (int sub = 0; sub < NSH; ++sub) mbar_wait_tight(fb + 8u * sub, phb);
            }
            tc_fence_after();
            if (issuer) {
#pragma unroll
              for (int sub = 0; sub < NSH; ++sub) {
                // mode3, tap t: start advanced by t rows of 128 B
                const uint32_t bt = MODE3 ? bl0 + sub * b_step + (uint32_t)(8 * t) : b_lo + sub * b_step;
                umma_bf16_lo(d_tmem[sub], a_lo, bt, desc_hi, idesc, acc);
                umma_bf16_lo(d_tmem[sub], a_lo + 2, bt + 2, desc_hi, idesc, 1u);
                umma_bf16_lo(d_tmem[sub], a_lo + 4, bt + 4, desc_hi, idesc, 1u);
                umma_bf16_lo(d_tmem[sub], a_lo + 6, bt + 6, desc_hi, idesc, 1u);
                if (!MODE3) umma_commit(eb + 8u * sub);
              }
              umma_commit(ea);
            }
            acc = 1u;
            if (!MODE3) {
              b_lo += NSH * b_step; fb += 8 * NSH; eb += 8 * NSH; sb += NSH;
              if (sb == b_stages) {
                sb = 0; phb ^= 1u; b_lo = b_lo0; fb = fullb(0); eb = emptyb(0);
              }
            }
            a_lo += a_step; fa += 8; ea += 8;
            if (++sa == a_stages) {
              sa = 0; pha ^= 1u; a_lo = a_lo0; fa = fulla(0); ea = emptya(0);
            }
          }
          if (MODE3 && issuer) {
#pragma unroll
            for (int sub = 0; sub < NSH; ++sub) umma_commit(eb0 + 8u * sub);
          }
        }
        if (issuer) {
#pragma unroll
          for (int sub = 0; sub < NSH; ++sub) umma_commit(tfull[sub]);
        }
        __syncwarp();
      }
      }
    }
  } else if (warp < 10) {
    // =========================== drain warps (2..9): TMEM -> y (global), moments ===========================
    const int ew = warp - 2;
    const int quarter = warp & 3;  // TMEM lanes [32*quarter, +32)
    const int half = ew >> 2;      // the two warps of a quarter alternate over the 16-column chunks
    const int cl = quarter * 32 + lane;
    const int n_chunks = p.n_cols >> 4;
    __nv_bfloat16* tr = reinterpret_cast<__nv_bfloat16*>(tail + CB_OFF_TR) + ew * 512;  // this warp's transpose scratch
    // number of real positions among this thread's columns of one sub-tile
    float cnt_sub = 0.f;
    for (int ch = half; ch < n_chunks; ch += 2)
      for (int j = 0; j < 16; ++j) cnt_sub += crow[(ch << 4) + j] != 0xFFFFFFFFu ? 1.f : 0.f;
    int ebuf = 0;        // TMEM ring position, walked exactly like the MMA warp's
    uint32_t ebph = 0;
    int jc = 0;          // jobs done by this CTA
    for (int job = blockIdx.x; job < total_jobs; job += gridDim.x, ++jc) {
      const int pos_job = job / p.n_co_tiles;
      const int co0 = (job % p.n_co_tiles) * 128, nj = pos_job * job_breaths;
      const int co = co0 + cl;
      const bool co_ok = co < p.c_out;
      const int par = jc & 1;
      (void)co_ok;
      // the moments slot of two jobs ago must have been read by the apply warps
      if (EPI == CB_FUSED && jc >= 2) named_bar_sync(4 + par, 2 * CB_EPI_THREADS);
      float s = 0.f, ss = 0.f, shift = 0.f;
      for (int sub = 0; sub < p.nsub; ++sub) {
        const int buf = ebuf;
        mbar_wait(tfull_bar(buf), ebph);
        if (++ebuf == p.n_bufs) {
          ebuf = 0;
          ebph ^= 1u;
        }
        tc_fence_after();
        const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * p.n_cols);
        // position q of breath n lives at row n*y_l + q*y_mul + y_off of y.  A chunk (16 columns x this warp's 32
        // channels) is transposed through 1 KB of shared memory so that a lane stores 16 bytes (8 channels of one
        // column) instead of 16 times 2 bytes: lane = (column within the pass) * 4 + (group of 8 channels)
        const int cv = lane & 3, lc = lane >> 2;
        const int cbase = co0 + quarter * 32 + cv * 8;
        const bool c_ok = cbase < p.c_out;
        __nv_bfloat16* ysub = p.y + ((size_t)(nj + sub * p.nb) * p.y_l + p.y_off) * p.y_stride + cbase;
        const bool first = (sub % p.spg) == 0;
        if (first) s = ss = 0.f;
        // software pipeline: the TMEM load of the next chunk is in flight while this one is converted and stored
        uint32_t va[16], vb[16];
        tmem_ld16(t_row + (uint32_t)(half << 4), va);
        auto chunk = [&](int ch, const uint32_t (&v)[16]) {
          const uint32_t* cr = crow + (ch << 4);
          if (EPI != CB_PLAIN && first && ch == half) {
            // any sample of the channel's data will do, but only a real column is one: the chunk's first column can be a
            // halo column (L = 16: column 16 of the second half), and a junk column may hold anything, NaN included
            shift = 0.f;
#pragma unroll
            for (int j = 15; j >= 0; --j)
              if (cr[j] != 0xFFFFFFFFu) shift = __uint_as_float(v[j]);
          }
          if (EPI != CB_PLAIN) {
            const uint4* cr4 = reinterpret_cast<const uint4*>(cr);
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const uint4 r4 = cr4[j4];
              const uint32_t rr[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) {
                // a junk column may hold anything, NaN included: select, never multiply
                const float d = rr[jj] != 0xFFFFFFFFu ? __uint_as_float(v[4 * j4 + jj]) - shift : 0.f;
                s += d;
                ss = fmaf(d, d, ss);
              }
            }
          }
          __syncwarp();  // the previous chunk's reads of the scratch are done
#pragma unroll
          for (int j = 0; j < 16; ++j) tr[j * 32 + lane] = __float2bfloat16_rn(__uint_as_float(v[j]));
          __syncwarp();
#pragma unroll
          for (int pass = 0; pass < 2; ++pass) {
            const int col = pass * 8 + lc;
            const uint32_t r = cr[col];
            if (r != 0xFFFFFFFFu && c_ok) {
              uint4 val = *reinterpret_cast<const uint4*>(tr + col * 32 + cv * 8);
              uint4* dst = reinterpret_cast<uint4*>(ysub + r);
              if (ACC) {
                float a[8], b[8];
                unpack8(val, a);
                unpack8(*dst, b);
#pragma unroll
                for (int k = 0; k < 8; ++k) a[k] += b[k];
                val = pack8(a);
              }
              *dst = val;
            }
          }
        };
        for (int ch = half; ch < n_chunks; ch += 4) {
          tmem_ld_wait();
          if (ch + 2 < n_chunks) tmem_ld16(t_row + (uint32_t)((ch + 2) << 4), vb);
          chunk(ch, va);
          if (ch + 2 < n_chunks) {
            tmem_ld_wait();
            if (ch + 4 < n_chunks) tmem_ld16(t_row + (uint32_t)((ch + 4) << 4), va);
            chunk(ch + 2, vb);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(buf));  // the accumulator may be overwritten
        if (EPI == CB_FUSED && (sub % p.spg) == p.spg - 1) {
          float* m = mom + (((par * 2 + sub / p.spg) * 2 + half) * 4) * 128 + cl;
          m[0] = cnt_sub * (float)p.spg;
          m[128] = s;
          m[256] = ss;
          m[384] = shift;
        }
      }
      if (EPI == CB_PARTIAL && co_ok) {
        // this thread's moments of its columns -> part[pos job][half][cnt, mean, M2][channel]   (nsub == 1)
        const float n = cnt_sub;
        const float inv = n > 0.f ? 1.f / n : 0.f;
        float* dst = p.part + ((size_t)(pos_job * 2 + half) * 3) * p.c_out + co;
        dst[0] = n;
        dst[p.c_out] = shift + s * inv;
        dst[2 * p.c_out] = fmaxf(ss - s * s * inv, 0.f);
      }
      if (EPI == CB_FUSED) {
        __threadfence_block();                         // y stores and moments before the hand-over
        named_bar_arrive(2 + par, 2 * CB_EPI_THREADS);  // the apply warps take the job from here
      }
    }
  } else {
    // =========================== apply warps (10..17, FUSED only): out = relu(y * scale + shift + res) ===============
    // y of the job was written by this CTA a moment ago: the re-read is an L2 hit, row-wise with 16-byte accesses.
    const int aw = warp - 10;
    const int at = threadIdx.x - (64 + CB_EPI_THREADS);
    const int cl = (aw & 3) * 32 + lane;
    const int sub_rows = p.nb * p.l;
    const int group_rows = p.spg * sub_rows;
    const int gpj = p.nsub / p.spg;
    const int vec = at & 15, rl = at >> 4;  // 16 vectors of 8 channels x 16 row lanes
    int jc = 0;
    for (int job = blockIdx.x; job < total_jobs; job += gridDim.x, ++jc) {
      const int pos_job = job / p.n_co_tiles;
      const int co0 = (job % p.n_co_tiles) * 128, nj = pos_job * job_breaths;
      const int par = jc & 1;
      named_bar_sync(2 + par, 2 * CB_EPI_THREADS);  // drain warps: y and the moments of this job are complete
      float* sc_tab = scsh + par * 512;
      if (aw < 4 * gpj) {
        // merge the two drain threads of every channel (Chan) -> scale / shift
        const int gi = aw >> 2;  // warps 0-3 take group 0, warps 4-7 group 1 (if the job has two)
        const int co = co0 + cl;
        const float* m0 = mom + (((par * 2 + gi) * 2 + 0) * 4) * 128 + cl;
        const float* m1 = mom + (((par * 2 + gi) * 2 + 1) * 4) * 128 + cl;
        const float n0 = m0[0], n1 = m1[0];
        const float i0 = n0 > 0.f ? 1.f / n0 : 0.f, i1 = n1 > 0.f ? 1.f / n1 : 0.f;
        const float s0 = m0[128], s1 = m1[128];
        const float e0 = m0[384] + s0 * i0, e1 = m1[384] + s1 * i1;
        const float q0 = fmaxf(m0[256] - s0 * s0 * i0, 0.f), q1 = fmaxf(m1[256] - s1 * s1 * i1, 0.f);
        const float n = n0 + n1, dlt = e1 - e0;
        const float mean = n1 > 0.f ? e0 + dlt * (n1 / n) : e0;
        const float m2 = n1 > 0.f ? q0 + q1 + dlt * dlt * (n0 * n1 / n) : q0;
        const float var = fmaxf(m2 / n, 0.f) + p.eps;
        float rstd = rsqrtf(var);
        rstd = rstd * (1.5f - 0.5f * var * rstd * rstd);  // one Newton step: the reference divides by sqrt()
        float sc = 0.f, sh = 0.f;
        if (co < p.c_out) {
          const size_t g = (size_t)pos_job * gpj + gi;
          sc = rstd * p.gamma[co];
          sh = p.beta[co] - mean * sc;
          p.save_mean[g * p.c_out + co] = mean;
          p.save_rstd[g * p.c_out + co] = rstd;
        }
        sc_tab[gi * 256 + cl] = sc;
        sc_tab[gi * 256 + 128 + cl] = sh;
      }
      named_bar_sync(6, CB_EPI_THREADS);                 // scale / shift visible to all apply threads
      named_bar_arrive(4 + par, 2 * CB_EPI_THREADS);     // the moments slot may be reused
      const int c = co0 + vec * 8;
      if (c < p.c_out) {
        for (int gi = 0; gi < gpj; ++gi) {
          float sc[8], sh[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            sc[j] = sc_tab[gi * 256 + vec * 8 + j];
            sh[j] = sc_tab[gi * 256 + 128 + vec * 8 + j];
          }
          const size_t grow0 = (size_t)nj * p.l + (size_t)gi * group_rows;
          const __nv_bfloat16* yp = p.y + grow0 * p.y_stride + c;
          __nv_bfloat16* op = p.out + grow0 * p.out_stride + c;
          const __nv_bfloat16* rp = p.res ? p.res + grow0 * p.res_stride + c : nullptr;
          auto one = [&](int row, const uint4& yy, const uint4& rr) {
            float v[8];
            unpack8(yy, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc[j], sh[j]);
            if (rp) {
              float e[8];
              unpack8(rr, e);
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] += e[j];
            }
            if (p.relu) {
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            *reinterpret_cast<uint4*>(op + (size_t)row * p.out_stride) = pack8(v);
          };
          const uint4 none = make_uint4(0u, 0u, 0u, 0u);
          int row = rl;
          for (; row + 48 < group_rows; row += 64) {  // 4 rows per thread in flight
            uint4 yy[4], rr[4] = {none, none, none, none};
#pragma unroll
            for (int u2 = 0; u2 < 4; ++u2) {
              yy[u2] = __ldcg(reinterpret_cast<const uint4*>(yp + (size_t)(row + 16 * u2) * p.y_stride));
              if (rp) rr[u2] = *reinterpret_cast<const uint4*>(rp + (size_t)(row + 16 * u2) * p.res_stride);
            }
#pragma unroll
            for (int u2 = 0; u2 < 4; ++u2) one(row + 16 * u2, yy[u2], rr[u2]);
          }
          for (; row < group_rows; row += 16) {
            const uint4 yy = __ldcg(reinterpret_cast<const uint4*>(yp + (size_t)row * p.y_stride));
            uint4 rr = none;
            if (rp) rr = *reinterpret_cast<const uint4*>(rp + (size_t)row * p.res_stride);
            one(row, yy, rr);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
struct CbPlan {
  CbParams p;
  int mode;      // 0 unsupported, 1 partial statistics, 2 fused
  int smem;
};

// `unit`: breaths that must stay together (the BatchNorm group; 1 for a plain convolution).  want_bn: statistics wanted.
static CbPlan cb_plan(int n_breaths, int unit, bool want_bn, int l_out, int c_red, int c_cols, int n_taps, bool mode3) {
  CbPlan w{};
  CbParams& p = w.p;
  w.mode = 0;
  if (unit <= 0 || n_breaths <= 0 || n_breaths % unit != 0) return w;
  if (c_red % 8 || c_cols % 8 || n_taps > CB_MAX_TAPS || n_taps < 1) return w;
  p.mode3 = mode3 ? 1 : 0;
  p.n_taps = n_taps;
  p.l = l_out;
  p.lp = mode3 ? l_out + 1 : l_out;
  const int slack = mode3 ? 1 : 0;  // the last breath of a tile has no junk column
  // breaths per sub-tile: the largest divisor of the unit whose columns fit one accumulator.  A plain convolution has
  // no unit: any count works as long as it divides the number of breaths.
  int nb = 0;
  const int lim = want_bn ? unit : n_breaths;
  for (int d = 1; d <= lim && d * p.lp - slack <= CB_MAX_COLS; ++d)
    if (lim % d == 0) nb = d;
  if (!want_bn && g_dbg_cb_wide != 1) {
    // two position tiles that share every weight tile need three accumulators: tiles of at most 170 columns
    int nb2 = 0;
    for (int d = 1; d <= lim && d * p.lp - slack <= 512 / 3; ++d)
      if (lim % d == 0 && (lim / d) % 2 == 0) nb2 = d;
    if (nb2 > 0 && nb2 * p.lp - slack >= 96) nb = nb2;
  }
  if (nb == 0) return w;
  p.nb = nb;
  p.n_cols = (nb * p.lp - slack + 15) / 16 * 16;
  if (p.n_cols < 64) return w;  // tiny tiles: the plain kernels + the BatchNorm kernel are the better path
  p.k_chunks = ceil_div(c_red, 64);
  p.n_co_tiles = ceil_div(c_cols, 128);
  p.c_out = c_cols;
  // staged rows read by the MMAs: n_cols (+ 2 for the shifted taps)
  p.b_bytes = ((p.n_cols + (mode3 ? 2 : 0)) * 128 + 1023) / 1024 * 1024;
  p.n_bufs = 512 / p.n_cols;
  if (p.n_bufs > 4) p.n_bufs = 4;
  const int min_rings = 3 * CB_A_BYTES;
  const int budget = CB_SMEM_LIMIT - 1024 - CB_TAIL_BYTES;
  if (want_bn) {
    const int spg = unit / nb;  // sub-tiles per group
    // the group's sub-tiles are accumulated together and the next job needs a free accumulator to start with
    const bool fits = spg <= CB_MAX_SUB && spg < p.n_bufs + (spg == 1 ? 1 : 0) && min_rings + 2 * spg * p.b_bytes <= budget;
    if (fits) {
      p.epi = CB_FUSED;
      p.spg = spg;
      p.nsub = spg;
      // a one-sub-tile group leaves room for a second group in the job: the weight tile then feeds both
      if (spg == 1 && p.n_bufs >= 3 && (n_breaths / unit) % 2 == 0 && min_rings + 4 * p.b_bytes <= budget) p.nsub = 2;
    } else {
      p.epi = CB_PARTIAL;
      p.spg = 1;
      p.nsub = 1;
    }
  } else {
    p.epi = CB_PLAIN;
    p.spg = 1;
    p.nsub = 1;
    if (p.n_bufs >= 3 && (n_breaths / nb) % 2 == 0 && min_rings + 4 * p.b_bytes <= budget) p.nsub = 2;
  }
  p.n_pos_jobs = n_breaths / (nb * p.nsub);
  // Sharing a weight tile between the job's two sub-tiles halves the L2 -> SM weight stream, but both accumulators then
  // finish together and the next job cannot start before the first is drained; one after the other, the third TMEM
  // buffer lets the MMAs of the next sub-tile overlap the drain.  The kernel is not L2-bound: default = sequential.
  p.nshare = (p.nsub == 2 && g_dbg_cb_share == 1) ? 2 : 1;
  int left = budget;
  if (mode3) {
    // activation tiles: two chunks of look-ahead; weight tiles take the rest (a weight tile lasts 4*nsub MMAs)
    p.b_stages = p.nshare == 2 ? 4 : 3;
    if (g_dbg_cb_bstages > 0) p.b_stages = g_dbg_cb_bstages / p.nshare * p.nshare;
    while (p.b_stages > 2 * p.nshare && left - p.b_stages * p.b_bytes < 3 * CB_A_BYTES) p.b_stages -= p.nshare;
    left -= p.b_stages * p.b_bytes;
    p.a_stages = left / CB_A_BYTES;
    if (p.a_stages > CB_MAX_A) p.a_stages = CB_MAX_A;
  } else {
    // per-tap loads consume one weight tile with nsub activation tiles
    int st = left / (CB_A_BYTES + p.nshare * p.b_bytes);
    if (st > CB_MAX_A) st = CB_MAX_A;
    if (st * p.nshare > CB_MAX_B) st = CB_MAX_B / p.nshare;
    p.a_stages = st;
    p.b_stages = st * p.nshare;
  }
  if (p.a_stages < 2 || p.b_stages < 2 * p.nshare || p.b_stages % p.nshare != 0 || p.b_stages > CB_MAX_B) return w;
  w.smem = p.b_stages * p.b_bytes + p.a_stages * CB_A_BYTES + CB_TAIL_BYTES + 1024;
  w.mode = p.epi == CB_FUSED ? 2 : 1;
  return w;
}

static bool cb_forward_taps(CbParams& p, int l_in, int l_out, int ktaps, int stride, int pad, bool* mode3) {
  if (stride != 1 && stride != 2) return false;
  if (ktaps > CB_MAX_TAPS || l_in % stride != 0 || l_out != (l_in + 2 * pad - ktaps) / stride + 1) return false;
  *mode3 = (ktaps == 3 && stride == 1 && pad == 1 && l_out >= 2) && g_dbg_cb_pertap != 1;
  for (int t = 0; t < ktaps; ++t) {
    // source position = q*stride + (t - pad) = stride*(q + floor((t-pad)/stride)) + ((t-pad) mod stride)
    const int d = t - pad;
    const int fl = d >= 0 ? d / stride : -((-d + stride - 1) / stride);
    p.w_tap[t] = t;
    p.in_par[t] = d - fl * stride;
    p.in_start[t] = fl;
  }
  return true;
}

static CbPlan cb_plan_fwd(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride, int pad) {
  CbParams taps{};
  bool mode3 = false;
  if (!cb_forward_taps(taps, l_in, l_out, ktaps, stride, pad, &mode3)) return CbPlan{};
  CbPlan w = cb_plan(n_breaths, group, true, l_out, c_in, c_out, ktaps, mode3);
  for (int t = 0; t < ktaps; ++t) {
    w.p.w_tap[t] = taps.w_tap[t];
    w.p.in_par[t] = taps.in_par[t];
    w.p.in_start[t] = taps.in_start[t];
  }
  return w;
}

int tc_conv_bn_mode(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride, int pad) {
  return cb_plan_fwd(n_breaths, group, l_in, l_out, c_in, c_out, ktaps, stride, pad).mode;
}

// PARTIAL mode: number of (count, mean, M2) records per group and channel
int tc_conv_bn_part_entries(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride, int pad) {
  CbPlan w = cb_plan_fwd(n_breaths, group, l_in, l_out, c_in, c_out, ktaps, stride, pad);
  if (w.mode != 1) return 0;
  return 2 * (group / w.p.nb);
}

static int cb_launch(CbPlan& w, const void* src, const void* wts, int n_breaths, int c_red, int c_cols, int ktaps_total,
                     int l_src, int src_planes, int src_stride, cudaStream_t st) {
  CbParams& p = w.p;
  CUtensorMap tm_w, tm_x;
  {
    cuuint64_t dims[3] = {(cuuint64_t)c_red, (cuuint64_t)c_cols, (cuuint64_t)ktaps_total};
    cuuint64_t str[2] = {(cuuint64_t)c_red * 2, (cuuint64_t)c_red * c_cols * 2};
    cuuint32_t box[3] = {64, 128, 1};
    int rc = make_bf16_map(&tm_w, wts, 3, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const int l_plane = l_src / src_planes;
    cuuint64_t dims[4] = {(cuuint64_t)c_red, (cuuint64_t)src_planes, (cuuint64_t)l_plane, (cuuint64_t)n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)src_stride * 2, (cuuint64_t)src_stride * src_planes * 2, (cuuint64_t)src_stride * l_src * 2};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)p.lp, (cuuint32_t)p.nb};
    int rc = make_bf16_map(&tm_x, src, 4, dims, str, box, true);
    if (rc) return rc;
  }
  const int jobs = p.n_pos_jobs * p.n_co_tiles;
  const int grid = jobs < sm_count() ? jobs : sm_count();
  static int attr_smem[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#define CB_RUN(IDX, E, A, M3, NS)                                                                                      \
  do {                                                                                                                 \
    if (w.smem > attr_smem[IDX]) {                                                                                     \
      cudaError_t e = cudaFuncSetAttribute(tc_conv_bn_kernel<E, A, M3, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, w.smem); \
      if (e != cudaSuccess) {                                                                                          \
        set_error("conv+bn: cannot opt in to %d bytes of shared memory: %s", w.smem, cudaGetErrorString(e));           \
        return DARDS_ERR_CUDA;                                                                                         \
      }                                                                                                                \
      attr_smem[IDX] = w.smem;                                                                                         \
    }                                                                                                                  \
    tc_conv_bn_kernel<E, A, M3, NS><<<grid, (E) == CB_FUSED ? CB_THREADS_FUSED : CB_THREADS, w.smem, st>>>(tm_w, tm_x, p);                                   \
  } while (0)
  const bool m3 = p.mode3 != 0, two = p.nshare == 2;
  if (p.epi == CB_FUSED) {
    if (m3 && two) CB_RUN(0, CB_FUSED, false, true, 2);
    else if (m3) CB_RUN(1, CB_FUSED, false, true, 1);
    else if (two) CB_RUN(2, CB_FUSED, false, false, 2);
    else CB_RUN(3, CB_FUSED, false, false, 1);
  } else if (p.epi == CB_PARTIAL) {
    if (m3) CB_RUN(4, CB_PARTIAL, false, true, 1);
    else CB_RUN(5, CB_PARTIAL, false, false, 1);
  } else if (p.accumulate) {
    if (two) CB_RUN(6, CB_PLAIN, true, true, 2);
    else CB_RUN(7, CB_PLAIN, true, true, 1);
  } else {
    if (two) CB_RUN(8, CB_PLAIN, false, true, 2);
    else CB_RUN(9, CB_PLAIN, false, true, 1);
  }
#undef CB_RUN
  DARDS_CHECK_LAUNCH("tc_conv_bn");
  return DARDS_OK;
}

int tc_conv_bn_fwd(const void* in, const void* w_koi, void* y, void* out, const void* res, const float* gamma,
                   const float* beta, float* save_mean, float* save_rstd, float* part, int n_breaths, int group, int l_in,
                   int l_out, int c_in, int c_out, int in_stride, int y_stride, int out_stride, int res_stride, int ktaps,
                   int stride, int pad, float eps, int relu, int src_last_use, cudaStream_t st) {
  CbPlan w = cb_plan_fwd(n_breaths, group, l_in, l_out, c_in, c_out, ktaps, stride, pad);
  if (w.mode == 0) {
    set_error("conv+bn: unsupported shape (n=%d group=%d l=%d->%d cin=%d cout=%d k=%d s=%d p=%d)", n_breaths, group, l_in,
              l_out, c_in, c_out, ktaps, stride, pad);
    return DARDS_ERR_UNSUPPORTED;
  }
  DARDS_CHECK_ARG(in_stride % 8 == 0 && y_stride % 8 == 0, "conv+bn: row strides must be multiples of 8");
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_koi) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                  "conv+bn: operands must be 16-byte aligned");
  CbParams& p = w.p;
  if (w.mode == 2) {
    DARDS_CHECK_ARG(out && gamma && beta && save_mean && save_rstd, "conv+bn (fused): null pointer");
    DARDS_CHECK_ARG(out_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "conv+bn: `out` must be 16-byte aligned rows");
    DARDS_CHECK_ARG(!res || (res_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(res) & 15) == 0),
                    "conv+bn: `res` must be 16-byte aligned rows");
  } else {
    DARDS_CHECK_ARG(part, "conv+bn (partial statistics): null `part`");
  }
  p.eps = eps;
  p.relu = relu ? 1 : 0;
  p.accumulate = 0;
  p.y = static_cast<__nv_bfloat16*>(y);
  p.y_stride = y_stride;
  p.y_l = l_out;
  p.y_mul = 1;
  p.y_off = 0;
  p.gamma = gamma;
  p.beta = beta;
  p.save_mean = save_mean;
  p.save_rstd = save_rstd;
  p.part = part;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.res = static_cast<const __nv_bfloat16*>(res);
  p.out_stride = out_stride;
  p.res_stride = res_stride;
  p.x_evict_first = (src_last_use && p.n_co_tiles == 1 && p.mode3 && g_dbg_l2_hint != 0) ? 1 : 0;
  return cb_launch(w, in, w_koi, n_breaths, c_in, c_out, ktaps, l_in, stride, in_stride, st);
}

// Plain k = 3 / stride 1 / pad 1 convolution (forward or data gradient: `reverse_taps`) through the same main loop:
// the wide layers (reduction over >= 256 channels), where conv_tc.cu's one-load-per-tap kernel is bound by the L2 -> SM
// operand stream.  Returns DARDS_ERR_UNSUPPORTED when the shape does not tile (the caller falls back).
int tc_conv3_shared(const void* src, const void* wts, void* dst, int n_breaths, int l, int c_red, int c_cols, int src_stride,
                    int dst_stride, bool reverse_taps, bool accumulate, cudaStream_t st) {
  if (l < 2) return DARDS_ERR_UNSUPPORTED;
  CbPlan w = cb_plan(n_breaths, 1, false, l, c_red, c_cols, 3, true);
  if (w.mode == 0) return DARDS_ERR_UNSUPPORTED;
  if (src_stride % 8 || dst_stride % 8 || (reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(wts) & 15) ||
      (reinterpret_cast<uintptr_t>(dst) & 15))
    return DARDS_ERR_UNSUPPORTED;
  CbParams& p = w.p;
  for (int t = 0; t < 3; ++t) {
    p.w_tap[t] = reverse_taps ? 2 - t : t;
    p.in_par[t] = 0;
    p.in_start[t] = 0;
  }
  p.accumulate = accumulate ? 1 : 0;
  p.y = static_cast<__nv_bfloat16*>(dst);
  p.y_stride = dst_stride;
  p.y_l = l;
  p.y_mul = 1;
  p.y_off = 0;
  p.relu = 0;
  p.eps = 0.f;
  p.gamma = p.beta = nullptr;
  p.save_mean = p.save_rstd = p.part = nullptr;
  p.out = nullptr;
  p.res = nullptr;
  p.out_stride = p.res_stride = 0;
  p.x_evict_first = 0;
  return cb_launch(w, src, wts, n_breaths, c_red, c_cols, 3, l, 1, src_stride, st);
}

}  // namespace dards

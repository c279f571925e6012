// tcgen05 weight-gradient kernel for Conv1d (bf16 operands, fp32 accumulation in TMEM, fp32 output).
//
//   dW[t][co][ci] = sum over rows k=(breath n, position q) of dout[k, co] * in[k shifted by tap t, ci]
//
// GEMM view: D_t[co, ci] = A^T B_t with the REDUCTION over positions.  Channels-last activations make both
// operands "MN-major" in shared memory: a TMA box of (64 channels x R rows) lands as R rows of 128 bytes, row =
// reduction index, which is exactly the canonical SWIZZLE_128B MN-major UMMA layout (8-row groups 1024 B apart =
// SBO, 64-channel chunks LBO apart).  No transposition anywhere.
//
// One TMA load per operand serves all taps: each breath is staged with ONE zero halo row -- dout as
// [dout[0..L-1], 0], the input as [0, in[0..L-1]] -- the halo coming for free from the TMA out-of-bounds fill.
// Tap t then multiplies the SAME staged input tile, read through a descriptor whose start address is advanced by
// t rows (t * 128 B): dout row j meets staged input row j + t = in[j + t - 1].  Where the shifted rows run into the
// next breath they meet either its leading zero row (the conv padding) or this breath's zero dout row, so nothing
// leaks across breaths.  Stride-2 convolutions stage the two parity planes of the input (4-D view (C, 2, L/2, N))
// as two tiles.
//
// 64 input channels, 3 taps, stride 1: the three taps are ONE MMA with N = 192.  For an MN-major operand the
// descriptor's leading-byte-offset is the distance between consecutive 64-column chunks; LBO = 128 B (one row) makes
// chunk t the tile shifted by t rows, i.e. tap t, so D[co, t*64 + ci] comes out of a single instruction that reads
// the dout tile once instead of three times.
//
// Tile: 128 output channels (TMEM lanes) x up to 128 input channels (columns) x up to 3 taps (3 accumulators =
// 384 TMEM columns), or x 64 input channels x 7 taps (the stride-2 k7 convolution, tc_wgrad7_kernel).  Split-K over groups of breaths; every CTA writes its fp32 partial tile and a second kernel
// reduces the partials in a fixed order (deterministic) into the parameter's (Cout, Cin, K) layout.
#include <cstring>

#include "tc_common.cuh"

namespace dards {

int g_dbg_wgrad_pair = -1;  // debug key 19 = 0: C >= 256 layers stay on single CTAs instead of CTA pairs (cta_group::2)

constexpr int WG_TC_THREADS = 192;       // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int WG_RMAX = 128;             // reduction rows per stage (multiple of 16)
constexpr int WG_CHUNK_A = WG_RMAX * 128;          // bytes of one 64-channel chunk of the dout tile
constexpr int WG_CHUNK_B = (WG_RMAX + 8) * 128;    // input tile: + 8 zero rows for the shifted taps
constexpr int WG_A_BYTES = 2 * WG_CHUNK_A;         // 128 output channels
constexpr int WG_B_BYTES = 2 * WG_CHUNK_B;         // 128 input channels
constexpr int WG_MAX_TAPS = 3;
constexpr int WG_MAX_STAGES = 8;
constexpr int WG_SMEM_LIMIT = 227 * 1024;

struct WgTcParams {
  int n_btiles;                // 1 (stride 1) or 2 (stride 2: one per parity plane)
  int b_plane[2], b_start[2];  // plane / first-row coordinates of the staged input tiles
  int a_start;                 // first-row coordinate of the staged dout tile (-1 with halo, 0 without)
  int n_taps;
  int tap_btile[WG_MAX_TAPS], tap_shift[WG_MAX_TAPS];
  int p_rows;                  // rows staged per breath (L + 2*halo)
  int nb;                      // breaths per stage
  int r_pad;                   // nb*p_rows rounded up to 16
  int n_units;                 // ceil(n_breaths / nb): reduction units
  int units_per_split;
  int c_in, c_out;
  int n_ci_tiles, n_co_tiles;
  int stages, stage_bytes;
  int a_bytes, b_bytes;        // bytes of the dout tile / of one input tile inside a stage (1 or 2 64-channel chunks)
  int base_offset_mode;        // 1 (default): base_offset 0;  0: (start >> 7) & 7 -- kept for the probe only
  int fuse_taps;               // 1: the 3 taps are the 3 column chunks of one N = 192 MMA (c_in == 64, stride 1)
  int tap_cols;                // TMEM column distance between the taps' accumulators (128, or 64 when fused)
  int l2_hint;                 // 1: the saved input activations (their last use) are loaded with L2 evict_first priority
  int pair;                    // 1: CTA pairs (cta_group::2): two output-channel tiles share one input tile, half of it per CTA
  int accumulate_l2;           // 1: the CTA's tile is ADDED into dw_t[t][co][ci] with TMA reduce-add (no partials, no reduce kernel)
};

// PAIR: launched as clusters of 2 CTAs along blockIdx.x.  The pair takes the output-channel tiles (2j, 2j+1) of one
// input-channel tile and one split: M = 256 through tcgen05.mma.cta_group::2, each CTA stages its own dout tile and ONE of
// the two 64-channel chunks of the input tile (the B operand's N = 128 columns are split between the two CTAs), which cuts
// the operand stream from 66 to 49 KB per stage -- the single-CTA kernel needs 42 B/clk/SM, exactly the L2 -> SM limit.
// Barriers as in tc_conv_pair_kernel: full[] in the leader, empty[] / done in both (multicast commits).
//
// NT: the tap count the MMA issuer is compiled for.  WG_MAX_TAPS (tc_wgrad_kernel): 1 or 3 taps as p.n_taps says.
// 7 (tc_wgrad7_kernel): the k7 / stride 2 / pad 3 convolution of the two-convolution ResNet stem, c_in <= 64, single CTA.
// Its seven 64-column accumulators take 448 of the 512 TMEM columns, and its tap map is fixed: in[2q + t - 3] is, for odd
// t, plane 0 row q + (t - 3)/2 and, for even t, plane 1 row q + (t - 4)/2; both planes are staged from row -2, so tap t
// reads tile (t odd ? 0 : 1) shifted by (t + 1)/2 rows.
template <bool PAIR, int NT>
__device__ __forceinline__ void tc_wgrad_body(const CUtensorMap& tm_a, const CUtensorMap& tm_b, const CUtensorMap& tm_d,
                                              float* __restrict__ partial, const WgTcParams& p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + p.stages * p.stage_bytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (WG_MAX_STAGES + s); };
  const uint32_t done_bar = bar_base + 8u * (2 * WG_MAX_STAGES);
  const uint32_t tmem_slot = bar_base + 8u * (2 * WG_MAX_STAGES + 1);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x, split = blockIdx.y;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool lead = rank == 0;
  // pairs: (tile >> 1) enumerates (output-channel tile pair, input-channel tile), the rank picks the channel tile
  const int co0 = PAIR ? (2 * ((tile >> 1) / p.n_ci_tiles) + (int)rank) * 128 : (tile / p.n_ci_tiles) * 128;
  const int ci0 = PAIR ? ((tile >> 1) % p.n_ci_tiles) * 128 : (tile % p.n_ci_tiles) * 128;
  const int ci_n = (p.c_in - ci0) >= 128 ? 128 : ((p.c_in - ci0 + 63) / 64) * 64;  // MMA N: 64 or 128
  const int co_chunks = (p.c_out - co0) > 64 ? 2 : 1, ci_chunks = PAIR ? 1 : ci_n / 64;  // chunks THIS CTA stages
  const int u_begin = split * p.units_per_split;
  int u_end = u_begin + p.units_per_split;
  if (u_end > p.n_units) u_end = p.n_units;
  const int n_iters = u_end > u_begin ? u_end - u_begin : 0;

  // Rows that TMA never writes must be ZERO (dout: they multiply shifted input rows) or at least finite
  // (input): clear the whole operand area once.  generic-proxy writes -> fence -> visible to the async proxy.
  {
    uint4* z = reinterpret_cast<uint4*>(smem_gen);
    const int n16 = (p.stages * p.stage_bytes) / 16;
    for (int i = threadIdx.x; i < n16; i += WG_TC_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(done_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) {
      tmem_alloc_2sm(tmem_slot, 512);
      tmem_relinquish_2sm();
    } else {
      tmem_alloc(tmem_slot, 512);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // both CTAs' barriers exist and both operand areas are cleared
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int rows = p.nb * p.p_rows;  // rows written by TMA per chunk

  if (warp == 0) {
    // TMA producer: the whole warp runs the loop, one elected lane issues (tc_common.cuh: elect_one)
    {
      const bool issuer = elect_one();
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t tx = (uint32_t)rows * 128u * (uint32_t)(co_chunks + p.n_btiles * ci_chunks);
      const uint64_t pol_b = l2_policy(p.l2_hint != 0);
      for (int it = 0; it < n_iters; ++it) {
        const int n0 = (u_begin + it) * p.nb;
        mbar_wait_tight(empty_bar(stage), phase ^ 1u);
        if (issuer) {
          const uint32_t sa = smem_base + stage * p.stage_bytes;
          if (PAIR) {
            const uint32_t fb = full_bar(stage) & TC_PEER_MASK;  // the leader's barrier collects both CTAs' bytes
            if (lead) mbar_arrive_expect_tx(full_bar(stage), 2u * tx);
            for (int c = 0; c < co_chunks; ++c) tma_load_4d_2sm(sa + c * WG_CHUNK_A, &tm_a, fb, co0 + c * 64, 0, p.a_start, n0);
            for (int b = 0; b < p.n_btiles; ++b)
              tma_load_4d_2sm_pol(sa + p.a_bytes + b * p.b_bytes, &tm_b, fb, ci0 + (int)rank * 64, p.b_plane[b], p.b_start[b], n0,
                                  pol_b);
          } else {
            mbar_arrive_expect_tx(full_bar(stage), tx);
            for (int c = 0; c < co_chunks; ++c) tma_load_4d(sa + c * WG_CHUNK_A, &tm_a, full_bar(stage), co0 + c * 64, 0, p.a_start, n0);
            for (int b = 0; b < p.n_btiles; ++b) {
              const uint32_t sb = sa + p.a_bytes + b * p.b_bytes;
              for (int c = 0; c < ci_chunks; ++c)
                tma_load_4d_pol(sb + c * WG_CHUNK_B, &tm_b, full_bar(stage), ci0 + c * 64, p.b_plane[b], p.b_start[b], n0, pol_b);
            }
          }
        }
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1 && NT == 7) {
    const bool issuer = elect_one();
    // D=f32, A=B=bf16, both MN-major, N = 64, M = 128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) |
                           ((uint32_t)(128 >> 4) << 24);
    const uint64_t a_tmpl = make_sw128_desc(0, WG_CHUNK_A >> 4, 1024 >> 4, 1, 0);
    const uint64_t b_tmpl = make_sw128_desc(0, WG_CHUNK_B >> 4, 1024 >> 4, 1, 0);
    const uint32_t a_hi = (uint32_t)(a_tmpl >> 32), b_hi = (uint32_t)(b_tmpl >> 32);
    const int k_steps = p.r_pad / 16;
    const uint32_t stage16 = (uint32_t)p.stage_bytes >> 4;
    const uint32_t s16_0 = (smem_base & 0x3FFFFu) >> 4;
    uint32_t s16 = s16_0, fb = full_bar(0), eb = empty_bar(0);
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0; it < n_iters; ++it) {
      mbar_wait_tight(fb, phase);
      tc_fence_after();
      if (issuer) {
        uint32_t a_lo = (uint32_t)a_tmpl + s16;
        uint32_t b[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t)
          b[t] = (uint32_t)b_tmpl + s16 + ((uint32_t)(p.a_bytes + ((t & 1) ? 0 : p.b_bytes) + ((t + 1) >> 1) * 128) >> 4);
        uint32_t acc = it != 0 ? 1u : 0u;
        for (int kk = 0; kk < k_steps; ++kk) {
#pragma unroll
          for (int t = 0; t < NT; ++t) {
            umma_bf16_lo2(tmem_base + (uint32_t)(t * 64), a_lo, a_hi, b[t], b_hi, idesc, acc);
            b[t] += 128;
          }
          a_lo += 128;
          acc = 1u;
        }
        umma_commit(eb);
      }
      s16 += stage16; fb += 8; eb += 8;
      if (++stage == p.stages) {
        stage = 0; phase ^= 1u; s16 = s16_0; fb = full_bar(0); eb = empty_bar(0);
      }
    }
    if (issuer) umma_commit(done_bar);
  } else if (warp == 1) {
    // MMA issuer: whole warp, one elected lane issues; all descriptor arithmetic on the 32-bit low words
    if (!PAIR || lead) {
      const bool issuer = elect_one();
      // instruction descriptor: D=f32, A=B=bf16, A and B MN-major (bits 15, 16), N = ci_n, M = 128 (256 over a CTA pair)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                             ((uint32_t)(ci_n >> 3) << 17) | ((uint32_t)((PAIR ? 256 : 128) >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      const int k_steps = p.r_pad / 16;
      // Descriptors are built ONCE: everything but the 14-bit start-address field is loop-invariant, and the
      // start only moves by multiples of 16 bytes, so advancing is a single 32-bit add on the low word (the high words
      // of the three descriptor kinds differ only in LBO / base offset, which live in the low / high halves as below)
      const uint64_t a_tmpl = make_sw128_desc(0, WG_CHUNK_A >> 4, 1024 >> 4, 1, 0);
      uint64_t b_tmpl[WG_MAX_TAPS];
      uint32_t d_tmem[WG_MAX_TAPS];
#pragma unroll
      for (int t = 0; t < WG_MAX_TAPS; ++t) {
        const uint32_t off = p.a_bytes + p.tap_btile[t] * p.b_bytes + p.tap_shift[t] * 128;
        const uint32_t bo = p.base_offset_mode == 0 ? (uint32_t)(p.tap_shift[t] & 7) : 0u;
        b_tmpl[t] = make_sw128_desc(0, WG_CHUNK_B >> 4, 1024 >> 4, 1, bo) + (uint64_t)(off >> 4);
        d_tmem[t] = tmem_base + (uint32_t)t * 128u;
      }
      const int n_taps = p.n_taps;
      // fused taps: N = 192, chunk stride (LBO) = one 128-byte row
      const uint32_t idesc_f = (idesc & ~(0x3Fu << 17)) | ((uint32_t)(192 >> 3) << 17);
      const uint64_t bf_tmpl = make_sw128_desc(0, 128 >> 4, 1024 >> 4, 1, 0) + (uint64_t)(p.a_bytes >> 4);
      const uint32_t a_hi = (uint32_t)(a_tmpl >> 32), bf_hi = (uint32_t)(bf_tmpl >> 32);
      const uint32_t b_hi0 = (uint32_t)(b_tmpl[0] >> 32), b_hi1 = (uint32_t)(b_tmpl[1] >> 32), b_hi2 = (uint32_t)(b_tmpl[2] >> 32);
      const uint32_t stage16 = (uint32_t)p.stage_bytes >> 4;
      // the descriptors' 14-bit address field is CTA-relative: drop the cluster-rank bits of the shared-window address
      const uint32_t s16_0 = (smem_base & 0x3FFFFu) >> 4;
      uint32_t s16 = s16_0, fb = full_bar(0), eb = empty_bar(0);
      for (int it = 0; it < n_iters; ++it) {
        mbar_wait_tight(fb, phase);
        tc_fence_after();
        if (issuer) {
          uint32_t a_lo = (uint32_t)a_tmpl + s16;
          uint32_t b0 = (uint32_t)b_tmpl[0] + s16, b1 = (uint32_t)b_tmpl[1] + s16, b2 = (uint32_t)b_tmpl[2] + s16;
          uint32_t acc = it != 0 ? 1u : 0u;
          if (p.fuse_taps) {
            uint32_t bf = (uint32_t)bf_tmpl + s16;
#pragma unroll 4
            for (int kk = 0; kk < k_steps; ++kk) {
              umma_bf16_lo2(d_tmem[0], a_lo, a_hi, bf, bf_hi, idesc_f, acc);
              a_lo += 128; bf += 128;
              acc = 1u;
            }
          } else if (PAIR) {
            if (n_taps == 3) {
#pragma unroll 4
              for (int kk = 0; kk < k_steps; ++kk) {
                umma2_bf16_lo2(d_tmem[0], a_lo, a_hi, b0, b_hi0, idesc, acc);
                umma2_bf16_lo2(d_tmem[1], a_lo, a_hi, b1, b_hi1, idesc, acc);
                umma2_bf16_lo2(d_tmem[2], a_lo, a_hi, b2, b_hi2, idesc, acc);
                a_lo += 128; b0 += 128; b1 += 128; b2 += 128;
                acc = 1u;
              }
            } else {
#pragma unroll 4
              for (int kk = 0; kk < k_steps; ++kk) {
                umma2_bf16_lo2(d_tmem[0], a_lo, a_hi, b0, b_hi0, idesc, acc);
                a_lo += 128; b0 += 128;
                acc = 1u;
              }
            }
          } else if (n_taps == 3) {
#pragma unroll 4
            for (int kk = 0; kk < k_steps; ++kk) {
              umma_bf16_lo2(d_tmem[0], a_lo, a_hi, b0, b_hi0, idesc, acc);
              umma_bf16_lo2(d_tmem[1], a_lo, a_hi, b1, b_hi1, idesc, acc);
              umma_bf16_lo2(d_tmem[2], a_lo, a_hi, b2, b_hi2, idesc, acc);
              a_lo += 128; b0 += 128; b1 += 128; b2 += 128;  // 16 reduction rows = 2048 bytes
              acc = 1u;
            }
          } else {
#pragma unroll 4
            for (int kk = 0; kk < k_steps; ++kk) {
              umma_bf16_lo2(d_tmem[0], a_lo, a_hi, b0, b_hi0, idesc, acc);
              a_lo += 128; b0 += 128;
              acc = 1u;
            }
          }
          if (PAIR) umma2_commit_mc(eb, 3u);
          else umma_commit(eb);
        }
        s16 += stage16; fb += 8; eb += 8;
        if (++stage == p.stages) {
          stage = 0; phase ^= 1u; s16 = s16_0; fb = full_bar(0); eb = empty_bar(0);
        }
      }
      if (issuer) {
        if (PAIR) umma2_commit_mc(done_bar, 3u);
        else umma_commit(done_bar);
      }
    }
  } else if (p.accumulate_l2) {
    // epilogue, accumulate mode: the fp32 tile of every tap goes through shared memory (the operand ring is idle once the
    // last MMA has completed) as 128 x 32 sub-tiles in the TMA's SWIZZLE_128B layout -- thread = output channel = row, its
    // 16-byte chunk j lands at chunk j ^ (row & 7), so the 32 rows of a warp spread over all banks -- and is ADDED into
    // dw_t[t][co][ci] by cp.reduce.async.bulk at the L2.  143 CTAs x 196 KB of split-K partials no longer travel to HBM and
    // back, and there is no reduce kernel; the order of the fp32 additions is the arrival order (not bit-reproducible).
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const bool leader = (threadIdx.x == 64);
    if (n_iters > 0) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
      const int n_sub = ci_n / 32;
      for (int t = 0; t < p.n_taps; ++t) {
        if (t > 0) {
          if (leader) tma_store_wait_read();          // the previous tap's reduce operations have read the staging tiles
          named_bar_sync(1, 128);
        }
        for (int sb = 0; sb < n_sub; ++sb) {
          uint32_t v[32];
          tmem_ld16(t_row + (uint32_t)(t * p.tap_cols + sb * 32), *reinterpret_cast<uint32_t(*)[16]>(v));
          tmem_ld16(t_row + (uint32_t)(t * p.tap_cols + sb * 32 + 16), *reinterpret_cast<uint32_t(*)[16]>(v + 16));
          tmem_ld_wait();
          uint8_t* tile = smem_gen + sb * 16384 + row * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(tile + ((j ^ (row & 7)) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
        fence_proxy_async();
        named_bar_sync(1, 128);
        if (leader) {
          for (int sb = 0; sb < n_sub; ++sb) tma_reduce_add_3d(&tm_d, smem_base + sb * 16384, ci0 + sb * 32, co0, t);
          tma_store_commit();
        }
      }
      if (leader) tma_store_wait_all();
    }
  } else {
    // epilogue: partial[split][t][co][ci] (fp32); thread = output channel, 16 input channels per TMEM load
    const int quarter = warp & 3;
    const int co = co0 + quarter * 32 + lane;
    if (n_iters > 0) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
    }
    const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
    for (int t = 0; t < p.n_taps; ++t) {
      float* dst = partial + (((size_t)split * p.n_taps + t) * p.c_out + co) * p.c_in + ci0;
      for (int c0 = 0; c0 < ci_n; c0 += 32) {  // ci_n is 64 or 128: two 16-column TMEM loads per wait
        uint32_t v[32];
        if (n_iters > 0) {
          tmem_ld16(t_row + (uint32_t)(t * p.tap_cols) + (uint32_t)c0, *reinterpret_cast<uint32_t(*)[16]>(v));
          tmem_ld16(t_row + (uint32_t)(t * p.tap_cols) + (uint32_t)c0 + 16u, *reinterpret_cast<uint32_t(*)[16]>(v + 16));
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
        if (co < p.c_out) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            if (ci0 + c0 + j < p.c_in)  // c_in is a multiple of 16
              *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                     __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();  // the partner may still signal this CTA's barriers / read its operands until here
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}

template <bool PAIR>
__global__ void __launch_bounds__(WG_TC_THREADS, 1)
    tc_wgrad_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                    const __grid_constant__ CUtensorMap tm_d, float* __restrict__ partial, const WgTcParams p) {
  tc_wgrad_body<PAIR, WG_MAX_TAPS>(tm_a, tm_b, tm_d, partial, p);
}

__global__ void __launch_bounds__(WG_TC_THREADS, 1)
    tc_wgrad7_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b,
                     const __grid_constant__ CUtensorMap tm_d, float* __restrict__ partial, const WgTcParams p) {
  tc_wgrad_body<false, 7>(tm_a, tm_b, tm_d, partial, p);
}

// dw[co][ci][t] (+)= sum_s partial[s][t][co][ci].  256 threads = (256 / LANES) float4 columns x LANES split lanes; every
// lane sums its splits in order and the lane sums are combined in a fixed order -> deterministic.  LANES follows the
// split count so that every thread has ~8-16 independent 16-byte loads in flight: with 9 splits (C = 512) one lane per
// column reads all of them at once, with 143 splits (C <= 128) eight lanes read 18 each.
template <int LANES>
__global__ void __launch_bounds__(256) tc_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw,
                                                              int splits, int ktaps, int c_in, int c_out, int accumulate) {
  constexpr int COLS = 256 / LANES;
  __shared__ float4 red[LANES][COLS + 1];
  const int per = ktaps * c_in * c_out;  // multiple of 4 (c_in % 16 == 0)
  const int col = threadIdx.x % COLS, ln = threadIdx.x / COLS;
  const int i = (blockIdx.x * COLS + col) * 4;  // index into [t][co][ci], ci fastest
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < per) {
#pragma unroll 8
    for (int k = ln; k < splits; k += LANES) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(partial + (size_t)k * per + i));
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  }
  if (LANES > 1) {
    red[ln][col] = s;
    __syncthreads();
  }
  if (ln == 0 && i < per) {
    float4 t = s;
    if (LANES > 1) {
#pragma unroll
      for (int k = 1; k < LANES; ++k) {
        const float4 v = red[k][col];
        t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
      }
    }
    const int ci = i % c_in, co = (i / c_in) % c_out, tap = i / (c_in * c_out);
    float* o = dw + ((size_t)co * c_in + ci) * ktaps + tap;
    const float r[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j * ktaps] = accumulate ? o[j * ktaps] + r[j] : r[j];
  }
}

struct WgPlan {
  WgTcParams p;
  int splits;
  bool ok;
};

static WgPlan wg_plan(int n_breaths, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride, int pad) {
  WgPlan w{};
  w.ok = false;
  WgTcParams& p = w.p;
  const bool k7 = ktaps == 7 && pad == 3 && stride == 2;  // tc_wgrad7_kernel
  if (!((ktaps == 3 && pad == 1) || (ktaps == 1 && pad == 0) || k7)) return w;
  if (stride != 1 && stride != 2) return w;
  if (c_in % 16 || c_out % 8 || l_in != l_out * stride) return w;
  if (k7 && (c_in > 64 || g_dbg_base_offset_mode == 0)) return w;  // 7 x 64 TMEM columns; base offset 0 only
  const int halo = ktaps == 3 ? 1 : 0;
  p.p_rows = l_out + halo;     // dout rows [0, L] (row L = zero fill), input rows [-1, L-1] (row -1 = zero fill)
  p.a_start = 0;
  p.n_taps = ktaps;
  if (k7) {
    // dout rows [0, L+2] (3 zero rows), both parity planes staged from row -2 (two zero rows); the tap map is in the kernel
    p.p_rows = l_out + 3;
    p.n_btiles = 2;
    p.b_plane[0] = 0; p.b_start[0] = -2;
    p.b_plane[1] = 1; p.b_start[1] = -2;
  } else if (stride == 1) {
    p.n_btiles = 1;
    p.b_plane[0] = 0;
    p.b_start[0] = -halo;  // staged row i = in[i - 1]; tap t of dout row j pairs with staged row j + t
    for (int t = 0; t < ktaps; ++t) {
      p.tap_btile[t] = 0;
      p.tap_shift[t] = t;
    }
  } else if (ktaps == 3) {
    // in[2q + t - 1]: t = 1 -> plane 0 row q; t = 0 -> plane 1 row q-1; t = 2 -> plane 1 row q
    p.n_btiles = 2;
    p.b_plane[0] = 0; p.b_start[0] = 0;   // staged row i = plane0[i]: dout row q pairs with row q
    p.b_plane[1] = 1; p.b_start[1] = -1;  // staged row i = plane1[i - 1]: tap 0 -> row q, tap 2 -> row q + 1
    p.tap_btile[0] = 1; p.tap_shift[0] = 0;
    p.tap_btile[1] = 0; p.tap_shift[1] = 0;
    p.tap_btile[2] = 1; p.tap_shift[2] = 1;
  } else {
    p.n_btiles = 1;
    p.b_plane[0] = 0; p.b_start[0] = 0;
    p.tap_btile[0] = 0; p.tap_shift[0] = 0;
  }
  p.nb = WG_RMAX / p.p_rows;
  if (p.nb < 1) return w;
  if (p.nb > 256) p.nb = 256;
  p.r_pad = (p.nb * p.p_rows + 15) / 16 * 16;
  p.n_units = ceil_div(n_breaths, p.nb);
  p.c_in = c_in; p.c_out = c_out;
  p.n_ci_tiles = ceil_div(c_in, 128);
  p.n_co_tiles = ceil_div(c_out, 128);
  // a stage holds 1 or 2 64-channel chunks of each operand: narrow layers get a deeper ring out of the same shared
  // memory (they are load-latency bound: the reduction streams activations straight from HBM)
  p.fuse_taps = (ktaps == 3 && stride == 1 && c_in == 64 && g_dbg_wgrad_fuse != 0) ? 1 : 0;
  p.pair = (g_dbg_wgrad_pair != 0 && c_out % 256 == 0 && c_in % 128 == 0 && !p.fuse_taps) ? 1 : 0;
  p.a_bytes = (c_out > 64 ? 2 : 1) * WG_CHUNK_A;
  p.b_bytes = (c_in > 64 && !p.pair ? 2 : 1) * WG_CHUNK_B;
  p.stage_bytes = p.a_bytes + p.n_btiles * p.b_bytes;
  p.stages = (WG_SMEM_LIMIT - 2048) / p.stage_bytes;
  if (p.stages > WG_MAX_STAGES) p.stages = WG_MAX_STAGES;
  if (p.stages < 2) return w;
  const int tiles = p.n_ci_tiles * p.n_co_tiles;
  // exactly one wave: tiles * splits <= #SMs (1 CTA per SM: ~200 KB of shared memory each), so no tail wave
  int splits = tiles >= sm_count() ? 1 : sm_count() / tiles;
  const int max_by_units = (p.n_units + 3) / 4;       // at least 4 reduction units per CTA
  if (splits > max_by_units) splits = max_by_units;
  if (splits < 1) splits = 1;
  p.units_per_split = ceil_div(p.n_units, splits);
  w.splits = ceil_div(p.n_units, p.units_per_split);
  // Measured on B200 (tools/tc_probe.py, profiles/r01_tc_probe.txt): the 128B swizzle is applied to ABSOLUTE shared
  // memory address bits, so a descriptor whose start is advanced by whole 128-byte rows needs base_offset = 0;
  // base_offset = (start >> 7) & 7 gives wrong results for the shifted taps.
  p.base_offset_mode = g_dbg_base_offset_mode >= 0 ? g_dbg_base_offset_mode : 1;
  p.tap_cols = p.fuse_taps || k7 ? 64 : 128;
  p.l2_hint = g_dbg_l2_hint != 0 ? 1 : 0;
  w.ok = true;
  return w;
}

static int wg_launch(WgPlan& w, const void* in, const void* dout, float* partial, float* dw_t, int n_breaths, int l_in,
                     int l_out, int c_in, int c_out, int in_stride, int dout_stride, int ktaps, int stride, cudaStream_t st);

// dw_t[t][co][ci] += ... : accumulate mode (the buffer must be zeroed by the caller once per backward pass)
int tc_conv_wgrad_accum(const void* in, const void* dout, float* dw_t, int n_breaths, int l_in, int l_out, int c_in, int c_out,
                        int in_stride, int dout_stride, int ktaps, int stride, int pad, cudaStream_t st) {
  WgPlan w = wg_plan(n_breaths, l_in, l_out, c_in, c_out, ktaps, stride, pad);
  if (!w.ok) {
    set_error("tcgen05 wgrad: unsupported shape (k=%d s=%d p=%d cin=%d cout=%d l=%d)", ktaps, stride, pad, c_in, c_out, l_in);
    return DARDS_ERR_UNSUPPORTED;
  }
  DARDS_CHECK_ARG(in_stride % 8 == 0 && dout_stride % 8 == 0, "tcgen05 wgrad: row strides must be multiples of 8");
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(dw_t) & 15) == 0,
                  "tcgen05 wgrad: operands must be 16-byte aligned");
  DARDS_CHECK_ARG(c_in % 32 == 0, "tcgen05 wgrad (accumulate): input channels must be a multiple of 32");
  w.p.accumulate_l2 = 1;
  return wg_launch(w, in, dout, nullptr, dw_t, n_breaths, l_in, l_out, c_in, c_out, in_stride, dout_stride, ktaps, stride, st);
}

long long tc_wgrad_workspace_bytes(int n_breaths, int l_out, int c_in, int c_out, int ktaps) {
  // the split count depends on the rows staged per breath: the stride-1 plan shape gives them for k = 1 and 3; k = 7 has
  // one plan only (stride 2, pad 3)
  WgPlan w = ktaps == 7 ? wg_plan(n_breaths, 2 * l_out, l_out, c_in, c_out, 7, 2, 3)
                        : wg_plan(n_breaths, l_out, l_out, c_in, c_out, ktaps, 1, ktaps == 3 ? 1 : 0);
  if (!w.ok) return 0;
  return (long long)w.splits * ktaps * c_in * c_out * (long long)sizeof(float);
}

static int wg_launch(WgPlan& w, const void* in, const void* dout, float* partial, float* dw_t, int n_breaths, int l_in,
                     int l_out, int c_in, int c_out, int in_stride, int dout_stride, int ktaps, int stride, cudaStream_t st) {
  WgTcParams& p = w.p;
  CUtensorMap tm_a, tm_b, tm_d;
  if (dw_t) {
    cuuint64_t dims[3] = {(cuuint64_t)c_in, (cuuint64_t)c_out, (cuuint64_t)ktaps};
    cuuint64_t str[2] = {(cuuint64_t)c_in * 4, (cuuint64_t)c_in * c_out * 4};
    cuuint32_t box[3] = {32, 128, 1};
    int rc = make_f32_map(&tm_d, dw_t, 3, dims, str, box, true);
    if (rc) return rc;
  } else {
    memset(&tm_d, 0, sizeof(tm_d));
  }
  {
    cuuint64_t dims[4] = {(cuuint64_t)c_out, 1, (cuuint64_t)l_out, (cuuint64_t)n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)dout_stride * 2, (cuuint64_t)dout_stride * 2, (cuuint64_t)dout_stride * l_out * 2};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)p.p_rows, (cuuint32_t)p.nb};
    int rc = make_bf16_map(&tm_a, dout, 4, dims, str, box, true);
    if (rc) return rc;
  }
  {
    const int l_plane = l_in / stride;
    cuuint64_t dims[4] = {(cuuint64_t)c_in, (cuuint64_t)stride, (cuuint64_t)l_plane, (cuuint64_t)n_breaths};
    cuuint64_t str[3] = {(cuuint64_t)in_stride * 2, (cuuint64_t)in_stride * stride * 2, (cuuint64_t)in_stride * l_in * 2};
    cuuint32_t box[4] = {64, 1, (cuuint32_t)p.p_rows, (cuuint32_t)p.nb};
    int rc = make_bf16_map(&tm_b, in, 4, dims, str, box, true);
    if (rc) return rc;
  }
  const int smem = p.stages * p.stage_bytes + 1024 + 256;
  dim3 grid(p.n_ci_tiles * p.n_co_tiles, w.splits);
  if (p.n_taps == 7) {
    static int attr_smem7 = 0;
    if (smem > attr_smem7) {
      cudaError_t e = cudaFuncSetAttribute(tc_wgrad7_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
      if (e != cudaSuccess) {
        set_error("tcgen05 wgrad (7 taps): cannot opt in to %d bytes of shared memory: %s", smem, cudaGetErrorString(e));
        return DARDS_ERR_CUDA;
      }
      attr_smem7 = smem;
    }
    tc_wgrad7_kernel<<<grid, WG_TC_THREADS, smem, st>>>(tm_a, tm_b, tm_d, partial, p);
    DARDS_CHECK_LAUNCH("tc_wgrad7");
    return DARDS_OK;
  }
  static int attr_smem[2] = {0, 0};
  if (smem > attr_smem[p.pair]) {
    cudaError_t e = p.pair ? cudaFuncSetAttribute(tc_wgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)
                           : cudaFuncSetAttribute(tc_wgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) {
      set_error("tcgen05 wgrad: cannot opt in to %d bytes of shared memory: %s", smem, cudaGetErrorString(e));
      return DARDS_ERR_CUDA;
    }
    attr_smem[p.pair] = smem;
  }
  if (p.pair) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;                 // grid.x is even (c_out % 256 == 0): clusters of 2 along x share blockIdx.y
    cfg.blockDim = dim3(WG_TC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, tc_wgrad_kernel<true>, tm_a, tm_b, tm_d, partial, p);
    if (e != cudaSuccess) {
      set_error("tcgen05 wgrad (CTA pairs): launch failed: %s", cudaGetErrorString(e));
      return DARDS_ERR_CUDA;
    }
    count_launch();
    return DARDS_OK;
  }
  tc_wgrad_kernel<false><<<grid, WG_TC_THREADS, smem, st>>>(tm_a, tm_b, tm_d, partial, p);
  DARDS_CHECK_LAUNCH("tc_wgrad");
  return DARDS_OK;
}


int tc_conv_wgrad(const void* in, const void* dout, float* dw, int accumulate, void* workspace, long long workspace_bytes,
                  int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride, int dout_stride, int ktaps,
                  int stride, int pad, cudaStream_t st) {
  WgPlan w = wg_plan(n_breaths, l_in, l_out, c_in, c_out, ktaps, stride, pad);
  if (!w.ok) {
    set_error("tcgen05 wgrad: unsupported shape (k=%d s=%d p=%d cin=%d cout=%d l=%d)", ktaps, stride, pad, c_in, c_out, l_in);
    return DARDS_ERR_UNSUPPORTED;
  }
  DARDS_CHECK_ARG(in_stride % 8 == 0 && dout_stride % 8 == 0, "tcgen05 wgrad: row strides must be multiples of 8");
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(dout) & 15) == 0,
                  "tcgen05 wgrad: operands must be 16-byte aligned");
  const long long need = (long long)w.splits * ktaps * c_in * c_out * (long long)sizeof(float);
  DARDS_CHECK_ARG(workspace != nullptr && workspace_bytes >= need, "tcgen05 wgrad: workspace too small (%lld < %lld)",
                  workspace_bytes, need);
  w.p.accumulate_l2 = 0;
  int rc = wg_launch(w, in, dout, static_cast<float*>(workspace), nullptr, n_breaths, l_in, l_out, c_in, c_out, in_stride,
                     dout_stride, ktaps, stride, st);
  if (rc) return rc;
  const int per = ktaps * c_in * c_out;
  const float* part = static_cast<const float*>(workspace);
  if (w.splits <= 16)
    tc_wgrad_reduce_kernel<1><<<ceil_div(per, 4 * 256), 256, 0, st>>>(part, dw, w.splits, ktaps, c_in, c_out, accumulate);
  else if (w.splits <= 48)
    tc_wgrad_reduce_kernel<4><<<ceil_div(per, 4 * 64), 256, 0, st>>>(part, dw, w.splits, ktaps, c_in, c_out, accumulate);
  else
    tc_wgrad_reduce_kernel<8><<<ceil_div(per, 4 * 32), 256, 0, st>>>(part, dw, w.splits, ktaps, c_in, c_out, accumulate);
  DARDS_CHECK_LAUNCH("tc_wgrad_reduce");
  return DARDS_OK;
}

}  // namespace dards

/*
 * deepards_b200 -- C ABI of the B200 (sm_100a) backend for the deepards cnn_linear hot path.
 *
 * The reference (hahnicity/deepards) has NO native interface: its extension points are two
 * Python dicts, `base_networks` (deepards/train_ards_detector.py:45-69) and `network_map`
 * (deepards/train_ards_detector.py:1410-1436), and all arithmetic is torch.nn library calls.
 * This header is therefore the boundary that the replacement Python modules
 * (deepards_b200/resnet.py, densenet.py, torch_cnn_linear_network.py -- same names, ctor
 * signatures and state_dict keys as deepards/models/*) bind with ctypes; every entry point
 * cites the torch.nn call site in the reference that it replaces.
 *
 * Conventions
 *  - Plain C symbols, raw DEVICE pointers, int sizes, a dtype enum and a cudaStream_t passed
 *    as void*.  No torch types.  All buffers are owned by the caller (PyTorch's caching
 *    allocator); the library never allocates, frees or retains device memory.
 *  - Every function only ENQUEUES work on `stream` and returns; no implicit synchronisation.
 *  - Return value: DARDS_OK (0) or a negative dards_status; dards_last_error() gives the
 *    message of the last failure on the calling thread.  Nothing throws or aborts.
 *  - Activation layout: channels-last.  A tensor the reference holds as (N, C, L) lives here
 *    as (N, L, C) with a row stride `*_stride` >= C (in elements), so that a channel slice
 *    of a wider buffer (DenseNet concatenation, densenet.py:40) is addressable in place.
 *    `dtype` is the storage type of ACTIVATIONS and packed weights (fp32 or bf16); all
 *    accumulation, BatchNorm statistics, parameters and parameter gradients are fp32.
 *  - "group": BatchNorm statistics are taken over `group` consecutive breaths (20 = one
 *    sequence; deepards/models/torch_cnn_linear_network.py:104-113 calls the backbone once
 *    per sequence), i.e. over group*L rows per channel.
 */
#ifndef DEEPARDS_B200_H_
#define DEEPARDS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum dards_status {
  DARDS_OK = 0,
  DARDS_ERR_INVALID_ARGUMENT = -1,
  DARDS_ERR_CUDA = -2,
  DARDS_ERR_UNSUPPORTED = -3
} dards_status;

typedef enum dards_dtype { DARDS_F32 = 0, DARDS_BF16 = 1 } dards_dtype;

/* Optional flag, OR-ed into the `impl` argument of dards_conv1d_fwd / dards_conv1d_dgrad and into the `relu` argument of
 * dards_gbn_fwd: the source activation tensor of this call is not read again before it would leave the L2 anyway (its
 * last use in the forward or in the backward pass).  Kernels that read every source byte once load it with L2
 * evict_first priority, so that it does not displace tensors the following kernels re-read.  Purely a performance hint. */
#define DARDS_HINT_LAST_USE 0x100

/* ---- library ---------------------------------------------------------------------- */
int dards_version(void);                 /* ABI version, bumped on any signature change */
const char* dards_last_error(void);      /* thread-local, never NULL */
/* number of kernels this library has launched so far in this process (bench.py's gpu_launches) */
long long dards_launch_count(void);
/* 1 if the device behind the current context is compute capability 10.x (B200). */
int dards_device_supported(void);

/* Persistent kernels launch one CTA per SM.  n_sms > 0 makes them size their grids for n_sms SMs instead (0 restores
 * the device count): a data-parallel run leaves a few SMs to the NCCL kernels that overlap the backward pass, otherwise
 * every persistent kernel that meets them runs its last CTAs as a second wave. */
int dards_set_sm_limit(int n_sms);

/* ---- weights ---------------------------------------------------------------------- */
/* nn.Conv1d weight (Cout, Cin, K) fp32 [resnet.py:7,88,128; densenet.py:25,30,75,119] ->
 * the two packed forms the kernels read, in `dtype`:
 *   w_kio[t][ci][co]  (reduction over ci, outputs co contiguous)
 *   w_koi[t][co][ci]  (reduction over co, outputs ci contiguous)
 * either output pointer may be NULL. */
int dards_pack_conv_weight(const float* w, void* w_kio, void* w_koi, int c_out, int c_in, int ktaps,
                           int dtype, void* stream);

/* The same for every convolution of a network in ONE launch.  `descs_dev` is a DEVICE array of n_descs
 * descriptors (ktaps <= 8); descriptor j owns the blocks [first_block_j, first_block_j + ceil(c_out/32) *
 * ceil(c_in/32)) -- one 32 x 32 x ktaps tile each -- first_block_0 = 0, and total_blocks is their sum. */
typedef struct dards_pack_desc {
  const float* w;
  void* w_kio;
  void* w_koi;
  int c_out, c_in, ktaps, first_block;
} dards_pack_desc;
int dards_pack_conv_weights_batched(const dards_pack_desc* descs_dev, int n_descs, int total_blocks, int dtype,
                                    void* stream);

/* ---- convolution (nn.Conv1d, bias=False) ------------------------------------------ */
/* Forward: out[n,q,co] = sum_{t,ci} in[n, q*stride + t - pad, ci] * W[co,ci,t]  (+ addend[n,q,co]).
 * `w_packed`: w_kio for impl 0, w_koi for impl 1 (the MMA wants the reduction dim contiguous);
 * `addend` may be NULL.  Replaces nn.Conv1d.forward
 * at resnet.py:27,31,35 and densenet.py:25,30,75 (the stem conv has its own entry point).
 * impl: 0 = CUDA-core fp32-accumulate implicit GEMM (any dtype), 1 = tcgen05 (bf16 only). */
int dards_conv1d_fwd(const void* in, const void* w_packed, void* out, const void* addend, int n_breaths, int l_in,
                     int l_out, int c_in, int c_out, int in_stride, int out_stride, int addend_stride, int ktaps,
                     int stride, int pad, int dtype, int impl, void* stream);

/* Data gradient: din[n,p,ci] = sum_{t,co} dout[n,q,co] * W[co,ci,t] over all (q,t) with
 * q*stride + t - pad == p  (+ addend).  `w_packed`: w_koi for impl 0, w_kio for impl 1.
 * autograd of the calls above. */
int dards_conv1d_dgrad(const void* dout, const void* w_packed, void* din, const void* addend, int n_breaths,
                       int l_in, int l_out, int c_in, int c_out, int dout_stride, int din_stride,
                       int addend_stride, int ktaps, int stride, int pad, int dtype, int impl, void* stream);

/* Weight gradient: dW[co,ci,t] (+)= sum_{n,q} dout[n,q,co] * in[n, q*stride + t - pad, ci], fp32,
 * written in the parameter's own (Cout, Cin, K) layout.  Deterministic: split-K partial sums go to
 * `workspace` (dards_conv1d_wgrad_workspace_bytes) and are reduced in a fixed order. */
int dards_conv1d_wgrad(const void* in, const void* dout, float* dw, int accumulate, void* workspace,
                       long long workspace_bytes, int n_breaths, int l_in, int l_out, int c_in, int c_out,
                       int in_stride, int dout_stride, int ktaps, int stride, int pad, int dtype, int impl,
                       void* stream);
long long dards_conv1d_wgrad_workspace_bytes(int n_breaths, int l_out, int c_in, int c_out, int ktaps, int impl);

/* Accumulate-mode weight gradient (tcgen05, bf16): dw_t[t][co][ci] += sum_{n,q} dout * in -- fp32, TAP-major, added into
 * the buffer by TMA reduce operations at the L2.  No split-K partials travel to memory and no reduce kernel runs (the
 * deterministic entry point above writes and re-reads ~28 MB per layer at the BASELINE shapes); the price is that the
 * order of the fp32 additions is the CTAs' arrival order, so results are not bit-reproducible from run to run.  The
 * caller zeroes dw_t once per backward pass (dards_memset_zero) and converts all layers to the parameter layout
 * (Cout, Cin, K) with ONE dards_unpack_wgrad_batched launch.  c_in % 32 == 0. */
int dards_conv1d_wgrad_accum(const void* in, const void* dout, float* dw_t, int n_breaths, int l_in, int l_out, int c_in,
                             int c_out, int in_stride, int dout_stride, int ktaps, int stride, int pad, int dtype,
                             void* stream);
typedef struct dards_unpack_desc {
  const float* dw_t; /* [ktaps][c_out][c_in] */
  float* dw;         /* [c_out][c_in][ktaps], the nn.Conv1d weight layout */
  int c_out, c_in, ktaps, first_block;
} dards_unpack_desc;
/* descriptor j owns ceil(c_out/32) * ceil(c_in/32) blocks starting at first_block_j; ktaps <= 8 */
int dards_unpack_wgrad_batched(const dards_unpack_desc* descs_dev, int n_descs, int total_blocks, void* stream);
/* cudaMemsetAsync(ptr, 0, bytes) on the stream (capturable; the accumulation buffers of a backward pass) */
int dards_memset_zero(void* ptr, long long bytes, void* stream);

/* ---- convolution with the BatchNorm that follows it, in one kernel (tcgen05, bf16) -------------- */
/* conv -> bn -> relu [-> += residual -> relu] (resnet.py:27-38) and conv -> norm -> relu (densenet.py:25-29):
 * y = conv(in) is stored (the backward needs it); its per-group statistics are taken from the fp32 accumulators in
 * the convolution epilogue.  dards_conv1d_bn_mode() says what the kernel can do for a shape:
 *   2  FUSED: a whole group's output fits on chip; the call also writes
 *        out = [relu](bn(y) [+ res]) and save_mean / save_rstd [n_groups][C]   (no BatchNorm launch at all)
 *   1  PARTIAL: the call writes y and per-tile moments (count, mean, M2) to `part`
 *        ([n_groups * entries][3][C] floats, entries = dards_conv1d_bn_part_entries()); dards_gbn_apply_fwd() below
 *        merges them and does the elementwise normalisation in one streaming pass
 *   0  unsupported (fp32 storage, or the group does not tile): use dards_conv1d_fwd + dards_gbn_fwd.
 * `relu` may carry DARDS_HINT_LAST_USE for `in`.  `out`, `res`, gamma ... save_rstd are unused in mode 1, `part` in
 * mode 2.  n_breaths must be a multiple of `group`. */
int dards_conv1d_bn_mode(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride,
                         int pad, int dtype);
int dards_conv1d_bn_part_entries(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps,
                                 int stride, int pad);
int dards_conv1d_bn_fwd(const void* in, const void* w_koi, void* y, void* out, const void* res, const float* gamma,
                        const float* beta, float* save_mean, float* save_rstd, float* part, int n_breaths, int group,
                        int l_in, int l_out, int c_in, int c_out, int in_stride, int y_stride, int out_stride,
                        int res_stride, int ktaps, int stride, int pad, float eps, int relu, int dtype, void* stream);
/* Mode-1 consumer: out = [relu]( bn(x) [+ res] [+ bn2(x2)] ), statistics merged from `part` (fixed order).  The
 * optional second normalised operand is the downsample branch of a ResNet block (resnet.py:34-38), so
 * relu(bn2(conv2(..)) + bn_d(conv_d(x))) is one pass.  Writes save_mean / save_rstd (and the pair of x2). */
int dards_gbn_apply_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta,
                        const float* part, int entries, float* save_mean, float* save_rstd, const void* x2,
                        const float* gamma2, const float* beta2, const float* part2, int entries2, float* save_mean2,
                        float* save_rstd2, int n_groups, int rows_per_group, int c, int x_stride, int out_stride,
                        int res_stride, int x2_stride, float eps, int relu, int dtype, void* stream);

/* ---- grouped BatchNorm1d (+ residual add, + ReLU) ---------------------------------- */
/* Training-mode nn.BatchNorm1d over groups of `rows_per_group` = group*L rows: biased variance, eps;
 * out = [relu]( (x-mean)*rstd*gamma + beta [+ res] ).  Saves mean/rstd as [n_groups][C] fp32.
 * Replaces bn/relu/"out += residual" at resnet.py:28-29,32,37-38,146-153 and norm/relu at
 * densenet.py:23-24,28-29,73-74,121-122,149,182.  x and out may alias. */
int dards_gbn_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta,
                  float* save_mean, float* save_rstd, int n_groups, int rows_per_group, int c, int x_stride,
                  int out_stride, int res_stride, float eps, int relu, int dtype, void* stream);

/* Backward of the above.  g = dout * relu_mask; dx (+)= gamma*rstd*(g - mean(g) - xhat*mean(g*xhat)).
 * relu_mode: 0 none, 1 recompute mask from x (xhat*gamma+beta > 0), 2 mask = (mask_src > 0).
 * dres (optional) receives g (gradient of the residual branch).  Per-group partial sums
 * dgamma_part/dbeta_part [n_groups][C] are reduced with dards_reduce_rows[_batched]. */
int dards_gbn_bwd(const void* dout, const void* x, const void* mask_src, const float* gamma, const float* beta,
                  const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx, void* dres,
                  float* dgamma_part, float* dbeta_part, int n_groups, int rows_per_group, int c,
                  int dout_stride, int x_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode,
                  int dtype, void* stream);

/* out[c] (+)= sum_r part[r][c]   (fixed order -> deterministic) */
int dards_reduce_rows(const float* part, float* out, int rows, int c, int accumulate, void* stream);
/* The same for a whole table of tensors in ONE launch (all BatchNorm dgamma/dbeta of a backward segment).
 * `descs_dev`: DEVICE array; c % 4 == 0, part/out 16-byte aligned; descriptor j owns ceil(c/64) blocks
 * starting at first_block_j (first_block_0 = 0); total_blocks = their sum. */
typedef struct dards_reduce_desc {
  const float* part;
  float* out;
  int rows, c, accumulate, first_block;
} dards_reduce_desc;
int dards_reduce_rows_batched(const dards_reduce_desc* descs_dev, int n_descs, int total_blocks, void* stream);

/* nn.BatchNorm1d running statistics, updated once per group IN ORDER (momentum, unbiased variance;
 * SURVEY.md hard part 6); num_batches_tracked (int64) += n_groups.  c % 4 == 0. */
int dards_bn_running_update(const float* save_mean, const float* save_rstd, float* running_mean,
                            float* running_var, long long* num_batches_tracked, int n_groups,
                            int rows_per_group, int c, float momentum, float eps, void* stream);
/* The same for every BatchNorm layer of a network in ONE launch (block bookkeeping as above). */
typedef struct dards_running_desc {
  const float* save_mean;
  const float* save_rstd;
  float* running_mean;
  float* running_var;
  long long* num_batches_tracked; /* nullable */
  int n_groups, rows_per_group, c;
  float momentum;
  int first_block, reserved;
} dards_running_desc;
int dards_bn_running_update_batched(const dards_running_desc* descs_dev, int n_descs, int total_blocks, float eps,
                                    void* stream);

/* ---- eval-mode BatchNorm (running statistics) ------------------------------------------ */
/* nn.BatchNorm1d in eval() is a fixed per-channel affine map y*scale[c] + shift[c].  For every layer of a network in ONE
 * launch:  scale = gamma / sqrt(running_var + eps),  shift = beta - running_mean * scale  (fp32).  Descriptor j owns
 * ceil(c/64) blocks starting at first_block_j (first_block_0 = 0); total_blocks is their sum.  Meant to run at the start
 * of every eval forward: the running buffers may have been edited in place since the last one. */
typedef struct dards_eval_coeff_desc {
  const float* gamma;
  const float* beta;
  const float* running_mean;
  const float* running_var;
  float* scale;
  float* shift;
  int c, first_block;
} dards_eval_coeff_desc;
int dards_bn_eval_coeffs_batched(const dards_eval_coeff_desc* descs_dev, int n_descs, int total_blocks, float eps,
                                 void* stream);

/* Convolution with eval-mode BatchNorm, residual add and ReLU in its epilogue (resnet.py:27-38 under eval()):
 *   out[n,q,co] = [relu]( conv(in)[n,q,co] * scale[co] + shift[co] [+ res[n,q,co]] )
 * computed in fp32 on the accumulator and rounded to the storage type once.  `res` may be NULL and must not overlap
 * `out`; `relu` is 0 or 1 and may carry DARDS_HINT_LAST_USE for `in`.  Shapes, strides and `w_packed` as for
 * dards_conv1d_fwd: impl 0 = CUDA cores (fp32 or bf16), impl 1 = tcgen05 (bf16). */
int dards_conv1d_affine_fwd(const void* in, const void* w_packed, void* out, const void* res, const float* scale,
                            const float* shift, int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride,
                            int out_stride, int res_stride, int ktaps, int stride, int pad, int relu, int dtype, int impl,
                            void* stream);

/* ---- BatchNorm with constant statistics under training (frozen BatchNorm) ------------- */
/* A network in train() whose nn.BatchNorm1d layers are in eval() (the usual fine-tuning idiom, resnet.py:27-38 and
 * 146-153 with running statistics): the forward is the eval-mode affine map, and the backward reaches gamma, beta and
 * the convolutions through it.
 * Elementwise forward: out = [relu]( y*scale[c] + shift[c] [+ res] [+ y2*scale2[c] + shift2[c]] ) over `rows` rows,
 * in fp32, rounded once; scale / shift as from dards_bn_eval_coeffs_batched.  The second operand is the downsample
 * branch of a ResNet block (resnet.py:34-38), so relu(bn2(y2) + bn_d(y_d)) is one pass.  fp32 or bf16; c and every
 * stride a multiple of 4 (fp32) / 8 (bf16), tensors 16-byte aligned; `out` must not overlap y, res or y2. */
int dards_bn_affine_apply(const void* y, void* out, const void* res, const float* scale, const float* shift,
                          const void* y2, const float* scale2, const float* shift2, int rows, int c, int y_stride,
                          int out_stride, int res_stride, int y2_stride, int relu, int dtype, void* stream);
/* Its backward, rows split into n_tiles tiles of rows_per_tile rows (any split: tiles only shape the partial sums):
 *   g = dout [* (mask)]    relu_mode 0: none, 1: y*scale + shift > 0 (recomputed), 2: mask_src > 0
 *   dres (optional) = g;   dx (+)= g * scale     (scale = gamma * rstd: no mean-of-gradient terms)
 *   dbeta_part[t][c] = sum over tile t of g,   dgamma_part[t][c] = sum over tile t of g * (y - running_mean) * rstd
 * with rstd = 1/sqrt(running_var + eps), which dards_bn_eval_coeffs_batched computes as `scale` for gamma = 1, beta = 0.
 * The partials are summed with dards_reduce_rows[_batched] (fixed order: deterministic).  dx may alias dout. */
int dards_bn_frozen_bwd(const void* dout, const void* y, const void* mask_src, const float* scale, const float* shift,
                        const float* running_mean, const float* rstd, void* dx, int accumulate_dx, void* dres,
                        float* dgamma_part, float* dbeta_part, int n_tiles, int rows_per_tile, int c, int dout_stride,
                        int y_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype,
                        void* stream);

/* ---- stem: Conv1d(1->C0,k7,s2,p3) + BN + ReLU + Max/AvgPool1d(3,2,1) ---------------- */
/* resnet.py:143-153 / densenet.py:119-123 fused: x (N,224) fp32 -> out (N,56,C0).  Nothing but the
 * group statistics is saved; the backward recomputes the convolution from x. pool: 0 max, 1 avg.
 * A BatchNorm group of up to 226 breaths (the sequence heads use 20) is one kernel and needs no workspace.  Larger groups
 * -- a flat batch through ResNet.forward / DenseNet.forward / CNNRegressor is ONE group (resnet.py:141-163) -- run in
 * chunks of 64 breaths through two passes and need `workspace` of dards_stem_workspace_bytes(...) bytes (0 otherwise;
 * the pointer may then be NULL). */
long long dards_stem_workspace_bytes(int n_groups, int group, int c0, int backward);
int dards_stem_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out,
                   float* save_mean, float* save_rstd, int n_groups, int group, int c0, int out_stride,
                   float eps, int pool, void* workspace, long long workspace_bytes, int dtype, void* stream);
/* Eval-mode stem: conv -> y*scale[c] + shift[c] (dards_bn_eval_coeffs_batched) -> ReLU -> pool, x (N,224) fp32 ->
 * out (N,56,C0).  Every breath is independent of the others: any n_breaths >= 1, no workspace. */
int dards_stem_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out, int n_breaths,
                        int c0, int out_stride, int pool, int dtype, void* stream);
/* Backward of dards_stem_eval_fwd for a network in train() with the stem's BatchNorm in eval(): dout (N,56,C0) ->
 * partials dw_part [n_chunks][C0][7], dgamma_part / dbeta_part [n_chunks][C0] over chunks of 64 breaths,
 * n_chunks = dards_stem_frozen_chunks(n_breaths), summed with dards_reduce_rows[_batched].  scale / shift: the
 * forward's; rstd = 1/sqrt(running_var + eps) (see dards_bn_frozen_bwd).  Any n_breaths, no workspace. */
int dards_stem_frozen_chunks(int n_breaths);
int dards_stem_frozen_bwd(const void* dout, const float* x, const float* w, const float* scale, const float* shift,
                          const float* running_mean, const float* rstd, float* dw_part, float* dgamma_part,
                          float* dbeta_part, int n_breaths, int c0, int dout_stride, int pool, int dtype, void* stream);
/* dout (N,56,C0) -> per-group partials dw_part [n_groups][C0][7], dgamma_part/dbeta_part [n_groups][C0]. */
int dards_stem_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* beta,
                   const float* save_mean, const float* save_rstd, float* dw_part, float* dgamma_part,
                   float* dbeta_part, int n_groups, int group, int c0, int dout_stride, int pool, void* workspace,
                   long long workspace_bytes, int dtype, void* stream);
/* Input gradient of the stem, run after dards_stem_bwd on the same dout: dx (N,224) fp32, N = n_groups * group.  The pool
 * arg-max and the ReLU mask are recomputed exactly as dards_stem_bwd recomputes them; dgamma_part / dbeta_part are the
 * group totals [n_groups][C0] that dards_stem_bwd wrote.  Deterministic (no atomics), no workspace. */
int dards_stem_dgrad(const void* dout, const float* x, const float* w, const float* gamma, const float* beta,
                     const float* save_mean, const float* save_rstd, const float* dgamma_part, const float* dbeta_part,
                     float* dx, int n_groups, int group, int c0, int dout_stride, int pool, int dtype, void* stream);
/* Input gradient of dards_stem_eval_fwd (running statistics): dx (N,224) fp32, with the forward's scale / shift. */
int dards_stem_frozen_dgrad(const void* dout, const float* x, const float* w, const float* scale, const float* shift,
                            float* dx, int n_breaths, int c0, int dout_stride, int pool, int dtype, void* stream);

/* ---- stage 1 of the two-convolution stem: Conv1d(1->C0,k3,s1,p1) + BN (ResNet double_conv_first) ------------- */
/* resnet.py:145-147: x (N,224) fp32 -> a0 = bn1(conv1_alt(x)) (N,224,C0) in `dtype`, no ReLU, no pool; the batch statistics
 * of every group go to save_mean / save_rstd [n_groups][C0].  The following Conv1d(C0,C0,k7,s2,p3) runs on
 * dards_conv1d_fwd and zero-pads a0, and the first pool is dards_pool3s2_fwd.  Groups of more than 226 breaths run in
 * chunks and need `workspace` of dards_stem_alt_workspace_bytes(...) bytes (0 otherwise; the pointer may then be NULL).
 * C0 must be a multiple of 16. */
long long dards_stem_alt_workspace_bytes(int n_groups, int group, int c0, int backward);
int dards_stem_alt_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out,
                       float* save_mean, float* save_rstd, int n_groups, int group, int c0, int out_stride, float eps,
                       void* workspace, long long workspace_bytes, int dtype, void* stream);
/* Eval mode: a0 = conv1_alt(x)*scale[c] + shift[c] (dards_bn_eval_coeffs_batched), every breath on its own, any n_breaths. */
int dards_stem_alt_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out,
                            int n_breaths, int c0, int out_stride, int dtype, void* stream);
/* d a0 (N,224,C0) + x -> per-group partials dw_part [n_groups][C0][3], dgamma_part / dbeta_part [n_groups][C0] of
 * conv1_alt and bn1, summed with dards_reduce_rows[_batched].  No gradient w.r.t. x. */
int dards_stem_alt_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* save_mean,
                       const float* save_rstd, float* dw_part, float* dgamma_part, float* dbeta_part, int n_groups,
                       int group, int c0, int dout_stride, void* workspace, long long workspace_bytes, int dtype,
                       void* stream);
/* Input gradient of stage 1, run after dards_stem_alt_bwd on the same d a0: dx (N,224) fp32, N = n_groups * group, from the
 * group totals dgamma_part / dbeta_part [n_groups][C0] that dards_stem_alt_bwd wrote.  Deterministic, no workspace. */
int dards_stem_alt_dgrad(const void* dout, const float* x, const float* w, const float* gamma, const float* save_mean,
                         const float* save_rstd, const float* dgamma_part, const float* dbeta_part, float* dx, int n_groups,
                         int group, int c0, int dout_stride, int dtype, void* stream);

/* ---- pooling, dropout --------------------------------------------------------------- */
/* nn.MaxPool1d / AvgPool1d(3, 2, padding 1) (resnet.py:101-104, 151-153): (N,L,C) -> (N,(L-1)/2+1,C).  pool: 0 max
 * (-inf padding), 1 avg (padding counted, divisor 3).  The backward takes the forward's input `in` (max: the gradient goes
 * to the first maximum of each window, recomputed from `in`; avg: `in` is not read and may be NULL) and writes every
 * element of din (N,L,C).  C and the strides must be multiples of 4. */
int dards_pool3s2_fwd(const void* in, void* out, int n_breaths, int l_in, int c, int in_stride, int out_stride, int pool,
                      int dtype, void* stream);
int dards_pool3s2_bwd(const void* dout, const void* in, void* din, int n_breaths, int l_in, int c, int dout_stride,
                      int in_stride, int din_stride, int pool, int dtype, void* stream);
/* nn.AvgPool1d(2,2) (densenet.py:77): (N,L,C) -> (N,L/2,C) and its backward. */
int dards_avgpool2_fwd(const void* in, void* out, int n_breaths, int l_in, int c, int in_stride, int out_stride,
                       int dtype, void* stream);
int dards_avgpool2_bwd(const void* dout, void* din, int n_breaths, int l_in, int c, int dout_stride,
                       int din_stride, int dtype, void* stream);
/* nn.AvgPool1d(7) + flatten (resnet.py:160-161, densenet.py:183-184): (N,7,C) -> feat (N,C) fp32. */
int dards_avgpool_full_fwd(const void* in, float* feat, int n_breaths, int l, int c, int in_stride, int dtype,
                           void* stream);
int dards_avgpool_full_bwd(const float* dfeat, void* din, int n_breaths, int l, int c, int din_stride, int dtype,
                           void* stream);
/* F.dropout(p, training=True) (densenet.py:37-39) in place on a channel slice; the keep-mask is Philox4x32-10 keyed by
 * (seed, step, GLOBAL element index), so the backward regenerates it and it does not depend on how a batch is sharded over
 * ranks (SURVEY.md 8e(iv)).  seed_offset_dev (nullable) points to TWO 64-bit words on the device: [0] a step counter mixed
 * into the key (a captured CUDA graph draws a fresh mask on every replay), [1] the index of this rank's first sequence in
 * the global batch; rows_per_seq = rows of x per sequence (group * L; 0 = ignore [1]). */
int dards_dropout(void* x, int n_rows, int c, int stride, float p, unsigned long long seed,
                  const unsigned long long* seed_offset_dev, int rows_per_seq, int dtype, void* stream);

/* ---- linear head --------------------------------------------------------------------- */
/* nn.Linear(K,2) on flattened features (torch_cnn_linear_network.py:102,110 and :55,63):
 * logits[r][j] = bias[j] + sum_k feat[r][k] * w[j][k], rows r = sequences (K = 20*F) or breaths (K = F). */
int dards_linear_fwd(const float* feat, const float* w, const float* bias, float* logits, int rows, int k,
                     int n_out, void* stream);
/* dfeat[r][k] = sum_j dlogits[r][j] w[j][k];  dw[j][k] (+)= sum_r dlogits[r][j] feat[r][k];  db[j] (+)= sum_r ... */
int dards_linear_bwd(const float* dlogits, const float* feat, const float* w, float* dfeat, float* dw, float* db,
                     int accumulate, int rows, int k, int n_out, void* stream);

/* torch.nn.BCEWithLogitsLoss() (train_ards_detector.py:530, 929-930), mean over n elements:
 * loss[0] = mean(softplus(z) - t*z);  dlogits = grad_scale * (sigmoid(z) - t) / n.  One CTA. */
int dards_bce_with_logits(const float* logits, const float* target, float* loss, float* dlogits, int n,
                          float grad_scale, void* stream);

/* ---- optimizer (after the gradient all-reduce) ---------------------------------------- */
/* g = clamp(grad*grad_scale, -clip, +clip) [clip<=0: no clamp]  (train_ards_detector.py:474-476, applied
 * AFTER the reduction like nn.DataParallel does -- SURVEY.md 8e); then torch.optim.SGD(momentum,
 * weight_decay, nesterov=True) (train_ards_detector.py:421) on flat fp32 buffers.
 * first_step != 0: momentum buffer is initialised with the gradient (torch semantics). */
int dards_clamp_sgd_nesterov(float* param, const float* grad, float* momentum_buf, long long n, float lr,
                             float momentum, float weight_decay, float clip, float grad_scale, int first_step,
                             void* stream);
/* torch.optim.Adam(lr) defaults (train_ards_detector.py:419): betas (0.9,0.999), eps 1e-8. step is 1-based. */
int dards_clamp_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                     float beta1, float beta2, float eps, float clip, float grad_scale, int step, void* stream);

/* ---- input contract ------------------------------------------------------------------- */
/* ARDSRawDataset.__getitem__ scaling + the trainer's .float() (dataset.py:1375-1379, train_ards_detector.py:150-151):
 * out[i] = (float)((raw[i] - mu) / std), float64 arithmetic, one rounding -- bit-exact with numpy.  `raw` is a DEVICE
 * array of n float64 (raw_f64 != 0) or float32 samples.  padded != 0 is the padded_breath_by_breath rule
 * (_get_padding_mask, dataset.py:1406-1409): mu is subtracted only where raw[i] != 0, so zero padding stays zero. */
int dards_scale_windows(const void* raw, int raw_f64, float* out, long long n, double mu, double std, int padded,
                        void* stream);

/* ---- GradCAM maps ---------------------------------------------------------------------- */
/* gradcam.py:40-65, 83-107 (forward through ReLU/AvgPool/Linear + one-hot backward to the norm5 output A) and the
 * numpy reductions of MaxMinNormCam / UnNormalizedCam (gradcam.py:125-162, 195-205), one CTA per sequence.
 * dA is taken in closed form, dA[n,c,l] = (A[n,c,l] > 0) ? W[target][n*F+c] / L : 0, so no convolution backward runs.
 *   a            (n_groups*group, L, F) channels-last feature map in `dtype`, row stride a_stride (L <= 8)
 *   w, bias      linear_final of CNNLinearNetwork: (n_out, group*F), (n_out)
 *   target_dev   per-sequence class index on the DEVICE (nullable); else `target` for every sequence;
 *                a value < 0 means "the predicted class" (np.argmax of the logits, gradcam.py:101-102)
 * outputs (every pointer except logits may be NULL):
 *   logits (n_groups, n_out); target_used (n_groups)
 *   read_raw / read_u8   (n_groups*group, L): generate_read_cam before / after normalize()
 *   seq_raw / seq_u8     (n_groups, L):       generate_cam before / after normalize() (max(seq_raw,0) = UnNormalizedCam)
 *   read_resized / seq_resized  (.., resized_len) uint8: cv2.resize(cam, (1, resized_len)) (patient_gradcam.py:217, 229)
 *   conv_out / grad_out  (n_groups*group, F, L) fp32: A and dA in the reference's layout
 *                        (generate_one_hot_grad_and_output, gradcam.py:83-99) */
typedef struct dards_gradcam_desc {
  const void* a;
  const float* w;
  const float* bias;
  const int* target_dev;
  float* logits;
  int* target_used;
  float* read_raw;
  uint8_t* read_u8;
  float* seq_raw;
  uint8_t* seq_u8;
  uint8_t* read_resized;
  uint8_t* seq_resized;
  float* conv_out;
  float* grad_out;
  int a_stride, target, n_groups, group, l, f, n_out, resized_len, dtype, reserved;
} dards_gradcam_desc;
int dards_gradcam(const dards_gradcam_desc* desc /* HOST struct, read during the call */, void* stream);

/* ---- debugging ----------------------------------------------------------------------- */
/* Kernel-variant switches used by the unit tests, the probes and the A/B measurements in DESIGN.md section 6
 * (value < 0 restores the default):
 *    0 / 1 / 2  LBO / version / SBO field of the K-major shared-memory descriptors
 *    4          epilogue of the per-tap conv kernel: 0 direct stores, 1 TMA store (default)
 *    5          0 | 1: single-load 3-tap kernel off | on for every k3/s1 layer (default: reductions over <= 128 channels)
 *    6          3: operand ring pinned to 3 stages
 *    7          0: the 3 wgrad taps of 64-channel layers as 3 MMAs instead of one N = 192 MMA
 *    8          1: wave-balanced position-tile width of the wide conv kernel
 *    9          0: no L2 evict_first hint on last-use operands
 *   10          1 | 2: wide | all k3/s1 convolutions through the main loop of conv_bn_tc.cu (plain store epilogue)
 *   11 / 12 / 13 / 14   fused conv+BatchNorm kernel: one activation load per tap / activation-ring depth / one 256-column
 *              tile per plain job / two sub-tiles share the weight tiles
 *   15 / 16    grouped BatchNorm: skip the widest tile configurations / resident CTAs chosen for the fullest last wave
 *   17         0: wide forward / dgrad convolutions on the single-CTA kernel instead of CTA pairs (cta_group::2)
 *   18         operand-ring depth of the CTA-pair conv kernel (default 6)
 *   19         0: weight gradients of >= 256-channel layers on single CTAs instead of CTA pairs */
int dards_tc_debug_set(int key, int value);

#ifdef __cplusplus
}
#endif
#endif /* DEEPARDS_B200_H_ */

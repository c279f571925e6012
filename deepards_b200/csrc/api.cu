// C ABI (include/deepards_b200.h): argument validation + dispatch to the kernel launchers.
#include <cstdarg>
#include <cstdio>

#include "common.cuh"

namespace dards {

static thread_local char g_err[512] = "";

static long long g_launches = 0;
void count_launch() { ++g_launches; }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- launchers implemented in the other translation units -----------------------------------------------
int simt_pack_conv_weight(const float*, void*, void*, int, int, int, int, cudaStream_t);
int simt_pack_conv_weights_batched(const dards_pack_desc*, int, int, int, cudaStream_t);
int simt_conv_gemm(const ConvGemmArgs&, int, cudaStream_t);
int simt_conv_wgrad(const void*, const void*, float*, int, void*, long long, int, int, int, int, int, int, int, int, int,
                    int, int, cudaStream_t);
long long simt_wgrad_workspace_bytes(int, int, int, int, int);

int tc_conv_fwd(const void* in, const void* w_koi, void* out, const void* addend, int n_breaths, int l_in, int l_out,
                int c_in, int c_out, int in_stride, int out_stride, int addend_stride, int ktaps, int stride, int pad,
                int src_last_use, cudaStream_t st);
int tc_conv_dgrad(const void* dout, const void* w_kio, void* din, const void* addend, int n_breaths, int l_in, int l_out,
                  int c_in, int c_out, int dout_stride, int din_stride, int addend_stride, int ktaps, int stride, int pad,
                  int src_last_use, cudaStream_t st);
int tc_conv_wgrad(const void* in, const void* dout, float* dw, int accumulate, void* workspace, long long workspace_bytes,
                  int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride, int dout_stride, int ktaps,
                  int stride, int pad, cudaStream_t st);
long long tc_wgrad_workspace_bytes(int n_breaths, int l_out, int c_in, int c_out, int ktaps);
int tc_conv_affine_fwd(const void* in, const void* w_koi, void* out, const void* res, const float* scale, const float* shift,
                       int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride, int out_stride, int res_stride,
                       int ktaps, int stride, int pad, int relu, int src_last_use, cudaStream_t st);
int launch_bn_eval_coeffs_batched(const dards_eval_coeff_desc*, int, int, float, cudaStream_t);
int launch_stem_eval_fwd(const float*, const float*, const float*, const float*, void*, int, int, int, int, int,
                         cudaStream_t);
int launch_bn_affine_apply(const void*, void*, const void*, const float*, const float*, const void*, const float*,
                           const float*, int, int, int, int, int, int, int, int, cudaStream_t);
int launch_bn_frozen_bwd(const void*, const void*, const void*, const float*, const float*, const float*, const float*,
                         void*, int, void*, float*, float*, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int stem_frozen_chunks(int n_breaths);
int launch_stem_frozen_bwd(const void*, const float*, const float*, const float*, const float*, const float*, const float*,
                           float*, float*, float*, int, int, int, int, int, cudaStream_t);
int tc_conv_wgrad_accum(const void* in, const void* dout, float* dw_t, int n_breaths, int l_in, int l_out, int c_in, int c_out,
                        int in_stride, int dout_stride, int ktaps, int stride, int pad, cudaStream_t st);
int simt_unpack_wgrad_batched(const dards_unpack_desc*, int, int, cudaStream_t);
int tc_debug_set(int key, int value);
int set_sm_limit(int n);
int tc_conv_bn_mode(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride, int pad);
int tc_conv_bn_part_entries(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride,
                            int pad);
int tc_conv_bn_fwd(const void* in, const void* w_koi, void* y, void* out, const void* res, const float* gamma,
                   const float* beta, float* save_mean, float* save_rstd, float* part, int n_breaths, int group, int l_in,
                   int l_out, int c_in, int c_out, int in_stride, int y_stride, int out_stride, int res_stride, int ktaps,
                   int stride, int pad, float eps, int relu, int src_last_use, cudaStream_t st);
int launch_gbn_apply_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta, const float* part,
                         int entries, float* save_mean, float* save_rstd, const void* x2, const float* gamma2,
                         const float* beta2, const float* part2, int entries2, float* save_mean2, float* save_rstd2,
                         int n_groups, int rows, int c, int x_stride, int out_stride, int res_stride, int x2_stride, float eps,
                         int relu, cudaStream_t st);

int launch_gbn_fwd(const void*, void*, const void*, const float*, const float*, float*, float*, int, int, int, int, int,
                   int, float, int, int, cudaStream_t);
int launch_gbn_bwd(const void*, const void*, const void*, const float*, const float*, const float*, const float*, void*,
                   int, void*, float*, float*, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int launch_reduce_rows_batched(const dards_reduce_desc*, int, int, cudaStream_t);
int launch_bn_running_update_batched(const dards_running_desc*, int, int, float, cudaStream_t);
int launch_reduce_rows(const float*, float*, int, int, int, cudaStream_t);
int launch_bn_running_update(const float*, const float*, float*, float*, long long*, int, int, int, float, float,
                             cudaStream_t);
int launch_stem_fwd(const float*, const float*, const float*, const float*, void*, float*, float*, int, int, int, int,
                    float, int, void*, long long, int, cudaStream_t);
int launch_stem_bwd(const void*, const float*, const float*, const float*, const float*, const float*, const float*,
                    float*, float*, float*, int, int, int, int, int, void*, long long, int, cudaStream_t);
long long stem_workspace_bytes(int n_groups, int group, int c0, int backward);
int launch_avgpool2(int, const void*, void*, int, int, int, int, int, int, cudaStream_t);
long long stem_alt_workspace_bytes(int n_groups, int group, int c0, int backward);
int launch_stem_alt_fwd(const float*, const float*, const float*, const float*, void*, float*, float*, int, int, int, int,
                        float, void*, long long, int, cudaStream_t);
int launch_stem_alt_eval_fwd(const float*, const float*, const float*, const float*, void*, int, int, int, int,
                             cudaStream_t);
int launch_stem_alt_bwd(const void*, const float*, const float*, const float*, const float*, const float*, float*, float*,
                        float*, int, int, int, int, void*, long long, int, cudaStream_t);
int launch_pool3s2(int, const void*, const void*, void*, int, int, int, int, int, int, int, int, cudaStream_t);
int launch_avgpool_full_fwd(const void*, float*, int, int, int, int, int, cudaStream_t);
int launch_avgpool_full_bwd(const float*, void*, int, int, int, int, int, cudaStream_t);
int launch_dropout(void*, int, int, int, float, unsigned long long, const unsigned long long*, int, int, cudaStream_t);
int launch_bce(const float*, const float*, float*, float*, int, float, cudaStream_t);
int launch_linear_fwd(const float*, const float*, const float*, float*, int, int, int, cudaStream_t);
int launch_linear_bwd(const float*, const float*, const float*, float*, float*, float*, int, int, int, int,
                      cudaStream_t);
int launch_clamp_sgd(float*, const float*, float*, long long, float, float, float, float, float, int, cudaStream_t);
int launch_clamp_adam(float*, const float*, float*, float*, long long, float, float, float, float, float, float, int,
                      cudaStream_t);

int launch_gradcam(const dards_gradcam_desc&, cudaStream_t);
int launch_scale_windows(const void*, int, float*, long long, double, double, int, cudaStream_t);

static inline cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }

static int conv_out_len(int l_in, int ktaps, int stride, int pad) { return (l_in + 2 * pad - ktaps) / stride + 1; }

}  // namespace dards

using namespace dards;

extern "C" {

int dards_version(void) { return 8; }

const char* dards_last_error(void) { return g_err; }

long long dards_launch_count(void) { return g_launches; }

int dards_device_supported(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10;
}

int dards_pack_conv_weight(const float* w, void* w_kio, void* w_koi, int c_out, int c_in, int ktaps, int dtype,
                           void* stream) {
  DARDS_CHECK_ARG(w && (w_kio || w_koi), "pack_conv_weight: null pointer");
  DARDS_CHECK_ARG(c_out > 0 && c_in > 0 && ktaps > 0, "pack_conv_weight: bad shape");
  return simt_pack_conv_weight(w, w_kio, w_koi, c_out, c_in, ktaps, dtype, S(stream));
}

int dards_pack_conv_weights_batched(const dards_pack_desc* descs_dev, int n_descs, int total_blocks, int dtype,
                                    void* stream) {
  DARDS_CHECK_ARG(descs_dev && n_descs >= 0 && total_blocks >= 0, "pack_conv_weights_batched: bad argument");
  DARDS_CHECK_ARG(dtype == DARDS_F32 || dtype == DARDS_BF16, "pack_conv_weights_batched: unknown dtype");
  return simt_pack_conv_weights_batched(descs_dev, n_descs, total_blocks, dtype, S(stream));
}

int dards_conv1d_fwd(const void* in, const void* w_packed, void* out, const void* addend, int n_breaths, int l_in,
                     int l_out, int c_in, int c_out, int in_stride, int out_stride, int addend_stride, int ktaps,
                     int stride, int pad, int dtype, int impl, void* stream) {
  const int src_last_use = (impl & DARDS_HINT_LAST_USE) ? 1 : 0;
  impl &= 0xff;
  DARDS_CHECK_ARG(in && w_packed && out, "conv1d_fwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_fwd: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_fwd: l_out %d != (l_in+2p-k)/s+1 = %d", l_out,
                  conv_out_len(l_in, ktaps, stride, pad));
  DARDS_CHECK_ARG(in_stride >= c_in && out_stride >= c_out, "conv1d_fwd: row stride smaller than channel count");
  if (impl == 1) {
    DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_fwd: the tcgen05 path is bf16 only");
    return tc_conv_fwd(in, w_packed, out, addend, n_breaths, l_in, l_out, c_in, c_out, in_stride, out_stride,
                       addend_stride, ktaps, stride, pad, src_last_use, S(stream));
  }
  DARDS_CHECK_ARG(impl == 0, "conv1d_fwd: unknown impl %d", impl);
  ConvGemmArgs a{};
  a.in = in; a.w = w_packed; a.out = out; a.addend = addend;
  a.m_total = (long long)n_breaths * l_out;
  a.l_src = l_in; a.l_dst = l_out; a.c_red = c_in; a.c_cols = c_out;
  a.src_stride = in_stride; a.dst_stride = out_stride; a.addend_stride = addend_stride;
  a.ktaps = ktaps; a.q_mul = stride; a.t_mul = 1; a.off = -pad; a.div = 1;
  return simt_conv_gemm(a, dtype, S(stream));
}

int dards_conv1d_affine_fwd(const void* in, const void* w_packed, void* out, const void* res, const float* scale,
                            const float* shift, int n_breaths, int l_in, int l_out, int c_in, int c_out, int in_stride,
                            int out_stride, int res_stride, int ktaps, int stride, int pad, int relu, int dtype, int impl,
                            void* stream) {
  const int src_last_use = (relu & DARDS_HINT_LAST_USE) ? 1 : 0;
  relu &= 0xff;
  DARDS_CHECK_ARG(in && w_packed && out && scale && shift, "conv1d_affine_fwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_affine_fwd: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_affine_fwd: l_out %d != (l_in+2p-k)/s+1 = %d",
                  l_out, conv_out_len(l_in, ktaps, stride, pad));
  DARDS_CHECK_ARG(in_stride >= c_in && out_stride >= c_out && (!res || res_stride >= c_out),
                  "conv1d_affine_fwd: row stride smaller than channel count");
  DARDS_CHECK_ARG(relu == 0 || relu == 1, "conv1d_affine_fwd: relu must be 0 or 1");
  if (res) {
    const size_t esz = dtype == DARDS_BF16 ? 2 : 4;
    const char* r0 = static_cast<const char*>(res);
    const char* o0 = static_cast<const char*>(out);
    const size_t rows = (size_t)n_breaths * l_out;
    const char* r1 = r0 + (rows ? ((rows - 1) * res_stride + c_out) * esz : 0);
    const char* o1 = o0 + (rows ? ((rows - 1) * out_stride + c_out) * esz : 0);
    DARDS_CHECK_ARG(r1 <= o0 || o1 <= r0, "conv1d_affine_fwd: the residual must not overlap the output");
  }
  if (impl == 1) {
    DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_affine_fwd: the tcgen05 path is bf16 only");
    return tc_conv_affine_fwd(in, w_packed, out, res, scale, shift, n_breaths, l_in, l_out, c_in, c_out, in_stride,
                              out_stride, res_stride, ktaps, stride, pad, relu, src_last_use, S(stream));
  }
  DARDS_CHECK_ARG(impl == 0, "conv1d_affine_fwd: unknown impl %d", impl);
  DARDS_CHECK_ARG((reinterpret_cast<uintptr_t>(scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(shift) & 15) == 0,
                  "conv1d_affine_fwd: scale / shift must be 16-byte aligned");
  ConvGemmArgs a{};
  a.in = in; a.w = w_packed; a.out = out; a.addend = res;
  a.m_total = (long long)n_breaths * l_out;
  a.l_src = l_in; a.l_dst = l_out; a.c_red = c_in; a.c_cols = c_out;
  a.src_stride = in_stride; a.dst_stride = out_stride; a.addend_stride = res_stride;
  a.ktaps = ktaps; a.q_mul = stride; a.t_mul = 1; a.off = -pad; a.div = 1;
  a.scale = scale; a.shift = shift; a.relu = relu;
  return simt_conv_gemm(a, dtype, S(stream));
}

int dards_conv1d_dgrad(const void* dout, const void* w_packed, void* din, const void* addend, int n_breaths, int l_in,
                       int l_out, int c_in, int c_out, int dout_stride, int din_stride, int addend_stride, int ktaps,
                       int stride, int pad, int dtype, int impl, void* stream) {
  const int src_last_use = (impl & DARDS_HINT_LAST_USE) ? 1 : 0;
  impl &= 0xff;
  DARDS_CHECK_ARG(dout && w_packed && din, "conv1d_dgrad: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_dgrad: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_dgrad: l_out %d != (l_in+2p-k)/s+1 = %d",
                  l_out, conv_out_len(l_in, ktaps, stride, pad));
  DARDS_CHECK_ARG(dout_stride >= c_out && din_stride >= c_in, "conv1d_dgrad: row stride smaller than channel count");
  if (impl == 1) {
    DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_dgrad: the tcgen05 path is bf16 only");
    return tc_conv_dgrad(dout, w_packed, din, addend, n_breaths, l_in, l_out, c_in, c_out, dout_stride, din_stride,
                         addend_stride, ktaps, stride, pad, src_last_use, S(stream));
  }
  DARDS_CHECK_ARG(impl == 0, "conv1d_dgrad: unknown impl %d", impl);
  ConvGemmArgs a{};
  a.in = dout; a.w = w_packed; a.out = din; a.addend = addend;
  a.m_total = (long long)n_breaths * l_in;
  a.l_src = l_out; a.l_dst = l_in; a.c_red = c_out; a.c_cols = c_in;
  a.src_stride = dout_stride; a.dst_stride = din_stride; a.addend_stride = addend_stride;
  // q*stride + t - pad == p  <=>  q = (p + pad - t) / stride
  a.ktaps = ktaps; a.q_mul = 1; a.t_mul = -1; a.off = pad; a.div = stride;
  return simt_conv_gemm(a, dtype, S(stream));
}

int dards_conv1d_wgrad(const void* in, const void* dout, float* dw, int accumulate, void* workspace,
                       long long workspace_bytes, int n_breaths, int l_in, int l_out, int c_in, int c_out,
                       int in_stride, int dout_stride, int ktaps, int stride, int pad, int dtype, int impl,
                       void* stream) {
  DARDS_CHECK_ARG(in && dout && dw, "conv1d_wgrad: null pointer");
  DARDS_CHECK_ARG(n_breaths > 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_wgrad: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_wgrad: l_out mismatch");
  DARDS_CHECK_ARG(in_stride >= c_in && dout_stride >= c_out, "conv1d_wgrad: row stride smaller than channel count");
  if (impl == 1) {
    DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_wgrad: the tcgen05 path is bf16 only");
    return tc_conv_wgrad(in, dout, dw, accumulate, workspace, workspace_bytes, n_breaths, l_in, l_out, c_in, c_out,
                         in_stride, dout_stride, ktaps, stride, pad, S(stream));
  }
  DARDS_CHECK_ARG(impl == 0, "conv1d_wgrad: unknown impl %d", impl);
  return simt_conv_wgrad(in, dout, dw, accumulate, workspace, workspace_bytes, n_breaths, l_in, l_out, c_in, c_out,
                         in_stride, dout_stride, ktaps, stride, pad, dtype, S(stream));
}

int dards_conv1d_wgrad_accum(const void* in, const void* dout, float* dw_t, int n_breaths, int l_in, int l_out, int c_in,
                             int c_out, int in_stride, int dout_stride, int ktaps, int stride, int pad, int dtype,
                             void* stream) {
  DARDS_CHECK_ARG(in && dout && dw_t, "conv1d_wgrad_accum: null pointer");
  DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_wgrad_accum: the tcgen05 path is bf16 only");
  DARDS_CHECK_ARG(n_breaths > 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_wgrad_accum: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_wgrad_accum: l_out mismatch");
  DARDS_CHECK_ARG(in_stride >= c_in && dout_stride >= c_out, "conv1d_wgrad_accum: row stride smaller than channel count");
  return tc_conv_wgrad_accum(in, dout, dw_t, n_breaths, l_in, l_out, c_in, c_out, in_stride, dout_stride, ktaps, stride, pad,
                             S(stream));
}

int dards_unpack_wgrad_batched(const dards_unpack_desc* descs_dev, int n_descs, int total_blocks, void* stream) {
  DARDS_CHECK_ARG(descs_dev && n_descs >= 0 && total_blocks >= 0, "unpack_wgrad_batched: bad argument");
  return simt_unpack_wgrad_batched(descs_dev, n_descs, total_blocks, S(stream));
}

int dards_memset_zero(void* ptr, long long bytes, void* stream) {
  DARDS_CHECK_ARG(ptr && bytes >= 0, "memset_zero: bad argument");
  if (bytes == 0) return DARDS_OK;
  cudaError_t e = cudaMemsetAsync(ptr, 0, (size_t)bytes, S(stream));
  if (e != cudaSuccess) {
    set_error("memset_zero: %s", cudaGetErrorString(e));
    return DARDS_ERR_CUDA;
  }
  count_launch();
  return DARDS_OK;
}

long long dards_conv1d_wgrad_workspace_bytes(int n_breaths, int l_out, int c_in, int c_out, int ktaps, int impl) {
  if (impl == 1) return tc_wgrad_workspace_bytes(n_breaths, l_out, c_in, c_out, ktaps);
  return simt_wgrad_workspace_bytes(n_breaths, l_out, c_in, c_out, ktaps);
}

int dards_conv1d_bn_mode(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps, int stride,
                         int pad, int dtype) {
  if (dtype != DARDS_BF16) return 0;
  return tc_conv_bn_mode(n_breaths, group, l_in, l_out, c_in, c_out, ktaps, stride, pad);
}

int dards_conv1d_bn_part_entries(int n_breaths, int group, int l_in, int l_out, int c_in, int c_out, int ktaps,
                                 int stride, int pad) {
  return tc_conv_bn_part_entries(n_breaths, group, l_in, l_out, c_in, c_out, ktaps, stride, pad);
}

int dards_conv1d_bn_fwd(const void* in, const void* w_koi, void* y, void* out, const void* res, const float* gamma,
                        const float* beta, float* save_mean, float* save_rstd, float* part, int n_breaths, int group,
                        int l_in, int l_out, int c_in, int c_out, int in_stride, int y_stride, int out_stride,
                        int res_stride, int ktaps, int stride, int pad, float eps, int relu, int dtype, void* stream) {
  const int src_last_use = (relu & DARDS_HINT_LAST_USE) ? 1 : 0;
  relu &= 0xff;
  DARDS_CHECK_ARG(in && w_koi && y, "conv1d_bn_fwd: null pointer");
  DARDS_CHECK_ARG(dtype == DARDS_BF16, "conv1d_bn_fwd: the fused tcgen05 path is bf16 only");
  DARDS_CHECK_ARG(n_breaths > 0 && group > 0 && l_in > 0 && c_in > 0 && c_out > 0 && ktaps > 0 && stride > 0 && pad >= 0,
                  "conv1d_bn_fwd: bad shape");
  DARDS_CHECK_ARG(l_out == conv_out_len(l_in, ktaps, stride, pad), "conv1d_bn_fwd: l_out %d != (l_in+2p-k)/s+1 = %d", l_out,
                  conv_out_len(l_in, ktaps, stride, pad));
  DARDS_CHECK_ARG(in_stride >= c_in && y_stride >= c_out && (!out || out_stride >= c_out) && (!res || res_stride >= c_out),
                  "conv1d_bn_fwd: row stride smaller than channel count");
  return tc_conv_bn_fwd(in, w_koi, y, out, res, gamma, beta, save_mean, save_rstd, part, n_breaths, group, l_in, l_out, c_in,
                        c_out, in_stride, y_stride, out_stride, res_stride, ktaps, stride, pad, eps, relu, src_last_use,
                        S(stream));
}

int dards_gbn_apply_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta,
                        const float* part, int entries, float* save_mean, float* save_rstd, const void* x2,
                        const float* gamma2, const float* beta2, const float* part2, int entries2, float* save_mean2,
                        float* save_rstd2, int n_groups, int rows_per_group, int c, int x_stride, int out_stride,
                        int res_stride, int x2_stride, float eps, int relu, int dtype, void* stream) {
  DARDS_CHECK_ARG(dtype == DARDS_BF16, "gbn_apply_fwd: bf16 only (it follows the fused tcgen05 convolution)");
  DARDS_CHECK_ARG(x_stride >= c && out_stride >= c, "gbn_apply_fwd: row stride smaller than channel count");
  return launch_gbn_apply_fwd(x, out, res, gamma, beta, part, entries, save_mean, save_rstd, x2, gamma2, beta2, part2,
                              entries2, save_mean2, save_rstd2, n_groups, rows_per_group, c, x_stride, out_stride, res_stride,
                              x2_stride, eps, relu, S(stream));
}

int dards_gbn_fwd(const void* x, void* out, const void* res, const float* gamma, const float* beta, float* save_mean,
                  float* save_rstd, int n_groups, int rows_per_group, int c, int x_stride, int out_stride,
                  int res_stride, float eps, int relu, int dtype, void* stream) {
  DARDS_CHECK_ARG(x && out && gamma && beta && save_mean && save_rstd, "gbn_fwd: null pointer");
  DARDS_CHECK_ARG(x_stride >= c && out_stride >= c, "gbn_fwd: row stride smaller than channel count");
  return launch_gbn_fwd(x, out, res, gamma, beta, save_mean, save_rstd, n_groups, rows_per_group, c, x_stride,
                        out_stride, res_stride, eps, relu, dtype, S(stream));
}

int dards_gbn_bwd(const void* dout, const void* x, const void* mask_src, const float* gamma, const float* beta,
                  const float* save_mean, const float* save_rstd, void* dx, int accumulate_dx, void* dres,
                  float* dgamma_part, float* dbeta_part, int n_groups, int rows_per_group, int c, int dout_stride,
                  int x_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype,
                  void* stream) {
  DARDS_CHECK_ARG(dout && x && gamma && beta && save_mean && save_rstd && dx, "gbn_bwd: null pointer");
  DARDS_CHECK_ARG(relu_mode >= 0 && relu_mode <= 2, "gbn_bwd: relu_mode must be 0, 1 or 2");
  return launch_gbn_bwd(dout, x, mask_src, gamma, beta, save_mean, save_rstd, dx, accumulate_dx, dres, dgamma_part,
                        dbeta_part, n_groups, rows_per_group, c, dout_stride, x_stride, mask_stride, dx_stride,
                        dres_stride, relu_mode, dtype, S(stream));
}

int dards_reduce_rows(const float* part, float* out, int rows, int c, int accumulate, void* stream) {
  DARDS_CHECK_ARG(part && out && rows >= 0 && c >= 0, "reduce_rows: bad argument");
  return launch_reduce_rows(part, out, rows, c, accumulate, S(stream));
}

int dards_reduce_rows_batched(const dards_reduce_desc* descs_dev, int n_descs, int total_blocks, void* stream) {
  DARDS_CHECK_ARG(descs_dev && n_descs >= 0 && total_blocks >= 0, "reduce_rows_batched: bad argument");
  return launch_reduce_rows_batched(descs_dev, n_descs, total_blocks, S(stream));
}

int dards_bn_running_update_batched(const dards_running_desc* descs_dev, int n_descs, int total_blocks, float eps,
                                    void* stream) {
  DARDS_CHECK_ARG(descs_dev && n_descs >= 0 && total_blocks >= 0, "bn_running_update_batched: bad argument");
  return launch_bn_running_update_batched(descs_dev, n_descs, total_blocks, eps, S(stream));
}

int dards_bn_eval_coeffs_batched(const dards_eval_coeff_desc* descs_dev, int n_descs, int total_blocks, float eps,
                                 void* stream) {
  DARDS_CHECK_ARG(descs_dev && n_descs >= 0 && total_blocks >= 0, "bn_eval_coeffs_batched: bad argument");
  return launch_bn_eval_coeffs_batched(descs_dev, n_descs, total_blocks, eps, S(stream));
}

int dards_bn_running_update(const float* save_mean, const float* save_rstd, float* running_mean, float* running_var,
                            long long* num_batches_tracked, int n_groups, int rows_per_group, int c, float momentum,
                            float eps, void* stream) {
  DARDS_CHECK_ARG(save_mean && save_rstd && running_mean && running_var, "bn_running_update: null pointer");
  return launch_bn_running_update(save_mean, save_rstd, running_mean, running_var, num_batches_tracked, n_groups,
                                  rows_per_group, c, momentum, eps, S(stream));
}

long long dards_stem_workspace_bytes(int n_groups, int group, int c0, int backward) {
  return stem_workspace_bytes(n_groups, group, c0, backward ? 1 : 0);
}

int dards_stem_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out, float* save_mean,
                   float* save_rstd, int n_groups, int group, int c0, int out_stride, float eps, int pool, void* workspace,
                   long long workspace_bytes, int dtype, void* stream) {
  DARDS_CHECK_ARG(x && w && gamma && beta && out && save_mean && save_rstd, "stem_fwd: null pointer");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "stem_fwd: pool must be 0 (max) or 1 (avg)");
  DARDS_CHECK_ARG(out_stride >= c0, "stem_fwd: row stride smaller than channel count");
  return launch_stem_fwd(x, w, gamma, beta, out, save_mean, save_rstd, n_groups, group, c0, out_stride, eps, pool, workspace,
                         workspace_bytes, dtype, S(stream));
}

int dards_stem_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out, int n_breaths,
                        int c0, int out_stride, int pool, int dtype, void* stream) {
  DARDS_CHECK_ARG(x && w && scale && shift && out, "stem_eval_fwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0, "stem_eval_fwd: negative number of breaths");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "stem_eval_fwd: pool must be 0 (max) or 1 (avg)");
  DARDS_CHECK_ARG(out_stride >= c0, "stem_eval_fwd: row stride smaller than channel count");
  return launch_stem_eval_fwd(x, w, scale, shift, out, n_breaths, c0, out_stride, pool, dtype, S(stream));
}

int dards_bn_affine_apply(const void* y, void* out, const void* res, const float* scale, const float* shift,
                          const void* y2, const float* scale2, const float* shift2, int rows, int c, int y_stride,
                          int out_stride, int res_stride, int y2_stride, int relu, int dtype, void* stream) {
  DARDS_CHECK_ARG(relu == 0 || relu == 1, "bn_affine_apply: relu must be 0 or 1");
  DARDS_CHECK_ARG(dtype == DARDS_F32 || dtype == DARDS_BF16, "bn_affine_apply: unknown dtype %d", dtype);
  return launch_bn_affine_apply(y, out, res, scale, shift, y2, scale2, shift2, rows, c, y_stride, out_stride, res_stride,
                                y2_stride, relu, dtype, S(stream));
}

int dards_bn_frozen_bwd(const void* dout, const void* y, const void* mask_src, const float* scale, const float* shift,
                        const float* running_mean, const float* rstd, void* dx, int accumulate_dx, void* dres,
                        float* dgamma_part, float* dbeta_part, int n_tiles, int rows_per_tile, int c, int dout_stride,
                        int y_stride, int mask_stride, int dx_stride, int dres_stride, int relu_mode, int dtype,
                        void* stream) {
  DARDS_CHECK_ARG(dout && y && scale && shift && running_mean && rstd && dx, "bn_frozen_bwd: null pointer");
  DARDS_CHECK_ARG(relu_mode >= 0 && relu_mode <= 2, "bn_frozen_bwd: relu_mode must be 0, 1 or 2");
  DARDS_CHECK_ARG(n_tiles >= 0 && rows_per_tile > 0 && c > 0, "bn_frozen_bwd: bad shape");
  return launch_bn_frozen_bwd(dout, y, mask_src, scale, shift, running_mean, rstd, dx, accumulate_dx, dres, dgamma_part,
                              dbeta_part, n_tiles, rows_per_tile, c, dout_stride, y_stride, mask_stride, dx_stride,
                              dres_stride, relu_mode, dtype, S(stream));
}

int dards_stem_frozen_chunks(int n_breaths) { return stem_frozen_chunks(n_breaths); }

int dards_stem_frozen_bwd(const void* dout, const float* x, const float* w, const float* scale, const float* shift,
                          const float* running_mean, const float* rstd, float* dw_part, float* dgamma_part,
                          float* dbeta_part, int n_breaths, int c0, int dout_stride, int pool, int dtype, void* stream) {
  DARDS_CHECK_ARG(dout && x && w && scale && shift && running_mean && rstd && dw_part && dgamma_part && dbeta_part,
                  "stem_frozen_bwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0, "stem_frozen_bwd: negative number of breaths");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "stem_frozen_bwd: pool must be 0 (max) or 1 (avg)");
  DARDS_CHECK_ARG(dout_stride >= c0, "stem_frozen_bwd: row stride smaller than channel count");
  return launch_stem_frozen_bwd(dout, x, w, scale, shift, running_mean, rstd, dw_part, dgamma_part, dbeta_part, n_breaths,
                                c0, dout_stride, pool, dtype, S(stream));
}

int dards_stem_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* beta,
                   const float* save_mean, const float* save_rstd, float* dw_part, float* dgamma_part,
                   float* dbeta_part, int n_groups, int group, int c0, int dout_stride, int pool, void* workspace,
                   long long workspace_bytes, int dtype, void* stream) {
  DARDS_CHECK_ARG(dout && x && w && gamma && beta && save_mean && save_rstd && dw_part && dgamma_part && dbeta_part,
                  "stem_bwd: null pointer");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "stem_bwd: pool must be 0 (max) or 1 (avg)");
  return launch_stem_bwd(dout, x, w, gamma, beta, save_mean, save_rstd, dw_part, dgamma_part, dbeta_part, n_groups, group,
                         c0, dout_stride, pool, workspace, workspace_bytes, dtype, S(stream));
}

long long dards_stem_alt_workspace_bytes(int n_groups, int group, int c0, int backward) {
  return stem_alt_workspace_bytes(n_groups, group, c0, backward ? 1 : 0);
}

int dards_stem_alt_fwd(const float* x, const float* w, const float* gamma, const float* beta, void* out, float* save_mean,
                       float* save_rstd, int n_groups, int group, int c0, int out_stride, float eps, void* workspace,
                       long long workspace_bytes, int dtype, void* stream) {
  DARDS_CHECK_ARG(x && w && gamma && beta && out && save_mean && save_rstd, "stem_alt_fwd: null pointer");
  DARDS_CHECK_ARG(n_groups >= 0, "stem_alt_fwd: negative number of groups");
  DARDS_CHECK_ARG(out_stride >= c0, "stem_alt_fwd: row stride smaller than channel count");
  return launch_stem_alt_fwd(x, w, gamma, beta, out, save_mean, save_rstd, n_groups, group, c0, out_stride, eps, workspace,
                             workspace_bytes, dtype, S(stream));
}

int dards_stem_alt_eval_fwd(const float* x, const float* w, const float* scale, const float* shift, void* out,
                            int n_breaths, int c0, int out_stride, int dtype, void* stream) {
  DARDS_CHECK_ARG(x && w && scale && shift && out, "stem_alt_eval_fwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0, "stem_alt_eval_fwd: negative number of breaths");
  DARDS_CHECK_ARG(out_stride >= c0, "stem_alt_eval_fwd: row stride smaller than channel count");
  return launch_stem_alt_eval_fwd(x, w, scale, shift, out, n_breaths, c0, out_stride, dtype, S(stream));
}

int dards_stem_alt_bwd(const void* dout, const float* x, const float* w, const float* gamma, const float* save_mean,
                       const float* save_rstd, float* dw_part, float* dgamma_part, float* dbeta_part, int n_groups, int group,
                       int c0, int dout_stride, void* workspace, long long workspace_bytes, int dtype, void* stream) {
  DARDS_CHECK_ARG(dout && x && w && gamma && save_mean && save_rstd && dw_part && dgamma_part && dbeta_part,
                  "stem_alt_bwd: null pointer");
  DARDS_CHECK_ARG(n_groups >= 0, "stem_alt_bwd: negative number of groups");
  DARDS_CHECK_ARG(dout_stride >= c0, "stem_alt_bwd: row stride smaller than channel count");
  return launch_stem_alt_bwd(dout, x, w, gamma, save_mean, save_rstd, dw_part, dgamma_part, dbeta_part, n_groups, group, c0,
                             dout_stride, workspace, workspace_bytes, dtype, S(stream));
}

int dards_pool3s2_fwd(const void* in, void* out, int n_breaths, int l_in, int c, int in_stride, int out_stride, int pool,
                      int dtype, void* stream) {
  DARDS_CHECK_ARG(in && out, "pool3s2_fwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0, "pool3s2_fwd: negative number of breaths");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "pool3s2_fwd: pool must be 0 (max) or 1 (avg)");
  return launch_pool3s2(0, in, nullptr, out, n_breaths, l_in, c, in_stride, in_stride, out_stride, pool, dtype, S(stream));
}

int dards_pool3s2_bwd(const void* dout, const void* in, void* din, int n_breaths, int l_in, int c, int dout_stride,
                      int in_stride, int din_stride, int pool, int dtype, void* stream) {
  DARDS_CHECK_ARG(dout && din && (in || pool == 1), "pool3s2_bwd: null pointer");
  DARDS_CHECK_ARG(n_breaths >= 0, "pool3s2_bwd: negative number of breaths");
  DARDS_CHECK_ARG(pool == 0 || pool == 1, "pool3s2_bwd: pool must be 0 (max) or 1 (avg)");
  return launch_pool3s2(1, dout, in, din, n_breaths, l_in, c, dout_stride, in_stride, din_stride, pool, dtype, S(stream));
}

int dards_avgpool2_fwd(const void* in, void* out, int n_breaths, int l_in, int c, int in_stride, int out_stride,
                       int dtype, void* stream) {
  DARDS_CHECK_ARG(in && out, "avgpool2_fwd: null pointer");
  return launch_avgpool2(0, in, out, n_breaths, l_in, c, in_stride, out_stride, dtype, S(stream));
}

int dards_avgpool2_bwd(const void* dout, void* din, int n_breaths, int l_in, int c, int dout_stride, int din_stride,
                       int dtype, void* stream) {
  DARDS_CHECK_ARG(dout && din, "avgpool2_bwd: null pointer");
  return launch_avgpool2(1, dout, din, n_breaths, l_in, c, dout_stride, din_stride, dtype, S(stream));
}

int dards_avgpool_full_fwd(const void* in, float* feat, int n_breaths, int l, int c, int in_stride, int dtype,
                           void* stream) {
  DARDS_CHECK_ARG(in && feat && l > 0, "avgpool_full_fwd: bad argument");
  return launch_avgpool_full_fwd(in, feat, n_breaths, l, c, in_stride, dtype, S(stream));
}

int dards_avgpool_full_bwd(const float* dfeat, void* din, int n_breaths, int l, int c, int din_stride, int dtype,
                           void* stream) {
  DARDS_CHECK_ARG(dfeat && din && l > 0, "avgpool_full_bwd: bad argument");
  return launch_avgpool_full_bwd(dfeat, din, n_breaths, l, c, din_stride, dtype, S(stream));
}

int dards_dropout(void* x, int n_rows, int c, int stride, float p, unsigned long long seed,
                  const unsigned long long* seed_offset_dev, int rows_per_seq, int dtype, void* stream) {
  DARDS_CHECK_ARG(x, "dropout: null pointer");
  DARDS_CHECK_ARG(rows_per_seq >= 0, "dropout: negative rows_per_seq");
  return launch_dropout(x, n_rows, c, stride, p, seed, seed_offset_dev, rows_per_seq, dtype, S(stream));
}

int dards_bce_with_logits(const float* logits, const float* target, float* loss, float* dlogits, int n,
                          float grad_scale, void* stream) {
  DARDS_CHECK_ARG(logits && target && (loss || dlogits) && n >= 0, "bce_with_logits: bad argument");
  return launch_bce(logits, target, loss, dlogits, n, grad_scale, S(stream));
}

int dards_linear_fwd(const float* feat, const float* w, const float* bias, float* logits, int rows, int k, int n_out,
                     void* stream) {
  DARDS_CHECK_ARG(feat && w && bias && logits && k > 0, "linear_fwd: bad argument");
  return launch_linear_fwd(feat, w, bias, logits, rows, k, n_out, S(stream));
}

int dards_linear_bwd(const float* dlogits, const float* feat, const float* w, float* dfeat, float* dw, float* db,
                     int accumulate, int rows, int k, int n_out, void* stream) {
  DARDS_CHECK_ARG(dlogits && feat && w && k > 0, "linear_bwd: bad argument");
  return launch_linear_bwd(dlogits, feat, w, dfeat, dw, db, accumulate, rows, k, n_out, S(stream));
}

int dards_clamp_sgd_nesterov(float* param, const float* grad, float* momentum_buf, long long n, float lr,
                             float momentum, float weight_decay, float clip, float grad_scale, int first_step,
                             void* stream) {
  DARDS_CHECK_ARG(param && grad && momentum_buf && n >= 0, "clamp_sgd_nesterov: bad argument");
  return launch_clamp_sgd(param, grad, momentum_buf, n, lr, momentum, weight_decay, clip, grad_scale, first_step,
                          S(stream));
}

int dards_clamp_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                     float beta1, float beta2, float eps, float clip, float grad_scale, int step, void* stream) {
  DARDS_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && n >= 0, "clamp_adam: bad argument");
  return launch_clamp_adam(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, clip, grad_scale, step, S(stream));
}

int dards_scale_windows(const void* raw, int raw_f64, float* out, long long n, double mu, double std, int padded,
                        void* stream) {
  DARDS_CHECK_ARG(n >= 0, "scale_windows: negative size");
  return launch_scale_windows(raw, raw_f64, out, n, mu, std, padded, S(stream));
}

int dards_gradcam(const dards_gradcam_desc* d, void* stream) {
  DARDS_CHECK_ARG(d != nullptr, "gradcam: null descriptor");
  DARDS_CHECK_ARG(d->n_groups >= 0, "gradcam: negative size");
  DARDS_CHECK_ARG(d->resized_len >= 0 && ((d->read_resized == nullptr && d->seq_resized == nullptr) || d->resized_len > 0),
                  "gradcam: resized outputs need resized_len > 0");
  return launch_gradcam(*d, S(stream));
}

int dards_tc_debug_set(int key, int value) { return tc_debug_set(key, value); }

int dards_set_sm_limit(int n_sms) { return set_sm_limit(n_sms); }

}  // extern "C"

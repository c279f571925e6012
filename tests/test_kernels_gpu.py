"""GPU: every C-ABI kernel against the same operation done by PyTorch in fp32 (and, for bf16 storage,
against PyTorch on the bf16-rounded inputs).  Tolerances are written next to each check.

These are the per-kernel parity tests; tests/test_model_parity_gpu.py checks whole networks against the oracle
and the golden vectors recorded from the reference.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from tests.helpers import rel_err  # noqa: E402


def K():
    from deepards_b200 import kernels
    return kernels


def cl(x):  # (N, C, L) -> channels-last (N, L, C)
    return x.permute(0, 2, 1).contiguous()


def ncl(x):
    return x.permute(0, 2, 1).contiguous()


DEV = "cuda"

CONV_CASES = [
    # n, cin, cout, l, k, stride, pad
    (40, 64, 64, 56, 3, 1, 1),
    (40, 64, 128, 56, 3, 2, 1),
    (40, 64, 128, 56, 1, 2, 0),
    (20, 128, 128, 28, 3, 1, 1),
    (23, 256, 512, 14, 3, 2, 1),   # ragged number of breaths
    (33, 512, 512, 7, 3, 1, 1),
    (20, 96, 128, 28, 1, 1, 0),    # DenseNet conv1 (Cin = 96)
    (20, 128, 32, 14, 3, 1, 1),    # DenseNet conv2 (Cout = 32)
    (20, 16, 32, 56, 3, 2, 1),     # 16-plane ResNet
    (4, 64, 64, 224, 7, 2, 3),     # generic 7-tap
]


def _conv_inputs(case, seed=0):
    n, cin, cout, l, k, s, p = case
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(n, cin, l, generator=g).to(DEV)
    w = (torch.randn(cout, cin, k, generator=g) / (cin * k) ** 0.5).to(DEV)
    lo = (l + 2 * p - k) // s + 1
    dy = torch.randn(n, cout, lo, generator=g).to(DEV)
    return x, w, dy


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_simt_fp32(case):
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case)
    x.requires_grad_(True)
    w.requires_grad_(True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    y_ref = F.conv1d(x, w, stride=s, padding=p)
    dx_ref, dw_ref = torch.autograd.grad(y_ref, [x, w], dy)
    y = K().conv1d_fwd(cl(x.detach()), w.detach(), s, p, impl=0)
    assert rel_err(ncl(y), y_ref) < 2e-5
    dx = K().conv1d_dgrad(cl(dy), w.detach(), l, s, p, impl=0)
    assert rel_err(ncl(dx), dx_ref) < 2e-5
    dw = K().conv1d_wgrad(cl(x.detach()), cl(dy), k, s, p, impl=0)
    assert rel_err(dw, dw_ref) < 5e-5


def test_conv_simt_strided_views_and_addend():
    """channel slices of wider buffers (DenseNet concat) and the fused `+ addend` epilogue."""
    case = (20, 64, 32, 28, 3, 1, 1)
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 3)
    wide_in = torch.randn(n, l, 128, device=DEV)
    wide_in[:, :, :cin] = cl(x)
    wide_out = torch.zeros(n, l, 128, device=DEV)
    add = torch.randn(n, l, cout, device=DEV)
    K().conv1d_fwd(wide_in[:, :, :cin], w, s, p, impl=0, out=wide_out[:, :, 96:128], addend=add)
    ref = cl(F.conv1d(x, w, stride=s, padding=p)) + add
    assert rel_err(wide_out[:, :, 96:128], ref) < 2e-5
    assert float(wide_out[:, :, :96].abs().max()) == 0.0  # nothing outside the slice was touched


@pytest.mark.parametrize("case", CONV_CASES[:8])
def test_conv_simt_bf16_storage(case):
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 1)
    xb, wb, dyb = x.bfloat16(), w.bfloat16(), dy.bfloat16()
    xr = xb.float().requires_grad_(True)
    wr = wb.float().requires_grad_(True)
    y_ref = F.conv1d(xr, wr, stride=s, padding=p)
    dx_ref, dw_ref = torch.autograd.grad(y_ref, [xr, wr], dyb.float())
    # bf16 output rounding: 2^-8 relative per element
    y = K().conv1d_fwd(cl(xb), w, s, p, impl=0)
    assert rel_err(ncl(y).float(), y_ref) < 6e-3
    dx = K().conv1d_dgrad(cl(dyb), w, l, s, p, impl=0)
    assert rel_err(ncl(dx).float(), dx_ref) < 6e-3
    dw = K().conv1d_wgrad(cl(xb), cl(dyb), k, s, p, impl=0)  # fp32 output, bf16-rounded weights not involved
    assert rel_err(dw, dw_ref) < 1e-4


@pytest.mark.parametrize("case", CONV_CASES[:9])
def test_conv_tcgen05_forward(case):
    """tcgen05/TMEM/TMA implicit GEMM == CUDA-core kernel on identical bf16 operands (fp32 accumulation both)."""
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 2)
    xb = cl(x.bfloat16())
    y_simt = K().conv1d_fwd(xb, w, s, p, impl=0)
    y_tc = K().conv1d_fwd(xb, w, s, p, impl=1)
    torch.cuda.synchronize()
    # both round the same fp32 sums (different summation order) to bf16: at most one bf16 ulp apart
    assert rel_err(y_tc.float(), y_simt.float()) < 8e-3
    ref = cl(F.conv1d(xb.permute(0, 2, 1).float(), w.bfloat16().float(), stride=s, padding=p))
    assert rel_err(y_tc.float(), ref) < 6e-3


@pytest.mark.parametrize("case", CONV_CASES[:9])
@pytest.mark.parametrize("with_addend", [False, True])
def test_conv_tcgen05_dgrad(case, with_addend):
    """stride 1 and stride 2 (one launch per output parity plane); in-place accumulation = TMA reduce-add."""
    n, cin, cout, l, k, s, p = case
    if k == 1 and s == 2 and not with_addend:
        pytest.skip("1x1 stride-2 dgrad leaves the odd plane untouched: only defined as an accumulation")
    x, w, dy = _conv_inputs(case, 4)
    dyb = cl(dy.bfloat16())
    add = torch.randn(n, l, cin, device=DEV).bfloat16() if with_addend else None
    d_simt = K().conv1d_dgrad(dyb, w, l, s, p, impl=0, addend=add)
    d_tc = K().conv1d_dgrad(dyb, w, l, s, p, impl=1, addend=add)
    torch.cuda.synchronize()
    # accumulate path: the TMA unit adds two bf16 values (result rounded once more) -> 2 bf16 ulps
    assert rel_err(d_tc.float(), d_simt.float()) < (1.6e-2 if with_addend else 8e-3)


@pytest.mark.parametrize("case", [(5120, 512, 512, 7, 3, 1, 1), (5120, 256, 256, 14, 3, 1, 1), (5120, 256, 512, 14, 3, 2, 1),
                                  (5120, 128, 256, 28, 1, 2, 0), (1000, 256, 256, 14, 3, 1, 1), (37, 512, 512, 7, 3, 1, 1)])
def test_conv_tcgen05_wave_balanced_tile_width(case):
    """Opt-in tile width that follows the persistent schedule (e.g. 36 x 7 = 252 columns issued as N = 256 MMAs, 3.9
    waves instead of 4.3; measured slower, so not the default): same per-column accumulation order, so forward, dgrad
    and in-place dgrad are bit-identical to the widest-multiple-of-16 tiling; the direct-store epilogue agrees too."""
    from deepards_b200 import _lib
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 3)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    add = torch.randn(n, l, cin, device=DEV).bfloat16()
    outs = {}
    for mode in (-1, 1):  # -1: default (widest multiple of 16 columns); 1: wave-balanced
        _lib.call("dards_tc_debug_set", 8, mode)
        try:
            outs[mode] = (K().conv1d_fwd(xb, w, s, p, impl=1), K().conv1d_dgrad(dyb, w, l, s, p, impl=1, addend=add))
            if mode == 1 and n < 100:
                _lib.call("dards_tc_debug_set", 4, 0)
                outs["direct"] = K().conv1d_fwd(xb, w, s, p, impl=1)
        finally:
            _lib.call("dards_tc_debug_set", 8, -1)
            _lib.call("dards_tc_debug_set", 4, -1)
    torch.cuda.synchronize()
    assert torch.equal(outs[1][0], outs[-1][0]) and torch.equal(outs[1][1], outs[-1][1])
    if "direct" in outs:
        assert torch.equal(outs["direct"], outs[-1][0])
    if n <= 1000:
        ref = cl(F.conv1d(xb.permute(0, 2, 1).float(), w.bfloat16().float(), stride=s, padding=p))
        assert rel_err(outs[-1][0].float(), ref) < 6e-3


PAIR_CASES = [
    (23, 256, 512, 14, 3, 2, 1),    # stride 2, ragged: the second CTA's half tile is partly / entirely out of bounds
    (33, 512, 512, 7, 3, 1, 1),
    (640, 256, 256, 14, 3, 1, 1),   # 80 pair jobs: several rounds of the 6-stage ring and of the TMEM double buffer
]


@pytest.mark.parametrize("case", PAIR_CASES)
def test_conv_tcgen05_cta_pair_kernel_equals_single_cta_kernel(case):
    """tcgen05.mma.cta_group::2 (two CTAs = two output-channel tiles sharing one activation tile, half of it staged by
    each) accumulates every output element over the same K order as the single-CTA kernel: forward, dgrad and in-place
    dgrad (TMA reduce-add) are bit-identical; the weight-gradient kernel's pair mode likewise (deterministic reduce)."""
    from deepards_b200 import _lib
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 5)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    add = torch.randn(n, l, cin, device=DEV).bfloat16()
    outs = {}
    for mode in (0, 1):
        _lib.call("dards_tc_debug_set", 17, mode)
        _lib.call("dards_tc_debug_set", 19, mode)
        try:
            outs[mode] = (K().conv1d_fwd(xb, w, s, p, impl=1), K().conv1d_dgrad(dyb, w, l, s, p, impl=1),
                          K().conv1d_dgrad(dyb, w, l, s, p, impl=1, addend=add), K().conv1d_wgrad(xb, dyb, k, s, p, impl=1))
        finally:
            _lib.call("dards_tc_debug_set", 17, -1)
            _lib.call("dards_tc_debug_set", 19, -1)
    torch.cuda.synchronize()
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)
    ref = cl(F.conv1d(xb.permute(0, 2, 1).float(), w.bfloat16().float(), stride=s, padding=p))
    assert rel_err(outs[1][0].float(), ref) < 6e-3


def test_conv_tcgen05_direct_store_epilogue_matches_tma_store():
    from deepards_b200 import _lib
    case = CONV_CASES[3]
    n, cin, cout, l, k, s, p = case
    x, w, _ = _conv_inputs(case, 6)
    xb = cl(x.bfloat16())
    _lib.call("dards_tc_debug_set", 5, 0)  # the one-load-per-tap kernel (the only one with a direct-store fallback)
    try:
        y_tma = K().conv1d_fwd(xb, w, s, p, impl=1)
        _lib.call("dards_tc_debug_set", 4, 0)
        y_direct = K().conv1d_fwd(xb, w, s, p, impl=1)
    finally:
        _lib.call("dards_tc_debug_set", 4, -1)
        _lib.call("dards_tc_debug_set", 5, -1)
    torch.cuda.synchronize()
    assert torch.equal(y_tma, y_direct)


@pytest.mark.parametrize("case", [(40, 64, 64, 56, 3, 1, 1), (45, 128, 128, 28, 3, 1, 1), (70, 256, 256, 14, 3, 1, 1),
                                  (61, 512, 512, 7, 3, 1, 1), (20, 128, 32, 14, 3, 1, 1), (9, 96, 160, 20, 3, 1, 1),
                                  (1, 64, 64, 56, 3, 1, 1), (1030, 64, 64, 7, 3, 1, 1)])
def test_conv_tcgen05_three_tap_single_load_kernel(case):
    """k3/s1/p1 kernel with ONE staged activation tile for the three taps (halo rows + row-shifted descriptors)
    against the one-load-per-tap kernel (3- and 4-stage variants, whole- and half-tile epilogues), forward,
    dgrad and in-place dgrad; ragged breath counts (partial last tile), channel counts that are not tile multiples."""
    from deepards_b200 import _lib
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 12)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    add = torch.randn(n, l, cin, device=DEV).bfloat16()
    outs = {}
    for mode in (0, 1):  # 0: one load per tap (the wide-layer kernel), 1: single load (default for <= 128 channels)
        _lib.call("dards_tc_debug_set", 5, mode)
        try:
            outs[mode] = (K().conv1d_fwd(xb, w, s, p, impl=1), K().conv1d_dgrad(dyb, w, l, s, p, impl=1),
                          K().conv1d_dgrad(dyb, w, l, s, p, impl=1, addend=add))
        finally:
            _lib.call("dards_tc_debug_set", 5, -1)
    (y2, d2, a2), (y3, d3, a3) = outs[0], outs[1]
    torch.cuda.synchronize()
    ref = cl(F.conv1d(xb.permute(0, 2, 1).float(), w.bfloat16().float(), stride=s, padding=p))
    assert rel_err(y3.float(), ref) < 6e-3
    # fp32 accumulation order differs (tap-major vs chunk-major): at most one bf16 ulp
    assert rel_err(y3.float(), y2.float()) < 8e-3
    assert rel_err(d3.float(), d2.float()) < 8e-3
    assert rel_err(a3.float(), a2.float()) < 1.6e-2


WGRAD_CASES = [c for c in CONV_CASES[:9]] + [(256, 64, 64, 56, 3, 1, 1), (37, 128, 256, 28, 3, 2, 1),
                                             # BASELINE batch (5120 breaths): one wave of split-K CTAs
                                             (5120, 512, 512, 7, 3, 1, 1), (5120, 256, 256, 14, 3, 1, 1),
                                             (5120, 64, 64, 56, 3, 1, 1), (5120, 256, 512, 14, 3, 2, 1),
                                             (5120, 128, 256, 28, 1, 2, 0), (2000, 128, 32, 14, 3, 1, 1)]


@pytest.mark.parametrize("case", WGRAD_CASES)
def test_conv_tcgen05_wgrad(case):
    """tcgen05 weight gradient (MN-major operands, shifted-descriptor taps) == CUDA-core wgrad on the same bf16 data."""
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 7)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    ref = K().conv1d_wgrad(xb, dyb, k, s, p, impl=0)
    got = K().conv1d_wgrad(xb, dyb, k, s, p, impl=1)
    torch.cuda.synchronize()
    assert rel_err(got, ref) < 2e-4, rel_err(got, ref)  # both accumulate exact bf16 products in fp32
    assert torch.equal(got, K().conv1d_wgrad(xb, dyb, k, s, p, impl=1))  # deterministic (fixed-order split-K reduction)


@pytest.mark.parametrize("case", [(40, 64, 64, 56, 3, 1, 1), (40, 64, 128, 56, 3, 2, 1), (40, 64, 128, 56, 1, 2, 0),
                                  (300, 128, 128, 28, 3, 1, 1), (23, 256, 512, 14, 3, 2, 1), (333, 512, 512, 7, 3, 1, 1),
                                  (60, 96, 128, 28, 1, 1, 0), (60, 128, 32, 14, 3, 1, 1), (5120, 256, 256, 14, 3, 1, 1)])
def test_conv_tcgen05_wgrad_accumulate_mode(case):
    """The accumulate path (TMA reduce-add of every CTA's fp32 tile into a tap-major buffer at the L2 + one unpack launch)
    against the deterministic split-K path: same products, fp32 additions in a different (arrival) order."""
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 13)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    ref = K().conv1d_wgrad(xb, dyb, k, s, p, impl=1)
    got = K().conv1d_wgrad_accum(xb, dyb, k, s, p)
    assert rel_err(got, ref) < 1e-5, rel_err(got, ref)
    assert rel_err(got, K().conv1d_wgrad(xb, dyb, k, s, p, impl=0)) < 2e-4


@pytest.mark.parametrize("case", [(40, 64, 64, 56, 3, 1, 1), (333, 64, 128, 28, 3, 1, 1), (2000, 64, 32, 7, 3, 1, 1)])
def test_conv_tcgen05_wgrad_fused_taps(case):
    """64 input channels: the three taps issued as ONE N = 192 MMA (descriptor chunk stride = one row) accumulate the
    same products in the same order as three N = 64 MMAs -> bit-identical weight gradients."""
    from deepards_b200 import _lib
    n, cin, cout, l, k, s, p = case
    x, w, dy = _conv_inputs(case, 9)
    xb, dyb = cl(x.bfloat16()), cl(dy.bfloat16())
    fused = K().conv1d_wgrad(xb, dyb, k, s, p, impl=1)
    _lib.call("dards_tc_debug_set", 7, 0)
    try:
        three = K().conv1d_wgrad(xb, dyb, k, s, p, impl=1)
    finally:
        _lib.call("dards_tc_debug_set", 7, -1)
    torch.cuda.synchronize()
    assert torch.equal(fused, three)
    assert rel_err(fused, K().conv1d_wgrad(xb, dyb, k, s, p, impl=0)) < 2e-4


def test_conv_tcgen05_into_channel_slice():
    case = (20, 128, 32, 14, 3, 1, 1)
    n, cin, cout, l, k, s, p = case
    x, w, _ = _conv_inputs(case, 5)
    xb = cl(x.bfloat16())
    wide = torch.zeros(n, l, 128, device=DEV, dtype=torch.bfloat16)
    K().conv1d_fwd(xb, w, s, p, impl=1, out=wide[:, :, 64:96])
    ref = K().conv1d_fwd(xb, w, s, p, impl=0)
    torch.cuda.synchronize()
    assert rel_err(wide[:, :, 64:96].float(), ref.float()) < 8e-3
    assert float(wide[:, :, :64].abs().max()) == 0.0 and float(wide[:, :, 96:].abs().max()) == 0.0


def _bn_ref(x, gamma, beta, group, relu, res=None):
    """x (N, C, L); per-group training-mode batch norm with autograd."""
    outs = []
    for i in range(0, x.shape[0], group):
        y = F.batch_norm(x[i:i + group], None, None, gamma, beta, True, 0.0, 1e-5)
        outs.append(y)
    y = torch.cat(outs)
    if res is not None:
        y = y + res
    return F.relu(y) if relu else y


@pytest.mark.parametrize("n,c,l,group", [(40, 64, 56, 20), (60, 128, 7, 20), (24, 16, 28, 8), (20, 96, 14, 20)])
@pytest.mark.parametrize("variant", ["relu", "plain", "res_relu"])
def test_gbn_forward_backward_fp32(n, c, l, group, variant):
    g = torch.Generator().manual_seed(7)
    x = (torch.randn(n, c, l, generator=g) * 2 + 0.5).to(DEV).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV).requires_grad_(True)
    beta = (0.2 * torch.randn(c, generator=g)).to(DEV).requires_grad_(True)
    res = torch.randn(n, c, l, generator=g).to(DEV).requires_grad_(True) if variant == "res_relu" else None
    dy = torch.randn(n, c, l, generator=g).to(DEV)
    relu = variant != "plain"
    y_ref = _bn_ref(x, gamma, beta, group, relu, res)
    ins = [x, gamma, beta] + ([res] if res is not None else [])
    grads = torch.autograd.grad(y_ref, ins, dy)
    out, mean, rstd = K().gbn_fwd(cl(x.detach()), gamma.detach(), beta.detach(), group * l, relu,
                                  res=cl(res.detach()) if res is not None else None)
    assert rel_err(ncl(out), y_ref) < 1e-5
    mode = 0 if variant == "plain" else (1 if variant == "relu" else 2)
    dx, dgamma, dbeta, dres = K().gbn_bwd(cl(dy), cl(x.detach()), gamma.detach(), beta.detach(), mean, rstd, group * l,
                                          mode, mask_src=out if mode == 2 else None, want_dres=res is not None)
    assert rel_err(ncl(dx), grads[0]) < 2e-5
    assert rel_err(dgamma, grads[1]) < 2e-5
    assert rel_err(dbeta, grads[2]) < 2e-5
    if res is not None:
        assert rel_err(ncl(dres), grads[3]) < 1e-6


def test_gbn_bf16_storage():
    n, c, l, group = 40, 64, 28, 20
    g = torch.Generator().manual_seed(8)
    x = torch.randn(n, c, l, generator=g).to(DEV).bfloat16()
    gamma = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV)
    beta = (0.2 * torch.randn(c, generator=g)).to(DEV)
    y_ref = _bn_ref(x.float(), gamma, beta, group, True)
    out, mean, rstd = K().gbn_fwd(cl(x), gamma, beta, group * l, True)
    assert out.dtype == torch.bfloat16
    assert rel_err(ncl(out).float(), y_ref) < 6e-3


def test_bn_running_update_matches_sequential_torch():
    from deepards_b200 import _lib
    n, c, l, group = 60, 32, 14, 20
    g = torch.Generator().manual_seed(9)
    x = torch.randn(n, c, l, generator=g).to(DEV)
    bn = torch.nn.BatchNorm1d(c).to(DEV).train()
    for i in range(0, n, group):
        bn(x[i:i + group])
    gamma, beta = torch.ones(c, device=DEV), torch.zeros(c, device=DEV)
    _, mean, rstd = K().gbn_fwd(cl(x), gamma, beta, group * l, False)
    rm, rv = torch.zeros(c, device=DEV), torch.ones(c, device=DEV)
    nbt = torch.zeros((), dtype=torch.long, device=DEV)
    _lib.call("dards_bn_running_update", mean.data_ptr(), rstd.data_ptr(), rm.data_ptr(), rv.data_ptr(), nbt.data_ptr(),
              n // group, group * l, c, 0.1, 1e-5, torch.cuda.current_stream().cuda_stream)
    assert rel_err(rm, bn.running_mean) < 1e-5
    assert rel_err(rv, bn.running_var) < 1e-5
    assert int(nbt) == 3


@pytest.mark.parametrize("n,c,l,group,dtype", [(120, 64, 14, 20, torch.float32), (5120, 512, 7, 20, torch.bfloat16),
                                               (5120, 64, 56, 20, torch.bfloat16), (60, 96, 28, 20, torch.bfloat16),
                                               (40, 128, 28, 20, torch.bfloat16), (30, 64, 56, 30, torch.bfloat16)])
def test_gbn_layer_shapes_cached_and_streaming_kernels(n, c, l, group, dtype):
    """Every tile configuration of the cached kernels (and the streaming fallback for the 30-breath group) against
    torch, forward and backward, residual + mask variant included."""
    g = torch.Generator().manual_seed(21)
    x = torch.randn(n, c, l, generator=g).to(DEV).to(dtype)
    res = torch.randn(n, c, l, generator=g).to(DEV).to(dtype)
    gamma = (1 + 0.2 * torch.randn(c, generator=g)).to(DEV).requires_grad_(True)
    beta = (0.2 * torch.randn(c, generator=g)).to(DEV).requires_grad_(True)
    dy = torch.randn(n, c, l, generator=g).to(DEV).to(dtype)
    tol = 1e-5 if dtype == torch.float32 else 1.2e-2
    xr, rr = x.float().requires_grad_(True), res.float().requires_grad_(True)
    y_ref = _bn_ref(xr, gamma, beta, group, True, rr)
    gx, gg, gb, gr = torch.autograd.grad(y_ref, [xr, gamma, beta, rr], dy.float())
    out, mean, rstd = K().gbn_fwd(cl(x), gamma.detach(), beta.detach(), group * l, True, res=cl(res))
    assert rel_err(ncl(out).float(), y_ref) < tol
    # the mask comes from the reference output so that bf16 rounding of `out` cannot flip a decision
    mask = cl((y_ref > 0).to(dtype))
    dx, dgamma, dbeta, dres = K().gbn_bwd(cl(dy), cl(x), gamma.detach(), beta.detach(), mean, rstd, group * l, 2,
                                          mask_src=mask, want_dres=True)
    assert rel_err(ncl(dx).float(), gx) < tol
    assert rel_err(dgamma, gg) < tol and rel_err(dbeta, gb) < tol
    assert rel_err(ncl(dres).float(), gr) < (1e-6 if dtype == torch.float32 else 1e-2)
    # determinism
    dx2, dgamma2, dbeta2, _ = K().gbn_bwd(cl(dy), cl(x), gamma.detach(), beta.detach(), mean, rstd, group * l, 2,
                                          mask_src=mask, want_dres=True)
    assert torch.equal(dx, dx2) and torch.equal(dgamma, dgamma2) and torch.equal(dbeta, dbeta2)


def test_batched_running_update_reduce_rows_and_pack():
    from deepards_b200 import _lib
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(22)
    # ---- running statistics of several BatchNorm layers in one launch == torch's sequential update ----
    layers, rows_tab = [], []
    for (n, c, l, group) in [(100, 64, 14, 20), (100, 96, 7, 20), (60, 512, 7, 20)]:
        x = torch.randn(n, c, l, generator=g).to(DEV)
        bn = torch.nn.BatchNorm1d(c).to(DEV).train()
        for i in range(0, n, group):
            bn(x[i:i + group])
        _, mean, rstd = K().gbn_fwd(cl(x), torch.ones(c, device=DEV), torch.zeros(c, device=DEV), group * l, False)
        rm, rv = torch.zeros(c, device=DEV), torch.ones(c, device=DEV)
        nbt = torch.zeros((), dtype=torch.long, device=DEV)
        layers.append((bn, rm, rv, nbt, n // group, mean, rstd))
        rows_tab.append((mean.data_ptr(), rstd.data_ptr(), rm.data_ptr(), rv.data_ptr(), nbt.data_ptr(), n // group,
                         group * l, c, 0.1))
    tab, total = _lib.desc_table(_lib.RunningDesc, rows_tab, DEV)
    _lib.call("dards_bn_running_update_batched", tab.data_ptr(), len(rows_tab), total, 1e-5, st)
    for bn, rm, rv, nbt, ng, _, _ in layers:
        assert rel_err(rm, bn.running_mean) < 2e-5 and rel_err(rv, bn.running_var) < 2e-5 and int(nbt) == ng
    # ---- batched row reduction ----
    parts = [torch.randn(r, c, generator=g).to(DEV) for r, c in [(256, 64), (256, 448), (7, 12), (300, 512)]]
    outs = [torch.full((p.shape[1],), 3.0, device=DEV) for p in parts]
    rows_tab = [(p.data_ptr(), o.data_ptr(), p.shape[0], p.shape[1], 1 if i == 2 else 0)
                for i, (p, o) in enumerate(zip(parts, outs))]
    tab, total = _lib.desc_table(_lib.ReduceDesc, rows_tab, DEV)
    _lib.call("dards_reduce_rows_batched", tab.data_ptr(), len(parts), total, st)
    for i, (p, o) in enumerate(zip(parts, outs)):
        assert rel_err(o, p.sum(0) + (3.0 if i == 2 else 0.0)) < 1e-5
    # ---- batched weight packing == per-tensor packing ----
    shapes = [(64, 64, 3), (128, 64, 1), (512, 256, 3), (32, 128, 3), (40, 24, 5)]
    ws = [torch.randn(s, generator=g).to(DEV) for s in shapes]
    rows_tab, outs = [], []
    for wt in ws:
        co, ci, k = wt.shape
        kio = torch.zeros((k, ci, co), dtype=torch.bfloat16, device=DEV)
        koi = torch.zeros((k, co, ci), dtype=torch.bfloat16, device=DEV)
        outs.append((kio, koi))
        rows_tab.append((wt.data_ptr(), kio.data_ptr(), koi.data_ptr(), co, ci, k))
    tab, total = _lib.desc_table(_lib.PackDesc, rows_tab, DEV)
    _lib.call("dards_pack_conv_weights_batched", tab.data_ptr(), len(ws), total, _lib.BF16, st)
    for wt, (kio, koi) in zip(ws, outs):
        r_kio, r_koi = K().pack_conv_weight(wt, torch.bfloat16)
        assert torch.equal(kio, r_kio) and torch.equal(koi, r_koi)


@pytest.mark.parametrize("c0,group,pool", [(64, 20, 0), (16, 20, 0), (64, 20, 1), (32, 7, 0), (64, 60, 0),
                                           (64, 226, 0),     # the largest group of the one-kernel path
                                           (64, 227, 0),     # chunked path: 3 chunks of 64 + one of 35 breaths
                                           (32, 300, 1), (16, 640, 0)])
def test_stem_forward_backward(c0, group, pool):
    """group <= 226: one fused kernel per direction; above: STATS + APPLY chunk passes forward, PARTIAL + combine backward
    (a flat batch is one BatchNorm group: ResNet.forward(x) / DenseNet.forward(x) / CNNRegressor, ADVICE r1)."""
    n = group * (3 if group <= 226 else 2)
    g = torch.Generator().manual_seed(10)
    x = torch.randn(n, 1, 224, generator=g).to(DEV)
    w = (torch.randn(c0, 1, 7, generator=g) * 0.3).to(DEV).requires_grad_(True)
    gamma = (1 + 0.2 * torch.randn(c0, generator=g)).to(DEV).requires_grad_(True)
    beta = (0.2 * torch.randn(c0, generator=g)).to(DEV).requires_grad_(True)
    dy = torch.randn(n, c0, 56, generator=g).to(DEV)
    outs = []
    for i in range(0, n, group):
        y = F.conv1d(x[i:i + group], w, stride=2, padding=3)
        y = F.relu(F.batch_norm(y, None, None, gamma, beta, True, 0.0, 1e-5))
        y = F.max_pool1d(y, 3, 2, 1) if pool == 0 else F.avg_pool1d(y, 3, 2, 1)
        outs.append(y)
    y_ref = torch.cat(outs)
    gw, gg, gb = torch.autograd.grad(y_ref, [w, gamma, beta], dy)
    out, mean, rstd = K().stem_fwd(x.view(n, 224), w.detach(), gamma.detach(), beta.detach(), group, pool, torch.float32)
    assert rel_err(ncl(out), y_ref) < 1e-5
    dw, dgamma, dbeta = K().stem_bwd(cl(dy), x.view(n, 224), w.detach(), gamma.detach(), beta.detach(), mean, rstd, group,
                                     pool)
    assert rel_err(dw, gw) < 5e-5
    assert rel_err(dgamma, gg) < 5e-5
    assert rel_err(dbeta, gb) < 5e-5


def test_pools_and_linear_and_bce():
    g = torch.Generator().manual_seed(11)
    x = torch.randn(40, 64, 28, generator=g).to(DEV)
    assert rel_err(ncl(K().avgpool2(cl(x))), F.avg_pool1d(x, 2, 2)) < 1e-6
    dy = torch.randn(40, 64, 14, generator=g).to(DEV)
    xr = x.clone().requires_grad_(True)
    (gx,) = torch.autograd.grad(F.avg_pool1d(xr, 2, 2), xr, dy)
    assert rel_err(ncl(K().avgpool2(cl(dy), backward=True)), gx) < 1e-6
    x7 = torch.randn(40, 128, 7, generator=g).to(DEV)
    feat = K().avgpool_full(cl(x7))
    assert rel_err(feat, F.avg_pool1d(x7, 7, 1).view(40, -1)) < 1e-6
    dfeat = torch.randn(40, 128, generator=g).to(DEV)
    assert rel_err(ncl(K().avgpool_full_bwd(dfeat, 7, torch.float32)), (dfeat / 7).unsqueeze(-1).expand(40, 128, 7)) < 1e-6
    # linear head: rows = sequences, K = 20*F
    f = torch.randn(6, 20 * 128, generator=g).to(DEV).requires_grad_(True)
    w = (torch.randn(2, 20 * 128, generator=g) * 0.02).to(DEV).requires_grad_(True)
    b = torch.randn(2, generator=g).to(DEV).requires_grad_(True)
    t = torch.tensor([[1., 0.]] * 3 + [[0., 1.]] * 3, device=DEV)
    out_ref = F.linear(f, w, b)
    loss_ref = F.binary_cross_entropy_with_logits(out_ref, t)
    gf, gw, gb = torch.autograd.grad(loss_ref, [f, w, b])
    out = K().linear_fwd(f.detach(), w.detach(), b.detach())
    assert rel_err(out, out_ref) < 1e-5
    loss, dl = K().bce_with_logits(out, t)
    assert abs(float(loss) - float(loss_ref)) < 1e-6
    dfeat, dw, db = K().linear_bwd(dl, f.detach(), w.detach())
    assert rel_err(dfeat, gf) < 1e-5 and rel_err(dw, gw) < 1e-5 and rel_err(db, gb) < 1e-5


def test_dropout_mask_is_reproducible_and_unbiased():
    x = torch.ones(64, 28, 32, device=DEV)
    a = K().dropout_(x.clone(), 0.2, 1234)
    b = K().dropout_(x.clone(), 0.2, 1234)
    c = K().dropout_(x.clone(), 0.2, 99)
    assert torch.equal(a, b) and not torch.equal(a, c)
    kept = (a > 0).float().mean().item()
    assert abs(kept - 0.8) < 0.01
    assert abs(float(a.max()) - 1.25) < 1e-6
    off = torch.tensor([5, 0], dtype=torch.int64, device=DEV)     # [step counter, first sequence]
    d = K().dropout_(x.clone(), 0.2, 1234, off)
    assert not torch.equal(a, d)
    # keyed by the GLOBAL element index (SURVEY.md 8e(iv)): the second half of the batch, run as its own shard with
    # first_sequence = 2 (of 4 sequences x 16 breaths x 28 rows), draws exactly the masks it has inside the whole batch;
    # a channel slice of a wider buffer and bf16 storage do not change them either
    rows_per_seq = 16 * 28
    whole = K().dropout_(x.clone(), 0.2, 1234, torch.tensor([7, 0], dtype=torch.int64, device=DEV), rows_per_seq)
    shard = K().dropout_(x[32:].clone(), 0.2, 1234, torch.tensor([7, 2], dtype=torch.int64, device=DEV), rows_per_seq)
    assert torch.equal(whole[32:], shard)
    wide = torch.ones(64, 28, 96, device=DEV)
    K().dropout_(wide[:, :, 64:96], 0.2, 1234, torch.tensor([7, 0], dtype=torch.int64, device=DEV), rows_per_seq)
    assert torch.equal(wide[:, :, 64:96], whole) and float(wide[:, :, :64].min()) == 1.0
    hb = K().dropout_(x.clone().bfloat16(), 0.2, 1234, torch.tensor([7, 0], dtype=torch.int64, device=DEV), rows_per_seq)
    assert torch.equal(hb > 0, whole > 0)


def test_fused_optimizers_match_torch():
    from deepards_b200 import _lib
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(12)
    p0 = torch.randn(10007, generator=g).to(DEV)
    grads = [(torch.randn(10007, generator=g) * 0.05).to(DEV) for _ in range(3)]
    # SGD nesterov with the reference's clamp hook
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.SGD([p_ref], lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    p = p0.clone()
    m = torch.zeros_like(p)
    for i, gr in enumerate(grads):
        p_ref.grad = gr.clamp(-0.01, 0.01)
        opt.step()
        _lib.call("dards_clamp_sgd_nesterov", p.data_ptr(), gr.data_ptr(), m.data_ptr(), p.numel(), 1e-3, 0.9, 1e-4, 0.01,
                  1.0, 1 if i == 0 else 0, st)
    assert rel_err(p, p_ref.detach()) < 1e-6
    # Adam
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([p_ref], lr=1e-3)
    p = p0.clone()
    ea, es = torch.zeros_like(p), torch.zeros_like(p)
    for i, gr in enumerate(grads):
        p_ref.grad = gr.clone()
        opt.step()
        _lib.call("dards_clamp_adam", p.data_ptr(), gr.data_ptr(), ea.data_ptr(), es.data_ptr(), p.numel(), 1e-3, 0.9,
                  0.999, 1e-8, 0.0, 1.0, i + 1, st)
    assert rel_err(p, p_ref.detach()) < 1e-5


# ---------------------------------------------------------------------------------------------------------------
# convolution + grouped BatchNorm (+ residual) (+ ReLU) in one tcgen05 kernel (conv_bn_tc.cu, bn_apply.cu)
# ---------------------------------------------------------------------------------------------------------------
CONV_BN_CASES = [
    # n, group, cin, cout, l, k, stride, pad, relu, residual, expected mode
    (40, 20, 64, 64, 56, 3, 1, 1, True, False, 1),      # ResNet layer 1: partial statistics + streaming apply
    (40, 20, 64, 64, 56, 3, 1, 1, True, True, 1),
    (40, 20, 64, 128, 56, 3, 2, 1, True, False, 1),     # layer2.0.conv1 (stride 2, per-tap loads)
    (60, 20, 128, 128, 28, 3, 1, 1, True, True, 1),
    (40, 20, 128, 256, 28, 3, 2, 1, True, False, 2),    # layer3.0.conv1: the group fits on chip
    (60, 20, 256, 256, 14, 3, 1, 1, True, True, 2),     # layer 3: fused, 2 sub-tiles, 2 channel tiles
    (40, 20, 128, 256, 28, 1, 2, 0, False, False, 2),   # layer3 downsample (no ReLU)
    (40, 20, 256, 512, 14, 3, 2, 1, True, False, 2),
    (80, 20, 512, 512, 7, 3, 1, 1, True, True, 2),      # layer 4: fused, 1 sub-tile, 4 channel tiles
    (40, 20, 96, 128, 14, 1, 1, 0, True, False, 2),     # DenseNet conv1 + norm2 (Cin = 96)
    (40, 20, 64, 128, 56, 1, 1, 0, True, False, 1),     # DenseNet block 1 conv1 + norm2
    (60, 20, 512, 512, 7, 3, 1, 1, True, True, 2),      # odd number of groups: one group per job
    (3000, 20, 512, 512, 7, 3, 1, 1, True, True, 2),    # many jobs per CTA (persistent schedule, park reuse)
]


def _bn_group_ref(y, gamma, beta, group, eps=1e-5):
    """y (N, C, L) fp32 -> grouped training-mode BatchNorm (biased variance) + the statistics."""
    n, c, l = y.shape
    g = n // group
    yg = y.view(g, group, c, l)
    mean = yg.mean(dim=(1, 3))
    var = yg.var(dim=(1, 3), unbiased=False)
    rstd = (var + eps).rsqrt()
    out = (yg - mean[:, None, :, None]) * rstd[:, None, :, None] * gamma[None, None, :, None] + beta[None, None, :, None]
    return out.view(n, c, l), mean, rstd


@pytest.mark.parametrize("case", CONV_BN_CASES)
def test_conv_bn_tcgen05_fused(case):
    """y, statistics and the normalised output against torch on the same bf16 operands.  The statistics come from the
    fp32 accumulators (not from the bf16-rounded y), the normalisation is applied to the stored bf16 y."""
    n, group, cin, cout, l, k, s, p, relu, has_res, want_mode = case
    gen = torch.Generator(device="cpu").manual_seed(7)
    x = torch.randn(n, cin, l, generator=gen).to(DEV).bfloat16()
    w = (torch.randn(cout, cin, k, generator=gen) / (cin * k) ** 0.5).to(DEV)
    gamma = (1.0 + 0.2 * torch.randn(cout, generator=gen)).to(DEV)
    beta = (0.3 * torch.randn(cout, generator=gen)).to(DEV)
    lo = (l + 2 * p - k) // s + 1
    res = torch.randn(n, cout, lo, generator=gen).to(DEV).bfloat16() if has_res else None
    mode, y, out, mean, rstd, _ = K().conv1d_bn_fwd(cl(x), w, gamma, beta, group, s, p, relu,
                                                    res=cl(res) if has_res else None)
    torch.cuda.synchronize()
    assert mode == want_mode
    y_ref = F.conv1d(x.float(), w.bfloat16().float(), stride=s, padding=p)
    assert rel_err(ncl(y).float(), y_ref) < 6e-3          # bf16 rounding of the stored convolution output
    bn_ref, mean_ref, rstd_ref = _bn_group_ref(y_ref, gamma, beta, group)
    assert rel_err(mean, mean_ref) < 2e-5 and rel_err(rstd, rstd_ref) < 2e-5   # fp32 statistics of the fp32 sums
    # the kernel normalises the bf16-rounded y with those statistics
    yb = ncl(y).float().view(n // group, group, cout, lo)
    o_ref = ((yb - mean[:, None, :, None]) * rstd[:, None, :, None] * gamma[None, None, :, None] +
             beta[None, None, :, None]).view(n, cout, lo)
    if has_res:
        o_ref = o_ref + res.float()
    if relu:
        o_ref = o_ref.relu()
    assert rel_err(ncl(out).float(), o_ref) < 6e-3        # one bf16 rounding of the output
    full = bn_ref + (res.float() if has_res else 0)
    assert rel_err(ncl(out).float(), full.relu() if relu else full) < 2e-2


def test_conv_bn_tcgen05_downsample_branch_merged():
    """layer2.0 of ResNet-18: out = relu(bn2(conv2(a1)) + bn_d(conv1x1_s2(x))) -- both BatchNorms in ONE elementwise pass."""
    n, group = 40, 20
    gen = torch.Generator(device="cpu").manual_seed(11)
    a1 = torch.randn(n, 128, 28, generator=gen).to(DEV).bfloat16()
    xin = torch.randn(n, 64, 56, generator=gen).to(DEV).bfloat16()
    w2 = (torch.randn(128, 128, 3, generator=gen) / 384 ** 0.5).to(DEV)
    wd = (torch.randn(128, 64, 1, generator=gen) / 8.0).to(DEV)
    g2, b2 = (1 + 0.1 * torch.randn(128, generator=gen)).to(DEV), (0.1 * torch.randn(128, generator=gen)).to(DEV)
    gd, bd = (1 + 0.1 * torch.randn(128, generator=gen)).to(DEV), (0.1 * torch.randn(128, generator=gen)).to(DEV)
    mode, y, out, mean, rstd, ex = K().conv1d_bn_fwd(cl(a1), w2, g2, b2, group, 1, 1, True,
                                                     ds=(cl(xin), wd, gd, bd, 2, 0))
    torch.cuda.synchronize()
    assert mode == 1
    y2 = F.conv1d(a1.float(), w2.bfloat16().float(), padding=1)
    yd = F.conv1d(xin.float(), wd.bfloat16().float(), stride=2)
    o2, m2, r2 = _bn_group_ref(y2, g2, b2, group)
    od, md, rd = _bn_group_ref(yd, gd, bd, group)
    assert rel_err(mean, m2) < 2e-5 and rel_err(rstd, r2) < 2e-5
    assert rel_err(ex["mean_d"], md) < 2e-5 and rel_err(ex["rstd_d"], rd) < 2e-5
    assert rel_err(ncl(ex["y_d"]).float(), yd) < 6e-3
    assert rel_err(ncl(out).float(), (o2 + od).relu()) < 2e-2


@pytest.mark.parametrize("shape", [(256, 14, 3, 1, 1), (512, 7, 3, 1, 1), (128, 14, 1, 1, 0), (64, 56, 3, 1, 1)])
def test_conv_bn_tcgen05_is_slice_invariant(shape):
    """Groups are independent and every reduction has a fixed order: a group's results do not depend on how many other
    groups the launch holds, which CTA ran it, or which other group shared its job (bit for bit)."""
    c, l, k, s, p = shape
    group = 20
    gen = torch.Generator(device="cpu").manual_seed(3)
    n_big = 20 * 330                                  # more jobs than SMs: several jobs per CTA
    x = torch.randn(n_big, l, c, generator=gen).to(DEV).bfloat16()
    w = (torch.randn(c, c, k, generator=gen) / (c * k) ** 0.5).to(DEV)
    gamma = (1.0 + 0.2 * torch.randn(c, generator=gen)).to(DEV)
    beta = (0.3 * torch.randn(c, generator=gen)).to(DEV)
    _, y, out, mean, rstd, _ = K().conv1d_bn_fwd(x, w, gamma, beta, group, s, p, True)
    for lo, hi in ((0, 2), (100, 103), (327, 330)):   # even / odd number of groups in the small launch
        xs = x[lo * group:hi * group].contiguous()
        _, y2, out2, mean2, rstd2, _ = K().conv1d_bn_fwd(xs, w, gamma, beta, group, s, p, True)
        torch.cuda.synchronize()
        assert torch.equal(y[lo * group:hi * group], y2)
        assert torch.equal(mean[lo:hi], mean2) and torch.equal(rstd[lo:hi], rstd2)
        assert torch.equal(out[lo * group:hi * group], out2)
    assert bool(torch.isfinite(out.float()).all())

"""GPU: BatchNorm and stem kernels against float64 on the data where one-pass and folded formulas lose digits.

Every case runs a kernel through deepards_b200.kernels and compares it with the same operation done in float64 by
tests/numerics_reference.py on the kernel's own inputs (for bf16 storage: the bf16 values, upcast).  The data families
are the edges of the statistics: a mean large against the spread (x = m + s*z), exactly constant and all-zero channels
(var = 0, rstd = 1/sqrt(eps)), near-constant channels (var ~ 1e-8, far below eps), and whole zero breaths (what the
padded-breath rule feeds the network), for the stem also a group made of zero breaths.

Gates (constants below):
- fp32 results: err_kernel <= max(CAL * err_torch32, FLOOR), where err_torch32 is the error of the same closed form
  evaluated by torch in fp32 (TF32 off) on the same device against the same float64 reference.  A kernel may lose what
  fp32 itself loses on such data, not more.
- bf16 outputs: elementwise, one bf16 rounding of the float64 value: |out - ref| <= 2^-8 |ref| + BF16_ATOL * max |ref|.
ReLU and max-pool decisions are kept out of the arithmetic: the ReLU is either off, fed a mask taken from the
reference, or provably inactive (gamma in [0.1, 0.3], beta >= 2, or >= 4 for the stem, asserted on the reference),
and the stem uses the average pool.  Backward kernels get the float64 statistics rounded to fp32, so the error measured
is the backward's own.  `pytest -s` prints the per-case table of kernel and torch fp32 errors.
"""
import pytest
import torch
import torch.nn.functional as F

from tests import numerics_reference as R
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
CAL = 4.0          # the kernel may be this many times worse than torch fp32 on the same data
# fp32 accumulation-order noise of the kernels' reductions (1e2 .. 1e5 terms): torch reduces with cascaded sums, the kernels
# per thread and then across lanes, and on centred data a statistic can come out ~20x further from float64 than torch's
# (B200, offset 0: up to 3e-6 relative in rstd) without anything wrong.  80 ulps; 1/20 of the fp32 parity target below.
FLOOR = 5e-6
# A reduction (mean, rstd, dgamma, dbeta, dW) sums 1e3 .. 1e4 terms per thread lane in fp32 before the lanes combine:
# same-sign sums (sum of squares) of that length drift by up to n ulps; 2e-5 is what the stem statistics of a constant
# group reached (B200: 1.1e-5 in rstd, 226-breath group), 1/5 of the fp32 parity target.
STAT_FLOOR = 2e-5
PARITY = 1e-4      # the fp32 path's accuracy target against float64: the stem weight gradient must meet it at any offset
BF16_ATOL = 1e-4   # absolute slack of the bf16 gate, relative to the largest reference value
FP32_OFFSETS = (0.0, 10.0, 1e2, 1e3)
BF16_OFFSETS = (0.0, 10.0, 1e2)


def K():
    from deepards_b200 import kernels
    return kernels


@pytest.fixture(autouse=True, scope="module")
def _no_tf32():
    """The torch fp32 calibration must be fp32: TF32 convolutions would loosen every gate."""
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def cl(x):  # (N, C, L) -> channels-last (N, L, C)
    return x.permute(0, 2, 1).contiguous()


def ncl(x):
    return x.permute(0, 2, 1).contiguous()


# ---- error measures ---------------------------------------------------------------------------------------------------
def chan_err(a, ref, slack=None):
    """Worst channel's max |a - ref| / max |ref|: a channel with a large scale (rstd = 1/sqrt(eps)) cannot hide the
    others.  (N, C, L) or (C, ...) tensors; `slack` (broadcast to ref) is an allowed absolute error taken off first."""
    a, ref = a.double(), ref.double()
    d = (a - ref).abs()
    if slack is not None:
        d = torch.where(torch.isnan(d), d, (d - slack).clamp_min(0))
    if ref.dim() == 3:
        d, ref = d.transpose(0, 1), ref.transpose(0, 1)
    d, ref = d.reshape(ref.shape[0], -1), ref.reshape(ref.shape[0], -1)
    num, den = d.amax(1), ref.abs().amax(1)
    return float(torch.where(den > 0, num / den.clamp_min(1e-300), num).max())


def mean_err(a, mean, rstd):
    """|a - mean| in units of max(|mean|, std): a mean can be no better than its own fp32 rounding."""
    a = a.double()
    return float(((a - mean).abs() / (mean.abs() + 1.0 / rstd)).max())


def rstd_err(a, rstd):
    return float(((a.double() - rstd).abs() / rstd).max())


class Table:
    """Prints one line per check and collects the failures, so that a case reports every quantity before it fails."""

    def __init__(self, case, fails=None):
        self.case, self.fails = case, ([] if fails is None else fails)

    def cal(self, what, e_kernel, e_torch, floor=FLOOR):
        ok = e_kernel <= max(CAL * e_torch, floor)  # False for NaN
        print("%-46s %-10s kernel %9.2e  torch32 %9.2e  %s" % (self.case, what, e_kernel, e_torch, "ok" if ok else "FAIL"))
        if not ok:
            self.fails.append("%s %s: kernel %.3e > max(%g * torch32 %.3e, %g)" % (self.case, what, e_kernel, CAL, e_torch, floor))

    def bf16(self, what, out, ref, slack=0.0):
        out, ref = out.double(), ref.double()
        bound = 2.0 ** -8 * ref.abs() + BF16_ATOL * float(ref.abs().max()) + slack
        worst = float(((out - ref).abs() / bound).max())
        ok = bool(torch.isfinite(out).all()) and worst <= 1.0
        print("%-46s %-10s bf16 max |out-ref| / bound %.3f  %s" % (self.case, what, worst, "ok" if ok else "FAIL"))
        if not ok:
            self.fails.append("%s %s: bf16 elementwise gate exceeded (%.3f of the bound)" % (self.case, what, worst))

    def parity(self, what, e_kernel, bound=PARITY):
        ok = e_kernel <= bound
        print("%-46s %-10s kernel %9.2e  <= %g  %s" % (self.case, what, e_kernel, bound, "ok" if ok else "FAIL"))
        if not ok:
            self.fails.append("%s %s: kernel %.3e > %g" % (self.case, what, e_kernel, bound))

    def exact(self, what, ok):
        print("%-46s %-10s exact %s" % (self.case, what, "ok" if ok else "FAIL"))
        if not ok:
            self.fails.append("%s %s: not exact" % (self.case, what))

    def check(self):
        assert not self.fails, "\n  ".join(self.fails)


def _out(t, what, out, ref, ref32, dtype, slack=None):
    if dtype == BF16:
        t.bf16(what, out, ref, 0.0 if slack is None else slack)
    else:
        t.cal(what, chan_err(out, ref, slack), chan_err(ref32, ref))


def _vec(t, what, out, ref, ref32):
    t.cal(what, rel_err(out, ref), rel_err(ref32, ref), STAT_FLOOR)


def _stats(t, mean, rstd, mean32, rstd32, mean64, rstd64, prefix=""):
    t.cal(prefix + "mean", mean_err(mean, mean64, rstd64), mean_err(mean32, mean64, rstd64), STAT_FLOOR)
    t.cal(prefix + "rstd", rstd_err(rstd, rstd64), rstd_err(rstd32, rstd64), STAT_FLOOR)


# ---- grouped BatchNorm: gbn_fwd / gbn_bwd -----------------------------------------------------------------------------
def _bn_families(dtype):
    offsets = FP32_OFFSETS if dtype == F32 else BF16_OFFSETS
    return ["offset %g" % r for r in offsets] + ["constant channels", "zero breaths"]


def _bn_data(family, n, c, l, group, gen):
    """(N, C, L) float64 on the CPU."""
    z = torch.randn(n, c, l, generator=gen, dtype=F64)
    s = 0.5 + 1.5 * torch.rand(c, generator=gen, dtype=F64)
    sign = torch.where(torch.arange(c) % 2 == 0, 1.0, -1.0).to(F64)
    if family.startswith("offset"):
        r = float(family.split()[1])
        return (r * sign * s)[None, :, None] + s[None, :, None] * z
    if family == "constant channels":
        x = s[None, :, None] * z
        ch = torch.arange(c) % 8
        x[:, ch == 0] = 0.0                                             # all zero: var = 0
        x[:, ch == 1] = 3.0                                             # constant
        x[:, ch == 2] = -1e3                                            # constant, large
        x[:, ch == 3] = 5.0 + 1e-4 * z[:, ch == 3]                      # var ~ 1e-8 << eps (constant once in bf16)
        x[:, ch == 4] = 1e-4 * z[:, ch == 4]                            # var ~ 1e-8 around zero
        return x
    x = (10.0 * sign * s)[None, :, None] + s[None, :, None] * z         # zero breaths in offset data
    b = torch.arange(n) % group
    x[(b == 1) | (b == group - 1) | (b == group // 2)] = 0.0
    return x


GBN_SHAPES = [(120, 64, 14, 20), (5120, 512, 7, 20), (5120, 64, 56, 20), (60, 96, 28, 20), (40, 128, 28, 20),
              (30, 64, 56, 30)]   # the tile configurations of the cached kernels, and the streaming fallback (group 30)


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("n,c,l,group", GBN_SHAPES)
def test_gbn_forward_backward_against_float64(n, c, l, group, dtype):
    rows = group * l
    fails = []
    for family in _bn_families(dtype):
        gen = torch.Generator().manual_seed(31)
        xq = _bn_data(family, n, c, l, group, gen).to(DEV).to(dtype)
        g32 = (0.1 + 0.2 * torch.rand(c, generator=gen)).to(DEV)
        b32 = (2.0 + torch.rand(c, generator=gen)).to(DEV)
        res = (0.3 * (2 * torch.rand(n, c, l, generator=gen, dtype=F64) - 1)).to(DEV).to(dtype)
        dout = torch.randn(n, c, l, generator=gen, dtype=F64).to(DEV).to(dtype)
        mask_src = (torch.rand(n, c, l, generator=gen) < 0.7).to(DEV).to(dtype)   # relu_mode 2 reads mask_src > 0
        x64, x32 = xq.double(), xq.float()
        gamma, beta = g32.double(), b32.double()
        t = Table("gbn %s n%d c%d l%d g%d %s" % (str(dtype)[6:], n, c, l, group, family), fails)

        out64, pre64, mean64, rstd64 = R.gbn_forward(x64, gamma, beta, group, res=res.double(), relu=True)
        assert float(pre64.min()) > 0.05, "the ReLU must be inactive"
        out32, _, mean32, rstd32 = R.gbn_forward(x32, g32, b32, group, res=res.float(), relu=True)
        out, mean, rstd = K().gbn_fwd(cl(xq), g32, b32, rows, True, res=cl(res))
        # The forward evaluates fmaf(x, sc, beta - mean*sc) (sc = rstd*gamma): the rounding of the folded shift, 4 ulps of
        # mean*sc allowed here, is a loss torch's (x - mean)*sc does not have.  It shows where var << eps and |mean| >>
        # sqrt(eps): a constant channel at -1e3 (rstd = 1/sqrt(eps)) is off by ~1e-3 of the output.  A centred forward
        # would also have to move relu_mode 1's ReLU decision and the conv+BN epilogues, which share this arithmetic.
        fold = 2.0 ** -22 * (mean64 * rstd64 * gamma).abs().repeat_interleave(group, 0)[:, :, None]
        _out(t, "fwd out", ncl(out), out64, out32, dtype, slack=fold)
        _stats(t, mean, rstd, mean32, rstd32, mean64, rstd64, "fwd ")

        # backward with the float64 statistics rounded to fp32
        mean_f, rstd_f = mean64.float(), rstd64.float()
        xhat = (x64 - mean_f.double().repeat_interleave(group, 0)[:, :, None]) * \
            rstd_f.double().repeat_interleave(group, 0)[:, :, None]
        assert float((beta[None, :, None] + gamma[None, :, None] * xhat).min()) > 0.05, "relu_mode 1 must pass everything"
        for mode in (0, 1, 2):
            mask = None if mode == 0 else (torch.ones_like(x64) if mode == 1 else (mask_src > 0).double())
            dx64, dg64, db64, dres64 = R.gbn_backward(dout.double(), x64, gamma, mean_f.double(), rstd_f.double(), group,
                                                      mask)
            dx32, dg32, db32, _ = R.gbn_backward(dout.float(), x32, g32, mean_f, rstd_f, group,
                                                 None if mask is None else mask.float())
            dx, dg, db, dres = K().gbn_bwd(cl(dout), cl(xq), g32, b32, mean_f, rstd_f, rows, mode,
                                           mask_src=cl(mask_src) if mode == 2 else None, want_dres=True)
            _out(t, "bwd%d dx" % mode, ncl(dx), dx64, dx32, dtype)
            _vec(t, "bwd%d dgam" % mode, dg, dg64, dg32)
            _vec(t, "bwd%d dbet" % mode, db, db64, db32)
            t.exact("bwd%d dres" % mode, torch.equal(ncl(dres), dres64.to(dtype)))
    t.check()


# ---- running statistics and eval coefficients ------------------------------------------------------------------------
def test_running_update_small_and_zero_variance():
    """var in {1, 1e-3, 1e-8, 0}: running_var = mix of 1/rstd^2 - eps must stay >= 0 and within 1e-6 (var + eps) of the
    float64 closed form, through the single-layer and the batched entry points."""
    from deepards_b200 import _lib
    st = torch.cuda.current_stream().cuda_stream
    gen = torch.Generator().manual_seed(41)
    n_groups, rows, momentum = 3, 280, 0.1
    tab, layers = [], []
    for c in (64, 128):
        base = torch.tensor([1.0, 1e-3, 1e-8, 0.0], dtype=F64).repeat(c // 4)
        var64 = base[None, :] * (0.5 + torch.rand(n_groups, c, generator=gen, dtype=F64))
        mean_f = (1e3 * (2 * torch.rand(n_groups, c, generator=gen, dtype=F64) - 1)).float().to(DEV)
        rstd_f = (var64 + R.EPS).rsqrt().float().to(DEV)
        var64 = var64.to(DEV)
        zeros = torch.zeros(c, dtype=F64, device=DEV)
        rm64, rv64 = R.running_update(mean_f.double(), var64, rows, momentum, zeros, zeros)
        bound = 1e-6 * (var64.amax(0) + R.EPS)
        outs = []
        for _ in range(2):   # single-layer, batched
            rm, rv = torch.zeros(c, device=DEV), torch.zeros(c, device=DEV)
            nbt = torch.zeros((), dtype=torch.long, device=DEV)
            outs.append((rm, rv, nbt))
        rm, rv, nbt = outs[0]
        _lib.call("dards_bn_running_update", mean_f.data_ptr(), rstd_f.data_ptr(), rm.data_ptr(), rv.data_ptr(),
                  nbt.data_ptr(), n_groups, rows, c, momentum, R.EPS, st)
        rm, rv, nbt = outs[1]
        tab.append((mean_f.data_ptr(), rstd_f.data_ptr(), rm.data_ptr(), rv.data_ptr(), nbt.data_ptr(), n_groups, rows, c,
                    momentum))
        layers.append((c, mean_f, rstd_f, rm64, rv64, bound, outs))
    t_dev, total = _lib.desc_table(_lib.RunningDesc, tab, DEV)
    _lib.call("dards_bn_running_update_batched", t_dev.data_ptr(), len(tab), total, R.EPS, st)
    torch.cuda.synchronize()
    for c, mean_f, _, rm64, rv64, bound, outs in layers:
        for name, (rm, rv, nbt) in zip(("single", "batched"), outs):
            worst = float(((rv.double() - rv64).abs() / bound).max())
            print("running update c%-4d %-8s min running_var %.3e  max |rv - ref| / (1e-6 (var + eps)) %.3f"
                  % (c, name, float(rv.min()), worst))
            assert float(rv.min()) >= 0.0
            assert worst <= 1.0
            assert float((rm.double() - rm64).abs().max()) <= 1e-6 * float(mean_f.abs().max())
            assert int(nbt) == n_groups


def test_eval_coeffs_small_running_var_and_large_mean():
    gen = torch.Generator().manual_seed(42)
    layers, refs = [], []
    for c in (64, 128):
        gamma = (0.1 + 1.9 * torch.rand(c, generator=gen, dtype=F64)).float().to(DEV)
        beta = torch.randn(c, generator=gen, dtype=F64).float().to(DEV)
        rm = torch.tensor([0.0, 10.0, -1e3, 1e3], dtype=F64).repeat(c // 4) * (0.5 + torch.rand(c, generator=gen,
                                                                                              dtype=F64))
        rv = torch.tensor([0.0, 1e-8, 1e-3, 1.0, 1e4, 0.0, 1e-8, 2.0], dtype=F64).repeat(c // 8)
        rm, rv = rm.float().to(DEV), rv.float().to(DEV)
        layers.append((gamma, beta, rm, rv))
        refs.append((R.eval_coeffs(gamma.double(), beta.double(), rm.double(), rv.double()),
                     R.eval_coeffs(gamma, beta, rm, rv)))
    outs = K().bn_eval_coeffs(layers)
    t = Table("bn_eval_coeffs")
    for (gamma, beta, rm, rv), (sc, sh), ((sc64, sh64), (sc32, sh32)) in zip(layers, outs, refs):
        scale_of_shift = beta.double().abs() + (rm.double() * sc64).abs()
        t.cal("scale c%d" % sc.numel(), float(((sc.double() - sc64).abs() / sc64).max()),
              float(((sc32.double() - sc64).abs() / sc64).max()))
        t.cal("shift c%d" % sc.numel(), float(((sh.double() - sh64).abs() / scale_of_shift).max()),
              float(((sh32.double() - sh64).abs() / scale_of_shift).max()))
    t.check()


# ---- convolution + BatchNorm (tcgen05, bf16) --------------------------------------------------------------------------
def _offset_conv_weight(cout, cin, k, gen):
    """Weights whose centre tap has a positive per-channel sum and whose other taps sum to zero over the input channels,
    so that an input offset moves every output position's mean alike (zero padding adds no edge outliers)."""
    w = torch.randn(cout, cin, k, generator=gen, dtype=F64) / (cin * k) ** 0.5
    w = w - w.mean(dim=1, keepdim=True)
    w[:, :, k // 2] += 2.0 / cin ** 0.5 * (0.5 + torch.rand(cout, 1, generator=gen, dtype=F64))
    return w


def _conv_bn_input(family, n, cin, l, group, w, gen):
    """bf16 input (N, Cin, L) and the target |mean| / std of the convolution output (None: not an offset family)."""
    z = torch.randn(n, cin, l, generator=gen, dtype=F64)
    if family.startswith("offset"):
        r = float(family.split()[1])
        wb = w.to(BF16).double()
        per_c = wb.flatten(1).norm(dim=1) / wb[:, :, wb.shape[2] // 2].sum(1)
        return (r * float(per_c.median()) + z).to(BF16), r
    if family == "zero breaths":
        x = 3.0 + z
        b = torch.arange(n) % group
        x[(b == 1) | (b == group - 1)] = 0.0
        return x.to(BF16), None
    return z.to(BF16), None


def _conv_bn_weight(family, cout, cin, k, gen):
    w = _offset_conv_weight(cout, cin, k, gen)
    if family == "constant channels":
        ch = torch.arange(cout) % 8
        w[ch == 0] = 0.0                      # y = 0: var = 0
        w[ch == 1] *= 1e-4                    # var ~ 1e-8 * |w|^2
    return w


CONV_BN_SHAPES = [
    # n, group, cin, cout, l, k, stride, pad, expected mode (1 = PARTIAL statistics + streaming apply, 2 = FUSED)
    (40, 20, 64, 64, 56, 3, 1, 1, 1),
    (40, 20, 64, 64, 16, 3, 1, 1, 1),       # L = 16: the second drain half's first column (16) is a halo column
    (40, 20, 64, 128, 56, 1, 1, 0, 1),
    (60, 20, 256, 256, 14, 3, 1, 1, 2),
    (40, 20, 128, 256, 28, 1, 2, 0, 2),
]


def _conv_bn_check(t, y, mean, rstd, x, w, gamma, beta, group, s, p, target):
    """y: one bf16 rounding of the float64 convolution of the bf16 operands; mean / rstd: the statistics of the fp32
    accumulators against float64 (calibrated by a torch fp32 convolution); out: the stored y normalised with the
    float64 statistics, one bf16 rounding."""
    wb = w.to(BF16)
    y64 = F.conv1d(x.double(), wb.double(), stride=s, padding=p)
    mean64, rstd64 = R.group_stats(y64, group)
    if target is not None:
        achieved = float((mean64.abs() * rstd64).median())
        print("%-46s |mean|/std of y: %.1f (target %g)" % (t.case, achieved, target))
        assert 0.5 * target <= achieved <= 2.0 * target
    mean32, rstd32 = R.group_stats(F.conv1d(x.float(), wb.float(), stride=s, padding=p), group)
    t.bf16("y", ncl(y), y64)
    _stats(t, mean, rstd, mean32, rstd32, mean64, rstd64)
    o64, _, _, _ = R.gbn_forward(ncl(y).double(), gamma.double(), beta.double(), group, stats=(mean64, rstd64))
    return o64


@pytest.mark.parametrize("case", CONV_BN_SHAPES)
def test_conv_bn_statistics_against_float64(case):
    n, group, cin, cout, l, k, s, p, want_mode = case
    fails = []
    for family in ["offset %g" % r for r in BF16_OFFSETS[1:]] + ["centred", "constant channels", "zero breaths"]:
        gen = torch.Generator().manual_seed(51)
        w = _conv_bn_weight(family, cout, cin, k, gen)
        x, target = _conv_bn_input(family, n, cin, l, group, w, gen)
        gamma = (0.5 + torch.rand(cout, generator=gen)).to(DEV)
        beta = (0.3 * torch.randn(cout, generator=gen)).to(DEV)
        x, w = x.to(DEV), w.float().to(DEV)
        t = Table("conv_bn n%d cin%d cout%d l%d k%d s%d %s" % (n, cin, cout, l, k, s, family), fails)
        mode, y, out, mean, rstd, _ = K().conv1d_bn_fwd(cl(x), w, gamma, beta, group, s, p, False)
        torch.cuda.synchronize()
        assert mode == want_mode
        o64 = _conv_bn_check(t, y, mean, rstd, x, w, gamma, beta, group, s, p, target)
        t.bf16("out", ncl(out), o64)
    t.check()


@pytest.mark.parametrize("offset", BF16_OFFSETS)
def test_conv_bn_downsample_branch_merged_against_float64(offset):
    """layer2.0 of ResNet-18: out = bn2(conv2(a1)) + bn_d(conv1x1_s2(x)) in one elementwise pass, on offset inputs."""
    n, group = 40, 20
    gen = torch.Generator().manual_seed(52)
    w2, wd = _offset_conv_weight(128, 128, 3, gen), _offset_conv_weight(128, 64, 1, gen)
    fam = "offset %g" % offset if offset else "centred"
    a1, t2 = _conv_bn_input(fam, n, 128, 28, group, w2, gen)
    xin, td = _conv_bn_input(fam, n, 64, 56, group, wd, gen)
    g2, b2 = (0.5 + torch.rand(128, generator=gen)).to(DEV), (0.3 * torch.randn(128, generator=gen)).to(DEV)
    gd, bd = (0.5 + torch.rand(128, generator=gen)).to(DEV), (0.3 * torch.randn(128, generator=gen)).to(DEV)
    a1, xin, w2, wd = a1.to(DEV), xin.to(DEV), w2.float().to(DEV), wd.float().to(DEV)
    mode, y, out, mean, rstd, ex = K().conv1d_bn_fwd(cl(a1), w2, g2, b2, group, 1, 1, False, ds=(cl(xin), wd, gd, bd, 2, 0))
    torch.cuda.synchronize()
    assert mode == 1
    t = Table("conv_bn downsample merged %s" % fam)
    t.case += " main"
    o2 = _conv_bn_check(t, y, mean, rstd, a1, w2, g2, b2, group, 1, 1, t2)
    t.case = t.case[:-5] + " ds"
    od = _conv_bn_check(t, ex["y_d"], ex["mean_d"], ex["rstd_d"], xin, wd, gd, bd, group, 2, 0, td)
    t.bf16("out", ncl(out), o2 + od)
    t.check()


# ---- stem: conv(1 -> C0, k7 s2 p3) + grouped BatchNorm + ReLU + average pool --------------------------------------------
def _stem_families(dtype):
    offsets = FP32_OFFSETS if dtype == F32 else BF16_OFFSETS
    return ["offset %g" % r for r in offsets] + ["constant group", "zero breaths"]


def _stem_input(family, n, group, gen):
    """(N, 224) fp32 on the CPU; the zero-breath family appends one all-zero group."""
    z = torch.randn(n, 224, generator=gen, dtype=F64)
    if family.startswith("offset"):
        return (float(family.split()[1]) + z).float()
    if family == "constant group":
        x = 10.0 + z
        x[:group] = 7.0
        return x.float()
    x = 10.0 + z
    b = torch.arange(n) % group
    x[(b == 1) | (b == group - 1) | (b == 63) | (b == 64)] = 0.0   # 63 / 64: either side of a chunk boundary
    return torch.cat([x, torch.zeros(group, 224, dtype=F64)]).float()


STEM_CASES = [
    # c0, group, groups, storage of the pooled output / its gradient
    (64, 20, 3, F32), (64, 20, 3, BF16),
    (64, 226, 2, F32),                        # the largest group of the one-kernel path
    (64, 227, 2, F32),                        # chunked: 3 chunks of 64 + one of 35
    (32, 640, 1, F32), (64, 640, 1, BF16),
    (64, 3000, 1, F32),                       # a flat batch: one BatchNorm group of 3000 breaths, 47 chunks
]


@pytest.mark.parametrize("c0,group,groups,dtype", STEM_CASES)
def test_stem_forward_backward_against_float64(c0, group, groups, dtype):
    pool = 1
    fails = []
    for family in _stem_families(dtype):
        gen = torch.Generator().manual_seed(61)
        x = _stem_input(family, group * groups, group, gen).to(DEV)
        n = x.shape[0]
        w = (0.3 * torch.randn(c0, 1, 7, generator=gen)).to(DEV)
        gamma = (0.1 + 0.2 * torch.rand(c0, generator=gen)).to(DEV)
        beta = (4.0 + torch.rand(c0, generator=gen)).to(DEV)
        dout = torch.randn(n, c0, 56, generator=gen).to(DEV).to(dtype)
        t = Table("stem c%d g%d x%d %s %s" % (c0, group, n // group, str(dtype)[6:], family), fails)
        x64, w64, g64, b64 = x.double(), w.double(), gamma.double(), beta.double()
        out64, pre64, mean64, rstd64 = R.stem_forward(x64, w64, g64, b64, group, pool)
        assert float(pre64.min()) > 0.1, "the ReLU must be inactive"
        out32, _, mean32, rstd32 = R.stem_forward(x, w, gamma, beta, group, pool)
        out, mean, rstd = K().stem_fwd(x, w, gamma, beta, group, pool, dtype)
        _out(t, "fwd out", ncl(out), out64, out32, dtype)
        _stats(t, mean, rstd, mean32, rstd32, mean64, rstd64, "fwd ")

        mean_f, rstd_f = mean64.float(), rstd64.float()
        dw64, dg64, db64 = R.stem_backward(dout.double(), x64, w64, g64, mean_f.double(), rstd_f.double(), group, pool,
                                           pre64)
        dw32, dg32, db32 = R.stem_backward(dout.float(), x, w, gamma, mean_f, rstd_f, group, pool, pre64.float())
        dw, dg, db = K().stem_bwd(cl(dout), x, w, gamma, beta, mean_f, rstd_f, group, pool)
        e_dw = chan_err(dw.view(c0, 7), dw64.view(c0, 7))
        t.cal("bwd dW", e_dw, chan_err(dw32.view(c0, 7), dw64.view(c0, 7)), STAT_FLOOR)
        # torch's own fp32 weight gradient (an uncentred sum of dy * x) misses PARITY at the larger offsets; the kernel's
        # input moments are taken about the mean of the group's first breath once it exceeds that breath's spread, and
        # must not
        t.parity("bwd dW", e_dw)
        _vec(t, "bwd dgam", dg, dg64, dg32)
        _vec(t, "bwd dbet", db, db64, db32)
    t.check()


# ---- eval / frozen BatchNorm on offset inputs --------------------------------------------------------------------------
def _running(y64, gen, c):
    """Running statistics of y (the offset passes into the running mean) and gamma / beta that keep the ReLU off."""
    rm = y64.mean(dim=(0, 2)).float()
    rv = y64.var(dim=(0, 2)).float()
    gamma = (0.1 + 0.2 * torch.rand(c, generator=gen)).to(DEV)
    beta = (2.0 + torch.rand(c, generator=gen)).to(DEV)
    return gamma, beta, rm, rv


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
def test_eval_and_frozen_bn_against_float64(dtype):
    """conv1d_affine_fwd, bn_affine_apply and bn_frozen_bwd with running statistics of offset data."""
    n, cin, cout, l = 40, 64, 64, 56
    impl = 0 if dtype == F32 else 1
    fails = []
    for r in (FP32_OFFSETS if dtype == F32 else BF16_OFFSETS):
        gen = torch.Generator().manual_seed(71)
        w = _offset_conv_weight(cout, cin, 3, gen)
        x, _ = _conv_bn_input("offset %g" % r if r else "centred", n, cin, l, 20, w, gen)
        x, w = x.to(DEV).to(dtype), w.float().to(DEV).to(dtype).float()
        t = Table("eval/frozen %s offset %g" % (str(dtype)[6:], r), fails)
        y64 = F.conv1d(x.double(), w.double(), padding=1)
        gamma, beta, rm, rv = _running(y64, gen, cout)
        sc64, sh64 = R.eval_coeffs(gamma.double(), beta.double(), rm.double(), rv.double())
        sc, sh = sc64.float(), sh64.float()
        # convolution with the affine BatchNorm in its epilogue
        o64 = y64 * sc64[None, :, None] + sh64[None, :, None]
        assert float(o64.min()) > 0.05, "the ReLU must be inactive"
        o32 = F.conv1d(x.float(), w, padding=1) * sc[None, :, None] + sh[None, :, None]
        out = K().conv1d_affine_fwd(cl(x), w, sc, sh, 1, 1, impl=impl, relu=True)
        _out(t, "conv+aff", ncl(out), o64, o32, dtype)
        # elementwise affine on a stored offset activation
        yq = (rm[None, :, None].double() + rv.sqrt()[None, :, None].double() *
              torch.randn(n, cout, l, generator=gen, dtype=F64).to(DEV)).to(dtype)
        a64 = yq.double() * sc64[None, :, None] + sh64[None, :, None]
        a32 = yq.float() * sc[None, :, None] + sh[None, :, None]
        out = K().bn_affine_apply(cl(yq), sc, sh, relu=False)
        _out(t, "affine", ncl(out), a64, a32, dtype)
        # frozen backward: dx = scale * g, dgamma = sum g * (y - running_mean) * rstd, dbeta = sum g
        rstd_f = (rv.double() + R.EPS).rsqrt().float()
        dout = torch.randn(n, cout, l, generator=gen).to(DEV).to(dtype)
        dx, dg, db, _ = K().bn_frozen_bwd(cl(dout), cl(yq), sc, sh, rm, rstd_f, 0)
        xh64 = (yq.double() - rm.double()[None, :, None]) * rstd_f.double()[None, :, None]
        xh32 = (yq.float() - rm[None, :, None]) * rstd_f[None, :, None]
        _out(t, "frz dx", ncl(dx), dout.double() * sc[None, :, None].double(), dout.float() * sc[None, :, None], dtype)
        _vec(t, "frz dgam", dg, (dout.double() * xh64).sum(dim=(0, 2)), (dout.float() * xh32).sum(dim=(0, 2)))
        _vec(t, "frz dbet", db, dout.double().sum(dim=(0, 2)), dout.float().sum(dim=(0, 2)))
    t.check()


@pytest.mark.parametrize("dtype", [F32, BF16], ids=["fp32", "bf16"])
def test_stem_eval_and_frozen_against_float64(dtype):
    n, c0, pool = 300, 64, 1
    fails = []
    for r in (FP32_OFFSETS if dtype == F32 else BF16_OFFSETS):
        gen = torch.Generator().manual_seed(72)
        x = (r + torch.randn(n, 224, generator=gen)).to(DEV)
        w = (0.3 * torch.randn(c0, 1, 7, generator=gen)).to(DEV)
        t = Table("stem eval/frozen %s offset %g" % (str(dtype)[6:], r), fails)
        y64 = R.stem_conv(x.double(), w.double())
        gamma, beta, rm, rv = _running(y64, gen, c0)
        beta = beta + 2.0     # the stem's edge positions are far from the running mean at large offsets
        sc64, sh64 = R.eval_coeffs(gamma.double(), beta.double(), rm.double(), rv.double())
        sc, sh = sc64.float(), sh64.float()
        out64, pre64 = R.stem_eval_forward(x.double(), w.double(), sc.double(), sh.double(), pool)
        assert float(pre64.min()) > 0.1, "the ReLU must be inactive"
        out32, _ = R.stem_eval_forward(x, w, sc, sh, pool)
        out = K().stem_eval_fwd(x, w, sc, sh, pool, dtype)
        _out(t, "fwd out", ncl(out), out64, out32, dtype)
        rstd_f = (rv.double() + R.EPS).rsqrt().float()
        dout = torch.randn(n, c0, 56, generator=gen).to(DEV).to(dtype)
        dw64, dg64, db64 = R.stem_frozen_backward(dout.double(), x.double(), w.double(), sc.double(), rm.double(),
                                                  rstd_f.double(), pool, pre64)
        dw32, dg32, db32 = R.stem_frozen_backward(dout.float(), x, w, sc, rm, rstd_f, pool, pre64.float())
        dw, dg, db = K().stem_frozen_bwd(cl(dout), x, w, sc, sh, rm, rstd_f, pool)
        t.cal("bwd dW", chan_err(dw.view(c0, 7), dw64.view(c0, 7)), chan_err(dw32.view(c0, 7), dw64.view(c0, 7)),
              STAT_FLOOR)
        _vec(t, "bwd dgam", dg, dg64, dg32)
        _vec(t, "bwd dbet", db, db64, db32)
    t.check()

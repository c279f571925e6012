"""GPU: ResNet in eval() -- BatchNorm with the running statistics, applied in the convolution epilogues.

  * the three kernels (convolution + affine epilogue, eval stem, coefficients) against PyTorch in fp32
  * whole networks against tests/eval_reference.py (F.batch_norm(training=False)) with non-trivial running statistics
  * semantics: batch independence, untouched running buffers, in-place edits seen by graph replays, train() unchanged,
    a loud backward error, the recorded call list and the plan's memory
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import cnn_linear_oracle as O  # noqa: E402
from tests import eval_reference as R  # noqa: E402
from tests.helpers import rel_err  # noqa: E402

DEV = "cuda"
FP32_TOL = 1e-4         # whole-network fp32 logits, as in test_model_parity_gpu.py
BF16_LOGIT_TOL = 1e-1   # whole-network bf16 logits (the existing bf16 gate is 8e-2; the eval gate is stated as 1e-1)


def K():
    from deepards_b200 import kernels
    return kernels


def cl(x):  # (N, C, L) <-> (N, L, C)
    return x.permute(0, 2, 1).contiguous()


# every convolution shape of ResNet-18 (n_breaths is varied inside the test): cin, cout, l_in, k, stride, pad
RESNET18_CONVS = [
    (64, 64, 56, 3, 1, 1),
    (64, 128, 56, 3, 2, 1), (64, 128, 56, 1, 2, 0), (128, 128, 28, 3, 1, 1),
    (128, 256, 28, 3, 2, 1), (128, 256, 28, 1, 2, 0), (256, 256, 14, 3, 1, 1),
    (256, 512, 14, 3, 2, 1), (256, 512, 14, 1, 2, 0), (512, 512, 7, 3, 1, 1),
]
VARIANTS = [(0, torch.float32), (0, torch.bfloat16), (1, torch.bfloat16)]  # (impl, storage dtype)


def _affine_inputs(n, cin, cout, l, k, s, p, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    lo = (l + 2 * p - k) // s + 1
    x = torch.randn(n, l, cin, generator=g).to(DEV, dtype)
    w = (torch.randn(cout, cin, k, generator=g) / (cin * k) ** 0.5).to(DEV)
    scale = (torch.rand(cout, generator=g) * 2 + 0.2).to(DEV)
    shift = torch.randn(cout, generator=g).to(DEV)
    res = torch.randn(n, lo, cout, generator=g).to(DEV, dtype)
    return x, w, scale, shift, res


def _affine_ref(x, w, scale, shift, s, p, res, relu, impl):
    # reference on exactly the operands the kernel sees: bf16 storage rounds x / res, bf16 packing rounds w
    wr = w.to(x.dtype).float()
    y = F.conv1d(x.float().permute(0, 2, 1), wr, stride=s, padding=p) * scale.view(1, -1, 1) + shift.view(1, -1, 1)
    y = cl(y)
    if res is not None:
        y = y + res.float()
    return F.relu(y) if relu else y


@pytest.mark.parametrize("case", RESNET18_CONVS)
@pytest.mark.parametrize("variant", VARIANTS, ids=["simt_fp32", "simt_bf16", "tcgen05_bf16"])
def test_conv_affine_epilogue_matches_torch(case, variant):
    impl, dtype = variant
    cin, cout, l, k, s, p = case
    torch.backends.cudnn.allow_tf32 = False
    tol = 3e-5 if dtype == torch.float32 else 6e-3   # bf16: one rounding of the stored output (2^-9 of the element)
    for n in (1, 7, 20, 333):
        x, w, scale, shift, res = _affine_inputs(n, cin, cout, l, k, s, p, dtype, seed=n + cin + k)
        for use_res in (False, True):
            for relu in (False, True):
                r = res if use_res else None
                out = K().conv1d_affine_fwd(x, w, scale, shift, s, p, impl=impl, res=r, relu=relu)
                ref = _affine_ref(x, w, scale, shift, s, p, r, relu, impl)
                err = rel_err(out.float(), ref)
                assert err < tol, (n, use_res, relu, err)


@pytest.mark.parametrize("variant", VARIANTS, ids=["simt_fp32", "simt_bf16", "tcgen05_bf16"])
def test_conv_affine_into_wider_rows(variant):
    """out_stride wider than c_out (an output slice of a wider buffer): nothing outside the slice is written."""
    impl, dtype = variant
    n, (cin, cout, l, k, s, p) = 37, RESNET18_CONVS[1]
    x, w, scale, shift, res = _affine_inputs(n, cin, cout, l, k, s, p, dtype, seed=5)
    lo = res.shape[1]
    wide = torch.zeros(n, lo, cout + 64, device=DEV, dtype=dtype)
    K().conv1d_affine_fwd(x, w, scale, shift, s, p, impl=impl, res=res, relu=True, out=wide[:, :, 32:32 + cout])
    ref = _affine_ref(x, w, scale, shift, s, p, res, True, impl)
    assert rel_err(wide[:, :, 32:32 + cout].float(), ref) < (3e-5 if dtype == torch.float32 else 6e-3)
    assert float(wide[:, :, :32].float().abs().max()) == 0.0 and float(wide[:, :, 32 + cout:].float().abs().max()) == 0.0


@pytest.mark.parametrize("case", [c for c in RESNET18_CONVS if c[1] >= 256])
def test_conv_affine_cta_pair_kernel_equals_single_cta_kernel(case):
    """The cta_group::2 kernel's affine epilogue is bit-identical to the single-CTA kernel's (debug key 17 = 0)."""
    from deepards_b200 import _lib
    cin, cout, l, k, s, p = case
    x, w, scale, shift, res = _affine_inputs(333, cin, cout, l, k, s, p, torch.bfloat16, seed=17)
    outs = []
    for mode in (-1, 0):
        _lib.call("dards_tc_debug_set", 17, mode)
        try:
            outs.append(K().conv1d_affine_fwd(x, w, scale, shift, s, p, impl=1, res=res, relu=True))
            torch.cuda.synchronize()
        finally:
            _lib.call("dards_tc_debug_set", 17, -1)
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("n", [1, 37, 300])
@pytest.mark.parametrize("pool", [0, 1])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_stem_eval_matches_torch(n, pool, dtype):
    c0 = 64
    g = torch.Generator().manual_seed(n + pool)
    x = torch.randn(n, 224, generator=g).to(DEV)
    w = (torch.randn(c0, 1, 7, generator=g) * 0.3).to(DEV)
    gamma, beta = (1 + 0.2 * torch.randn(c0, generator=g)).to(DEV), (0.2 * torch.randn(c0, generator=g)).to(DEV)
    rm, rv = (0.3 * torch.randn(c0, generator=g)).to(DEV), (torch.rand(c0, generator=g) + 0.05).to(DEV)
    y = F.relu(F.batch_norm(F.conv1d(x.view(n, 1, 224), w, stride=2, padding=3), rm, rv, gamma, beta, False, 0.0, 1e-5))
    ref = cl(F.max_pool1d(y, 3, 2, 1) if pool == 0 else F.avg_pool1d(y, 3, 2, 1))
    (sc, sh), = K().bn_eval_coeffs([(gamma, beta, rm, rv)])
    out = K().stem_eval_fwd(x, w, sc, sh, pool, dtype)
    assert rel_err(out.float(), ref) < (1e-5 if dtype == torch.float32 else 6e-3)


def test_eval_coefficients_match_torch():
    g = torch.Generator().manual_seed(3)
    layers = []
    for c in (64, 128, 256, 512, 100):
        gamma, beta = 1 + 0.5 * torch.randn(c, generator=g), torch.randn(c, generator=g)
        rm = torch.randn(c, generator=g)
        rv = torch.exp(torch.empty(c).uniform_(np.log(1e-3), np.log(10.0), generator=g))
        rv[:4] = torch.tensor([1e-3, 2e-3, 5e-3, 1e-2])
        layers.append(tuple(t.to(DEV) for t in (gamma, beta, rm, rv)))
    got = K().bn_eval_coeffs(layers)
    for (gamma, beta, rm, rv), (sc, sh) in zip(layers, got):
        ref_sc = gamma.double() / torch.sqrt(rv.double() + 1e-5)
        ref_sh = beta.double() - rm.double() * ref_sc
        assert rel_err(sc, ref_sc) < 1e-6 and rel_err(sh, ref_sh) < 1e-6
        # the same numbers as torch's own eval-mode BatchNorm on a unit impulse
        x = torch.stack([torch.zeros_like(rm), torch.ones_like(rm)]).unsqueeze(-1)
        y = F.batch_norm(x, rm, rv, gamma, beta, False, 0.0, 1e-5)[..., 0]
        assert rel_err(sh, y[0]) < 1e-5 and rel_err(sc + sh, y[1]) < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# whole networks vs the eval-mode reference (tests/eval_reference.py)
# ---------------------------------------------------------------------------------------------------------------------
def _trained_state(initial_planes=64, seed=0, pool="max"):
    """A ResNet-18 whose running statistics are far from their zeros / ones: three training-mode forwards on synthetic
    breaths (each updates the running buffers), then a per-channel perturbation of every BatchNorm's buffers and affine
    parameters -- a wrong mean, variance or eps cannot hide behind the initial state."""
    import deepards_b200 as D
    torch.manual_seed(seed)
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=initial_planes, first_pool_type=pool), 20, 0).to(DEV)
    net.precision = "fp32"
    net.train()
    with torch.no_grad():
        for i in range(3):
            net(O.synthetic_breaths(2, seed=300 + i).to(DEV), None)
        g = torch.Generator(device="cpu").manual_seed(seed + 1)
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                c = m.num_features
                m.running_mean.add_((0.3 * torch.randn(c, generator=g)).to(DEV))
                m.running_var.mul_(torch.exp(0.5 * torch.randn(c, generator=g)).to(DEV))
                m.weight.mul_((1 + 0.2 * torch.randn(c, generator=g)).to(DEV))
                m.bias.add_((0.1 * torch.randn(c, generator=g)).to(DEV))
    sd = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    assert float(sd["breath_block.layer2.0.bn1.running_var"].sub(1).abs().max()) > 0.1
    return sd


def _backbone_sd(sd):
    return {k[len("breath_block."):]: v for k, v in sd.items() if k.startswith("breath_block.")}


@pytest.fixture(scope="module")
def trained():
    return _trained_state()


def _net(kind, sd, precision):
    import deepards_b200 as D
    bb = D.resnet18()
    if kind == "cnn_linear":
        net = D.CNNLinearNetwork(bb, 20, 0)
    elif kind == "per_breath":
        net = D.CNNSingleBreathLinearNetwork(bb)
    elif kind == "flat":
        net = bb
    else:
        net = D.CNNRegressor(bb, 3)
    if kind == "flat":
        net.load_state_dict(_backbone_sd(sd))
    elif kind == "regressor":
        torch.manual_seed(5)
        lin = torch.nn.Linear(512, 3)
        full = dict(sd)
        full.pop("linear_final.weight")
        full.pop("linear_final.bias")
        full["linear_final.weight"], full["linear_final.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
        net.load_state_dict(full)
    else:
        if kind == "per_breath":
            full = dict(sd)
            torch.manual_seed(6)
            lin = torch.nn.Linear(512, 2)
            full["linear_final.weight"], full["linear_final.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
            net.load_state_dict(full)
        else:
            net.load_state_dict(sd)
    net = net.to(DEV).eval()
    net.precision = precision
    return net


def _run_both(kind, sd, precision):
    net = _net(kind, sd, precision)
    full = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    if kind in ("cnn_linear", "per_breath"):
        x = O.synthetic_breaths(3, seed=71)
        with torch.no_grad():
            got = net(x.to(DEV), None).cpu()
        ref = R.cnn_linear_forward(full, x, per_breath=kind == "per_breath")
    elif kind == "flat":
        x = O.synthetic_breaths(17, seed=72).reshape(-1, 1, 224)[:333]
        with torch.no_grad():
            got = net(x.to(DEV)).cpu()
        ref = R.resnet_forward(full, x)
    else:
        x = O.synthetic_breaths(3, seed=73).reshape(-1, 1, 224)[:57]
        with torch.no_grad():
            got = net(x.to(DEV)).cpu()
        ref = R.regressor_forward(full, x)
    return got, ref


@pytest.mark.parametrize("kind", ["cnn_linear", "per_breath", "flat", "regressor"])
def test_eval_fp32_matches_reference(trained, kind):
    got, ref = _run_both(kind, trained, "fp32")
    assert got.shape == ref.shape
    assert rel_err(got, ref) <= FP32_TOL, rel_err(got, ref)


@pytest.mark.parametrize("kind", ["cnn_linear", "per_breath", "flat", "regressor"])
def test_eval_bf16_matches_reference(trained, kind):
    got, ref = _run_both(kind, trained, "bf16")
    err = rel_err(got, ref)
    print("bf16 eval logits vs fp32 reference (%s): %.3e" % (kind, err))
    assert err <= BF16_LOGIT_TOL, err


def test_eval_bf16_vs_fp32_at_65536_breaths(trained):
    """The single-breath classifier at the largest configs[3] size: bf16 / tcgen05 eval against the fp32 eval plan."""
    x = O.synthetic_breaths(64, seed=80).repeat(52, 1, 1, 1)[:3277]  # 65 540 breaths
    x = (x * (1 + 0.05 * torch.randn(x.shape[0], 1, 1, 1, generator=torch.Generator().manual_seed(1)))).to(DEV)
    outs = {}
    for precision in ("fp32", "bf16"):
        net = _net("per_breath", trained, precision)
        with torch.no_grad():
            outs[precision] = net(x, None).float()
        del net
        torch.cuda.empty_cache()
    err = rel_err(outs["bf16"], outs["fp32"])
    print("bf16 vs fp32 eval logits at %d breaths: %.3e" % (x.shape[0] * 20, err))
    assert err <= BF16_LOGIT_TOL, err


# ---------------------------------------------------------------------------------------------------------------------
# semantics
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_output_does_not_depend_on_the_rest_of_the_batch(trained, precision):
    net = _net("cnn_linear", trained, precision)
    x = O.synthetic_breaths(7, seed=90).to(DEV)
    with torch.no_grad():
        whole = net(x, None)
        single = torch.cat([net(x[i:i + 1], None) for i in range(x.shape[0])])
    err = rel_err(whole, single)
    print("%s: batch vs per-sequence eval logits: max rel %.3e, bit-identical: %s" % (precision, err,
                                                                                      torch.equal(whole, single)))
    assert err <= 1e-6


def test_eval_leaves_running_buffers_untouched_and_sees_in_place_edits(trained):
    net = _net("cnn_linear", trained, "fp32")
    before = {k: v.clone() for k, v in net.state_dict().items()}
    x = O.synthetic_breaths(2, seed=91)
    bb = net.breath_block
    for call in range(5):
        if call == 3:   # the plan replays a CUDA graph from the third call on
            with torch.no_grad():
                bb.layer3[1].bn2.running_var.mul_(1.7)
                bb.layer1[0].bn1.running_mean.add_(0.25)
                bb.layer2[0].conv2.weight.mul_(0.9)
                bb.bn1.weight.mul_(1.1)
            before = {k: v.clone() for k, v in net.state_dict().items()}
        with torch.no_grad():
            got = net(x.to(DEV), None).cpu()
        ref = R.cnn_linear_forward({k: v.cpu() for k, v in net.state_dict().items()}, x)
        assert rel_err(got, ref) <= FP32_TOL, (call, rel_err(got, ref))
        for k, v in net.state_dict().items():
            assert torch.equal(v, before[k]), (call, k)   # running_*, num_batches_tracked: bit-identical


def test_train_eval_train_round_trip_leaves_training_unchanged(trained):
    """fp32 path: gradients and running statistics after train(), eval() forward, train() are bit-identical to a module
    that never left train()."""
    import deepards_b200 as D
    nets = []
    for _ in range(2):
        net = D.CNNLinearNetwork(D.resnet18(), 20, 0)
        net.load_state_dict(trained)
        net = net.to(DEV).train()
        net.precision = "fp32"
        nets.append(net)
    x, t = O.synthetic_breaths(2, seed=92).to(DEV), O.synthetic_targets(2, seed=92).to(DEV)
    grads = []
    for i, net in enumerate(nets):
        for step in range(2):
            net.zero_grad()
            F.binary_cross_entropy_with_logits(net(x, None), t).backward()
            if i == 1 and step == 0:
                net.eval()
                with torch.no_grad():
                    net(x, None)
                net(x, None)  # grad enabled: the output is attached, but nothing runs backward
                net.train()
        grads.append({n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None})
    assert grads[0].keys() == grads[1].keys()
    for n in grads[0]:
        assert torch.equal(grads[0][n], grads[1][n]), n
    s0, s1 = nets[0].state_dict(), nets[1].state_dict()
    for k in s0:
        assert torch.equal(s0[k], s1[k]), k


def test_backward_in_eval_raises(trained):
    net = _net("cnn_linear", trained, "fp32")
    x = O.synthetic_breaths(2, seed=93).to(DEV)
    out = net(x, None)
    assert out.requires_grad
    with pytest.raises(NotImplementedError, match="running-statistics BatchNorm .*train\\(\\)"):
        out.sum().backward()
    with pytest.raises(NotImplementedError):   # the input-gradient refusal is unchanged
        net(x.clone().requires_grad_(True), None)


def _eval_plan(net):
    plans = [p for p in net.__dict__["_dards_plans"].values() if p.bn == "eval"]
    assert len(plans) == 1
    return plans[0]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_plan_records_no_batch_statistics_and_bounded_memory(trained, precision):
    net = _net("per_breath", trained, precision)
    x = O.synthetic_breaths(50, seed=94).to(DEV)   # 1000 breaths
    with torch.no_grad():
        net(x, None)
    plan = _eval_plan(net)
    names = [c[0] for c in plan.fwd.calls]
    forbidden = [n for n in names if n.startswith("dards_gbn_") or n in ("dards_conv1d_bn_fwd", "dards_stem_fwd")
                 or n.startswith("dards_bn_running_update")]
    assert not forbidden, forbidden
    assert names[0] == "dards_bn_eval_coeffs_batched" and names[1] == "dards_stem_eval_fwd"
    assert names.count("dards_conv1d_affine_fwd") == 19 and len(plan.bwd) == 0
    n = plan.N
    esz = 4 if precision == "fp32" else 2
    largest = n * 56 * 64 * esz                      # every ResNet-18 stage activation has N * 3584 elements
    assert plan.act_bytes == 4 * largest
    packed = sum(c.kio.numel() * c.kio.element_size() + c.koi.numel() * c.koi.element_size() for c in plan.convs)
    total = sum(t.numel() * t.element_size() for t in plan.bufs)
    # four activations of the largest stage + the packed weights + input, pooled features, logits and small tables
    bound = 4 * largest + packed + n * (224 + 512 + 8) * 4 + (1 << 20)
    print("%s eval plan at %d breaths: %.1f MB (bound %.1f MB)" % (precision, n, total / 2**20, bound / 2**20))
    assert total <= bound

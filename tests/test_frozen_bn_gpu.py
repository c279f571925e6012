"""GPU: ResNet fine-tuning with frozen BatchNorm -- the network in train(), its BatchNorm layers in eval().

  * the three kernels (affine apply, constant-statistics BatchNorm backward, frozen stem backward) against torch autograd
    of F.batch_norm(training=False) (+ residual, + ReLU), fp32 and bf16
  * whole networks against the oracle with its BatchNorm normalising with the running statistics (decisions pinned)
  * semantics: untouched running buffers, batch independence, agreement with the eval plan, in-place edits, the way back
    to train(), refusal of mixed states, determinism, and the data-parallel trainer
"""

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import cnn_linear_oracle as O  # noqa: E402
from tests.helpers import cosine, pinned_decision_check, plan_of, rel_err  # noqa: E402
from tests.test_eval_gpu import _backbone_sd, _trained_state  # noqa: E402
from tests.test_frozen_bn_cpu import frozen_oracle  # noqa: E402

DEV = "cuda"
EPS = 1e-5


def K():
    from deepards_b200 import kernels
    return kernels


def _freeze(net):
    net.train()
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.eval()
    return net


def _bn_consts(c, seed, small_var=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    gamma = 1 + 0.3 * torch.randn(c, generator=g)
    beta = 0.2 * torch.randn(c, generator=g)
    rm = 0.5 * torch.randn(c, generator=g)
    rv = torch.exp(0.7 * torch.randn(c, generator=g))
    if small_var:
        rv[::7] = 1e-3
    return [t.to(DEV) for t in (gamma, beta, rm, rv)]


def _coeffs(gamma, beta, rm, rv):
    (sc, sh), (rs, _) = K().bn_eval_coeffs([(gamma, beta, rm, rv), (torch.ones_like(gamma), torch.zeros_like(beta), rm, rv)])
    return sc, sh, rs


# ---------------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------------
# every BatchNorm shape of ResNet-18: (C, L)
RESNET18_BN = [(64, 56), (128, 28), (256, 14), (512, 7)]
TOL = {torch.float32: 2e-5, torch.bfloat16: 2e-2}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c,l", RESNET18_BN)
@pytest.mark.parametrize("variant", ["relu", "res_relu", "second", "plain"])
def test_affine_apply_and_frozen_bwd(dtype, c, l, variant):
    """out = [relu](bn(y) [+ res] [+ bn_d(y2)]) with running statistics and its backward, against torch autograd, ragged N
    (333 breaths) and a channel slice of a wider row."""
    n = 333
    torch.manual_seed(c + l)
    wide = torch.randn(n, l, c + 16, device=DEV).to(dtype)
    y = wide[:, :, 8:8 + c]
    gamma, beta, rm, rv = _bn_consts(c, 1, small_var=True)
    sc, sh, rs = _coeffs(gamma, beta, rm, rv)
    res = torch.randn(n, l, c, device=DEV).to(dtype) if variant == "res_relu" else None
    second = None
    if variant == "second":
        y2 = torch.randn(n, l, c, device=DEV).to(dtype)
        g2, b2, rm2, rv2 = _bn_consts(c, 2)
        sc2, sh2, rs2 = _coeffs(g2, b2, rm2, rv2)
        second = (y2, sc2, sh2)
    relu = variant != "plain"
    out = K().bn_affine_apply(y, sc, sh, res=res, relu=relu, second=second)

    # torch reference in fp32 on the stored values
    yr = y.float().permute(0, 2, 1).requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    z = F.batch_norm(yr, rm, rv, gr, br, False, 0.1, EPS)
    if res is not None:
        z = z + res.float().permute(0, 2, 1)
    if second is not None:
        g2r, b2r = g2.clone().requires_grad_(True), b2.clone().requires_grad_(True)
        z = z + F.batch_norm(y2.float().permute(0, 2, 1), rm2, rv2, g2r, b2r, False, 0.1, EPS)
    ref = F.relu(z) if relu else z
    assert rel_err(out.float().permute(0, 2, 1).cpu(), ref.detach().cpu()) <= TOL[dtype]

    dout = torch.randn(n, l, c, device=DEV).to(dtype)
    ref.backward(dout.float().permute(0, 2, 1))
    # relu mode 2 reads the decisions from the forward output (the plan's residual sites), mode 1 recomputes them
    mode = 0 if not relu else (2 if variant in ("res_relu", "second") else 1)
    dx, dgamma, dbeta, dres = K().bn_frozen_bwd(dout, y, sc, sh, rm, rs, mode, mask_src=out if mode == 2 else None,
                                                want_dres=mode == 2, tile_rows=[l, 9 * l, 37 * l][c % 3])
    assert rel_err(dx.float().permute(0, 2, 1).cpu(), yr.grad.cpu()) <= TOL[dtype]
    assert rel_err(dgamma.cpu(), gr.grad.cpu()) <= TOL[dtype]
    assert rel_err(dbeta.cpu(), br.grad.cpu()) <= TOL[dtype]
    if dres is not None:
        g = dout.float() * (out.float() > 0)
        assert torch.equal(dres.float(), g)  # the masked gradient is exact


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_frozen_bwd_accumulate(dtype):
    n, l, c = 40, 28, 128
    y = torch.randn(n, l, c, device=DEV).to(dtype)
    gamma, beta, rm, rv = _bn_consts(c, 3)
    sc, sh, rs = _coeffs(gamma, beta, rm, rv)
    dout = torch.randn(n, l, c, device=DEV).to(dtype)
    base = torch.randn(n, l, c, device=DEV).to(dtype)
    fresh, _, _, _ = K().bn_frozen_bwd(dout, y, sc, sh, rm, rs, 1)
    acc, _, _, _ = K().bn_frozen_bwd(dout, y, sc, sh, rm, rs, 1, dx=base.clone(), accumulate=True)
    want = fresh.float() + base.float()
    assert rel_err(acc.float().cpu(), want.cpu()) <= (1e-6 if dtype == torch.float32 else 1e-2)


def _stem_ref(x, w, gamma, beta, rm, rv, pool):
    y = F.conv1d(x.unsqueeze(1), w, stride=2, padding=3)
    z = F.relu(F.batch_norm(y, rm, rv, gamma, beta, False, 0.1, EPS))
    return F.max_pool1d(z, 3, 2, 1) if pool == 0 else F.avg_pool1d(z, 3, 2, 1)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c0", [16, 64])
@pytest.mark.parametrize("pool", [0, 1])
@pytest.mark.parametrize("n", [20, 333, 5120])
def test_stem_frozen_bwd(dtype, c0, pool, n):
    torch.manual_seed(n + c0)
    x = torch.randn(n, 224, device=DEV)
    w = 0.3 * torch.randn(c0, 1, 7, device=DEV)
    gamma, beta, rm, rv = _bn_consts(c0, 4, small_var=True)
    sc, sh, rs = _coeffs(gamma, beta, rm, rv)
    out = K().stem_eval_fwd(x, w, sc, sh, pool, dtype)
    dout = torch.randn(n, 56, c0, device=DEV).to(dtype)
    dw, dgamma, dbeta = K().stem_frozen_bwd(dout, x, w, sc, sh, rm, rs, pool)
    wr, gr, br = (t.clone().requires_grad_(True) for t in (w, gamma, beta))
    ref = _stem_ref(x, wr, gr, br, rm, rv, pool)
    if dtype == torch.float32:
        # the kernel recomputes the forward's pre-pool values bit for bit: pin torch's max-pool choice to the forward
        assert rel_err(out.permute(0, 2, 1).cpu(), ref.detach().cpu()) <= 1e-5
    ref.backward(dout.float().permute(0, 2, 1))
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    assert rel_err(dw.cpu(), wr.grad.cpu()) <= tol
    assert rel_err(dgamma.cpu(), gr.grad.cpu()) <= tol
    assert rel_err(dbeta.cpu(), br.grad.cpu()) <= tol


# ---------------------------------------------------------------------------------------------------------------------
# whole networks
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def trained():
    return _trained_state()


@pytest.fixture(scope="module")
def trained16():
    return _trained_state(initial_planes=16, seed=2)


def _frozen_net(kind, sd, precision, planes=64):
    import deepards_b200 as D
    bb = D.resnet18(initial_planes=planes)
    if kind == "cnn_linear":
        net = D.CNNLinearNetwork(bb, 20, 0)
        net.load_state_dict(sd)
    elif kind == "per_breath":
        net = D.CNNSingleBreathLinearNetwork(bb)
        full = dict(sd)
        torch.manual_seed(6)
        lin = torch.nn.Linear(8 * planes, 2)
        full["linear_final.weight"], full["linear_final.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
        net.load_state_dict(full)
    elif kind == "flat":
        net = bb
        net.load_state_dict(_backbone_sd(sd))
    else:
        net = D.CNNRegressor(bb, 3)
        full = dict(sd)
        torch.manual_seed(5)
        lin = torch.nn.Linear(8 * planes, 3)
        full["linear_final.weight"], full["linear_final.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
        net.load_state_dict(full)
    net = _freeze(net.to(DEV))
    net.precision = precision
    return net


def _state_of(net):
    return {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}


@pytest.mark.parametrize("kind,planes", [("cnn_linear", 64), ("cnn_linear", 16), ("per_breath", 64)])
def test_fp32_sequence_heads_pinned(kind, planes, trained, trained16):
    sd = trained if planes == 64 else trained16
    net = _frozen_net(kind, sd, "fp32", planes)
    full = _state_of(net)
    b = 16
    x, t = O.synthetic_breaths(b, seed=21), O.synthetic_targets(b, seed=21)
    per_breath = kind == "per_breath"
    tt = t.unsqueeze(1).expand(-1, 20, -1).contiguous() if per_breath else t
    out = net(x.to(DEV), None)
    F.binary_cross_entropy_with_logits(out, tt.to(DEV)).backward()
    mine = {n: p.grad for n, p in net.named_parameters() if p.grad is not None}
    with frozen_oracle():
        ref_out, _, ref_g = O.forward_backward({k: v.clone() for k, v in full.items()}, x, tt, per_breath=per_breath)
        assert rel_err(out.detach().cpu(), ref_out) <= 1e-4
        assert set(mine) == set(ref_g)
        pinned_decision_check(plan_of(net, b * 20), full, x, tt, mine, 1e-4, kind, per_breath=per_breath)


def _flat_reference(plan, full, x, params, head):
    """Oracle ResNet (+ the regressor's linear head) for a flat batch, BatchNorm frozen and the ReLU decisions of the block
    sites pinned to the plan's (see helpers.pinned_decision_check).  Returns (output, leaves)."""
    masks = {s: (buf.float() > 0).permute(0, 2, 1).unsqueeze(0).cpu() for s, buf in plan.sites.items()}
    leaves = {k: (v.clone().requires_grad_(True) if k in params else v) for k, v in full.items()}
    with frozen_oracle():
        feat = O.resnet_forward(leaves, x, prefix="breath_block." if head else "", hooks=O.DecisionHooks(masks=masks))
    out = F.linear(feat, leaves["linear_final.weight"], leaves["linear_final.bias"]) if head else feat
    return out, leaves


@pytest.mark.parametrize("kind,planes", [("flat", 64), ("regressor", 64), ("regressor", 16)])
def test_fp32_flat_batches_pinned(kind, planes, trained, trained16):
    sd = trained if planes == 64 else trained16
    net = _frozen_net(kind, sd, "fp32", planes)
    full = _state_of(net)
    n = 333 if kind == "flat" else 57
    x = O.synthetic_breaths(17, seed=72).reshape(-1, 1, 224)[:n]
    out = net(x.to(DEV))
    gw = torch.randn(out.shape, generator=torch.Generator().manual_seed(3))
    (out * gw.to(DEV)).sum().backward()
    params = dict(net.named_parameters())
    names = [k for k, p in params.items() if p.grad is not None]
    # the regressor runs its backbone as a module of its own: the plan lives on breath_block
    plan = plan_of(net.breath_block if kind == "regressor" else net, n)
    ref, leaves = _flat_reference(plan, full, x, params, kind == "regressor")
    assert rel_err(out.detach().cpu(), ref.detach()) <= 1e-4
    grads = torch.autograd.grad((ref * gw).sum(), [leaves[k] for k in names])
    stem = ("conv1.weight", "bn1.weight", "bn1.bias")
    for k, g in zip(names, grads):
        e = rel_err(params[k].grad.cpu(), g)
        # the stem's ReLU + max-pool decisions are recomputed inside the kernel and cannot be pinned
        is_stem = k in stem or k in tuple("breath_block." + s for s in stem)
        assert e <= (5e-2 if is_stem else 1e-4), (k, e)


# bf16: logits within 1e-1 of the fp32 frozen reference, and the worst per-tensor gradient cosine against the oracle.
# Measured on an NVIDIA B200 (1000 W): B = 16 logits 1.09e-2, worst cosine 0.97094; B = 256 logits 1.56e-2, worst cosine
# 0.99812.  The gates leave room for the bf16 rounding of other inputs.
BF16_COS = {16: 0.95, 256: 0.99}


@pytest.mark.parametrize("b", [16, 256])
def test_bf16_whole_network(b, trained):
    net = _frozen_net("cnn_linear", trained, "bf16")
    full = _state_of(net)
    x, t = O.synthetic_breaths(b, seed=31), O.synthetic_targets(b, seed=31)
    out = net(x.to(DEV), None)
    F.binary_cross_entropy_with_logits(out, t.to(DEV)).backward()
    with frozen_oracle():
        ref_out, _, ref_g = O.forward_backward({k: v.clone() for k, v in full.items()}, x, t)
    err = rel_err(out.detach().cpu(), ref_out)
    params = dict(net.named_parameters())
    worst = min(cosine(params[k].grad.cpu(), g) for k, g in ref_g.items())
    print("bf16 frozen B=%d: logits rel err %.3e, worst gradient cosine %.6f" % (b, err, worst))
    assert err <= 1e-1
    assert worst >= BF16_COS[b]


# ---------------------------------------------------------------------------------------------------------------------
# semantics
# ---------------------------------------------------------------------------------------------------------------------
def _clamp_hooks(net):
    for p in net.parameters():
        if p.requires_grad:
            p.register_hook(lambda g: g.clamp(-0.01, 0.01))


def test_running_buffers_untouched_and_gradients(trained):
    net = _frozen_net("cnn_linear", trained, "fp32")
    bb = net.breath_block
    bb.layer2[0].bn1.weight.requires_grad_(False)
    bb.layer2[0].bn1.bias.requires_grad_(False)
    _clamp_hooks(net)
    before = {k: v.clone() for k, v in net.state_dict().items() if "running" in k or "num_batches" in k}
    opt = torch.optim.SGD([p for p in net.parameters() if p.requires_grad], lr=1e-3, momentum=0.9, nesterov=True)
    for i in range(3):
        opt.zero_grad()
        x, t = O.synthetic_breaths(4, seed=40 + i), O.synthetic_targets(4, seed=40 + i)
        F.binary_cross_entropy_with_logits(net(x.to(DEV), None), t.to(DEV)).backward()
        opt.step()
    after = net.state_dict()
    for k, v in before.items():
        assert torch.equal(v, after[k]), k
    for name in ("conv1_alt", "conv2", "bn2"):
        mod = getattr(bb, name, None)
        if mod is not None:
            assert all(p.grad is None for p in mod.parameters()), name
    assert bb.layer2[0].bn1.weight.grad is None and bb.layer2[0].bn1.bias.grad is None
    assert bb.layer2[0].bn2.weight.grad is not None and bb.bn1.bias.grad is not None


def test_batch_equals_per_sequence_and_eval_plan(trained):
    net = _frozen_net("cnn_linear", trained, "fp32")
    x = O.synthetic_breaths(5, seed=50).to(DEV)
    with torch.no_grad():
        batch = net(x, None)
        single = torch.cat([net(x[i:i + 1], None) for i in range(5)])
        net.eval()
        ev = net(x, None)
    assert torch.equal(batch, single)
    assert rel_err(batch.cpu(), ev.cpu()) <= 1e-6


def test_running_var_edit_after_capture(trained):
    net = _frozen_net("cnn_linear", trained, "fp32")
    x, t = O.synthetic_breaths(2, seed=60), O.synthetic_targets(2, seed=60)
    for _ in range(4):  # the third and later calls replay CUDA graphs
        net.zero_grad()
        F.binary_cross_entropy_with_logits(net(x.to(DEV), None), t.to(DEV)).backward()
    with torch.no_grad():
        net.breath_block.layer3[0].bn1.running_var.mul_(1.7)
        net.breath_block.bn1.running_mean.add_(0.05)
    net.zero_grad()
    out = net(x.to(DEV), None)
    F.binary_cross_entropy_with_logits(out, t.to(DEV)).backward()
    full = _state_of(net)
    with frozen_oracle():
        ref_out, _, ref_g = O.forward_backward({k: v.clone() for k, v in full.items()}, x, t)
    assert rel_err(out.detach().cpu(), ref_out) <= 1e-4
    g = net.breath_block.layer3[0].bn1.weight.grad.cpu()
    assert rel_err(g, ref_g["breath_block.layer3.0.bn1.weight"]) <= 1e-3


def test_back_to_train_is_the_training_step(trained):
    import deepards_b200 as D
    net = _frozen_net("cnn_linear", trained, "fp32")
    x, t = O.synthetic_breaths(3, seed=70), O.synthetic_targets(3, seed=70)
    F.binary_cross_entropy_with_logits(net(x.to(DEV), None), t.to(DEV)).backward()
    net.train()  # every BatchNorm back to batch statistics
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    fresh = D.CNNLinearNetwork(D.resnet18(), 20, 0).to(DEV)
    fresh.load_state_dict(sd)
    fresh.precision = "fp32"
    fresh.train()
    for m in (net, fresh):
        m.zero_grad()
        F.binary_cross_entropy_with_logits(m(x.to(DEV), None), t.to(DEV)).backward()
    for (n, p), (_, q) in zip(net.named_parameters(), fresh.named_parameters()):
        assert (p.grad is None) == (q.grad is None), n
        if p.grad is not None:
            assert torch.equal(p.grad, q.grad), n
    for k, v in net.state_dict().items():
        assert torch.equal(v, fresh.state_dict()[k]), k


def test_mixed_state_raises(trained):
    from deepards_b200.data_parallel import DataParallelTrainer
    net = _frozen_net("cnn_linear", trained, "fp32")
    net.breath_block.layer4[1].bn2.train()
    x = O.synthetic_breaths(2, seed=80).to(DEV)
    with pytest.raises(NotImplementedError, match="layer4.1.bn2"):
        net(x, None)
    with pytest.raises(NotImplementedError, match="layer4.1.bn2"):
        DataParallelTrainer(net).train_step(x, O.synthetic_targets(2, seed=80).to(DEV))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_deterministic(precision, trained, monkeypatch):
    if precision == "bf16":
        monkeypatch.setenv("DEEPARDS_B200_WGRAD", "deterministic")
    runs = []
    for _ in range(2):
        net = _frozen_net("cnn_linear", trained, precision)
        x, t = O.synthetic_breaths(16, seed=90), O.synthetic_targets(16, seed=90)
        F.binary_cross_entropy_with_logits(net(x.to(DEV), None), t.to(DEV)).backward()
        runs.append({n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None})
    for n in runs[0]:
        assert torch.equal(runs[0][n], runs[1][n]), n


# ---------------------------------------------------------------------------------------------------------------------
# trainer
# ---------------------------------------------------------------------------------------------------------------------
def test_trainer_matches_module_path(trained):
    from deepards_b200.data_parallel import DataParallelTrainer
    a = _frozen_net("cnn_linear", trained, "fp32")
    b = _frozen_net("cnn_linear", trained, "fp32")
    _clamp_hooks(b)
    tr = DataParallelTrainer(a, lr=1e-3, optimizer="sgd", momentum=0.9, weight_decay=1e-4, clip_val=0.01, use_graph=True)
    opt = torch.optim.SGD(b.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    before = {k: v.clone() for k, v in a.state_dict().items() if "running" in k or "num_batches" in k}
    for i in range(3):
        x, t = O.synthetic_breaths(4, seed=100 + i).to(DEV), O.synthetic_targets(4, seed=100 + i).to(DEV)
        tr.train_step(x, t)
        opt.zero_grad()
        F.binary_cross_entropy_with_logits(b(x, None), t).backward()
        opt.step()
    torch.cuda.synchronize()
    # measured on an NVIDIA B200 (1000 W): the stem convolution weight differs by 4.0e-6
    for (n, p), (_, q) in zip(a.named_parameters(), b.named_parameters()):
        assert rel_err(p.detach().cpu(), q.detach().cpu()) <= 1e-5, n
    for k, v in before.items():
        assert torch.equal(v, a.state_dict()[k]), k

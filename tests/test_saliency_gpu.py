"""GPU: input-gradient attributions (saliency.input_gradients) and the stem input-gradient kernels.

  * dards_stem_dgrad / dards_stem_frozen_dgrad / dards_stem_alt_dgrad against float64 torch autograd of conv -> BatchNorm ->
    ReLU -> pool (stage 1: conv -> BatchNorm), on randn, DC-offset, constant-breath and zero-breath data, groups of 20 and
    300 (chunked weight-gradient path), C0 16 and 64, max and avg pool, fp32 and bf16 gradients.  DC-offset data (40 +- 0.05)
    runs with avg pool only: there the gaps between max-pool window neighbours are at fp32 resolution of the forward's own
    conv output, so the float64 reference takes other arg-max decisions on many breaths
  * whole networks in fp32 against float64 autograd of the oracle with the ReLU decisions pinned from plan.sites
  * bf16 against fp32, no side effects, eager vs graph-replayed determinism, the integrated-gradients example, refusals
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import deepards_b200 as D  # noqa: E402
from oracle import cnn_linear_oracle as O  # noqa: E402
from tests import bottleneck_oracle as BO  # noqa: E402
from tests import eval_reference as E  # noqa: E402
from tests.helpers import cosine, rel_err  # noqa: E402

DEV = "cuda"
EPS = 1e-5
TIE = 1e-5   # relative gap below which a float64 decision may differ from the kernel's fp32 one


def _lib():
    from deepards_b200 import _lib
    return _lib


def _st():
    return torch.cuda.current_stream().cuda_stream


def _data(kind, n, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 224, generator=g)
    if kind == "offset":
        x = x * 0.05 + 40.0
    elif kind == "constant":
        x = torch.randn(n, 1, generator=g).expand(n, 224).contiguous() * 2.0
    elif kind == "zero":
        x[::3] = 0.0
    return x


def _params(c0, k, seed):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(c0, 1, k, generator=g) * 0.4
    gamma = 1 + 0.3 * torch.randn(c0, generator=g)
    beta = 0.2 * torch.randn(c0, generator=g)
    return w, gamma, beta


def _ref_stem(x, w, gamma, beta, group, pool, dout, frozen=None):
    """float64 autograd of the stem; returns (dx, pre-pool z, per-breath 'near-tie' flags)."""
    x = x.double().clone().requires_grad_(True)
    n, c0 = x.shape[0], w.shape[0]
    y = F.conv1d(x.view(n, 1, 224), w.double(), stride=2, padding=3)          # (N, C, 112)
    if frozen is None:
        yg = y.view(n // group, group, c0, 112).permute(0, 2, 1, 3).reshape(n // group, c0, -1)
        mean = yg.mean(-1, keepdim=True)
        var = yg.var(-1, unbiased=False, keepdim=True)
        z = (yg - mean) / torch.sqrt(var + EPS) * gamma.double()[:, None] + beta.double()[:, None]
        z = z.view(n // group, c0, group, 112).permute(0, 2, 1, 3).reshape(n, c0, 112)
    else:
        scale, shift = frozen
        z = y * scale.double()[:, None] + shift.double()[:, None]
    r = F.relu(z)
    p = F.max_pool1d(r, 3, 2, 1) if pool == 0 else F.avg_pool1d(r, 3, 2, 1)
    (dx,) = torch.autograd.grad(p, [x], dout.double().permute(0, 2, 1))
    return dx, _near_ties(z.detach(), pool)


def _near_ties(z, pool):
    """Breaths with a ReLU input, or (max pool) a pair of window neighbours, closer than TIE (relative) without being
    equal: there the fp32 kernel may take the other decision."""
    s = z.abs().mean()
    near = ((z.abs() < TIE * s) & (z != 0)).flatten(1).any(1)
    if pool == 0:
        r = F.relu(z)
        for a, b in ((r[..., :-1], r[..., 1:]), (r[..., :-2], r[..., 2:])):
            d = (a - b).abs()
            near |= ((d < TIE * s) & (d != 0) & ((a > 0) | (b > 0))).flatten(1).any(1)
    return near


def _check_dx(dx, ref, near, tol, what):
    keep = ~near.cpu()
    assert int(keep.sum()) >= 0.5 * keep.numel(), "%s: too many near-tie breaths (%d)" % (what, int(near.sum()))
    e = rel_err(dx.cpu()[keep], ref.cpu()[keep])
    assert e <= tol, "%s: dx rel err %.3e > %.1e" % (what, e, tol)
    return e


STEM_CASES = [(16, 0, torch.float32), (64, 0, torch.bfloat16), (64, 1, torch.float32), (16, 1, torch.bfloat16)]


@pytest.mark.parametrize("kind", ["randn", "offset", "constant", "zero"])
@pytest.mark.parametrize("group,n_groups", [(20, 3), (300, 1)])
@pytest.mark.parametrize("c0,pool,dtype", STEM_CASES)
def test_stem_dgrad_kernel(kind, group, n_groups, c0, pool, dtype):
    if kind == "offset" and pool == 0:
        pytest.skip("DC-offset data is checked with avg pool: max-pool window gaps are at fp32 resolution there")
    from deepards_b200 import kernels as K
    n = group * n_groups
    x = _data(kind, n, 11 + c0).to(DEV)
    w, gamma, beta = [t.to(DEV) for t in _params(c0, 7, 5 + pool)]
    out, mean, rstd = K.stem_fwd(x, w, gamma, beta, group, pool, dtype)
    dout = (torch.randn(n, 56, c0, generator=torch.Generator().manual_seed(3)) * 0.1).to(DEV).to(dtype)
    g = n // group
    dwp = torch.empty((g, c0 * 7), device=DEV)
    dgp = torch.empty((g, c0), device=DEV)
    dbp = torch.empty((g, c0), device=DEV)
    nbytes = _lib().fn("dards_stem_workspace_bytes")(g, group, c0, 1)
    ws = torch.empty(((nbytes + 3) // 4,), device=DEV) if nbytes else None
    dt = _lib().BF16 if dtype == torch.bfloat16 else _lib().F32
    _lib().call("dards_stem_bwd", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                mean.data_ptr(), rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), g, group, c0, c0, pool,
                ws.data_ptr() if ws is not None else None, nbytes, dt, _st())
    dx = torch.full((n, 224), float("nan"), device=DEV)
    _lib().call("dards_stem_dgrad", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                mean.data_ptr(), rstd.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), dx.data_ptr(), g, group, c0, c0, pool, dt,
                _st())
    torch.cuda.synchronize()
    ref, near = _ref_stem(x.cpu(), w.cpu(), gamma.cpu(), beta.cpu(), group, pool, dout.float().cpu())
    assert torch.isfinite(dx).all()
    _check_dx(dx, ref, near, 1e-4 if kind != "zero" else 2e-4, "stem %s g%d c%d p%d %s" % (kind, group, c0, pool, dtype))


@pytest.mark.parametrize("kind", ["randn", "offset", "constant", "zero"])
@pytest.mark.parametrize("c0,pool,dtype", STEM_CASES)
def test_stem_frozen_dgrad_kernel(kind, c0, pool, dtype):
    if kind == "offset" and pool == 0:
        pytest.skip("DC-offset data is checked with avg pool: max-pool window gaps are at fp32 resolution there")
    n = 150  # three chunk CTAs of the weight-gradient kernel, a partial one of the input-gradient kernel
    x = _data(kind, n, 21 + c0).to(DEV)
    w, scale, shift = [t.to(DEV) for t in _params(c0, 7, 9 + pool)]
    dout = (torch.randn(n, 56, c0, generator=torch.Generator().manual_seed(4)) * 0.1).to(DEV).to(dtype)
    dx = torch.full((n, 224), float("nan"), device=DEV)
    dt = _lib().BF16 if dtype == torch.bfloat16 else _lib().F32
    _lib().call("dards_stem_frozen_dgrad", dout.data_ptr(), x.data_ptr(), w.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                dx.data_ptr(), n, c0, c0, pool, dt, _st())
    torch.cuda.synchronize()
    ref, near = _ref_stem(x.cpu(), w.cpu(), None, None, 1, pool, dout.float().cpu(), frozen=(scale.cpu(), shift.cpu()))
    _check_dx(dx, ref, near, 1e-4, "frozen stem %s c%d p%d %s" % (kind, c0, pool, dtype))


@pytest.mark.parametrize("kind", ["randn", "offset", "constant", "zero"])
@pytest.mark.parametrize("group,n_groups", [(20, 3), (300, 1)])
@pytest.mark.parametrize("c0,dtype", [(16, torch.float32), (64, torch.bfloat16), (64, torch.float32)])
def test_stem_alt_dgrad_kernel(kind, group, n_groups, c0, dtype):
    from deepards_b200 import kernels as K
    n = group * n_groups
    x = _data(kind, n, 31 + c0).to(DEV)
    w, gamma, beta = [t.to(DEV) for t in _params(c0, 3, 13)]
    _, mean, rstd = K.stem_alt_fwd(x, w, gamma, beta, group, dtype)
    dout = (torch.randn(n, 224, c0, generator=torch.Generator().manual_seed(5)) * 0.1).to(DEV).to(dtype)
    g = n // group
    dwp = torch.empty((g, c0 * 3), device=DEV)
    dgp = torch.empty((g, c0), device=DEV)
    dbp = torch.empty((g, c0), device=DEV)
    nbytes = _lib().fn("dards_stem_alt_workspace_bytes")(g, group, c0, 1)
    ws = torch.empty(((nbytes + 3) // 4,), device=DEV) if nbytes else None
    dt = _lib().BF16 if dtype == torch.bfloat16 else _lib().F32
    _lib().call("dards_stem_alt_bwd", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), g, group, c0, c0,
                ws.data_ptr() if ws is not None else None, nbytes, dt, _st())
    dx = torch.full((n, 224), float("nan"), device=DEV)
    _lib().call("dards_stem_alt_dgrad", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                rstd.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), dx.data_ptr(), g, group, c0, c0, dt, _st())
    torch.cuda.synchronize()
    xr = x.cpu().double().requires_grad_(True)
    y = F.conv1d(xr.view(n, 1, 224), w.cpu().double(), padding=1)
    yg = y.view(g, group, c0, 224).permute(0, 2, 1, 3).reshape(g, c0, -1)
    z = (yg - yg.mean(-1, keepdim=True)) / torch.sqrt(yg.var(-1, unbiased=False, keepdim=True) + EPS)
    z = z * gamma.cpu().double()[:, None] + beta.cpu().double()[:, None]
    z = z.view(g, c0, group, 224).permute(0, 2, 1, 3).reshape(n, c0, 224)
    (ref,) = torch.autograd.grad(z, [xr], dout.float().cpu().double().permute(0, 2, 1))
    e = rel_err(dx.cpu(), ref)
    assert e <= 1e-4, "stage 1 %s g%d c%d %s: dx rel err %.3e" % (kind, group, c0, dtype, e)


# ---------------------------------------------------------------------------------------------------------------------
# networks
# ---------------------------------------------------------------------------------------------------------------------
def _net(sd, head="cnn_linear", precision="fp32", **bkw):
    rn = "breath_block.conv1.weight" in sd
    planes = sd["breath_block.conv1.weight"].shape[0] if rn else 64
    bb = D.resnet18(initial_planes=planes, **bkw) if rn else D.densenet18(drop_rate=0.0)
    net = {"cnn_linear": lambda: D.CNNLinearNetwork(bb, 20, 0),
           "per_breath": lambda: D.CNNSingleBreathLinearNetwork(bb),
           "to_mean": lambda: D.CNNLinearToMean(bb),
           "regressor": lambda: D.CNNRegressor(bb, 2)}[head]()
    net.load_state_dict(sd, strict=False)
    net = net.to(DEV)
    net.precision = precision
    return net


def _masks(plan, b, g):
    out = {}
    for site, buf in plan.sites.items():
        n, l, c = buf.shape
        out[site] = (buf.float() > 0).permute(0, 2, 1).reshape(b, g, c, l).cpu()
    return out


def _pinned_oracle_grad(sd, x, target, masks, head, regressor=False, dtype=torch.float64, forward=None, **kw):
    """autograd of the oracle (float64 by default) with the ReLU decisions pinned -> (dx, outputs, relu0 near-tie flag)."""
    sd64 = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    xr = x.to(dtype).clone().requires_grad_(True)
    rec = {}
    hooks = O.DecisionHooks(record=rec, masks=masks)
    if forward is not None:
        out = forward(sd64, xr, hooks=hooks, **kw)
    elif regressor:
        out = O.regressor_forward(sd64, xr, hooks=hooks, **kw)
    else:
        out = O.cnn_linear_forward(sd64, xr, head=head, hooks=hooks, **kw)
    seed = torch.zeros_like(out).scatter_(-1, target.cpu().unsqueeze(-1), 1.0)
    (dx,) = torch.autograd.grad(out, [xr], seed)
    z0 = torch.stack([rec["relu0"][i] for i in sorted(rec["relu0"])]) if "relu0" in rec else None
    near = z0 is not None and float(z0.abs().min() / z0.abs().mean()) < 1e-5
    return dx, out.detach(), near


NET_CASES = [
    ("resnet18_p64_max", dict(backbone="resnet18", seed=1, bn_perturb=0.1), {}, "cnn_linear"),
    ("resnet18_p16_avg", dict(backbone="resnet18", seed=3, bn_perturb=0.1, initial_planes=16),
     dict(first_pool_type="avg"), "cnn_linear"),
    ("resnet18_p16_double", dict(backbone="resnet18", seed=8, bn_perturb=0.1, initial_planes=16),
     dict(double_conv_first=True), "cnn_linear"),
    ("densenet18", dict(backbone="densenet18", seed=4, bn_perturb=0.1), {}, "cnn_linear"),
    ("resnet18_p16_per_breath", dict(backbone="resnet18", seed=6, bn_perturb=0.1, initial_planes=16, per_breath=True), {},
     "per_breath"),
]


@pytest.mark.parametrize("name,skw,fkw,head", NET_CASES, ids=[c[0] for c in NET_CASES])
def test_network_fp32_pinned(name, skw, fkw, head):
    sd = O.cnn_linear_state(**skw)
    net = _net(sd, head, **fkw)
    b = 2
    x = O.synthetic_breaths(b, seed=17).to(DEV)
    grad, out = D.input_gradients(net, x)
    plan = [p for p in net._dards_plans.values() if getattr(p, "input_grad", False)][0]
    target = out.argmax(-1)
    ref, ref_out, near = _pinned_oracle_grad(sd, x.cpu(), target, _masks(plan, b, 20), head, **fkw)
    assert grad.shape == x.shape and grad.dtype == torch.float32
    assert rel_err(out.cpu(), ref_out) <= 1e-4
    e = rel_err(grad.cpu(), ref)
    assert e <= (5e-2 if near else 1e-4), "%s: input gradient rel err %.3e (stem near-tie %s)" % (name, e, near)


def test_resnet50_fp32_pinned():
    """Bottleneck blocks (tests/bottleneck_oracle.py).  Gate: 1e-4 of the pinned float64 oracle, or -- the conditioned rule of
    test_bottleneck_gpu -- no further from it than 3x the pinned fp32 oracle's own distance."""
    sd = BO.cnn_linear_state("resnet50", seed=21, bn_perturb=0.1, initial_planes=16)
    net = D.CNNLinearNetwork(D.resnet50(initial_planes=16), 20, 0)
    net.load_state_dict(sd)
    net = net.to(DEV)
    net.precision = "fp32"
    b = 2
    x = O.synthetic_breaths(b, seed=23).to(DEV)
    grad, out = D.input_gradients(net, x)
    plan = [p for p in net._dards_plans.values() if p.input_grad][0]
    masks = _masks(plan, b, 20)
    target = out.argmax(-1)
    ref, ref_out, near = _pinned_oracle_grad(sd, x.cpu(), target, masks, None, forward=BO.cnn_linear_forward)
    ref32, _, _ = _pinned_oracle_grad(sd, x.cpu(), target, masks, None, dtype=torch.float32, forward=BO.cnn_linear_forward)
    e, e32 = rel_err(grad.cpu(), ref), rel_err(ref32, ref)
    print("resnet50 input gradient: rel err %.3e, fp32 oracle %.3e, stem near-tie %s" % (e, e32, near))
    assert e <= max(5e-2 if near else 1e-4, 3 * e32), (e, e32, near)


def test_sibling_head_and_target_forms():
    sd = O.cnn_linear_state(backbone="resnet18", seed=2, bn_perturb=0.1, initial_planes=16, per_breath=True)
    net = _net(sd, "to_mean")
    x = O.synthetic_breaths(3, seed=5).to(DEV)
    g_none, out = D.input_gradients(net, x)
    masks = _masks([p for p in net._dards_plans.values() if p.input_grad][0], 3, 20)
    ref, ref_out, near = _pinned_oracle_grad(sd, x.cpu(), out.argmax(-1), masks, "to_mean")
    assert rel_err(g_none.cpu(), ref) <= (5e-2 if near else 1e-4)
    g1, _ = D.input_gradients(net, x, 1)
    g1t, _ = D.input_gradients(net, x, torch.ones(3, dtype=torch.long))
    assert torch.equal(g1, g1t)
    g0, _ = D.input_gradients(net, x, 0)
    ref0, _, _ = _pinned_oracle_grad(sd, x.cpu(), torch.zeros(3, dtype=torch.long), masks, "to_mean")
    assert rel_err(g0.cpu(), ref0) <= (5e-2 if near else 1e-4)
    assert not torch.equal(g0, g1)


def test_regressor_flat_batch_300():
    sd = O.cnn_linear_state(backbone="resnet18", seed=9, bn_perturb=0.1, initial_planes=16, per_breath=True)
    net = _net(sd, "regressor")
    x = O.synthetic_breaths(15, seed=3).reshape(300, 1, 224).to(DEV)
    grad, out = D.input_gradients(net, x)
    plan = [p for p in net._dards_plans.values() if p.input_grad][0]
    assert plan.group == 300
    ref, ref_out, near = _pinned_oracle_grad(sd, x.cpu(), out.argmax(-1), _masks(plan, 1, 300), None, regressor=True)
    e = rel_err(grad.cpu(), ref)
    assert e <= (5e-2 if near else 1e-4), "regressor: rel err %.3e" % e


def _running_state(seed, planes=16):
    sd = O.cnn_linear_state(backbone="resnet18", seed=seed, bn_perturb=0.1, initial_planes=planes)
    g = torch.Generator().manual_seed(seed)
    for k in list(sd):
        if k.endswith("running_mean"):
            sd[k] = 0.3 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = torch.exp(0.5 * torch.randn(sd[k].shape, generator=g))
    return sd


def test_eval_and_frozen_against_running_statistics_oracle():
    sd = _running_state(41)
    net = _net(sd)
    x = O.synthetic_breaths(2, seed=8).to(DEV)
    net.eval()
    g_eval, out_eval = D.input_gradients(net, x)
    net.train()   # frozen BatchNorm: the network in train(), its BatchNorm layers in eval()
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.eval()
    g_frozen, out_frozen = D.input_gradients(net, x)
    # eval() runs the frozen plan: the same arithmetic
    assert torch.equal(g_eval, g_frozen) and torch.equal(out_eval, out_frozen)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    xr = x.cpu().double().requires_grad_(True)
    ref_out = E.cnn_linear_forward(sd64, xr)
    seed = torch.zeros_like(ref_out).scatter_(-1, out_eval.argmax(-1).cpu().unsqueeze(-1), 1.0)
    (ref,) = torch.autograd.grad(ref_out, [xr], seed)
    e = rel_err(g_eval.cpu(), ref)
    # decisions are not pinned here (the eval restatement has no hooks); measured error stated in the summary
    assert e <= 1e-4, "eval/frozen input gradient rel err %.3e" % e


def test_double_conv_first_eval_refused():
    sd = O.cnn_linear_state(backbone="resnet18", seed=8, bn_perturb=0.1, initial_planes=16)
    net = _net(sd, double_conv_first=True).eval()
    with pytest.raises(NotImplementedError, match="double_conv_first"):
        D.input_gradients(net, O.synthetic_breaths(1, seed=1).to(DEV))


def test_bf16_against_fp32():
    sd = O.cnn_linear_state(backbone="resnet18", seed=1, bn_perturb=0.1)
    x = O.synthetic_breaths(16, seed=2).to(DEV)
    g32, o32 = D.input_gradients(_net(sd, precision="fp32"), x)
    g16, o16 = D.input_gradients(_net(sd, precision="bf16"), x, o32.argmax(-1))
    c = cosine(g16.cpu(), g32.cpu())
    print("bf16 vs fp32 input-gradient cosine %.4f" % c)
    # measured on an NVIDIA B200: 0.9281 (ResNet-18, 64 planes, B = 16, at initialisation); the gate leaves that margin
    assert c >= 0.9, c


def test_no_side_effects_and_determinism():
    sd = O.cnn_linear_state(backbone="resnet18", seed=1, bn_perturb=0.1, initial_planes=16)
    net = _net(sd)
    x = O.synthetic_breaths(2, seed=4).to(DEV)
    with torch.no_grad():
        before = net(x).clone()   # (a train() forward: it updates the running buffers itself)
    bufs = {k: v.clone() for k, v in net.state_dict().items() if "running" in k or "num_batches" in k}
    grads = [D.input_gradients(net, x)[0] for _ in range(4)]   # calls 3 and 4 replay CUDA graphs
    torch.cuda.synchronize()
    for g in grads[1:]:
        assert torch.equal(g, grads[0])
    for p in net.parameters():
        assert p.grad is None
    for k, v in net.state_dict().items():
        if k in bufs:
            assert torch.equal(v, bufs[k]), k
    with torch.no_grad():
        after = net(x)
    assert torch.equal(before, after)
    # the module path still refuses autograd input gradients
    with pytest.raises(NotImplementedError):
        net(x.clone().requires_grad_(True))


def test_refusals():
    with pytest.raises(TypeError):
        D.input_gradients(torch.nn.Linear(224, 2).to(DEV), torch.zeros(2, 224, device=DEV))
    sd = O.cnn_linear_state(backbone="resnet18", seed=1, initial_planes=16)
    net = _net(sd)
    with pytest.raises(RuntimeError):
        D.input_gradients(net, torch.zeros(1, 20, 1, 224))
    meta = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 3).to(DEV)
    with pytest.raises(NotImplementedError, match="metadata"):
        D.input_gradients(meta, torch.zeros(1, 20, 1, 224, device=DEV))
    with pytest.raises(ValueError):
        D.input_gradients(net, torch.zeros(1, 20, 1, 224, device=DEV), torch.zeros(3, dtype=torch.long))


def test_integrated_gradients_completeness():
    """The INTEGRATION.md example: a ResNet in eval(), 256 alpha-scaled copies stacked on the batch dimension, one call."""
    sd = _running_state(43, planes=64)
    net = _net(sd).eval()
    x = O.synthetic_breaths(1, seed=6).to(DEV)          # (1, 20, 1, 224)
    base = torch.zeros_like(x)
    steps = 256   # 32 midpoint steps measured sum 0.02635 against 0.03494: the Riemann sum over the ReLU kinks
    alphas = (torch.arange(steps, device=DEV, dtype=torch.float32) + 0.5) / steps
    path = base + alphas.view(-1, 1, 1, 1) * (x - base)
    target = int(D.input_gradients(net, x)[1].argmax())
    g, _ = D.input_gradients(net, path, target)
    attr = (x - base) * g.mean(0, keepdim=True)
    with torch.no_grad():
        f = D.input_gradients(net, torch.cat([x, base]), target)[1][:, target]
    gap = float(f[0] - f[1])
    err = abs(float(attr.sum()) - gap)
    print("integrated gradients: sum %.5f, f(x) - f(base) %.5f, |diff| %.2e" % (float(attr.sum()), gap, err))
    # measured on an NVIDIA B200 with 256 steps: sum 0.03538 against 0.03494, |diff| 4.3e-4 (1.2 % of the gap)
    assert err <= 0.05 * abs(gap)


def test_eval_plan_refuses_input_grad():
    from deepards_b200 import engine
    net = _net(O.cnn_linear_state(backbone="resnet18", seed=1, initial_planes=16)).eval()
    with pytest.raises(ValueError, match="input_grad"):
        engine.Plan(net, net.breath_block, None, 20, 20, "fp32", "backbone", (), False, bn="eval", input_grad=True)


def _scalars(args):
    """The recorded arguments that are not device pointers (shapes, strides, flags, dtypes)."""
    return tuple(a for a in args if not (isinstance(a, int) and abs(a) >= 1 << 32))


@pytest.mark.parametrize("backbone", ["resnet18", "densenet18", "resnet50", "resnet18_double"])
@pytest.mark.parametrize("bn", ["train", "frozen"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_input_grad_plan_adds_only_the_dgrad_call(backbone, bn, precision):
    """An input_grad plan records the calls of the plan without it, plus one stem dgrad call right after the stem
    backward; the plan without it is cached under the key it always had."""
    from deepards_b200 import engine
    if backbone.startswith("densenet") and bn == "frozen":
        pytest.skip("DenseNet has no frozen BatchNorm")
    if backbone == "resnet18_double" and bn == "frozen":
        pytest.skip("double_conv_first has no frozen plan")
    bb = {"resnet18": lambda: D.resnet18(initial_planes=16), "densenet18": lambda: D.densenet18(drop_rate=0.0),
          "resnet50": lambda: D.resnet50(initial_planes=16),
          "resnet18_double": lambda: D.resnet18(initial_planes=16, double_conv_first=True)}[backbone]()
    net = D.CNNLinearNetwork(bb, 20, 0).to(DEV)
    if bn == "frozen":
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.eval()
    plain = engine.get_plan(net, bb, None, 40, 20, precision, "backbone", (), False, bn=bn)
    grad = engine.get_plan(net, bb, None, 40, 20, precision, "backbone", (), False, bn=bn, input_grad=True)
    assert plain is not grad and plain.dx is None and grad.dx.shape == (40, 224)
    key = [k for k, v in net._dards_plans.items() if v is plain][0]
    assert "input_grad" not in key
    a = [(n, _scalars(args)) for n, _, args in plain.bwd.calls]
    b = [(n, _scalars(args)) for n, _, args in grad.bwd.calls]
    extra = [i for i, (n, _) in enumerate(b) if n.startswith("dards_stem") and n.endswith("_dgrad")]
    assert len(extra) == 1
    i = extra[0]
    assert b[i - 1][0] in ("dards_stem_bwd", "dards_stem_frozen_bwd", "dards_stem_alt_bwd")
    assert b[:i] + b[i + 1:] == a
    assert [(n, _scalars(x)) for n, _, x in plain.fwd.calls] == [(n, _scalars(x)) for n, _, x in grad.fwd.calls]

"""GPU: DataParallelTrainer on every head of the package.  The sibling heads (and CNNLinearNetwork /
CNNSingleBreathLinearNetwork with a caller-supplied criterion) take the generic step: backbone plan forward, the head's
torch arithmetic and the criterion under autograd, backbone plan backward, the fused clamp + optimizer update.  Held
against the module path with torch.optim (the reference's loop), against float64 autograd on the oracle, and eager
against CUDA-graph replay."""
import copy
import warnings

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import cnn_linear_oracle as O  # noqa: E402
from tests.helpers import cosine, rel_err  # noqa: E402

DEV = "cuda"
HEADS = ["to_mean", "compr_to_rf", "double_linear", "regressor", "lstm", "transformer"]
STEM_UNUSED = ("breath_block.conv1_alt.weight", "breath_block.conv2.weight", "breath_block.bn2.weight",
               "breath_block.bn2.bias")
# the package's bf16 gates (tests/test_model_parity_gpu.py)
BF16_LOSS_TOL, BF16_GRAD_COS, BF16_GRAD_COS_MEAN = 5e-3, 0.82, 0.93


def _make(kind, seed=0, precision="fp32", backbone="resnet18"):
    import deepards_b200 as D
    torch.manual_seed(seed)
    bb = D.resnet18(initial_planes=16) if backbone == "resnet18" else D.densenet18(drop_rate=0.0)
    net = {"to_mean": lambda: D.CNNLinearToMean(bb), "compr_to_rf": lambda: D.CNNLinearComprToRF(bb),
           "double_linear": lambda: D.CNNDoubleLinearNetwork(bb, 20, 0), "regressor": lambda: D.CNNRegressor(bb, 3),
           "lstm": lambda: D.CNNLSTMNetwork(bb, 0, False, 32),
           "transformer": lambda: D.CNNTransformerNetwork(bb, 0, False, 64, 2),
           "cnn_linear": lambda: D.CNNLinearNetwork(bb, 20, 0),
           "per_breath": lambda: D.CNNSingleBreathLinearNetwork(bb)}[kind]()
    for m in net.modules():
        if isinstance(m, nn.Dropout):
            m.p = 0.0               # the transformer's dropout draws from torch's RNG: compared with dropout off
    net = net.to(DEV).train()
    net.precision = precision
    return net


def _pair(kind, seed=0, precision="fp32", backbone="resnet18"):
    a = _make(kind, seed, precision, backbone)
    b = _make(kind, seed, precision, backbone)
    b.load_state_dict(a.state_dict())
    return a, b


def _criterion(kind):
    return nn.MSELoss() if kind == "regressor" else nn.BCEWithLogitsLoss()


def _batch(kind, b, seed):
    """(x, target) as the module path takes them: sequences (B, 20, 1, 224), breaths (20 B, 1, 224) for the regressor;
    per-step targets (B, 20, 2) for the LSTM / transformer / per-breath heads."""
    x = O.synthetic_breaths(b, seed=seed)
    t = O.synthetic_targets(b, seed=seed)
    if kind == "regressor":
        x = x.reshape(-1, 1, 224)
        t = torch.randn(x.shape[0], 3, generator=torch.Generator().manual_seed(seed))
    elif kind in ("lstm", "transformer", "per_breath"):
        t = t.unsqueeze(1).repeat(1, 20, 1)
    return x.to(DEV), t.to(DEV)


def _out(out):
    return out[0] if isinstance(out, tuple) else out     # CNNLSTMNetwork: (per-step outputs, (hx, cx))


def _clamp_hooks(net, clip=0.01):
    for p in net.parameters():
        if p.requires_grad:
            p.register_hook(lambda g: torch.clamp(g, -clip, clip))


def _module_optimizer(net, optimizer):
    params = [p for p in net.parameters() if p.requires_grad]
    if optimizer == "sgd":
        return torch.optim.SGD(params, lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    return torch.optim.Adam(params, lr=1e-3)


def _module_step(net, opt, crit, x, t):
    opt.zero_grad()
    loss = crit(_out(net(x, None)), t)
    loss.backward()
    opt.step()
    return float(loss)


def _trainer(net, optimizer="sgd", use_graph=False, criterion=None, lr=1e-3):
    from deepards_b200.data_parallel import DataParallelTrainer
    return DataParallelTrainer(net, lr=lr, optimizer=optimizer, momentum=0.9, weight_decay=1e-4, clip_val=0.01,
                               use_graph=use_graph, criterion=criterion)


def _plan(tr, x):
    return tr.plan_for(x)


def _grads(tr, plan):
    """{name: gradient} of the latest step, read from the plan's flat buffer (before the clamp, which the update
    kernel applies on the fly)."""
    return {n: plan.grad_view(p).clone() for n, p, _ in tr.layout
            if id(p) in plan.grad_written or any(p is q for q in tr.head_params)}


def _sync_adam(tr, net, opt):
    """Start the module path's next Adam step from the trainer's weights and moments."""
    with torch.no_grad():
        for (_, p, off), q in zip(tr.layout, net.parameters()):
            q.copy_(p)
            st = opt.state.get(q)
            if st:
                st["exp_avg"].copy_(tr.state1[off:off + q.numel()].view_as(q))
                st["exp_avg_sq"].copy_(tr.state2[off:off + q.numel()].view_as(q))


# ---- the module path + torch.optim ----------------------------------------------------------------------------------
@pytest.mark.parametrize("optimizer", ["sgd", "adam"])
@pytest.mark.parametrize("kind", HEADS)
def test_trainer_steps_match_the_module_path(kind, optimizer):
    """Three steps: the reference's loop (model(x, meta) -> criterion -> backward -> clamp hooks +-0.01 -> torch.optim)
    on the module path against DataParallelTrainer with the same criterion: every parameter within 1e-5.  Parameters
    that get no gradient (the stem's conv1_alt / conv2 / bn2) stay unchanged, and the BatchNorm running statistics agree.

    Adam moves every weight by about lr per step whatever its gradient's size, so two fp32 trajectories that differ in
    the last bits after the first update (fused kernel against torch.optim, the same formula) take different ReLU and
    median decisions in the next forward and part: measured on an NVIDIA B200, up to 1.2e-3 after three steps, where SGD
    stays within 1e-8.  For Adam, steps 2 and 3 therefore start the module path from the trainer's weights and moments,
    and each step is held to 1e-5."""
    a, b = _pair(kind, seed=11)
    init = {n: p.detach().clone() for n, p in a.named_parameters()}
    crit = _criterion(kind)
    _clamp_hooks(b)
    opt = _module_optimizer(b, optimizer)
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        tr = _trainer(a, optimizer, criterion=crit if kind == "regressor" else None)
        for i in range(3):
            x, t = _batch(kind, 3, 700 + i)
            if optimizer == "adam" and i > 0:
                _sync_adam(tr, b, opt)
            lt = float(tr.train_step(x, t))
            lm = _module_step(b, opt, crit, x, t)
            assert abs(lt - lm) <= 1e-5 * max(1.0, abs(lm)), (i, lt, lm)
            d = max(float((p.detach() - q.detach()).abs().max()) for p, q in zip(a.parameters(), b.parameters()))
            assert d <= 1e-5, (i, d)
        torch.cuda.synchronize()
    # the head's LSTM runs ATen's LSTM (cuDNN is off in CNNLSTMNetwork._head), which reads the weights where the trainer's
    # flat buffer holds them: no per-call weight copy, no warning
    assert not [w for w in caught if "contiguous" in str(w.message)], [str(w.message) for w in caught]
    diff = torch.cat([(p.detach() - q.detach()).abs().reshape(-1) for p, q in zip(a.parameters(), b.parameters())])
    print("%s %s: parameters after 3 steps, max |trainer - module path| %.2e" % (kind, optimizer, float(diff.max())))
    for n, p in a.named_parameters():
        if n in STEM_UNUSED:
            assert torch.equal(p.detach(), init[n]), n
    for (n, p), (_, q) in zip(a.state_dict().items(), b.state_dict().items()):
        if "running" in n:
            assert rel_err(p.cpu(), q.cpu()) <= 1e-5, n


@pytest.mark.parametrize("kind", HEADS)
def test_eager_and_graph_replay_are_bit_identical(kind):
    out = {}
    for use_graph in (False, True):
        net = _make(kind, seed=12)
        tr = _trainer(net, "sgd", use_graph=use_graph, criterion=_criterion(kind))
        losses = [float(tr.train_step(*_batch(kind, 2, 710 + i % 2))) for i in range(5)]
        torch.cuda.synchronize()
        out[use_graph] = (losses, tr.param_flat.clone(), {k: v.clone() for k, v in net.state_dict().items()})
    assert tr.graph_launches > 0          # the step was replayed from a captured graph
    assert out[False][0] == out[True][0]
    assert torch.equal(out[False][1], out[True][1])
    for k in out[False][2]:
        assert torch.equal(out[False][2][k], out[True][2][k]), k


# ---- float64 oracle -------------------------------------------------------------------------------------------------
def _transformer_oracle(head, sd, x):
    """The transformer head restated on the oracle: the oracle's backbone per sequence, then `head`, a copy of the
    module's own transformer blocks, and the final linear (test_extra_gpu.py holds these modules against the
    reference's)."""
    feats = torch.stack([O.backbone_forward(sd, x[i]) for i in range(x.shape[0])])
    out = F.linear(head(feats), sd["linear_final.weight"], sd["linear_final.bias"])
    return out, {"transformer." + n: p for n, p in head.named_parameters()}


def _oracle_grads(kind, sd, head, x, t, names, dtype):
    """{name: gradient} of the criterion on the oracle (and, for the transformer, a copy of the module's own head)
    in `dtype`, by torch autograd."""
    sd = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in sd.items()}
    leaves = {k: sd[k].clone().requires_grad_(True) for k in names if k in sd}
    sd.update(leaves)
    x, t = x.to(dtype), t.to(dtype)
    params = dict(leaves)
    if kind == "regressor":
        out = O.regressor_forward(sd, x)
    elif kind == "transformer":
        h = copy.deepcopy(head).to(dtype)
        out, extra = _transformer_oracle(h, sd, x)
        params.update(extra)
    else:
        out = O.cnn_linear_forward(sd, x, head=kind)
    loss = _criterion(kind)(out, t)
    grads = torch.autograd.grad(loss, [params[k] for k in names])
    return float(loss.detach()), dict(zip(names, grads))


@pytest.mark.parametrize("kind", HEADS)
def test_first_step_gradients_match_the_float64_oracle(kind):
    """The first step's gradients (the trainer's flat buffer, before the clamp) against float64 autograd on the oracle:
    within 1e-4, or -- where the step is ill-conditioned -- as close to float64 as the oracle's own fp32 arithmetic gets
    on a few-ulp perturbation of the input (the package's gate, tests/helpers.py::conditioned_grad_check).  The
    regressor's 40 breaths are one BatchNorm group; its ReLU / max-pool near-ties move whole gradient tensors (measured
    on an NVIDIA B200: 1.0e-2 from float64 for layer4.0.bn1.bias, where the module path gives the same numbers)."""
    net = _make(kind, seed=13)
    sd = {k: v.detach().cpu().double().clone() for k, v in net.state_dict().items()}
    head = copy.deepcopy(net.transformer).cpu().double() if kind == "transformer" else None
    tr = _trainer(net, "sgd", criterion=_criterion(kind))
    x, t = _batch(kind, 2, 720)
    plan = _plan(tr, x)
    loss = float(tr.train_step(x, t))
    torch.cuda.synchronize()
    mine = {k: v.cpu() for k, v in _grads(tr, plan).items()}
    names = list(mine)
    x, t = x.cpu(), t.cpu()
    ref_loss, g64 = _oracle_grads(kind, sd, head, x, t, names, torch.float64)
    assert abs(loss - ref_loss) <= 1e-5 * max(1.0, abs(ref_loss))
    gmax = max(float(v.abs().max()) for v in g64.values())
    # a parameter whose exact gradient is zero (the transformer's key bias: a constant added to every key shifts each
    # softmax row uniformly) holds rounding noise on both sides: measured against 1e-3 of the largest gradient entry
    floor = dict((k, max(float(v.abs().max()), 1e-3 * gmax)) for k, v in g64.items())
    err = lambda a, k: float((a.double() - g64[k]).abs().max()) / floor[k]  # noqa: E731
    errs = dict((k, err(mine[k], k)) for k in names)
    worst = max(errs, key=errs.get)
    print("%s: first-step gradients vs float64, worst rel err %.2e (%s)" % (kind, errs[worst], worst))
    if errs[worst] <= 1e-4:
        return
    sens = 0.0
    for s_ in (0, 1, -1, 2, -2):
        _, g32 = _oracle_grads(kind, sd, head, x * (1.0 + s_ * 2.0 ** -21), t, names, torch.float32)
        sens = max(sens, max(err(g32[k], k) for k in names))
    allow = min(0.2, max(1e-4, 3.0 * sens))
    print("%s: the oracle's own fp32 sensitivity %.2e, allowance %.2e" % (kind, sens, allow))
    bad = dict((k, e) for k, e in errs.items() if e > allow)
    assert not bad, (allow, bad)


# ---- the regressor's flat batch ----------------------------------------------------------------------------------------
def test_regressor_normalises_the_whole_flat_batch_and_trains_with_mse():
    a, b = _pair("regressor", seed=14)
    tr = _trainer(a, "sgd", criterion=nn.MSELoss(), lr=1e-2)
    x, t = _batch("regressor", 4, 730)
    losses = [float(tr.train_step(x, t))]
    with torch.no_grad():
        b(x, None)                          # the module path: one BatchNorm group over all 80 breaths
    for (n, p), (_, q) in zip(a.state_dict().items(), b.state_dict().items()):
        if "running" in n:
            assert rel_err(p.cpu(), q.cpu()) <= 1e-6, n
    # ...which differs from normalising the two halves separately
    c = _make("regressor", seed=14)
    c.load_state_dict(b.state_dict())
    with torch.no_grad():
        c(x[:40], None)
        c(x[40:], None)
    assert rel_err(c.breath_block.bn1.running_mean.cpu(), b.breath_block.bn1.running_mean.cpu()) > 1e-4
    for _ in range(19):
        losses.append(float(tr.train_step(x, t)))
    assert losses[-1] < 0.9 * losses[0], losses


# ---- CNNLinearNetwork / CNNSingleBreathLinearNetwork with a caller-supplied criterion -------------------------------
@pytest.mark.parametrize("kind", ["cnn_linear", "per_breath"])
def test_custom_criterion_on_the_fused_heads_matches_the_module_path(kind):
    a, b = _pair(kind, seed=15)
    crit = nn.BCEWithLogitsLoss(pos_weight=torch.tensor([2.0, 0.5], device=DEV))
    _clamp_hooks(b)
    opt = _module_optimizer(b, "sgd")
    tr = _trainer(a, "sgd", criterion=crit)
    for i in range(3):
        x, t = _batch(kind, 3, 740 + i)
        assert tr.plan_for(x).mode == "backbone"
        lt = float(tr.train_step(x, t))
        lm = _module_step(b, opt, crit, x, t)
        assert abs(lt - lm) <= 1e-5, (lt, lm)
    torch.cuda.synchronize()
    for (n, p), (_, q) in zip(a.named_parameters(), b.named_parameters()):
        assert rel_err(p.detach().cpu(), q.detach().cpu()) <= 1e-5, n
    # the default criterion keeps the fused plan
    tr2 = _trainer(_make(kind, seed=15), "sgd")
    assert tr2.plan_for(_batch(kind, 3, 740)[0]).mode == kind


# ---- global_batch, raw windows, refusals -----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", HEADS)
def test_ragged_global_batch_weights_the_gradient(kind):
    """A rank holding 3 of 5 sequences (regressor: 60 of 100 breaths) back-propagates its local mean weighted by 3/5."""
    x, t = _batch(kind, 3, 750)
    grads = []
    for global_batch in (None, 5 * x.shape[0] // 3):
        net = _make(kind, seed=16)
        tr = _trainer(net, "sgd", criterion=_criterion(kind))
        plan = _plan(tr, x)
        tr.train_step(x, t, global_batch=global_batch)
        torch.cuda.synchronize()
        grads.append(plan.grad_flat.clone())
    assert rel_err(grads[1], grads[0] * 0.6) <= 1e-5


@pytest.mark.parametrize("kind", HEADS)
def test_train_step_raw_equals_train_step(kind):
    mu, std = 1.5, 7.0
    x, t = _batch(kind, 2, 760)
    raw = (x.double() * std + mu)
    scaled = ((raw - mu) / std).float()
    res = []
    for use_raw in (False, True):
        net = _make(kind, seed=17)
        tr = _trainer(net, "sgd", criterion=_criterion(kind))
        for _ in range(2):
            loss = tr.train_step_raw(raw, t, mu, std) if use_raw else tr.train_step(scaled, t)
        res.append((float(loss), tr.param_flat.clone()))
    assert res[0][0] == res[1][0] and torch.equal(res[0][1], res[1][1])


def test_unknown_nets_and_metadata_heads_are_refused():
    import deepards_b200 as D
    from deepards_b200.data_parallel import DataParallelTrainer
    with pytest.raises(TypeError, match="Sequential"):
        DataParallelTrainer(nn.Sequential(nn.Linear(4, 2)).to(DEV))
    with pytest.raises(TypeError, match="ResNet"):
        DataParallelTrainer(D.resnet18(initial_planes=16).to(DEV))
    x, t = _batch("to_mean", 2, 770)
    net = D.CNNDoubleLinearNetwork(D.resnet18(initial_planes=16), 20, 3).to(DEV)
    with pytest.raises(NotImplementedError, match="metadata"):
        DataParallelTrainer(net).train_step(x, t)
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 3).to(DEV)
    with pytest.raises(NotImplementedError, match="metadata"):
        DataParallelTrainer(net, criterion=nn.BCEWithLogitsLoss()).train_step(x, t)
    with pytest.raises(NotImplementedError, match="metadata"):
        D.CNNLSTMNetwork(D.resnet18(initial_planes=16), 3, False, 32)


# ---- bf16 -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", HEADS)
def test_bf16_step_agrees_with_the_module_path_and_trains(kind):
    a, b = _pair(kind, seed=18, precision="bf16")
    crit = _criterion(kind)
    tr = _trainer(a, "sgd", criterion=crit, lr=1e-2)
    x, t = _batch(kind, 4, 780)
    plan = _plan(tr, x)
    loss = float(tr.train_step(x, t))
    torch.cuda.synchronize()
    mine = _grads(tr, plan)
    ref_loss = crit(_out(b(x, None)), t)
    ref_loss.backward()
    assert abs(loss - float(ref_loss)) <= BF16_LOSS_TOL, (loss, float(ref_loss))
    cs = [cosine(mine[n].cpu(), p.grad.cpu()) for n, p in b.named_parameters()
          if p.grad is not None and p.numel() >= 64]
    assert min(cs) >= BF16_GRAD_COS and sum(cs) / len(cs) >= BF16_GRAD_COS_MEAN, (min(cs), sum(cs) / len(cs))
    losses = [loss]
    for _ in range(19):
        losses.append(float(tr.train_step(x, t)))
    assert losses[-1] < losses[0], losses

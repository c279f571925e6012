"""CPU: the frozen-BatchNorm reference and the rule that picks a plan from the modules' training flags.

A network in train() whose BatchNorm layers are in eval() normalises with the running statistics and back-propagates
through that fixed affine map.  The GPU tests (test_frozen_bn_gpu.py) check the backend against the oracle with its
BatchNorm replaced by F.batch_norm(training=False); here that patched oracle is checked against tests/eval_reference.py,
forward and gradients, on the same state.
"""
import contextlib

import pytest
import torch
import torch.nn.functional as F

from oracle import cnn_linear_oracle as O
from tests import eval_reference as R


def _frozen_bn(x, sd, name, running_update):
    return F.batch_norm(x, sd[name + ".running_mean"], sd[name + ".running_var"], sd[name + ".weight"], sd[name + ".bias"],
                        False, O.BN_MOMENTUM, O.BN_EPS)


@contextlib.contextmanager
def frozen_oracle():
    """The oracle with every BatchNorm normalising with its running statistics (nn.BatchNorm1d in eval())."""
    orig = O._batchnorm
    O._batchnorm = _frozen_bn
    try:
        yield
    finally:
        O._batchnorm = orig


def _state(seed, pool="max"):
    sd = O.cnn_linear_state("resnet18", seed=seed, bn_perturb=0.1)
    g = torch.Generator().manual_seed(seed + 1)
    for k in list(sd):
        if k.endswith("running_mean"):
            sd[k] = 0.3 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = torch.exp(0.5 * torch.randn(sd[k].shape, generator=g))
    return sd


@pytest.mark.parametrize("per_breath", [False, True])
def test_frozen_oracle_matches_eval_reference(per_breath):
    sd = _state(11)
    if per_breath:
        torch.manual_seed(6)
        lin = torch.nn.Linear(512, 2)
        sd["linear_final.weight"], sd["linear_final.bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
    x, t = O.synthetic_breaths(2, seed=5), O.synthetic_targets(2, seed=5)
    if per_breath:
        t = t.unsqueeze(1).expand(-1, 20, -1).contiguous()
    with frozen_oracle():
        out, loss, grads = O.forward_backward({k: v.clone() for k, v in sd.items()}, x, t, per_breath=per_breath)
    leaves = {k: (v.detach().clone().requires_grad_(True) if k in grads else v) for k, v in sd.items()}
    ref = R.cnn_linear_forward(leaves, x, per_breath=per_breath)
    ref_loss = O.bce_with_logits(ref, t)
    names = sorted(grads)
    ref_grads = torch.autograd.grad(ref_loss, [leaves[k] for k in names])
    ref = ref.detach()
    assert float((out - ref).abs().max()) <= 1e-6 * float(ref.abs().max())
    for k, g in zip(names, ref_grads):
        assert float((grads[k] - g).abs().max()) <= 1e-6 * float(g.abs().max()) + 1e-12, k
    # frozen statistics: the batch does not enter the normalisation, so the stem's unused bn2 / conv2 get no gradient
    assert not any(k.startswith(("breath_block.bn2", "breath_block.conv2", "breath_block.conv1_alt")) for k in grads)


def test_bn_mode_rule():
    import deepards_b200 as D
    from deepards_b200 import engine
    bb = D.resnet18()
    bb.train()
    assert engine.bn_mode(bb) == "train"
    for m in bb.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.eval()
    assert engine.bn_mode(bb) == "frozen"
    bb.bn2.train()  # the stem's bn2 takes no part in forward(): it does not count
    assert engine.bn_mode(bb) == "frozen"
    bb.layer3[1].bn2.train()
    with pytest.raises(NotImplementedError, match=r"in train\(\): .*layer3\.1\.bn2.*in eval\(\): bn1, layer1\.0\.bn1"):
        engine.bn_mode(bb)
    bb.eval()
    bb.layer3[1].bn2.train()
    assert engine.bn_mode(bb) == "eval"  # a backbone in eval() is inference, whatever its BatchNorm layers say
    names = [n for n, _ in engine.resnet_bn_layers(bb)]
    assert len(names) == 1 + 8 * 2 + 3 and "bn2" not in names


def test_densenet_ignores_bn_flags():
    """DenseNet's BatchNorm layers keep no running statistics: torch normalises with the batch statistics in train() and
    in eval() alike, so the training plan is the right one in either state."""
    import deepards_b200 as D
    from deepards_b200 import engine
    bb = D.densenet18(drop_rate=0.0)
    bns = [m for m in bb.modules() if isinstance(m, torch.nn.BatchNorm1d)]
    assert bns and all(m.running_mean is None for m in bns)
    x = torch.randn(6, 64, 14)
    m = bns[1]
    if m.num_features != 64:
        m = torch.nn.BatchNorm1d(64, track_running_stats=False)
    m.train()
    a = m(x)
    m.eval()
    b = m(x)
    assert torch.equal(a, b)
    bb.train()
    for n in bns:
        n.eval()
    assert engine.bn_mode(bb) == "train"
    bb.eval()
    assert engine.bn_mode(bb) == "train"

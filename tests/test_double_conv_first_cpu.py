"""CPU: the references for ResNet double_conv_first=True, and the plan rule for its stem's bn2.

With double_conv_first the stem is conv1_alt (k3, s1, p1) -> bn1 -> conv2 (k7, s2, p3) -> bn2 -> ReLU -> first pool
(resnet.py:141-163); conv1 is unused.  The GPU tests (test_double_conv_first_gpu.py) compare the backend with the oracle's
double path in train() and with `eval_forward` below in eval(); here both references are checked against the module's own
nn children run in plain torch.
"""
import pytest
import torch
import torch.nn.functional as F

import deepards_b200 as D
from deepards_b200 import engine
from oracle import cnn_linear_oracle as O
from tests.helpers import rel_err


def children_forward(m, x):
    """The reference ResNet.forward restated on the module's children (BasicBlock.forward is a stub here)."""
    if m.double_conv_first:
        y = m.bn1(m.conv1_alt(x))
        y = F.relu(m.bn2(m.conv2(y)))
    else:
        y = F.relu(m.bn1(m.conv1(x)))
    y = m.first_pool(y)
    for layer in (m.layer1, m.layer2, m.layer3, m.layer4):
        for blk in layer:
            out = F.relu(blk.bn1(blk.conv1(y)))
            out = blk.bn2(blk.conv2(out))
            res = blk.downsample(y) if blk.downsample is not None else y
            y = F.relu(out + res)
    return m.avgpool(y).flatten(1)


def _bn_eval(t, sd, name):
    """BatchNorm1d in eval() as the backend applies it: y * scale + shift, scale = gamma / sqrt(running_var + eps)."""
    scale = sd[name + ".weight"] / torch.sqrt(sd[name + ".running_var"] + O.BN_EPS)
    shift = sd[name + ".bias"] - sd[name + ".running_mean"] * scale
    return t * scale[None, :, None] + shift[None, :, None]


def eval_forward(sd, x, first_pool_type="max", prefix=""):
    """(N, 1, 224) -> (N, 8 * initial_planes): a double_conv_first ResNet in eval(), every breath on its own."""
    g = lambda k: sd[prefix + k]
    bn = lambda t, name: _bn_eval(t, {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}, name)
    y = bn(F.conv1d(x, g("conv1_alt.weight"), stride=1, padding=1), "bn1")
    y = F.relu(bn(F.conv1d(y, g("conv2.weight"), stride=2, padding=3), "bn2"))
    y = F.max_pool1d(y, 3, 2, 1) if first_pool_type == "max" else F.avg_pool1d(y, 3, 2, 1)
    li = 1
    while (prefix + "layer%d.0.conv1.weight" % li) in sd:
        bi = 0
        while (prefix + "layer%d.%d.conv1.weight" % (li, bi)) in sd:
            pre = "layer%d.%d." % (li, bi)
            stride = 2 if (li > 1 and bi == 0) else 1
            out = F.relu(bn(F.conv1d(y, g(pre + "conv1.weight"), stride=stride, padding=1), pre + "bn1"))
            out = bn(F.conv1d(out, g(pre + "conv2.weight"), stride=1, padding=1), pre + "bn2")
            if (prefix + pre + "downsample.0.weight") in sd:
                res = bn(F.conv1d(y, g(pre + "downsample.0.weight"), stride=stride), pre + "downsample.1")
            else:
                res = y
            y = F.relu(out + res)
            bi += 1
        li += 1
    return F.avg_pool1d(y, 7, 1).flatten(1)


def eval_cnn_linear_forward(sd, x, first_pool_type="max", per_breath=False):
    """cnn_linear / per_breath heads over `eval_forward` (torch_cnn_linear_network.py:57-67, 104-113)."""
    b, g = x.shape[0], x.shape[1]
    feat = eval_forward(sd, x.reshape(b * g, 1, 224), first_pool_type, prefix="breath_block.")
    w, bias = sd["linear_final.weight"], sd["linear_final.bias"]
    if per_breath:
        return F.linear(feat, w, bias).view(b, g, -1)
    return F.linear(feat.reshape(b, -1), w, bias)


def double_state(seed, initial_planes=64, pool="max", running=False):
    """A double_conv_first cnn_linear state dict: the module's He init with perturbed BatchNorm affine parameters, and,
    with running=True, random running statistics."""
    torch.manual_seed(seed)
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=initial_planes, first_pool_type=pool, double_conv_first=True), 20, 0)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(seed + 1)
    for k in list(sd):
        if k.endswith("bn1.weight") or k.endswith("bn2.weight") or k.endswith("downsample.1.weight"):
            sd[k] = 1 + 0.1 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("bn1.bias") or k.endswith("bn2.bias") or k.endswith("downsample.1.bias"):
            sd[k] = 0.1 * torch.randn(sd[k].shape, generator=g)
        elif running and k.endswith("running_mean"):
            sd[k] = 0.3 * torch.randn(sd[k].shape, generator=g)
        elif running and k.endswith("running_var"):
            sd[k] = torch.exp(0.5 * torch.randn(sd[k].shape, generator=g))
    return sd


def _backbone(sd, pool, initial_planes):
    m = D.resnet18(initial_planes=initial_planes, first_pool_type=pool, double_conv_first=True)
    m.load_state_dict({k[len("breath_block."):]: v for k, v in sd.items() if k.startswith("breath_block.")})
    return m


@pytest.mark.parametrize("pool,initial_planes", [("max", 64), ("avg", 16)])
def test_oracle_double_path_matches_module_children(pool, initial_planes):
    sd = double_state(3, initial_planes, pool)
    m = _backbone(sd, pool, initial_planes).train()
    x = O.synthetic_breaths(2, seed=4).reshape(40, 1, 224)
    bsd = {k[len("breath_block."):]: v.clone() for k, v in sd.items() if k.startswith("breath_block.")}
    leaves = {k: (v.requires_grad_(True) if v.is_floating_point() and "running" not in k else v) for k, v in bsd.items()}
    ref = O.resnet_forward(leaves, x, first_pool_type=pool, double_conv_first=True, running_update=True)
    out = children_forward(m, x)
    assert rel_err(ref.detach(), out.detach()) <= 1e-5
    gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(5))
    names = [k for k, v in leaves.items() if isinstance(v, torch.Tensor) and v.requires_grad]
    grads = dict(zip(names, torch.autograd.grad(ref, [leaves[k] for k in names], gout, allow_unused=True)))
    out.backward(gout)
    params = dict(m.named_parameters())
    assert grads["conv1.weight"] is None and params["conv1.weight"].grad is None
    for k in ("conv1_alt.weight", "bn1.weight", "bn1.bias", "conv2.weight", "bn2.weight", "bn2.bias",
              "layer1.0.conv1.weight", "layer4.1.bn2.weight"):
        assert grads[k] is not None, k
        assert rel_err(grads[k], params[k].grad) <= 1e-4, k
    # both stem BatchNorm layers update their running statistics once
    buffers = dict(m.named_buffers())
    for k in ("bn1", "bn2"):
        assert rel_err(leaves[k + ".running_mean"], buffers[k + ".running_mean"]) <= 1e-5
        assert rel_err(leaves[k + ".running_var"], buffers[k + ".running_var"]) <= 1e-5
        assert int(leaves[k + ".num_batches_tracked"]) == int(buffers[k + ".num_batches_tracked"]) == 1


@pytest.mark.parametrize("pool", ["max", "avg"])
def test_eval_restatement_matches_module_children_in_eval(pool):
    sd = double_state(7, 64, pool, running=True)
    m = _backbone(sd, pool, 64).eval()
    x = O.synthetic_breaths(1, seed=8).reshape(20, 1, 224)
    bsd = {k[len("breath_block."):]: v for k, v in sd.items() if k.startswith("breath_block.")}
    with torch.no_grad():
        assert rel_err(eval_forward(bsd, x, pool), children_forward(m, x)) <= 1e-5
        # every breath on its own
        assert rel_err(eval_forward(bsd, x[3:4], pool), children_forward(m, x)[3:4]) <= 1e-5


def test_bn_layers_include_the_stem_bn2_with_double_conv_first():
    names = [n for n, _ in engine.resnet_bn_layers(D.resnet18(double_conv_first=True))]
    assert names[:2] == ["bn1", "bn2"]
    assert "bn2" not in [n for n, _ in engine.resnet_bn_layers(D.resnet18())]


def test_bn_mode_with_double_conv_first():
    m = D.resnet18(double_conv_first=True).train()
    assert engine.bn_mode(m) == "train"
    m.bn2.eval()
    with pytest.raises(NotImplementedError, match=r"in eval\(\): bn2$"):
        engine.bn_mode(m)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm1d):
            mod.eval()
    assert engine.bn_mode(m) == "frozen"   # the plan then refuses it (test_double_conv_first_gpu.py)
    assert engine.bn_mode(m.eval()) == "eval"
    # the default stem never calls bn2: its state does not count
    d = D.resnet18().train()
    d.bn2.eval()
    assert engine.bn_mode(d) == "train"

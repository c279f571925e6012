"""CPU: Bottleneck ResNets (resnet50 / resnet101 / resnet152) -- module surface, oracle and plan rules.

  * the modules' state_dict keys, shapes and order against a torch restatement of the block (resnet.py:43-78,
    torchvision's layout), n_out_filters and the head it sizes, the init distribution, the registries, pickling
  * the Bottleneck oracle (tests/bottleneck_oracle.py) against a forward through the module's own nn.Conv1d /
    nn.BatchNorm1d children in float64, running statistics included, for both stems
  * eval_forward: the running-statistics restatement the GPU tests compare eval() plans with, checked the same way
  * bn_mode names the bn3 layers
"""
import pickle
import types

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import deepards_b200 as D
from deepards_b200 import engine
from oracle import cnn_linear_oracle as O
from tests import bottleneck_oracle as BO
from tests.helpers import rel_err

LAYERS = {"resnet50": (3, 4, 6, 3), "resnet101": (3, 4, 23, 3), "resnet152": (3, 8, 36, 3)}
FACTORIES = {"resnet50": D.resnet50, "resnet101": D.resnet101, "resnet152": D.resnet152}


# ---------------------------------------------------------------------------------------------------------------------
# a torch restatement of the reference's Bottleneck ResNet, for the key layout only
# ---------------------------------------------------------------------------------------------------------------------
class _RefBottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes, planes, stride, downsample):
        super().__init__()
        self.conv1 = nn.Conv1d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm1d(planes)
        self.conv2 = nn.Conv1d(planes, planes, 3, stride=stride, padding=1, bias=False)
        self.bn2 = nn.BatchNorm1d(planes)
        self.conv3 = nn.Conv1d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm1d(planes * 4)
        self.downsample = downsample


class _RefResNet(nn.Module):
    def __init__(self, layers, p=64):
        super().__init__()
        self.conv1 = nn.Conv1d(1, p, 7, stride=2, padding=3, bias=False)
        self.conv1_alt = nn.Conv1d(1, p, 3, stride=1, padding=1, bias=False)
        self.bn1 = nn.BatchNorm1d(p)
        self.conv2 = nn.Conv1d(p, p, 7, stride=2, padding=3, bias=False)
        self.bn2 = nn.BatchNorm1d(p)
        self.inplanes = p
        for i, (n, s) in enumerate(zip(layers, (1, 2, 2, 2))):
            setattr(self, "layer%d" % (i + 1), self._stage(p * 2 ** i, n, s))

    def _stage(self, planes, n, stride):
        ds = None
        if stride != 1 or self.inplanes != planes * 4:
            ds = nn.Sequential(nn.Conv1d(self.inplanes, planes * 4, 1, stride=stride, bias=False), nn.BatchNorm1d(planes * 4))
        blocks = [_RefBottleneck(self.inplanes, planes, stride, ds)]
        self.inplanes = planes * 4
        blocks += [_RefBottleneck(self.inplanes, planes, 1, None) for _ in range(1, n)]
        return nn.Sequential(*blocks)


@pytest.mark.parametrize("name", sorted(LAYERS))
def test_state_dict_layout_matches_restatement(name):
    m = FACTORIES[name]()
    ref = _RefResNet(LAYERS[name])
    got = [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
    want = [(k, tuple(v.shape)) for k, v in ref.state_dict().items()]
    assert got == want
    assert m.network_name == name
    assert m.expansion == 4
    assert isinstance(m.layer1[0], D.Bottleneck)
    # layer1's first block has a stride-1 downsample (64 -> 256 at L = 56); the other stages' first blocks stride 2
    assert m.layer1[0].downsample[0].stride == (1,) and m.layer1[0].downsample[0].out_channels == 256
    for li in (2, 3, 4):
        blk = getattr(m, "layer%d" % li)[0]
        assert blk.conv2.stride == (2,) and blk.downsample[0].stride == (2,) and blk.conv1.stride == (1,)
    with pytest.raises(RuntimeError, match="parameters only"):
        m.layer1[0](torch.zeros(1, 64, 56))


def test_n_out_filters_and_heads():
    assert D.resnet50().n_out_filters == 2048
    assert D.resnet50(initial_planes=16).n_out_filters == 512
    assert D.resnet152(initial_planes=16).n_out_filters == 512
    assert D.resnet18().n_out_filters == 512 and D.resnet34(initial_planes=16).n_out_filters == 128
    net = D.CNNLinearNetwork(D.resnet50(), 20, 0)
    assert (net.linear_final.in_features, net.linear_final.out_features) == (40960, 2)
    assert D.CNNSingleBreathLinearNetwork(D.resnet101()).linear_final.in_features == 2048
    sd = BO.cnn_linear_state("resnet50", seed=1, initial_planes=16)
    assert sd["linear_final.weight"].shape == (2, 512 * 20)
    net16 = D.CNNLinearNetwork(D.resnet50(initial_planes=16), 20, 0)
    assert [(k, tuple(v.shape)) for k, v in net16.state_dict().items()] == [(k, tuple(v.shape)) for k, v in sd.items()]


def test_init_distribution():
    torch.manual_seed(0)
    m = D.resnet50()
    for name, conv in (("layer4.0.conv2", m.layer4[0].conv2), ("layer3.2.conv3", m.layer3[2].conv3),
                       ("layer2.0.downsample.0", m.layer2[0].downsample[0]), ("layer4.1.conv1", m.layer4[1].conv1)):
        w = conv.weight.detach()
        std = (2.0 / (conv.kernel_size[0] * conv.out_channels)) ** 0.5   # He-normal, fan = k * Cout (resnet.py:115-118)
        assert abs(float(w.std()) / std - 1) < 0.02, name
        assert abs(float(w.mean())) < 0.02 * std, name
    for mod in m.modules():
        if isinstance(mod, nn.BatchNorm1d):
            assert torch.all(mod.weight == 1) and torch.all(mod.bias == 0)


def test_registry_install_and_exports():
    for name in LAYERS:
        assert D.base_networks[name] is FACTORIES[name]
        assert name in D.__all__
    assert "Bottleneck" in D.__all__
    tad = types.SimpleNamespace(base_networks={"resnet50": None})
    D.install(tad)
    assert tad.base_networks["resnet50"] is D.resnet50 and tad.base_networks["resnet152"] is D.resnet152


def test_pickling_drops_plans():
    net = D.CNNLinearNetwork(D.resnet50(initial_planes=16), 20, 0)
    net.__dict__["_dards_plans"] = {"x": object()}
    net.breath_block.__dict__["_dards_plans"] = {"y": object()}
    back = pickle.loads(pickle.dumps(net))
    assert "_dards_plans" not in back.__dict__ and "_dards_plans" not in back.breath_block.__dict__
    for (k, v), (k2, v2) in zip(net.state_dict().items(), back.state_dict().items()):
        assert k == k2 and torch.equal(v, v2)


def test_oracle_state_matches_module_layout():
    for name, f in FACTORIES.items():
        sd = BO.resnet_state(seed=3, layers=LAYERS[name], initial_planes=16)
        m = f(initial_planes=16)
        assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == [(k, tuple(v.shape)) for k, v in sd.items()]


# ---------------------------------------------------------------------------------------------------------------------
# the oracle against the module's own children, float64
# ---------------------------------------------------------------------------------------------------------------------
def children_forward(m, x):
    """ResNet forward (resnet.py:141-163) through the module's nn.Conv1d / nn.BatchNorm1d children."""
    if m.double_conv_first:
        y = F.relu(m.bn2(m.conv2(m.bn1(m.conv1_alt(x)))))
    else:
        y = F.relu(m.bn1(m.conv1(x)))
    y = F.max_pool1d(y, 3, 2, 1) if m.first_pool_type == "max" else F.avg_pool1d(y, 3, 2, 1)
    for layer in (m.layer1, m.layer2, m.layer3, m.layer4):
        for blk in layer:
            out = F.relu(blk.bn1(blk.conv1(y)))
            out = F.relu(blk.bn2(blk.conv2(out)))
            out = blk.bn3(blk.conv3(out))
            y = F.relu(out + (blk.downsample(y) if blk.downsample is not None else y))
    return F.avg_pool1d(y, 7, 1).flatten(1)


def _perturbed_module(factory, planes, seed, **kw):
    m = factory(initial_planes=planes, **kw)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, nn.BatchNorm1d):
                mod.weight.add_(0.1 * torch.randn(mod.weight.shape, generator=g))
                mod.bias.add_(0.1 * torch.randn(mod.bias.shape, generator=g))
                mod.running_mean.copy_(0.1 * torch.randn(mod.running_mean.shape, generator=g))
                mod.running_var.copy_(1 + 0.2 * torch.rand(mod.running_var.shape, generator=g))
    return m.double()


@pytest.mark.parametrize("double_conv_first,pool", [(False, "max"), (True, "avg")])
def test_oracle_bottleneck_matches_module_children(double_conv_first, pool):
    m = _perturbed_module(D.resnet50, 16, 5, double_conv_first=double_conv_first, first_pool_type=pool).train()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    x = O.synthetic_breaths(1, seed=6)[0].double()
    ref = children_forward(m, x)
    got = BO.resnet_forward(sd, x, first_pool_type=pool, double_conv_first=double_conv_first, running_update=True)
    assert got.shape == (20, 512)
    assert rel_err(got, ref.detach()) <= 1e-12
    for k, v in m.state_dict().items():
        if "running" in k or "num_batches" in k:
            assert rel_err(sd[k], v) <= 1e-12 if v.is_floating_point() else torch.equal(sd[k], v), k
    # decision sites of a Bottleneck: relu1 / relu2 / relu3 per block
    rec = {}
    BO.resnet_forward({k: v.clone() for k, v in m.state_dict().items()}, x, first_pool_type=pool,
                      double_conv_first=double_conv_first, hooks=O.DecisionHooks(record=rec))
    assert {"layer1.0.relu3", "layer4.2.relu1", "layer4.2.relu2", "layer4.2.relu3"} <= set(rec)


# ---------------------------------------------------------------------------------------------------------------------
# eval(): the running-statistics restatement (every BatchNorm F.batch_norm(training=False))
# ---------------------------------------------------------------------------------------------------------------------
def _bn(sd, name, t):
    return F.batch_norm(t, sd[name + ".running_mean"], sd[name + ".running_var"], sd[name + ".weight"], sd[name + ".bias"],
                        False, 0.0, O.BN_EPS)


def eval_forward(sd, x, prefix="", first_pool_type="max", double_conv_first=False):
    """(N, 1, 224) -> (N, 32 * initial_planes): a Bottleneck ResNet in eval()."""
    g = lambda k: sd[prefix + k]
    bn = lambda name, t: _bn(sd, prefix + name, t)
    if double_conv_first:
        y = bn("bn1", F.conv1d(x, g("conv1_alt.weight"), padding=1))
        y = F.relu(bn("bn2", F.conv1d(y, g("conv2.weight"), stride=2, padding=3)))
    else:
        y = F.relu(bn("bn1", F.conv1d(x, g("conv1.weight"), stride=2, padding=3)))
    y = F.max_pool1d(y, 3, 2, 1) if first_pool_type == "max" else F.avg_pool1d(y, 3, 2, 1)
    li = 1
    while (prefix + "layer%d.0.conv1.weight" % li) in sd:
        bi = 0
        while (prefix + "layer%d.%d.conv1.weight" % (li, bi)) in sd:
            pre = "layer%d.%d." % (li, bi)
            stride = 2 if (li > 1 and bi == 0) else 1
            out = F.relu(bn(pre + "bn1", F.conv1d(y, g(pre + "conv1.weight"))))
            out = F.relu(bn(pre + "bn2", F.conv1d(out, g(pre + "conv2.weight"), stride=stride, padding=1)))
            out = bn(pre + "bn3", F.conv1d(out, g(pre + "conv3.weight")))
            if (prefix + pre + "downsample.0.weight") in sd:
                res = bn(pre + "downsample.1", F.conv1d(y, g(pre + "downsample.0.weight"), stride=stride))
            else:
                res = y
            y = F.relu(out + res)
            bi += 1
        li += 1
    return F.avg_pool1d(y, 7, 1).flatten(1)


def eval_cnn_linear_forward(sd, x, **kw):
    """(B, 20, 1, 224) -> (B, 2): CNNLinearNetwork in eval()."""
    w, b = sd["linear_final.weight"], sd["linear_final.bias"]
    return torch.cat([F.linear(eval_forward(sd, x[i], "breath_block.", **kw).reshape(-1), w, b).unsqueeze(0)
                      for i in range(x.shape[0])], 0)


@pytest.mark.parametrize("double_conv_first", [False, True])
def test_eval_restatement_matches_module_children(double_conv_first):
    m = _perturbed_module(D.resnet50, 16, 7, double_conv_first=double_conv_first).eval()
    x = O.synthetic_breaths(1, seed=8)[0].double()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    with torch.no_grad():
        assert rel_err(eval_forward(sd, x, double_conv_first=double_conv_first), children_forward(m, x)) <= 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# plan rules
# ---------------------------------------------------------------------------------------------------------------------
def test_bn_layers_and_mode_name_bn3():
    m = D.resnet50(initial_planes=16)
    names = [n for n, _ in engine.resnet_bn_layers(m)]
    assert len(names) == 53 and names.count("bn1") == 1
    assert names[:5] == ["bn1", "layer1.0.bn1", "layer1.0.bn2", "layer1.0.bn3", "layer1.0.downsample.1"]
    assert len(engine.resnet_bn_layers(D.resnet50(double_conv_first=True))) == 54
    assert len(engine.resnet_bn_layers(D.resnet101())) == 104 and len(engine.resnet_bn_layers(D.resnet152())) == 155
    # BasicBlock lists are unchanged
    assert len(engine.resnet_bn_layers(D.resnet18())) == 20
    m.train()
    assert engine.bn_mode(m) == "train"
    m.layer3[5].bn3.eval()
    with pytest.raises(NotImplementedError, match=r"in eval\(\): layer3\.5\.bn3$"):
        engine.bn_mode(m)
    for mod in m.modules():
        if isinstance(mod, nn.BatchNorm1d):
            mod.eval()
    assert engine.bn_mode(m) == "frozen"
    m.layer1[0].bn3.train()
    with pytest.raises(NotImplementedError, match=r"in train\(\): layer1\.0\.bn3; in eval\(\): bn1, "):
        engine.bn_mode(m)
    m.eval()
    assert engine.bn_mode(m) == "eval"


def test_other_block_types_still_raise():
    class Odd(D.BasicBlock):
        pass

    with pytest.raises(NotImplementedError, match="BasicBlock and Bottleneck"):
        D.ResNet(Odd, [1, 1, 1, 1])

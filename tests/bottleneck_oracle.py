"""CPU oracle of the Bottleneck ResNets (resnet50 / resnet101 / resnet152), for the Bottleneck tests.

The same restatement as oracle/cnn_linear_oracle.py (torch.nn.functional calls in the reference's order on an explicit
state_dict), for the reference's Bottleneck block (deepards/models/resnet.py:43-78, the convolutions at :48-53,
torchvision's layout): conv1 1x1 inplanes -> planes, bn1, ReLU, conv2 k3 with the block's stride and padding 1, bn2,
ReLU, conv3 1x1 planes -> 4 * planes, bn3, plus the identity or the downsample (1x1 with the block's stride, BatchNorm),
ReLU.  Stem, pooling, BatchNorm, ReLU sites and the head are the oracle's own (its _batchnorm, _act, DecisionHooks), so
tests/test_frozen_bn_cpu.frozen_oracle() and decision pinning act on this forward too.  ReLU sites of a block:
"layerI.J.relu1", "relu2", "relu3".
"""
from collections import OrderedDict

import torch
import torch.nn.functional as F

from oracle import cnn_linear_oracle as O

LAYERS = {"resnet50": (3, 4, 6, 3), "resnet101": (3, 4, 23, 3), "resnet152": (3, 8, 36, 3)}   # resnet.py:188-222


def resnet_state(seed=0, layers=(3, 4, 6, 3), initial_planes=64, bn_perturb=0.0, prefix=""):
    """state_dict of the reference's Bottleneck ResNet (resnet.py:83-139, 43-78), stem parameters included, drawn with the
    reference's init distribution; keys in the module's order."""
    gen = torch.Generator().manual_seed(seed)
    sd = OrderedDict()
    p = initial_planes
    sd["conv1.weight"] = O._conv_w(gen, p, 1, 7)
    sd["conv1_alt.weight"] = O._conv_w(gen, p, 1, 3)
    O._bn(sd, "bn1", p, True, gen, bn_perturb)
    sd["conv2.weight"] = O._conv_w(gen, p, p, 7)
    O._bn(sd, "bn2", p, True, gen, bn_perturb)
    inpl = p
    for li, nb in enumerate(layers, 1):
        planes = p * 2 ** (li - 1)
        for bi in range(nb):
            stride = 2 if (li > 1 and bi == 0) else 1
            pre = "layer%d.%d." % (li, bi)
            sd[pre + "conv1.weight"] = O._conv_w(gen, planes, inpl, 1)
            O._bn(sd, pre + "bn1", planes, True, gen, bn_perturb)
            sd[pre + "conv2.weight"] = O._conv_w(gen, planes, planes, 3)
            O._bn(sd, pre + "bn2", planes, True, gen, bn_perturb)
            sd[pre + "conv3.weight"] = O._conv_w(gen, 4 * planes, planes, 1)
            O._bn(sd, pre + "bn3", 4 * planes, True, gen, bn_perturb)
            if stride != 1 or inpl != 4 * planes:
                sd[pre + "downsample.0.weight"] = O._conv_w(gen, 4 * planes, inpl, 1)
                O._bn(sd, pre + "downsample.1", 4 * planes, True, gen, bn_perturb)
            inpl = 4 * planes
    if prefix:
        sd = OrderedDict((prefix + k, v) for k, v in sd.items())
    return sd


def cnn_linear_state(backbone="resnet50", seed=0, sub_batch=20, bn_perturb=0.0, initial_planes=64):
    """state_dict of CNNLinearNetwork(backbone(initial_planes=...), sub_batch, 0): Linear(32 * planes * sub_batch, 2)."""
    sd = resnet_state(seed, LAYERS[backbone], initial_planes, bn_perturb, prefix="breath_block.")
    gen = torch.Generator().manual_seed(seed + 7919)
    O._linear(sd, "linear_final", 32 * initial_planes * sub_batch, 2, gen)
    return sd


def resnet_forward(sd, x, prefix="", first_pool_type="max", double_conv_first=False, running_update=False, hooks=None):
    """(N, 1, 224) -> (N, 32 * initial_planes); BatchNorm statistics over the whole N (resnet.py:141-163)."""
    g = lambda k: sd[prefix + k]
    view = O._Prefixed(sd, prefix)
    bn = lambda t, name: O._batchnorm(t, view, name, running_update)   # looked up per call: frozen_oracle() patches it
    if not double_conv_first:
        y = bn(F.conv1d(x, g("conv1.weight"), stride=2, padding=3), "bn1")
    else:
        y = bn(F.conv1d(x, g("conv1_alt.weight"), stride=1, padding=1), "bn1")
        y = bn(F.conv1d(y, g("conv2.weight"), stride=2, padding=3), "bn2")
    y = O._act(y, "relu0", hooks)
    y = F.max_pool1d(y, 3, 2, 1) if first_pool_type == "max" else F.avg_pool1d(y, 3, 2, 1)
    li = 1
    while (prefix + "layer%d.0.conv1.weight" % li) in sd:
        bi = 0
        while (prefix + "layer%d.%d.conv1.weight" % (li, bi)) in sd:
            pre = "layer%d.%d." % (li, bi)
            stride = 2 if (li > 1 and bi == 0) else 1
            out = O._act(bn(F.conv1d(y, g(pre + "conv1.weight")), pre + "bn1"), pre + "relu1", hooks)
            out = F.conv1d(out, g(pre + "conv2.weight"), stride=stride, padding=1)
            out = O._act(bn(out, pre + "bn2"), pre + "relu2", hooks)
            out = bn(F.conv1d(out, g(pre + "conv3.weight")), pre + "bn3")
            if (prefix + pre + "downsample.0.weight") in sd:
                res = bn(F.conv1d(y, g(pre + "downsample.0.weight"), stride=stride), pre + "downsample.1")
            else:
                res = y
            y = O._act(out + res, pre + "relu3", hooks)
            bi += 1
        li += 1
    y = F.avg_pool1d(y, 7, 1)
    return y.reshape(y.shape[0], -1)


def cnn_linear_forward(sd, x, **kw):
    """The reference's per-sequence loop (torch_cnn_linear_network.py:104-113): (B, 20, 1, 224) -> (B, 2)."""
    w, b = sd["linear_final.weight"], sd["linear_final.bias"]
    rows = []
    for i in range(x.shape[0]):
        if kw.get("hooks") is not None:
            kw["hooks"].seq = i
        feat = resnet_forward(sd, x[i], "breath_block.", **kw)
        rows.append(F.linear(feat.reshape(-1), w, b).unsqueeze(0))
    return torch.cat(rows, 0)


def forward_backward(sd, x, target, **kw):
    """One training step's forward + backward (O.forward_backward for this forward): (logits, loss, {name: grad}) on leaf
    copies of the floating-point parameters; parameters the forward does not use get no entry."""
    leaves = OrderedDict()
    for k, v in sd.items():
        if v.is_floating_point() and not k.endswith(("running_mean", "running_var")):
            leaves[k] = v.detach().clone().requires_grad_(True)
        else:
            leaves[k] = v
    out = cnn_linear_forward(leaves, x, **kw)
    loss = O.bce_with_logits(out, target)
    names = [k for k, v in leaves.items() if v.requires_grad]
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    return out.detach(), loss.detach(), OrderedDict((k, g) for k, g in zip(names, grads) if g is not None)

"""1-D ResNet backbones on the B200 backend -- drop-in for deepards/models/resnet.py.

Same factory names (resnet18/34 with BasicBlock, resnet50/101/152 with Bottleneck, resnet.py:166-222) and keyword
arguments (`resnet18(pretrained=False, initial_planes=64, first_pool_type='max', double_conv_first=False)`,
resnet.py:83,166-174), same attributes (`n_out_filters`, `network_name`,
`inplanes`, `expansion`) and the same `state_dict` keys -- including the stem's `conv1_alt`,
`conv2`, `bn2` (resnet.py:90-96), unused by the default stem -- so checkpoints move between the two implementations unchanged.

`double_conv_first=True` selects the two-convolution stem (resnet.py:145-150): conv1_alt -> bn1 -> conv2 -> bn2 -> ReLU ->
first pool, with `conv1` unused (its `.grad` stays None).  It runs in train() and eval(); train() with the BatchNorm layers
in eval() (frozen BatchNorm) raises NotImplementedError for it.

The `nn.Conv1d` / `nn.BatchNorm1d` children are parameter CONTAINERS only: `forward` does not call them, it
runs the recorded kernel plan (engine.Plan) through autograd.  BatchNorm statistics are taken over the whole
first dimension of the input, exactly like calling the reference module on that tensor; the cnn_linear heads
call the plan with group = 20 breaths instead (torch_cnn_linear_network.py:104-113).
"""
import math

import torch.nn as nn

from . import autograd as _ag


class _Picklable(object):
    """torch.save(model) pickles the module __dict__ (train_ards_detector.py:364,374): drop the plan cache."""

    def __getstate__(self):
        st = dict(self.__dict__)
        st.pop("_dards_plans", None)
        return st


def _conv3(cin, cout, stride=1):
    return nn.Conv1d(cin, cout, kernel_size=3, stride=stride, padding=1, bias=False)


class BasicBlock(_Picklable, nn.Module):
    """conv3-bn-relu-conv3-bn (+ downsampled identity) -relu; parameter container (resnet.py:11-40)."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super(BasicBlock, self).__init__()
        self.conv1 = _conv3(inplanes, planes, stride)
        self.bn1 = nn.BatchNorm1d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = _conv3(planes, planes)
        self.bn2 = nn.BatchNorm1d(planes)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        raise RuntimeError("deepards_b200.BasicBlock holds parameters only; call the enclosing ResNet")


class Bottleneck(_Picklable, nn.Module):
    """conv1x1-bn-relu-conv3(stride)-bn-relu-conv1x1(x4)-bn (+ downsampled identity) -relu; parameter container
    (resnet.py:43-78, the Bottleneck convolutions at :48-53, torchvision's layout): conv1 is 1x1 inplanes -> planes,
    conv2 is k3 / stride / padding 1 planes -> planes, conv3 is 1x1 planes -> 4 * planes; no bias anywhere."""
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super(Bottleneck, self).__init__()
        self.conv1 = nn.Conv1d(inplanes, planes, kernel_size=1, bias=False)
        self.bn1 = nn.BatchNorm1d(planes)
        self.conv2 = _conv3(planes, planes, stride)
        self.bn2 = nn.BatchNorm1d(planes)
        self.conv3 = nn.Conv1d(planes, planes * self.expansion, kernel_size=1, bias=False)
        self.bn3 = nn.BatchNorm1d(planes * self.expansion)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride

    def forward(self, x):
        raise RuntimeError("deepards_b200.Bottleneck holds parameters only; call the enclosing ResNet")


class ResNet(_Picklable, nn.Module):
    def __init__(self, block, layers, initial_planes=64, first_pool_type='max', double_conv_first=False):
        super(ResNet, self).__init__()
        if block not in (BasicBlock, Bottleneck):
            raise NotImplementedError("only BasicBlock and Bottleneck ResNets run on the B200 backend")
        if first_pool_type not in ('max', 'avg'):
            raise ValueError("first_pool_type must be 'max' or 'avg'")
        self.inplanes = initial_planes
        self.expansion = block.expansion
        self.first_pool_type = first_pool_type
        self.double_conv_first = double_conv_first
        p = initial_planes
        self.conv1 = nn.Conv1d(1, p, kernel_size=7, stride=2, padding=3, bias=False)
        self.conv1_alt = nn.Conv1d(1, p, kernel_size=3, stride=1, padding=1, bias=False)
        self.bn1 = nn.BatchNorm1d(p)
        self.conv2 = nn.Conv1d(p, p, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn2 = nn.BatchNorm1d(p)
        self.relu = nn.ReLU(inplace=True)
        pool_cls = nn.MaxPool1d if first_pool_type == 'max' else nn.AvgPool1d
        self.first_pool = pool_cls(kernel_size=3, stride=2, padding=1)
        self.layer1 = self._stage(block, p, layers[0], 1)
        self.layer2 = self._stage(block, p * 2, layers[1], 2)
        self.layer3 = self._stage(block, p * 4, layers[2], 2)
        self.layer4 = self._stage(block, p * 8, layers[3], 2)
        self.avgpool = nn.AvgPool1d(7, stride=1)
        for m in self.modules():
            if isinstance(m, nn.Conv1d):
                # He-normal, fan = kernel * out_channels (resnet.py:115-118)
                m.weight.data.normal_(0, math.sqrt(2.0 / (m.kernel_size[0] * m.out_channels)))
            elif isinstance(m, nn.BatchNorm1d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
        # the features the backbone returns: the last stage's output channels, 8 * initial_planes * expansion.  The
        # reference computes `self.inplanes * block.expansion` here, which is the same for BasicBlock (expansion 1) but
        # 4x too large for Bottleneck, where self.inplanes already includes the expansion.
        self.n_out_filters = self.inplanes
        self.network_name = 'resnet'
        self.precision = None  # None -> DEEPARDS_B200_PRECISION or 'bf16' (tcgen05 path); 'fp32' = the 1e-4 parity path

    def _stage(self, block, planes, n_blocks, stride):
        ds = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            ds = nn.Sequential(nn.Conv1d(self.inplanes, planes * block.expansion, kernel_size=1, stride=stride, bias=False),
                               nn.BatchNorm1d(planes * block.expansion))
        blocks = [block(self.inplanes, planes, stride, ds)]
        self.inplanes = planes * block.expansion
        blocks += [block(self.inplanes, planes) for _ in range(1, n_blocks)]
        return nn.Sequential(*blocks)

    def forward(self, x):
        """x: (N, 1, 224) -> (N, n_out_filters); in train() BatchNorm over all N breaths (resnet.py:141-163), in eval() with
        the running statistics (every breath on its own)."""
        if x.dim() != 3 or x.shape[1] != 1 or x.shape[2] != 224:
            raise RuntimeError("deepards_b200 ResNet expects (N, 1, 224), got %s" % (tuple(x.shape),))
        return _ag.run_plan(self, self, None, x, x.shape[0], "backbone")


def resnet18(pretrained=False, **kwargs):
    """1-D ResNet-18 (resnet.py:166-174).  `pretrained` is accepted and ignored, like the reference."""
    model = ResNet(BasicBlock, [2, 2, 2, 2], **kwargs)
    model.network_name = 'resnet18'
    return model


def resnet34(pretrained=False, **kwargs):
    """1-D ResNet-34 (resnet.py:178-186)."""
    model = ResNet(BasicBlock, [3, 4, 6, 3], **kwargs)
    model.network_name = 'resnet34'
    return model


def resnet50(pretrained=False, **kwargs):
    """1-D ResNet-50 (resnet.py:188-198): Bottleneck, [3, 4, 6, 3]."""
    model = ResNet(Bottleneck, [3, 4, 6, 3], **kwargs)
    model.network_name = 'resnet50'
    return model


def resnet101(pretrained=False, **kwargs):
    """1-D ResNet-101 (resnet.py:200-210): Bottleneck, [3, 4, 23, 3]."""
    model = ResNet(Bottleneck, [3, 4, 23, 3], **kwargs)
    model.network_name = 'resnet101'
    return model


def resnet152(pretrained=False, **kwargs):
    """1-D ResNet-152 (resnet.py:212-222): Bottleneck, [3, 8, 36, 3]."""
    model = ResNet(Bottleneck, [3, 8, 36, 3], **kwargs)
    model.network_name = 'resnet152'
    return model

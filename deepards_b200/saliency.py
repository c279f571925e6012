"""Input-gradient attributions: the gradient of a network output with respect to the breath waveform, at full resolution.

`input_gradients(net, x, target)` returns d sum(output[..., target]) / dx for any head of this package over any backbone,
224 values per breath.  Saliency maps, SmoothGrad and integrated gradients are all built from it (INTEGRATION.md shows the
compositions).  GradCAM (gradcam.py) gives 7 values per breath and needs a DenseNet; this works for every backbone.

How it runs, for every head: the head's "backbone" plan, built with input_grad=True, runs forward; `net._head` runs on
the pooled features under autograd; the one-hot seed is back-propagated into plan.dfeat; the plan's backward runs down to
the stem, whose input-gradient kernel writes plan.dx.  This is the trainer's generic step (DataParallelTrainer._head_step)
with the same plan choice (data_parallel.head_backbone_plan).

BatchNorm and dropout follow the network's own state, as for GradCAM: batch statistics in train(), the frozen plan for
frozen BatchNorm, and for a ResNet in eval() also the frozen plan (the same running-statistics arithmetic as the eval plan,
with a backward).  No running statistic, num_batches_tracked or parameter .grad changes; the module path's plans are not
touched.  `net(x)` with x.requires_grad still raises: this is an explicit explainer call, not autograd.
"""
import torch

from . import engine
from .data_parallel import head_backbone_plan


def _bn_rule(bb):
    bn = engine.bn_mode(bb)
    if bn == "eval":
        if bb.double_conv_first:
            raise NotImplementedError("deepards_b200: input gradients of a ResNet in eval() run the frozen-BatchNorm "
                                      "plan, which does not exist for double_conv_first=True; call train() on it for "
                                      "batch statistics")
        return "frozen"
    return bn


def _seed(out, target):
    """One-hot (out's shape) of the target class at every output position."""
    n_out = out.shape[-1]
    if target is None:
        idx = out.detach().argmax(dim=-1)
    elif isinstance(target, int) or (torch.is_tensor(target) and target.dim() == 0 and not target.is_floating_point()):
        t = int(target)
        if not 0 <= t < n_out:
            raise ValueError("target %d is not an output index (the output has %d)" % (t, n_out))
        idx = torch.full(out.shape[:-1], t, dtype=torch.long, device=out.device)
    else:
        idx = torch.as_tensor(target)
        if idx.is_floating_point() or idx.dtype == torch.bool:
            raise TypeError("target must be None, an int or an integer tensor, got %s" % (idx.dtype,))
        if tuple(idx.shape) != tuple(out.shape[:-1]):
            raise ValueError("target must be shaped like the output without its last dimension %s, got %s"
                             % (tuple(out.shape[:-1]), tuple(idx.shape)))
        idx = idx.to(device=out.device, dtype=torch.long)
        if bool(((idx < 0) | (idx >= n_out)).any()):
            raise ValueError("target holds indices outside [0, %d)" % n_out)
    return torch.zeros_like(out).scatter_(-1, idx.unsqueeze(-1), 1.0)


def input_gradients(net, x, target=None):
    """net: a head of registry.network_heads; x: what its forward takes ((B, S, 1, 224), CNNRegressor (N, 1, 224)) on the
    network's device.  target: None (the argmax of the output), an int, or an integer tensor shaped like the output without
    its last dimension.  Returns (grad, outputs): grad = d sum(output[..., target]) / dx, fp32 in x's shape, and what
    forward returns (for CNNLSTMNetwork the per-step outputs)."""
    from .torch_cnn_linear_network import CNNRegressor, _HeadBase
    if not isinstance(net, _HeadBase) or not hasattr(net, "_head"):
        raise TypeError("input_gradients explains the heads of deepards_b200 (registry.network_heads), not %s"
                        % type(net).__name__)
    if not torch.is_tensor(x):
        raise TypeError("x must be a tensor")
    if x.shape[-1] != engine.SEQ_LEN:
        raise Exception('input breaths must have sequence length of 224')
    flat = isinstance(net, CNNRegressor)
    if flat and (x.dim() != 3 or x.shape[1] != 1):
        raise NotImplementedError("CNNRegressor takes (N, 1, 224) breaths, got %s" % (tuple(x.shape),))
    if not flat:
        net._check(x)
    plan = head_backbone_plan(net, x, _bn_rule, False, input_grad=True)
    if x.device != plan.device:
        raise RuntimeError("input is on %s but the network is on %s" % (x.device, plan.device))
    with torch.no_grad():
        plan.load_input(x.detach() if x.dtype == torch.float32 else x.detach().float())
        plan.run_forward()
    feat = plan.feat.detach()
    if not flat:
        feat = feat.view(plan.G, plan.group, -1)
    feat.requires_grad_(True)
    with torch.enable_grad():
        out = net._head(feat)
        if isinstance(out, tuple):      # CNNLSTMNetwork: (per-step outputs, (hx, cx))
            out = out[0]
        seed = _seed(out, target)
        (dfeat,) = torch.autograd.grad(out, [feat], grad_outputs=seed)
    plan.dfeat.copy_(dfeat.reshape(plan.dfeat.shape))
    plan.run_backward()
    return plan.dx.view(x.shape).clone(), out.detach()

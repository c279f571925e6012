"""torch.autograd bridge: one Function per network call.

Gradients must arrive through autograd so that tensor hooks fire (the reference clamps gradients with
`p.register_hook`, train_ards_detector.py:474-476) and `.grad` is populated for `optimizer.step()`.  The
Function runs a whole recorded `Plan` in forward and the matching recorded backward, and hands autograd one
gradient per parameter (views of a fresh copy of the plan's flat gradient buffer).
"""
import torch

from . import engine


def module_precision(mod):
    return getattr(mod, "precision", None) or engine.default_precision()


class PlanFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, plan, x, *params):
        if x.requires_grad:
            raise NotImplementedError("deepards_b200: gradients w.r.t. the input waveform are not implemented "
                                      "(the reference never asks for them: the first conv skips dgrad)")
        if x.device != plan.device:
            raise RuntimeError("input is on %s but the network is on %s" % (x.device, plan.device))
        plan.load_input(x if x.dtype == torch.float32 else x.float())
        plan.run_forward()
        ctx.plan = plan
        ctx.serial = plan.fwd_serial
        ctx.n_params = len(params)
        if plan.mode == "features":
            # (N, L, F) channels-last -> the reference's (N, F, L) fp32
            out = plan.feat_map.permute(0, 2, 1).float().contiguous()
        elif plan.mode == "backbone":
            out = plan.feat.clone()
        elif plan.mode == "cnn_linear":
            out = plan.logits.clone()
        else:  # per_breath: (N, 2) -> (B, group, 2)
            out = plan.logits.view(plan.G, plan.group, -1).clone()
        if not any(ctx.needs_input_grad):
            plan.mark_no_backward()
        return out

    @staticmethod
    def backward(ctx, dout):
        plan = ctx.plan
        if plan.bn == "eval":
            raise NotImplementedError("deepards_b200: backward through running-statistics BatchNorm (ResNet in eval() "
                                      "mode) is not implemented; call train() on the network to train it")
        if ctx.serial != plan.fwd_serial:
            raise RuntimeError("deepards_b200: this network was called again before backward(); a plan keeps the "
                               "activations of its latest forward only")
        dout = dout.contiguous()
        if plan.mode == "features":
            plan.dfeat_map.copy_(dout.permute(0, 2, 1))
        elif plan.mode == "backbone":
            # the head lives outside the plan: seed the pooled-feature gradient directly
            plan.dfeat.copy_(dout)
        else:
            plan.dlogits.copy_(dout.reshape(plan.dlogits.shape))
        plan.run_backward()
        g = plan.grads()
        out = [None, None]
        for i, p in enumerate(plan.autograd_params()):
            out.append(g.get(id(p)) if ctx.needs_input_grad[2 + i] else None)
        return tuple(out)


def run_plan(net, backbone, linear, x, group, mode, dropout_key=()):
    """Common entry of every module forward: pick/build the plan, run it through autograd."""
    n = x.numel() // engine.SEQ_LEN
    training = backbone.training
    # A ResNet in eval() normalises with its running statistics: every breath is independent of the rest of the batch, and
    # `group` only shapes the heads.  A ResNet in train() with its BatchNorm layers in eval() does the same and trains
    # (frozen BatchNorm); mixed BatchNorm states raise.  DenseNet keeps no running statistics; its eval() only turns dropout
    # off.  engine.bn_mode states the rule.
    bn = engine.bn_mode(backbone)
    plan = engine.get_plan(net, backbone, linear, n, group, module_precision(net), mode,
                           dropout=dropout_key if training else (), update_running=training, bn=bn)
    # Only the parameters the backward writes are inputs of the autograd node.  ResNet's conv1_alt / conv2 / bn2 (conv1 with
    # double_conv_first=True) never take part in forward() (resnet.py:141-163): in the reference they are not in the graph, their hooks never fire and
    # their .grad stays None -- a None handed to a `p.register_hook(lambda g: g.clamp(...))` hook would raise.
    return PlanFunction.apply(plan, x, *plan.autograd_params())

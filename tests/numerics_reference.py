"""Closed-form references of the BatchNorm and stem arithmetic, written once for any floating dtype.

Called in float64 they are the references of tests/test_numerics_gpu.py; called in float32 on the same device they are
the torch fp32 calibration of the same gates.  Layout is torch's (N, C, L); grouped BatchNorm takes `group` consecutive
samples of the batch as one set of statistics (biased variance, as the training forward uses).
tests/test_numerics_cpu.py checks them against nn.BatchNorm1d / nn.Conv1d / the pooling modules.
"""
import torch
import torch.nn.functional as F

EPS = 1e-5


def group_stats(y, group, eps=EPS):
    """y (N, C, L) -> mean, rstd (G, C): two-pass (centred) statistics of every group."""
    n, c, l = y.shape
    yg = y.reshape(n // group, group, c, l)
    mean = yg.mean(dim=(1, 3))
    var = (yg - mean[:, None, :, None]).square().mean(dim=(1, 3))
    return mean, (var + eps).rsqrt()


def _bcast(t, group):
    """(G, C) -> (N, C, 1) with every group's row repeated over its samples."""
    return t.repeat_interleave(group, dim=0)[:, :, None]


def gbn_forward(x, gamma, beta, group, res=None, relu=False, eps=EPS, stats=None):
    """-> (out, pre-ReLU value, mean, rstd).  `stats` = (mean, rstd) normalises with given statistics."""
    mean, rstd = stats if stats is not None else group_stats(x, group, eps)
    pre = (x - _bcast(mean, group)) * _bcast(rstd, group) * gamma[None, :, None] + beta[None, :, None]
    if res is not None:
        pre = pre + res
    return (pre.clamp_min(0) if relu else pre), pre, mean, rstd


def gbn_backward(dout, x, gamma, mean, rstd, group, mask=None):
    """Training-mode BatchNorm backward with the given statistics: the gradient at the BatchNorm output is dout * mask
    (mask: the ReLU's pass-through, None = no ReLU).  -> (dx, dgamma, dbeta, g) with g the masked gradient (= dres)."""
    n, c, l = x.shape
    g = dout if mask is None else dout * mask
    xhat = (x - _bcast(mean, group)) * _bcast(rstd, group)
    gg, xg = g.reshape(n // group, group, c, l), xhat.reshape(n // group, group, c, l)
    s1 = gg.sum(dim=(1, 3))
    s2 = (gg * xg).sum(dim=(1, 3))
    cnt = group * l
    dx = gamma[None, :, None] * _bcast(rstd, group) * (g - _bcast(s1 / cnt, group) - xhat * _bcast(s2 / cnt, group))
    return dx, s2.sum(0), s1.sum(0), g


def running_update(means, variances, rows, momentum, running_mean, running_var):
    """nn.BatchNorm1d's update, one group after the other: r <- (1 - m) r + m v_g, the variance unbiased."""
    rm, rv = running_mean.clone(), running_var.clone()
    for mg, vg in zip(means, variances):
        rm = (1 - momentum) * rm + momentum * mg
        rv = (1 - momentum) * rv + momentum * vg * (rows / (rows - 1))
    return rm, rv


def eval_coeffs(gamma, beta, running_mean, running_var, eps=EPS):
    """BatchNorm with the running statistics as y * scale + shift."""
    scale = gamma / torch.sqrt(running_var + eps)
    return scale, beta - running_mean * scale


def stem_conv(x, w):
    """x (N, 224), w (C0, 1, 7) -> (N, C0, 112): the stem convolution (k7, s2, p3)."""
    return F.conv1d(x[:, None, :], w, stride=2, padding=3)


def _pool(z, pool):
    return F.max_pool1d(z, 3, 2, 1) if pool == 0 else F.avg_pool1d(z, 3, 2, 1)


def stem_forward(x, w, gamma, beta, group, pool, eps=EPS):
    """conv -> grouped BatchNorm -> ReLU -> pool.  -> (out (N, C0, 56), pre-ReLU value, mean, rstd)."""
    y = stem_conv(x, w)
    _, pre, mean, rstd = gbn_forward(y, gamma, beta, group, eps=eps)
    return _pool(pre.clamp_min(0), pool), pre, mean, rstd


def stem_eval_forward(x, w, scale, shift, pool):
    pre = stem_conv(x, w) * scale[None, :, None] + shift[None, :, None]
    return _pool(pre.clamp_min(0), pool), pre


def _pool_backward(dout, pre, pool):
    """Gradient at the pre-ReLU value of pool(relu(pre))."""
    z = pre.detach().clamp_min(0).requires_grad_(True)
    with torch.enable_grad():
        (g,) = torch.autograd.grad(_pool(z, pool), z, dout)
    return g * (pre > 0)


def stem_backward(dout, x, w, gamma, mean, rstd, group, pool, pre):
    """-> (dW, dgamma, dbeta) of stem_forward with the given statistics; `pre` decides the ReLU and the max-pool."""
    g = _pool_backward(dout, pre, pool)
    dy, dgamma, dbeta, _ = gbn_backward(g, stem_conv(x, w), gamma, mean, rstd, group)
    dw = torch.nn.grad.conv1d_weight(x[:, None, :], w.shape, dy, stride=2, padding=3)
    return dw, dgamma, dbeta


def stem_frozen_backward(dout, x, w, scale, running_mean, rstd, pool, pre):
    """Backward of stem_eval_forward with constant statistics: dy = scale * g.  -> (dW, dgamma, dbeta)."""
    g = _pool_backward(dout, pre, pool)
    xhat = (stem_conv(x, w) - running_mean[None, :, None]) * rstd[None, :, None]
    dw = torch.nn.grad.conv1d_weight(x[:, None, :], w.shape, g * scale[None, :, None], stride=2, padding=3)
    return dw, (g * xhat).sum(dim=(0, 2)), g.sum(dim=(0, 2))

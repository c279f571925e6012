"""CPU: the float64 references of tests/numerics_reference.py against torch's modules in float64.

The GPU numerics tests trust these closed forms as their ground truth, so they are checked here against
nn.BatchNorm1d / nn.Conv1d / the pooling modules and autograd, on the same offset, constant and zero data."""
import pytest
import torch
import torch.nn.functional as F

from tests import numerics_reference as R

D = torch.float64


def _data(n, c, l, offset, gen):
    x = offset + torch.randn(n, c, l, generator=gen, dtype=D)
    x[:, 0] = 0.0                                           # all-zero channel
    x[:, 1] = 3.0                                           # constant channel
    x[:, 2] = 5.0 + 1e-4 * torch.randn(n, l, generator=gen, dtype=D)   # var ~ 1e-8, far below eps
    x[1] = 0.0                                              # a zero breath
    return x


def _module_bn(x, gamma, beta, group):
    """Grouped training-mode BatchNorm: nn.BatchNorm1d's functional form, one call per group (differentiable in gamma and
    beta), and the module itself for the running statistics."""
    bn = torch.nn.BatchNorm1d(x.shape[1], dtype=D)
    with torch.no_grad():
        for i in range(0, x.shape[0], group):
            bn(x[i:i + group])
    y = torch.cat([F.batch_norm(x[i:i + group], None, None, gamma, beta, True, 0.0, R.EPS)
                   for i in range(0, x.shape[0], group)])
    return y, bn


@pytest.mark.parametrize("offset", [0.0, 1e3])
def test_grouped_bn_forward_backward_matches_module(offset):
    gen = torch.Generator().manual_seed(1)
    n, c, l, group = 12, 6, 9, 4
    x = _data(n, c, l, offset, gen).requires_grad_(True)
    gamma = (0.5 + torch.rand(c, generator=gen, dtype=D)).requires_grad_(True)
    beta = torch.randn(c, generator=gen, dtype=D).requires_grad_(True)
    res = torch.randn(n, c, l, generator=gen, dtype=D)
    dout = torch.randn(n, c, l, generator=gen, dtype=D)
    y, bn = _module_bn(x, gamma, beta, group)
    ref = (y + res).relu()
    gx, gg, gb = torch.autograd.grad(ref, [x, gamma, beta], dout)
    out, pre, mean, rstd = R.gbn_forward(x.detach(), gamma.detach(), beta.detach(), group, res=res, relu=True)
    torch.testing.assert_close(out, ref.detach(), rtol=1e-12, atol=1e-11)
    dx, dgamma, dbeta, dres = R.gbn_backward(dout, x.detach(), gamma.detach(), mean, rstd, group, mask=(pre > 0).to(D))
    torch.testing.assert_close(dx, gx, rtol=1e-10, atol=1e-9)
    torch.testing.assert_close(dgamma, gg, rtol=1e-10, atol=1e-9)
    torch.testing.assert_close(dbeta, gb, rtol=1e-12, atol=1e-11)
    torch.testing.assert_close(dres, dout * (ref > 0), rtol=0, atol=0)
    # var = 0 gives rstd = 1/sqrt(eps): channel 0 everywhere, channel 1 in the groups without the zero breath
    assert torch.all(rstd[:, 0] == R.EPS ** -0.5) and torch.all(rstd[1:, 1] == R.EPS ** -0.5)


def test_running_update_matches_module():
    gen = torch.Generator().manual_seed(2)
    n, c, l, group = 12, 5, 7, 3
    x = _data(n, c, l, 100.0, gen)
    _, bn = _module_bn(x, torch.ones(c, dtype=D), torch.zeros(c, dtype=D), group)
    xg = x.view(n // group, group, c, l)
    means = xg.mean(dim=(1, 3))
    variances = xg.var(dim=(1, 3), unbiased=False)
    rm, rv = R.running_update(means, variances, group * l, 0.1, torch.zeros(c, dtype=D), torch.ones(c, dtype=D))
    torch.testing.assert_close(rm, bn.running_mean, rtol=1e-13, atol=1e-14)
    torch.testing.assert_close(rv, bn.running_var, rtol=1e-13, atol=1e-14)


def test_eval_coeffs_match_module_in_eval():
    gen = torch.Generator().manual_seed(3)
    c = 4
    bn = torch.nn.BatchNorm1d(c, dtype=D).eval()
    with torch.no_grad():
        bn.weight.copy_(0.5 + torch.rand(c, generator=gen, dtype=D))
        bn.bias.copy_(torch.randn(c, generator=gen, dtype=D))
        bn.running_mean.copy_(torch.tensor([0.0, 1e3, -1e3, 3.0], dtype=D))
        bn.running_var.copy_(torch.tensor([0.0, 1e-8, 1.0, 1e4], dtype=D))
    y = bn.running_mean[None, :, None] + torch.randn(3, c, 8, generator=gen, dtype=D)
    scale, shift = R.eval_coeffs(bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var)
    torch.testing.assert_close(y * scale[None, :, None] + shift[None, :, None], bn(y).detach(), rtol=1e-10, atol=1e-10)


def _stem_module(c0, pool):
    conv = torch.nn.Conv1d(1, c0, 7, stride=2, padding=3, bias=False, dtype=D)
    p = torch.nn.MaxPool1d(3, 2, 1) if pool == 0 else torch.nn.AvgPool1d(3, 2, 1)
    return conv, p


@pytest.mark.parametrize("pool", [0, 1])
@pytest.mark.parametrize("offset", [0.0, 1e3])
def test_stem_chain_matches_modules(pool, offset):
    gen = torch.Generator().manual_seed(4)
    n, c0, group = 6, 8, 3
    x = offset + torch.randn(n, 224, generator=gen, dtype=D)
    x[1] = 0.0
    x[3:] = 0.0                                             # one all-zero group
    conv, p = _stem_module(c0, pool)
    with torch.no_grad():
        conv.weight.copy_(0.3 * torch.randn(c0, 1, 7, generator=gen, dtype=D))
    gamma = (0.5 + torch.rand(c0, generator=gen, dtype=D)).requires_grad_(True)
    beta = torch.randn(c0, generator=gen, dtype=D).requires_grad_(True)
    dout = torch.randn(n, c0, 56, generator=gen, dtype=D)
    y, _ = _module_bn(conv(x[:, None, :]), gamma, beta, group)
    ref = p(y.relu())
    gw, gg, gb = torch.autograd.grad(ref, [conv.weight, gamma, beta], dout)
    w = conv.weight.detach()
    out, pre, mean, rstd = R.stem_forward(x, w, gamma.detach(), beta.detach(), group, pool)
    torch.testing.assert_close(out, ref.detach(), rtol=1e-11, atol=1e-11)
    dw, dgamma, dbeta = R.stem_backward(dout, x, w, gamma.detach(), mean, rstd, group, pool, pre)
    torch.testing.assert_close(dw, gw, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(dgamma, gg, rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(dbeta, gb, rtol=1e-12, atol=1e-11)


@pytest.mark.parametrize("pool", [0, 1])
def test_stem_eval_and_frozen_chain_match_modules(pool):
    gen = torch.Generator().manual_seed(5)
    n, c0 = 4, 8
    x = 100.0 + torch.randn(n, 224, generator=gen, dtype=D)
    conv, p = _stem_module(c0, pool)
    bn = torch.nn.BatchNorm1d(c0, dtype=D).eval()
    with torch.no_grad():
        conv.weight.copy_(0.3 * torch.randn(c0, 1, 7, generator=gen, dtype=D))
        y = conv(x[:, None, :])
        bn.running_mean.copy_(y.mean(dim=(0, 2)))
        bn.running_var.copy_(y.var(dim=(0, 2)))
        bn.weight.copy_(0.5 + torch.rand(c0, generator=gen, dtype=D))
        bn.bias.copy_(torch.randn(c0, generator=gen, dtype=D))
    dout = torch.randn(n, c0, 56, generator=gen, dtype=D)
    ref = p(bn(conv(x[:, None, :])).relu())
    gw, gg, gb = torch.autograd.grad(ref, [conv.weight, bn.weight, bn.bias], dout)
    scale, shift = R.eval_coeffs(bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var)
    w = conv.weight.detach()
    out, pre = R.stem_eval_forward(x, w, scale, shift, pool)
    torch.testing.assert_close(out, ref.detach(), rtol=1e-10, atol=1e-10)
    rstd = (bn.running_var + R.EPS).rsqrt()
    dw, dgamma, dbeta = R.stem_frozen_backward(dout, x, w, scale, bn.running_mean, rstd, pool, pre)
    torch.testing.assert_close(dw, gw, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(dgamma, gg, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(dbeta, gb, rtol=1e-12, atol=1e-11)


def test_frozen_bn_backward_matches_module():
    """bn_frozen_bwd's reference: dx = scale * g, dgamma = sum g * xhat, dbeta = sum g (xhat from the running statistics)."""
    gen = torch.Generator().manual_seed(6)
    n, c, l = 5, 4, 11
    bn = torch.nn.BatchNorm1d(c, dtype=D).eval()
    with torch.no_grad():
        bn.running_mean.copy_(torch.tensor([0.0, 1e3, -10.0, 5.0], dtype=D))
        bn.running_var.copy_(torch.tensor([1.0, 1e-8, 0.0, 4.0], dtype=D))
        bn.weight.copy_(0.5 + torch.rand(c, generator=gen, dtype=D))
    x = (bn.running_mean[None, :, None] + torch.randn(n, c, l, generator=gen, dtype=D)).requires_grad_(True)
    dout = torch.randn(n, c, l, generator=gen, dtype=D)
    gx, gg, gb = torch.autograd.grad(bn(x), [x, bn.weight, bn.bias], dout)
    scale, _ = R.eval_coeffs(bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var)
    rstd = (bn.running_var + R.EPS).rsqrt()
    xhat = (x.detach() - bn.running_mean[None, :, None]) * rstd[None, :, None]
    torch.testing.assert_close(dout * scale[None, :, None], gx, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close((dout * xhat).sum(dim=(0, 2)), gg, rtol=1e-10, atol=1e-10)
    torch.testing.assert_close(dout.sum(dim=(0, 2)), gb, rtol=1e-12, atol=1e-12)

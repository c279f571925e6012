"""CPU: the input-gradient API's refusals, plan keys and ABI entries (no device needed)."""
import pytest
import torch

import deepards_b200 as D
from deepards_b200 import _lib, engine, saliency


def test_exported():
    assert D.input_gradients is saliency.input_gradients
    assert "input_gradients" in D.__all__


def test_abi_entries_declared():
    for name in ("dards_stem_dgrad", "dards_stem_frozen_dgrad", "dards_stem_alt_dgrad"):
        assert name in _lib._SIGNATURES


def test_not_a_head_refused():
    with pytest.raises(TypeError, match="Linear"):
        D.input_gradients(torch.nn.Linear(224, 2), torch.zeros(1, 20, 1, 224))
    with pytest.raises(TypeError):
        D.input_gradients(D.resnet18(initial_planes=16), torch.zeros(1, 20, 1, 224))


def test_cpu_network_refused():
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        D.input_gradients(net, torch.zeros(1, 20, 1, 224))


def test_shape_refusals():
    net = D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 0)
    with pytest.raises(Exception, match="224"):
        D.input_gradients(net, torch.zeros(1, 20, 1, 200))
    reg = D.CNNRegressor(D.resnet18(initial_planes=16), 2)
    with pytest.raises(NotImplementedError, match="N, 1, 224"):
        D.input_gradients(reg, torch.zeros(2, 20, 1, 224))


def test_double_conv_first_eval_rule():
    bb = D.resnet18(initial_planes=16, double_conv_first=True).eval()
    with pytest.raises(NotImplementedError, match="double_conv_first"):
        saliency._bn_rule(bb)
    assert saliency._bn_rule(D.resnet18(initial_planes=16).eval()) == "frozen"
    assert saliency._bn_rule(D.resnet18(initial_planes=16).train()) == "train"
    assert saliency._bn_rule(D.densenet18().eval()) == "train"


def test_seed_forms():
    out = torch.tensor([[0.1, 0.9], [0.8, 0.2]])
    assert torch.equal(saliency._seed(out, None), torch.tensor([[0., 1.], [1., 0.]]))
    assert torch.equal(saliency._seed(out, 0), torch.tensor([[1., 0.], [1., 0.]]))
    assert torch.equal(saliency._seed(out, torch.tensor([1, 1])), torch.tensor([[0., 1.], [0., 1.]]))
    for bad in (torch.tensor([1, 1, 0]), 2):
        with pytest.raises(ValueError):
            saliency._seed(out, bad)
    with pytest.raises(TypeError):
        saliency._seed(out, torch.tensor([0.5, 1.0]))


def test_plan_and_get_plan_take_input_grad():
    import inspect
    assert inspect.signature(engine.Plan.__init__).parameters["input_grad"].default is False
    assert inspect.signature(engine.get_plan).parameters["input_grad"].default is False

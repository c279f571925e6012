"""CPU: the parts of DataParallelTrainer's generic head step that need no GPU -- which nets it refuses, and the head run on
substitute parameter leaves (torch.func.functional_call over `net._head`), which must give the module's own numbers."""
import pytest
import torch
import torch.nn as nn


def test_a_net_the_trainer_does_not_know_raises_type_error_naming_its_class():
    import deepards_b200 as D
    from deepards_b200.data_parallel import DataParallelTrainer
    with pytest.raises(TypeError, match="Sequential"):
        DataParallelTrainer(nn.Sequential(nn.Linear(4, 2)))
    with pytest.raises(TypeError, match="ResNet"):
        DataParallelTrainer(D.resnet18(initial_planes=16))


@pytest.mark.parametrize("kind", ["to_mean", "compr_to_rf", "double_linear", "regressor", "lstm", "transformer",
                                  "cnn_linear", "per_breath"])
def test_head_on_fresh_leaves_equals_the_module_head(kind):
    import deepards_b200 as D
    from deepards_b200.data_parallel import _HeadCall
    torch.manual_seed(0)
    bb = D.resnet18(initial_planes=16)
    net = {"to_mean": lambda: D.CNNLinearToMean(bb), "compr_to_rf": lambda: D.CNNLinearComprToRF(bb),
           "double_linear": lambda: D.CNNDoubleLinearNetwork(bb, 20, 0), "regressor": lambda: D.CNNRegressor(bb, 3),
           "lstm": lambda: D.CNNLSTMNetwork(bb, 0, False, 32),
           "transformer": lambda: D.CNNTransformerNetwork(bb, 0, False, 64, 2),
           "cnn_linear": lambda: D.CNNLinearNetwork(bb, 20, 0),
           "per_breath": lambda: D.CNNSingleBreathLinearNetwork(bb)}[kind]()
    for m in net.modules():
        if isinstance(m, nn.Dropout):
            m.p = 0.0
    net.precision = "fp32"
    backbone = set(id(p) for p in bb.parameters())
    named = [("net." + n, p) for n, p in net.named_parameters() if id(p) not in backbone]
    feat = torch.randn((40, 128) if kind == "regressor" else (2, 20, 128))
    first = lambda o: o[0] if isinstance(o, tuple) else o  # noqa: E731
    f1 = feat.clone().requires_grad_(True)
    leaves = dict((n, p.detach().requires_grad_(True)) for n, p in named)
    out = first(torch.func.functional_call(_HeadCall(net), leaves, (f1,), strict=False, tie_weights=False))
    g = torch.autograd.grad(out.sum(), [f1] + list(leaves.values()))
    f2 = feat.clone().requires_grad_(True)
    ref = first(net._head(f2))
    r = torch.autograd.grad(ref.sum(), [f2] + [p for _, p in named])
    assert torch.equal(out, ref)
    assert all(torch.equal(a, b) for a, b in zip(g, r))
    # the module's own parameters are back in place afterwards (nn.LSTM's flat weight list included)
    assert all(p is q for (_, p), (_, q) in zip(named, [(n, p) for n, p in net.named_parameters() if id(p) not in backbone]))
    if kind == "lstm":
        lstm = net.lstm
        assert all(a is b for a, b in zip(lstm._flat_weights, [lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0,
                                                               lstm.bias_hh_l0]))

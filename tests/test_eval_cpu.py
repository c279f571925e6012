"""CPU: ResNet eval() at the boundary -- argument validation of the new entry points, the eval path's refusal of CPU
tensors, and the eval-mode reference the GPU tests compare with.  No kernel is launched here."""
import pytest
import torch
import torch.nn.functional as F

from oracle import cnn_linear_oracle as O
from tests import eval_reference as R
from tests.helpers import rel_err


def test_eval_entry_points_validate_their_arguments():
    import __graft_entry__ as g
    g.build()
    from deepards_b200 import _lib
    lib = _lib.load()
    # null pointers, a bad l_out, relu outside {0, 1}, the tcgen05 path without bf16
    rc = lib.dards_conv1d_affine_fwd(None, None, None, None, None, None, 1, 56, 56, 64, 64, 64, 64, 0, 3, 1, 1, 1, 0, 0, None)
    assert rc == -1 and "null pointer" in _lib.last_error()
    rc = lib.dards_conv1d_affine_fwd(16, 16, 16, None, 16, 16, 1, 56, 55, 64, 64, 64, 64, 0, 3, 1, 1, 1, 0, 0, None)
    assert rc == -1 and "l_out" in _lib.last_error()
    rc = lib.dards_conv1d_affine_fwd(16, 16, 16, None, 16, 16, 1, 56, 56, 64, 64, 64, 64, 0, 3, 1, 1, 2, 0, 0, None)
    assert rc == -1 and "relu" in _lib.last_error()
    rc = lib.dards_conv1d_affine_fwd(16, 16, 16, None, 16, 16, 1, 56, 56, 64, 64, 64, 64, 0, 3, 1, 1, 1, 0, 1, None)
    assert rc == -1 and "bf16" in _lib.last_error()
    # the residual must not overlap the output (the epilogue reads it while other tiles are being stored)
    rc = lib.dards_conv1d_affine_fwd(16, 16, 4096, 4096 + 64, 16, 16, 2, 56, 56, 64, 64, 64, 64, 64, 3, 1, 1, 1, 1, 1, None)
    assert rc == -1 and "overlap" in _lib.last_error()
    with pytest.raises(RuntimeError, match="multiple of 16"):   # C0 = 40: the stem works on 16-channel slabs
        _lib.call("dards_stem_eval_fwd", 16, 16, 16, 16, 16, 3, 40, 40, 0, 0, None)
    with pytest.raises(RuntimeError, match="pool"):
        _lib.call("dards_stem_eval_fwd", 16, 16, 16, 16, 16, 3, 64, 64, 2, 0, None)
    assert lib.dards_bn_eval_coeffs_batched(None, 1, 1, 1e-5, None) == -1


def test_eval_mode_takes_the_eval_path_and_still_refuses_cpu_tensors():
    import deepards_b200 as D
    for net in (D.CNNLinearNetwork(D.resnet18(initial_planes=16), 20, 0), D.resnet18(initial_planes=16)):
        net.eval()
        x = torch.zeros(2, 20, 1, 224) if isinstance(net, D.CNNLinearNetwork) else torch.zeros(7, 1, 224)
        with pytest.raises(RuntimeError, match="no CPU fallback"):   # not the former NotImplementedError
            net(x, None) if isinstance(net, D.CNNLinearNetwork) else net(x)


def _perturbed_resnet_state(seed):
    sd = O.cnn_linear_state("resnet18", seed=seed, initial_planes=16)
    g = torch.Generator().manual_seed(seed)
    for k in sd:
        if k.endswith("running_mean"):
            sd[k] = 0.3 * torch.randn(sd[k].shape, generator=g)
        elif k.endswith("running_var"):
            sd[k] = torch.exp(0.5 * torch.randn(sd[k].shape, generator=g))
    return sd


def _torch_modules_eval(bb, x):
    """The backbone's own nn.Conv1d / nn.BatchNorm1d children in eval(), composed as resnet.py:141-163 does."""
    y = bb.first_pool(F.relu(bb.bn1(bb.conv1(x))))
    for layer in (bb.layer1, bb.layer2, bb.layer3, bb.layer4):
        for blk in layer:
            out = blk.bn2(blk.conv2(F.relu(blk.bn1(blk.conv1(y)))))
            y = F.relu(out + (blk.downsample(y) if blk.downsample is not None else y))
    return bb.avgpool(y).reshape(y.shape[0], -1)


@pytest.mark.parametrize("pool", ["max", "avg"])
def test_eval_reference_matches_torch_batchnorm_modules_in_eval(pool):
    """tests/eval_reference.py (what the GPU eval plans are compared with) is nn.BatchNorm1d.eval() semantics: checked
    against torch's own modules, with running statistics far from their initial zeros / ones."""
    import deepards_b200 as D
    sd = _perturbed_resnet_state(11)
    bb_sd = {k[len("breath_block."):]: v for k, v in sd.items() if k.startswith("breath_block.")}
    bb = D.resnet18(initial_planes=16, first_pool_type=pool)
    bb.load_state_dict(bb_sd)
    bb.eval()
    x = O.synthetic_breaths(2, seed=12)
    flat = x.reshape(-1, 1, 224)
    before = {k: v.clone() for k, v in sd.items()}
    with torch.no_grad():
        ref = _torch_modules_eval(bb, flat)
    got = R.resnet_forward(bb_sd, flat, first_pool_type=pool)
    assert rel_err(got, ref) < 1e-5
    assert all(torch.equal(sd[k], before[k]) for k in sd)   # eval mode never touches the running buffers
    # the sequence head: one row of logits per sequence from its 20 breaths' features
    w, b = sd["linear_final.weight"], sd["linear_final.bias"]
    heads = R.cnn_linear_forward(sd, x, first_pool_type=pool)
    assert rel_err(heads, torch.stack([F.linear(ref[i * 20:(i + 1) * 20].reshape(-1), w, b) for i in range(2)])) < 1e-5
    # every breath is independent of the rest of its batch
    single = torch.cat([R.resnet_forward(bb_sd, flat[i:i + 1], first_pool_type=pool) for i in range(0, flat.shape[0], 13)])
    assert rel_err(got[::13], single) < 1e-5   # CPU convolutions sum in a batch-size dependent order

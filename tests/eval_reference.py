"""Reference of a ResNet-backed network in eval(): the forward of oracle/cnn_linear_oracle.py (resnet.py:141-163,
torch_cnn_linear_network.py:57-67, 104-113, torch_cnn_bm_regressor.py:14-19) with every BatchNorm normalising with its
running buffers, F.batch_norm(training=False) -- what nn.BatchNorm1d does after module.eval().

Plain torch on the CPU in fp32; the test files compare the B200 eval plans against it.  `sd` is a state_dict in the
reference's key layout (the oracle's cnn_linear_state(), or a module's own state_dict())."""
import torch
import torch.nn.functional as F

BN_EPS = 1e-5
SEQ_LEN = 224


def _bn(sd, name, t):
    return F.batch_norm(t, sd[name + ".running_mean"], sd[name + ".running_var"], sd[name + ".weight"], sd[name + ".bias"],
                        False, 0.0, BN_EPS)


def resnet_forward(sd, x, prefix="", first_pool_type="max"):
    """(N, 1, 224) -> (N, 8 * initial_planes); BasicBlock ResNet, double_conv_first=False."""
    g = lambda k: sd[prefix + k]
    bn = lambda name, t: _bn(sd, prefix + name, t)
    y = F.relu(bn("bn1", F.conv1d(x, g("conv1.weight"), stride=2, padding=3)))
    y = F.max_pool1d(y, 3, 2, 1) if first_pool_type == "max" else F.avg_pool1d(y, 3, 2, 1)
    li = 1
    while (prefix + "layer%d.0.conv1.weight" % li) in sd:
        bi = 0
        while (prefix + "layer%d.%d.conv1.weight" % (li, bi)) in sd:
            pre = "layer%d.%d." % (li, bi)
            stride = 2 if (li > 1 and bi == 0) else 1
            out = F.relu(bn(pre + "bn1", F.conv1d(y, g(pre + "conv1.weight"), stride=stride, padding=1)))
            out = bn(pre + "bn2", F.conv1d(out, g(pre + "conv2.weight"), stride=1, padding=1))
            if (prefix + pre + "downsample.0.weight") in sd:
                res = bn(pre + "downsample.1", F.conv1d(y, g(pre + "downsample.0.weight"), stride=stride))
            else:
                res = y
            y = F.relu(out + res)
            bi += 1
        li += 1
    y = F.avg_pool1d(y, 7, 1)
    return y.reshape(y.shape[0], -1)


def cnn_linear_forward(sd, x, per_breath=False, **kw):
    """(B, 20, 1, 224) -> (B, 2) (CNNLinearNetwork) or (B, 20, 2) (CNNSingleBreathLinearNetwork)."""
    if x.shape[-1] != SEQ_LEN:
        raise Exception("input breaths must have sequence length of 224")
    w, b = sd["linear_final.weight"], sd["linear_final.bias"]
    rows = []
    for i in range(x.shape[0]):
        feat = resnet_forward(sd, x[i], "breath_block.", **kw)
        rows.append((F.linear(feat, w, b) if per_breath else F.linear(feat.reshape(-1), w, b)).unsqueeze(0))
    return torch.cat(rows, 0)


def regressor_forward(sd, x, **kw):
    """CNNRegressor: the backbone on a flat batch (N, 1, 224), then Linear."""
    return F.linear(resnet_forward(sd, x, "breath_block.", **kw).squeeze(), sd["linear_final.weight"],
                    sd["linear_final.bias"])

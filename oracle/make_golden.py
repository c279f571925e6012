"""Generate tests/golden/*.npz from the UNMODIFIED reference modules.

TEST INFRASTRUCTURE ONLY (see oracle/cnn_linear_oracle.py).  Runs only in the build
container, where /root/reference is mounted:

    python oracle/make_golden.py

What it does: imports deepards.models.{resnet,densenet,torch_cnn_linear_network} from
/root/reference, instantiates the reference's nn.Modules, loads the oracle's seeded
state_dict into them with strict=True (this also pins the state_dict KEY NAMES, which are
an interface -- SURVEY.md section 8b), runs forward + BCEWithLogits + backward exactly as
train_ards_detector.py:153,162-163 does, and records logits / loss / parameter gradients /
running statistics / GradCAM tensors.  Big gradient tensors are recorded as a strided
sample (every 61st element) plus sum and L2 norm to keep the fixtures small.

Inputs: randn, the synthetic breath model (SURVEY.md section 8d) and two REAL sequences cut
from the reference's deepards/tests/test_dataset.pkl (z-scored with its stored mu/std).
"""
import os
import pickle
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference")

from oracle import cnn_linear_oracle as O  # noqa: E402

from deepards.models.resnet import resnet18 as ref_resnet18  # noqa: E402
from deepards.models.densenet import densenet18 as ref_densenet18  # noqa: E402
from deepards.models.torch_cnn_linear_network import (  # noqa: E402
    CNNLinearNetwork as RefCNNLinearNetwork,
    CNNSingleBreathLinearNetwork as RefCNNSingleBreathLinearNetwork,
)

OUT = os.path.join(ROOT, "tests", "golden")
SAMPLE_STRIDE = 61
FULL_LIMIT = 50_000  # tensors up to this many elements are stored whole
MAX_FILE_BYTES = 1_000_000  # fixtures stay small: beyond this the largest whole gradients are sampled as well


def real_sequences(n=2):
    """First n sequences of deepards/tests/test_dataset.pkl (py2 pickle of ARDSRawDataset)."""
    for m in ["ventmap", "ventmap.raw_utils", "ventmap.constants", "ventmap.SAM", "imblearn",
              "imblearn.under_sampling", "imblearn.over_sampling", "algorithms", "algorithms.breath_meta", "mock"]:
        sys.modules.setdefault(m, types.ModuleType(m))

    class _Any(object):
        def __init__(self, *a, **k):
            pass

        def __setstate__(self, st):
            if isinstance(st, dict):
                self.__dict__.update(st)

    class U(pickle.Unpickler):
        def find_class(self, module, name):
            try:
                return super().find_class(module, name)
            except Exception:
                return type(name, (_Any,), {})

    with open("/root/reference/deepards/tests/test_dataset.pkl", "rb") as f:
        d = U(f, encoding="latin1").load()
    mu, std = d.scaling_factors[None]
    seqs = np.stack([d.all_sequences[i][1] for i in range(n)])  # (n, 20, 1, 224) f64
    tgt = np.stack([d.all_sequences[i][2] for i in range(n)])
    # dataset.py:1379 then train_ards_detector.py:151 (.float())
    return ((seqs - mu) / std).astype(np.float32), tgt.astype(np.float32), float(mu), float(std)


def record_grads(rec, model):
    for name, p in model.named_parameters():
        if p.grad is None:
            rec["nograd/" + name] = np.zeros(0, np.float32)
            continue
        g = p.grad.detach().reshape(-1).numpy()
        if g.size <= FULL_LIMIT:
            rec["grad/" + name] = g.reshape(p.shape).copy()
        else:
            record_sample(rec, name, g)


def record_sample(rec, name, g):
    rec["gradsample/" + name] = g[::SAMPLE_STRIDE].copy()
    rec["gradstat/" + name] = np.array([g.sum(dtype=np.float64), np.sqrt((g.astype(np.float64) ** 2).sum())])


def save_within_limit(path, rec):
    """np.savez_compressed, sampling the largest whole gradients (as record_grads samples those beyond FULL_LIMIT)
    until the file fits in MAX_FILE_BYTES."""
    while True:
        np.savez_compressed(path, **rec)
        whole = [k for k in rec if k.startswith("grad/")]
        if os.path.getsize(path) <= MAX_FILE_BYTES or not whole:
            return
        key = max(whole, key=lambda k: rec[k].size)
        record_sample(rec, key[len("grad/"):], rec.pop(key).reshape(-1))


def run_case(name, model, sd, x, target, per_breath=False, extra=None):
    missing = model.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    model.train()
    model.zero_grad()
    xt = torch.from_numpy(x)
    out = model(xt, None)
    tt = torch.from_numpy(target)
    loss = torch.nn.BCEWithLogitsLoss()(out, tt)
    loss.backward()
    rec = {"x": x, "target": target, "logits": out.detach().numpy(), "loss": np.array(loss.item(), np.float64)}
    record_grads(rec, model)
    for k, v in model.state_dict().items():
        if k.endswith(("running_mean", "running_var", "num_batches_tracked")):
            rec["buf/" + k] = v.numpy().copy()
    # weight checksum: detects any drift of the oracle's seeded generator
    rec["wsum"] = np.array([float(v.double().abs().sum()) for k, v in sd.items() if v.is_floating_point()])
    if extra:
        rec.update(extra)
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    save_within_limit(path, rec)
    print("%-34s logits[0]=%s loss=%.6f  %.1f KB" % (name, out[0].detach().numpy().ravel()[:2], loss.item(),
                                                   os.path.getsize(path) / 1024))


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    g = torch.Generator().manual_seed(42)

    # 1. ResNet-18 (64 planes), randn, B=2
    sd = O.cnn_linear_state("resnet18", seed=1, bn_perturb=0.1)
    x = torch.randn(2, 20, 1, 224, generator=g).numpy()
    t = np.array([[1, 0], [0, 1]], np.float32)
    run_case("resnet18_p64_B2_randn", RefCNNLinearNetwork(ref_resnet18(), 20, 0), sd, x, t)

    # 2. ResNet-18 with 16 initial planes, synthetic breaths, B=3 (odd on purpose), full grads
    sd = O.cnn_linear_state("resnet18", seed=2, bn_perturb=0.1, initial_planes=16)
    x = O.synthetic_breaths(3, seed=77).numpy()
    t = O.synthetic_targets(3, seed=77).numpy()
    run_case("resnet18_p16_B3_synth", RefCNNLinearNetwork(ref_resnet18(initial_planes=16), 20, 0), sd, x, t)

    # 3. ResNet-18 avg first pool, logits + grads
    sd = O.cnn_linear_state("resnet18", seed=3, bn_perturb=0.1, initial_planes=16)
    x = torch.randn(2, 20, 1, 224, generator=g).numpy()
    run_case("resnet18_p16_B2_avgpool", RefCNNLinearNetwork(ref_resnet18(initial_planes=16, first_pool_type="avg"), 20, 0),
             sd, x, np.array([[0, 1], [1, 0]], np.float32))

    # 4. DenseNet-18 on REAL sequences; drop_rate 0 so the step is deterministic (SURVEY.md point 4)
    xr, tr, mu, std = real_sequences(2)
    sd = O.cnn_linear_state("densenet18", seed=4, bn_perturb=0.1)
    dn = ref_densenet18()
    for m in dn.modules():
        if hasattr(m, "drop_rate"):
            m.drop_rate = 0.0
    model = RefCNNLinearNetwork(dn, 20, 0)
    model.load_state_dict(sd, strict=True)
    # GradCAM tensors for sequence 0 (gradcam.py:40-65, 83-99), target = argmax
    a = model.breath_block.features(torch.from_numpy(xr[0]))
    grads = {}
    a.register_hook(lambda gr: grads.__setitem__("dA", gr))
    y = torch.nn.functional.relu(a)
    y = model.breath_block.avgpool(y).view(-1)
    mo = model.linear_final(y).unsqueeze(0)
    tgt = int(mo.argmax())
    model.zero_grad()
    mo[0, tgt].backward()
    extra = {"cam/A": a.detach().numpy(), "cam/dA": grads["dA"].numpy(), "cam/out": mo.detach().numpy(),
             "cam/target": np.array(tgt), "scaling": np.array([mu, std])}
    run_case("densenet18_B2_real", model, sd, xr, tr, extra=extra)

    # 5. DenseNet-18, synthetic, B=3
    sd = O.cnn_linear_state("densenet18", seed=5, bn_perturb=0.1)
    dn = ref_densenet18()
    for m in dn.modules():
        if hasattr(m, "drop_rate"):
            m.drop_rate = 0.0
    x = O.synthetic_breaths(3, seed=99).numpy()
    t = O.synthetic_targets(3, seed=99).numpy()
    run_case("densenet18_B3_synth", RefCNNLinearNetwork(dn, 20, 0), sd, x, t)

    # 6. per-breath head (config 4): CNNSingleBreathLinearNetwork, padded breaths
    sd = O.cnn_linear_state("resnet18", seed=6, bn_perturb=0.1, initial_planes=16, per_breath=True)
    x = O.synthetic_breaths(2, seed=5).numpy()
    lens = np.random.RandomState(5).randint(60, 201, size=(2, 20))
    for i in range(2):
        for j in range(20):
            x[i, j, 0, lens[i, j]:] = 0.0  # dataset.py:1233-1237 zero padding stays zero after scaling (:1375-1377)
    t = np.tile(np.array([[1, 0]], np.float32), (2, 20, 1))
    run_case("resnet18_p16_B2_perbreath", RefCNNSingleBreathLinearNetwork(ref_resnet18(initial_planes=16)), sd, x, t,
             per_breath=True)


if __name__ == "__main__":
    main()

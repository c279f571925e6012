"""Input-gradient attributions on one GPU: saliency.input_gradients for bf16 ResNet-18 and DenseNet-18 cnn_linear.

    python tools/bench_saliency.py [--out profiles/r08_saliency.jsonl] [--iters 20]

One JSON line per configuration:
  * call_ms: one input_gradients call (forward plan, torch head + one-hot backward, backward plan with the stem's input
    gradient), CUDA events around `iters` calls after warm-up (the plan's CUDA graphs are live by then);
  * dgrad_ms: the stem input-gradient kernel alone, the recorded call of the plan of that batch size replayed under CUDA
    events (the input, d(pool out) and the partial rows stay those of the plan's last call);
  * dgrad_gflop: its arithmetic from the shapes (recomputed convolution, BatchNorm / pool terms ignored, and the 7-tap
    transpose), 2 FLOP per FMA;
  * oracle_autograd_fp32_ms: torch autograd of the fp32 oracle (per-sequence Python loop) on the same GPU, for context;
  * integrated gradients over one 24-hour recording (720 sequences) in 32 alpha steps, as 4 calls of 8 stacked steps;
  * the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import deepards_b200 as D  # noqa: E402
from oracle import cnn_linear_oracle as O  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def events_ms(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def build(backbone):
    bb = D.resnet18() if backbone == "resnet18" else D.densenet18(drop_rate=0.0)
    net = D.CNNLinearNetwork(bb, 20, 0).cuda()
    net.precision = "bf16"
    return net


def dgrad_call(net, n_breaths):
    """The stem input-gradient call of the input_grad plan of n_breaths breaths (the net caches one plan per batch size)."""
    plan = [p for p in net._dards_plans.values() if getattr(p, "input_grad", False) and p.N == n_breaths][0]
    for name, f, args in plan.bwd.calls:
        if name.endswith("_dgrad") and name.startswith("dards_stem"):
            return plan, name, f, args
    raise RuntimeError("no stem dgrad call recorded")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_saliency.jsonl"))
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_saliency needs a GPU"
    name, power = card()
    rows = []
    for backbone in ("resnet18", "densenet18"):
        net = build(backbone)
        for b in (256, 720):
            x = O.synthetic_breaths(b, seed=1).cuda()
            for _ in range(4):
                D.input_gradients(net, x)
            ms = events_ms(lambda: D.input_gradients(net, x), a.iters)
            plan, cname, f, args = dgrad_call(net, b * 20)
            st = torch.cuda.current_stream().cuda_stream
            kms = events_ms(lambda: f(*args, st), 50)
            c0 = 64
            n = b * 20
            flop = 2.0 * n * (112 * 7 * c0 + 224 * 3.5 * c0)
            row = dict(bench="input_gradients", backbone=backbone, head="cnn_linear", precision="bf16", sequences=b,
                       breaths=n, call_ms=round(ms, 3), dgrad_kernel=cname, dgrad_ms=round(kms, 4),
                       dgrad_gflop=round(flop / 1e9, 3), dgrad_tflops=round(flop / kms / 1e9, 2), gpu=name,
                       power_limit=power)
            if b == 256:
                sd = {k: v.cuda() for k, v in net.state_dict().items()}
                xo = x.clone().requires_grad_(True)

                def oracle():
                    out = O.cnn_linear_forward(sd, xo, training=False) if backbone == "densenet18" else \
                        O.cnn_linear_forward(sd, xo)
                    torch.autograd.grad(out[:, 1].sum(), [xo])
                oracle()
                t0 = time.perf_counter()
                for _ in range(3):
                    oracle()
                torch.cuda.synchronize()
                row["oracle_autograd_fp32_ms"] = round((time.perf_counter() - t0) / 3 * 1e3, 2)
            rows.append(row)
            print(json.dumps(row), flush=True)
        # integrated gradients over one recording: 720 sequences, 32 alpha steps as 4 calls of 8 stacked steps
        x = O.synthetic_breaths(720, seed=2).cuda()
        alphas = (torch.arange(32, device="cuda", dtype=torch.float32) + 0.5) / 32

        def ig():
            tot = torch.zeros_like(x)
            for k in range(4):
                al = alphas[8 * k:8 * k + 8].view(8, 1, 1, 1, 1)
                g, _ = D.input_gradients(net, (al * x.unsqueeze(0)).reshape(-1, 20, 1, 224), 1)
                tot += g.view(8, 720, 20, 1, 224).sum(0)
            return tot * x / 32
        ig()
        ig()
        ms = events_ms(ig, 3)
        row = dict(bench="integrated_gradients", backbone=backbone, head="cnn_linear", precision="bf16", sequences=720,
                   steps=32, calls=4, breaths_per_call=8 * 720 * 20, total_ms=round(ms, 2), gpu=name, power_limit=power)
        rows.append(row)
        print(json.dumps(row), flush=True)
        del net
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        for r in rows:
            fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

"""Device-timed ResNet-18 training step with frozen BatchNorm (network in train(), BatchNorm layers in eval(): running
statistics, no statistics pass, no running-statistics update) against the ordinary training step (batch statistics).

Workload: CNNLinearNetwork(resnet18(), 20), bf16 / tcgen05, B = 256 sequences (5 120 breaths), the module path as a
training script drives it: net(x) -> BCEWithLogits -> backward() -> SGD-Nesterov with the clamp hooks.

    python tools/bench_frozen.py [--out FILE] [--reps R] [--steps S]

One JSON object per line (stdout, and FILE if given):
  * "device": the card's name and power limit, read in the same run;
  * "step": ms per step of each mode, the two modes alternated `reps` times in the same process (CUDA events around
    `steps` steps after 3 warm-up steps; each mode has its own module, so its plans and CUDA graphs stay warm);
  * "entry_points": per-entry-point device time of one eager forward + backward of each mode (CUDA events between the
    recorded calls, summed by entry-point name), so that a difference between the modes can be attributed.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import deepards_b200 as D  # noqa: E402
from oracle import cnn_linear_oracle as O  # noqa: E402  (synthetic inputs only)
from tools.bench_eval import device_info, timed  # noqa: E402

DEV = torch.device("cuda", 0)
B = 256


def make(frozen):
    torch.manual_seed(0)
    net = D.CNNLinearNetwork(D.resnet18(), 20, 0).to(DEV)
    net.precision = "bf16"
    net.train()
    if frozen:
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.eval()
    for p in net.parameters():
        p.register_hook(lambda g: g.clamp(-0.01, 0.01))
    opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    return net, opt


def step_fn(net, opt, xs, t):
    def fn(i):
        opt.zero_grad(set_to_none=True)
        F.binary_cross_entropy_with_logits(net(xs[i % len(xs)], None), t).backward()
        opt.step()
    return fn


def per_entry_point(plan):
    """{name: ms} over one eager forward + backward of `plan` (events between the recorded calls)."""
    st = torch.cuda.current_stream(DEV).cuda_stream
    out = {}
    for rec in (plan.pack, plan.fwd, plan.bwd):
        for name, f, args in rec.calls:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f(*args, st)
            e1.record()
            torch.cuda.synchronize()
            out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
    return {k: round(v, 4) for k, v in sorted(out.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    a = ap.parse_args()
    lines = [dict(device_info(), what="device")]
    xs = [O.synthetic_breaths(B, seed=s).to(DEV) for s in range(4)]
    t = O.synthetic_targets(B, seed=0).to(DEV)
    nets = {"train": make(False), "frozen": make(True)}
    fns = {k: step_fn(net, opt, xs, t) for k, (net, opt) in nets.items()}
    times = {k: [] for k in nets}
    for _ in range(a.reps):
        for k in ("train", "frozen"):
            times[k].append(round(timed(fns[k], a.steps), 4))
    lines.append(dict(what="step", workload="cnn_linear resnet18 bf16 B=%d (%d breaths), module path + SGD" % (B, B * 20),
                      ms_per_step=times, median={k: sorted(v)[len(v) // 2] for k, v in times.items()}))
    for k, (net, _) in nets.items():
        plan = max(net.__dict__["_dards_plans"].values(), key=lambda p: p.fwd_serial)
        plan.load_input(xs[0])
        per_entry_point(plan)  # warm
        lines.append(dict(what="entry_points", mode=k, bn=plan.bn, ms=per_entry_point(plan),
                          launches=len(plan.pack) + len(plan.fwd) + len(plan.bwd)))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

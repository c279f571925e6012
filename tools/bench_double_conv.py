"""Device-timed cost of ResNet-18 double_conv_first=True (the two-convolution stem) against the default stem.

    python tools/bench_double_conv.py [--out FILE] [--reps R] [--steps S] [--eval-breaths N]

One JSON object per line (stdout, and FILE if given):
  * "device": the card's name and power limit, read in the same run;
  * "flops": the stem's work computed from the shapes (no measurement): multiply-accumulates per sequence of 20 breaths
    for the default stem, the two-convolution stem and the whole ResNet-18 forward, and the size of a0 at B = 256;
  * "step": ms per training step of CNNLinearNetwork(resnet18(double_conv_first=d), 20), bf16 / tcgen05, B = 256 sequences,
    module path + SGD-Nesterov with the clamp hooks, for d = False and True alternated `reps` times in one process (CUDA
    events around `steps` steps after 3 warm-up steps);
  * "eval": ms per eval() forward of `eval_breaths` breaths (per-breath head, no_grad), both stems alternated;
  * "kernels": a torch.profiler run of its own (one training step of the double stem after warm-up): device time per
    kernel name, the stem's new kernels listed first.
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
NEW_KERNELS = ("stem_alt", "pool3s2", "tc_wgrad7")


def flops(p=64):
    """MACs per breath from the shapes: conv MACs = L_out * C_out * C_in * K."""
    stem = 112 * p * 1 * 7
    alt = 224 * p * 1 * 3 + 112 * p * p * 7
    blocks = 0
    L, cin = 56, p
    for planes, stride in ((p, 1), (2 * p, 2), (4 * p, 2), (8 * p, 2)):
        for bi in range(2):
            s = stride if bi == 0 else 1
            lo = (L + 2 - 3) // s + 1
            blocks += lo * planes * cin * 3 + lo * planes * planes * 3
            if bi == 0 and (s != 1 or cin != planes):
                blocks += lo * planes * cin
            cin, L = planes, lo
    head = 8 * p * 20 * 2 / 20
    per_seq = lambda x: 20 * x  # noqa: E731
    return dict(what="flops", unit="MAC per sequence (20 breaths), forward", default_stem=per_seq(stem),
                double_stem=per_seq(alt), conv2_only=per_seq(112 * p * p * 7), resnet18_default=per_seq(stem + blocks + head),
                resnet18_double=per_seq(alt + blocks + head),
                conv2_over_default_network=round(per_seq(112 * p * p * 7) / per_seq(stem + blocks + head), 4),
                a0_bytes_bf16_B256=B * 20 * 224 * p * 2,
                training_step_extra_gflop_B256=round(3 * 2 * B * per_seq(alt - stem) / 1e9, 2))


def make(double, eval_mode=False):
    torch.manual_seed(0)
    bb = D.resnet18(double_conv_first=double)
    net = (D.CNNSingleBreathLinearNetwork(bb) if eval_mode else D.CNNLinearNetwork(bb, 20, 0)).to(DEV)
    net.precision = "bf16"
    if eval_mode:
        return net.eval(), None
    net.train()
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


def eval_fn(net, x):
    def fn(i):
        with torch.no_grad():
            net(x, None)
    return fn


def kernel_table(fn):
    from torch.profiler import ProfilerActivity, profile
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(0)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            out[ev.key] = [round(t / 1000.0, 4), ev.count]
    new = {k: v for k, v in out.items() if any(s in k for s in NEW_KERNELS)}
    return dict(what="kernels", unit="ms device time, launches", step="one double_conv_first training step, B=%d" % B,
                new=dict(sorted(new.items(), key=lambda kv: -kv[1][0])),
                all=dict(sorted(out.items(), key=lambda kv: -kv[1][0])[:40]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--eval-breaths", type=int, default=65520)
    a = ap.parse_args()
    lines = [dict(device_info(), what="device"), flops()]
    xs = [O.synthetic_breaths(B, seed=s).to(DEV) for s in range(4)]
    t = O.synthetic_targets(B, seed=0).to(DEV)
    nets = {d: make(d) for d in (False, True)}
    fns = {d: step_fn(net, opt, xs, t) for d, (net, opt) in nets.items()}
    times = {"default": [], "double_conv_first": []}
    for _ in range(a.reps):
        for d, k in ((False, "default"), (True, "double_conv_first")):
            times[k].append(round(timed(fns[d], a.steps), 4))
    lines.append(dict(what="step", workload="cnn_linear resnet18 bf16 B=%d (%d breaths), module path + SGD" % (B, B * 20),
                      ms_per_step=times, median={k: sorted(v)[len(v) // 2] for k, v in times.items()}))
    del nets, fns
    torch.cuda.empty_cache()

    seqs = a.eval_breaths // 20
    xe = O.synthetic_breaths(seqs, seed=7).to(DEV)
    enets = {d: make(d, eval_mode=True)[0] for d in (False, True)}
    efns = {d: eval_fn(n, xe) for d, n in enets.items()}
    etimes = {"default": [], "double_conv_first": []}
    for _ in range(a.reps):
        for d, k in ((False, "default"), (True, "double_conv_first")):
            etimes[k].append(round(timed(efns[d], 5, warmup=2), 3))
    lines.append(dict(what="eval", workload="per-breath head, eval(), bf16, %d breaths" % (seqs * 20), ms_per_forward=etimes,
                      median={k: sorted(v)[len(v) // 2] for k, v in etimes.items()}))
    del enets, efns, xe
    torch.cuda.empty_cache()

    net, opt = make(True)
    lines.append(kernel_table(step_fn(net, opt, xs, t)))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

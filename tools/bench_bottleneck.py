"""Device-timed ResNet-50 (Bottleneck) training step and eval forward.

Workload: CNNLinearNetwork(resnet50(), 20, 0), bf16 / tcgen05, B = 256 sequences (5 120 breaths).

    python tools/bench_bottleneck.py [--out FILE] [--reps R] [--steps S]

One JSON object per line (stdout, and FILE if given):
  * "device": the card's name and power limit, read in the same run;
  * "macs": forward multiply-accumulates per sequence from the convolution shapes, for resnet18 / 50 / 101 / 152;
  * "step": ms per training step and sequences per second through DataParallelTrainer (one GPU, whole-step CUDA graph)
    and through the module path (net(x) -> BCEWithLogits -> backward() -> SGD-Nesterov with the clamp hooks), the two
    alternated `reps` times (CUDA events around `steps` steps after 3 warm-up steps); the peak memory of each; and the
    fraction of the dense bf16 tensor ceiling that the step's convolution FLOPs (forward + data gradient + weight
    gradient, from the shapes) reach at the data-sheet 2 250 TFLOP/s;
  * "entry_points": per-entry-point device time of one eager forward + backward (CUDA events between the recorded calls,
    summed by entry-point name);
  * "eval": the eval() forward of CNNSingleBreathLinearNetwork(resnet50()) at 65 520 breaths, ms and breaths per second.
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
from tools.bench_frozen import per_entry_point  # noqa: E402

DEV = torch.device("cuda", 0)
B = 256
GROUP = 20
EVAL_BREATHS = 65520
BF16_DENSE_TFLOPS = 2250.0   # NVIDIA HGX B200 data sheet, one GPU, dense BF16


def conv_macs(backbone):
    """(forward MACs per sequence, of which the stem's first convolution) from the convolution shapes that the forward
    uses: l_out * c_in * c_out * k per breath, times the 20 breaths of a sequence."""
    c = backbone.conv1   # the default stem: 224 -> 112
    stem = 112 * c.in_channels * c.out_channels * c.kernel_size[0]
    total, L = stem, 56
    for layer in (backbone.layer1, backbone.layer2, backbone.layer3, backbone.layer4):
        for blk in layer:
            convs = [blk.conv1, blk.conv2] + ([blk.conv3] if hasattr(blk, "conv3") else [])
            l = L
            for cv in convs:
                l = (l + 2 * cv.padding[0] - cv.kernel_size[0]) // cv.stride[0] + 1
                total += l * cv.in_channels * cv.out_channels * cv.kernel_size[0]
            if blk.downsample is not None:
                cv = blk.downsample[0]
                total += l * cv.in_channels * cv.out_channels
            L = l
    return total * GROUP, stem * GROUP


def make(seed=0):
    torch.manual_seed(seed)
    net = D.CNNLinearNetwork(D.resnet50(), GROUP, 0).to(DEV)
    net.precision = "bf16"
    return net.train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    a = ap.parse_args()
    from deepards_b200.data_parallel import DataParallelTrainer
    lines = [dict(device_info(), what="device")]
    macs = {n: conv_macs(f())[0] for n, f in (("resnet18", D.resnet18), ("resnet50", D.resnet50),
                                              ("resnet101", D.resnet101), ("resnet152", D.resnet152))}
    fwd50, stem50 = conv_macs(D.resnet50())
    # training step: forward + dgrad (not for the stem's convolution, whose input needs no gradient) + wgrad
    step_flops = 2.0 * B * (3 * fwd50 - stem50)
    lines.append(dict(what="macs", forward_macs_per_sequence=macs, resnet50_step_flops_B256=step_flops))

    xs = [O.synthetic_breaths(B, seed=s).to(DEV) for s in range(4)]
    t = O.synthetic_targets(B, seed=0).to(DEV)

    net_m = make()
    for p in net_m.parameters():
        p.register_hook(lambda g: g.clamp(-0.01, 0.01))
    opt = torch.optim.SGD(net_m.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)

    def module_step(i):
        opt.zero_grad(set_to_none=True)
        F.binary_cross_entropy_with_logits(net_m(xs[i % len(xs)], None), t).backward()
        opt.step()

    tr = DataParallelTrainer(make(), lr=1e-3, optimizer="sgd", momentum=0.9, weight_decay=1e-4, clip_val=0.01,
                             use_graph=True)

    def trainer_step(i):
        tr.train_step(xs[i % len(xs)], t)

    fns = {"trainer": trainer_step, "module": module_step}
    peak = {}
    for k, fn in fns.items():   # first use builds the plans and graphs; peak memory of each path on its own
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(DEV)
        timed(fn, 2)
        peak[k] = round(torch.cuda.max_memory_allocated(DEV) / 2 ** 30, 3)
    times = {k: [] for k in fns}
    for _ in range(a.reps):
        for k, fn in fns.items():
            times[k].append(round(timed(fn, a.steps), 4))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    lines.append(dict(what="step", workload="cnn_linear resnet50 bf16 B=%d (%d breaths)" % (B, B * GROUP),
                      ms_per_step=times, median_ms=med,
                      seq_per_s={k: round(B / (v / 1e3), 1) for k, v in med.items()},
                      peak_mem_gib=peak,
                      tensor_ceiling_fraction={k: round(step_flops / (v / 1e3) / (BF16_DENSE_TFLOPS * 1e12), 4)
                                               for k, v in med.items()}))

    plan = max(net_m.__dict__["_dards_plans"].values(), key=lambda p: p.fwd_serial)
    plan.load_input(xs[0])
    per_entry_point(plan)  # warm
    lines.append(dict(what="entry_points", bn=plan.bn, ms=per_entry_point(plan),
                      launches=len(plan.pack) + len(plan.fwd) + len(plan.bwd)))
    del tr, net_m, opt
    torch.cuda.empty_cache()

    torch.manual_seed(0)
    ev = D.CNNSingleBreathLinearNetwork(D.resnet50()).to(DEV)
    ev.precision = "bf16"
    ev.eval()
    xe = O.synthetic_breaths(EVAL_BREATHS // GROUP, seed=7).to(DEV)
    with torch.no_grad():
        ms = [round(timed(lambda i: ev(xe, None), 10), 3) for _ in range(3)]
        out = ev(xe, None)
    m = sorted(ms)[1]
    lines.append(dict(what="eval", workload="CNNSingleBreathLinearNetwork(resnet50()) eval() bf16, %d breaths" % EVAL_BREATHS,
                      ms=ms, median_ms=m, breaths_per_s=round(EVAL_BREATHS / (m / 1e3)), finite=bool(torch.isfinite(out).all())))
    text = "\n".join(json.dumps(x) for x in lines)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

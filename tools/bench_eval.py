"""Device-timed ResNet-18 inference in eval() (running-statistics BatchNorm in the convolution epilogues) against the
train-mode forward (batch statistics, today's `tools/bench_configs.py inference` path) on the same inputs.

Workload: BASELINE.json configs[3], the padded_breath_by_breath single-breath classifier (CNNSingleBreathLinearNetwork,
ResNet-18, bf16 / tcgen05), forward only, at 1 024 / 4 096 / 16 384 / 65 536 breaths.

    python tools/bench_eval.py [--out FILE] [--reps R]

One JSON object per line (stdout, and FILE if given):
  * "device": the card's name and power limit, read in the same run;
  * per size and mode: ms per call, breaths/s, kernel launches per forward, and the per-entry-point device time of one
    eager forward (CUDA events between the recorded calls);
  * "parity": bf16 eval logits against the fp32 eval plan (CUDA-core kernels) at the largest size.
Timing: CUDA events around `steps` calls after 3 warm-up calls, the two modes alternated `reps` times in the same process.
Inputs rotate over distinct batches whose total size exceeds twice the 126 MB L2, so no call finds its input in the L2;
the plan's own activation buffers are reused by every call, as in any inference loop (at 1 024 breaths they fit the L2).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import deepards_b200 as D  # noqa: E402
from deepards_b200 import _lib  # noqa: E402
from oracle import cnn_linear_oracle as O  # noqa: E402  (synthetic inputs only)

DEV = torch.device("cuda", 0)
L2_BYTES = 126 << 20
SIZES = (1024, 4096, 16384, 65536)


def device_info():
    info = {"device": torch.cuda.get_device_name(DEV)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power, clock = [s.strip() for s in q.strip().splitlines()[0].split(",")]
        info.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # a missing tool must not hide the timings; say so in the record
        info["power_limit"] = "not read (%s)" % (e,)
    return info


def timed(fn, steps, warmup=3):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def padded(x, seed):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(60, 201, (x.shape[0], x.shape[1]), generator=g)
    return x * (torch.arange(224).view(1, 1, 1, 224) < lens.view(x.shape[0], x.shape[1], 1, 1))


def plan_of(net, bn):
    return next(p for p in net.__dict__["_dards_plans"].values() if p.bn == bn)


def per_call_profile(plan, reps=3):
    """Launches of one eager forward (pack + recorded list) and the device time of each recorded entry point."""
    st = torch.cuda.current_stream(DEV)
    calls = [(n, f, a) for n, f, a in plan.pack.calls] + list(plan.fwd.calls)
    lib = _lib.load()
    torch.cuda.synchronize()
    before = lib.dards_launch_count()
    for n, f, a in calls:
        _lib.check(f(*a, st.cuda_stream), n)
    torch.cuda.synchronize()
    launches = lib.dards_launch_count() - before
    times = {}
    for _ in range(reps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(calls) + 1)]
        ev[0].record()
        for i, (n, f, a) in enumerate(calls):
            _lib.check(f(*a, st.cuda_stream), n)
            ev[i + 1].record()
        torch.cuda.synchronize()
        for i, (n, _, _) in enumerate(calls):
            times[n] = times.get(n, 0.0) + ev[i].elapsed_time(ev[i + 1]) / reps
    return launches, {k: round(v, 4) for k, v in sorted(times.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    out = open(args.out, "w") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit(dict(device_info(), torch=torch.__version__, cuda=torch.version.cuda))
    torch.manual_seed(0)
    net = D.CNNSingleBreathLinearNetwork(D.resnet18()).to(DEV)
    net.precision = "bf16"
    # non-trivial running statistics, as a trained checkpoint would have
    with torch.no_grad():
        net.train()
        for i in range(3):
            net(O.synthetic_breaths(8, seed=500 + i).to(DEV), None)
    flop = 76.26e6  # per breath, forward (SURVEY.md 8d)
    for n_breaths in SIZES:
        b = n_breaths // 20
        one = padded(O.synthetic_breaths(min(b, 512), seed=40), 7).repeat((b + 511) // 512, 1, 1, 1)[:b].contiguous()
        n_inputs = max(2, -(-2 * L2_BYTES // (one.numel() * 4)))
        xs = [(one * (1 + 0.01 * i)).to(DEV) for i in range(n_inputs)]
        res = {"train": [], "eval": []}
        steps = 20 if n_breaths <= 16384 else 8
        for rep in range(args.reps):
            for mode in ("eval", "train"):
                getattr(net, mode)()

                def call(i):
                    with torch.no_grad():
                        net(xs[i % n_inputs], None)
                res[mode].append(timed(call, steps))
        for mode in ("eval", "train"):
            getattr(net, mode)()
            with torch.no_grad():
                net(xs[0], None)
            launches, per_call = per_call_profile(plan_of(net, mode))
            ms = sorted(res[mode])
            emit({"config": "configs[3] single-breath classifier, ResNet-18 bf16", "mode": mode,
                  "batchnorm": "running statistics (eval)" if mode == "eval" else "batch statistics (train-mode forward)",
                  "breaths": b * 20, "ms_per_call_median": round(ms[len(ms) // 2], 4),
                  "ms_per_call_all": [round(v, 4) for v in res[mode]],
                  "breaths_per_s": round(b * 20 / ms[len(ms) // 2] * 1e3),
                  "tflops": round(b * 20 * flop / ms[len(ms) // 2] / 1e9, 1), "launches_per_forward": launches,
                  "eager_ms_per_entry_point": per_call, "inputs_rotated": n_inputs})
        net.train()
        del xs
        net.__dict__.pop("_dards_plans", None)
        torch.cuda.empty_cache()

    # bf16 eval logits vs the fp32 eval plan at the largest size
    b = SIZES[-1] // 20
    x = padded(O.synthetic_breaths(min(b, 512), seed=41), 8).repeat((b + 511) // 512, 1, 1, 1)[:b].to(DEV)
    net.eval()
    logits = {}
    for precision in ("fp32", "bf16"):
        net.precision = precision
        with torch.no_grad():
            logits[precision] = net(x, None).double()
        net.__dict__.pop("_dards_plans", None)
        torch.cuda.empty_cache()
    err = float((logits["bf16"] - logits["fp32"]).abs().max() / logits["fp32"].abs().max())
    emit({"parity": "bf16 eval logits vs fp32 eval plan", "breaths": b * 20, "max_abs_rel": err,
          "argmax_agreement": float((logits["bf16"].argmax(-1) == logits["fp32"].argmax(-1)).double().mean())})


if __name__ == "__main__":
    main()

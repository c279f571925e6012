"""Device-timed training step of the six torch heads: DataParallelTrainer's generic step against the module path.

Workload: bf16 resnet18() backbone (64 planes), B = 256 sequences of 20 breaths per GPU; CNNRegressor takes the same
5 120 breaths as one flat batch (one BatchNorm group) with nn.MSELoss(), the other heads nn.BCEWithLogitsLoss().

    python tools/bench_heads_dp.py [--out profiles/r07_heads_dp.jsonl] [--reps R] [--steps S] [--worlds 1,2,8]

One JSON object per line (stdout, and FILE if given):
  * "device": the card's name and power limit, read in the same run, and the number of visible GPUs;
  * "step" (one per head, world 1): ms per step and sequences per second through DataParallelTrainer (SGD, use_graph=True:
    one CUDA graph per step) and through the module path (net(x) -> criterion -> backward() -> torch.optim.SGD-Nesterov
    with the reference's clamp hooks), the two alternated `reps` times (CUDA events around `steps` steps after 3 warm-up
    steps); whether the trainer's step was replayed from a captured graph;
  * "step_dp" (one per head and world size > 1, when the machine has that many GPUs): the trainer's ms per step with B
    sequences per GPU (NCCL all-reduce, per-segment CUDA graphs), the slowest rank's time.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

import deepards_b200 as D  # noqa: E402
from oracle import cnn_linear_oracle as O  # noqa: E402  (synthetic inputs only)

B = 256
GROUP = 20
HEADS = ["cnn_linear_to_mean", "cnn_linear_compr_to_rf", "cnn_double_linear", "cnn_regressor", "cnn_lstm",
         "cnn_transformer"]


def make(kind, dev, seed=0):
    torch.manual_seed(seed)
    bb = D.resnet18()
    net = {"cnn_linear_to_mean": lambda: D.CNNLinearToMean(bb), "cnn_linear_compr_to_rf": lambda: D.CNNLinearComprToRF(bb),
           "cnn_double_linear": lambda: D.CNNDoubleLinearNetwork(bb, GROUP, 0), "cnn_regressor": lambda: D.CNNRegressor(bb, 1),
           "cnn_lstm": lambda: D.CNNLSTMNetwork(bb, 0, False, 32),
           "cnn_transformer": lambda: D.CNNTransformerNetwork(bb, 0, False, 64, 2)}[kind]()
    net = net.to(dev).train()
    net.precision = "bf16"
    return net


def batches(kind, dev, seed=0):
    xs, ts = [], []
    for s in range(4):
        x = O.synthetic_breaths(B, seed=seed + s)
        t = O.synthetic_targets(B, seed=seed + s)
        if kind == "cnn_regressor":
            x = x.reshape(-1, 1, 224)
            t = torch.randn(x.shape[0], 1, generator=torch.Generator().manual_seed(seed + s))
        elif kind in ("cnn_lstm", "cnn_transformer"):
            t = t.unsqueeze(1).repeat(1, GROUP, 1)
        xs.append(x.to(dev))
        ts.append(t.to(dev))
    return xs, ts


def criterion(kind):
    return nn.MSELoss() if kind == "cnn_regressor" else nn.BCEWithLogitsLoss()


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


def one_gpu(kind, reps, steps):
    from deepards_b200.data_parallel import DataParallelTrainer
    dev = torch.device("cuda", 0)
    xs, ts = batches(kind, dev)
    crit = criterion(kind)
    net_m = make(kind, dev)
    for p in net_m.parameters():
        p.register_hook(lambda g: g.clamp(-0.01, 0.01))
    opt = torch.optim.SGD(net_m.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)

    def module_step(i):
        opt.zero_grad(set_to_none=True)
        out = net_m(xs[i % 4], None)
        crit(out[0] if isinstance(out, tuple) else out, ts[i % 4]).backward()
        opt.step()

    tr = DataParallelTrainer(make(kind, dev), lr=1e-3, optimizer="sgd", momentum=0.9, weight_decay=1e-4, clip_val=0.01,
                             use_graph=True, criterion=crit)

    def trainer_step(i):
        tr.train_step(xs[i % 4], ts[i % 4])

    fns = {"trainer": trainer_step, "module": module_step}
    for fn in fns.values():
        timed(fn, 2)
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            times[k].append(round(timed(fn, steps), 4))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    out = dict(what="step", head=kind, world=1,
               workload="%s resnet18 bf16 B=%d (%d breaths)%s" % (kind, B, B * GROUP,
                                                                   ", one BatchNorm group" if kind == "cnn_regressor" else ""),
               ms_per_step=times, median_ms=med, seq_per_s={k: round(B / (v / 1e3), 1) for k, v in med.items()},
               trainer_speedup=round(med["module"] / med["trainer"], 3), trainer_graph_replayed=tr.graph_launches > 0)
    del tr, net_m, opt
    torch.cuda.empty_cache()
    return out


def _dp_worker(rank, world, port, kind, steps, q):
    import torch.distributed as dist
    from deepards_b200.data_parallel import DataParallelTrainer
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world, device_id=dev)
    xs, ts = batches(kind, dev, seed=100 * rank)
    tr = DataParallelTrainer(make(kind, dev), lr=1e-3, optimizer="sgd", momentum=0.9, weight_decay=1e-4, clip_val=0.01,
                             use_graph=True, criterion=criterion(kind))
    ms = [timed(lambda i: tr.train_step(xs[i % 4], ts[i % 4]), steps) for _ in range(3)]
    m = torch.tensor([sorted(ms)[1]], device=dev)
    dist.all_reduce(m, op=dist.ReduceOp.MAX)
    if rank == 0:
        q.put(float(m))
    dist.barrier()
    tr.close()
    dist.destroy_process_group()


def multi_gpu(kind, world, steps):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 32500 + (os.getpid() % 1000) + world
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, kind, steps, q)) for r in range(world)]
    for p in procs:
        p.start()
    ms = q.get(timeout=900)
    for p in procs:
        p.join(timeout=300)
        if p.exitcode != 0:
            raise RuntimeError("rank exited with %s" % p.exitcode)
    return dict(what="step_dp", head=kind, world=world, sequences_per_gpu=B, trainer_ms=round(ms, 4),
                seq_per_s=round(world * B / (ms / 1e3), 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--worlds", default="1,2,8", help="GPU counts to run (those above the visible count are skipped)")
    a = ap.parse_args()
    from tools.bench_eval import device_info
    n_gpu = torch.cuda.device_count()
    lines = [dict(device_info(), what="device", visible_gpus=n_gpu)]
    worlds = [int(w) for w in a.worlds.split(",")]
    for kind in HEADS:
        if 1 in worlds:
            lines.append(one_gpu(kind, a.reps, a.steps))
            print(json.dumps(lines[-1]), flush=True)
        for w in worlds:
            if 1 < w <= n_gpu:
                lines.append(multi_gpu(kind, w, a.steps))
                print(json.dumps(lines[-1]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()

"""Benchmark of the cnn_linear hot path (BASELINE.json metric: train sequences/sec, 20x224 breaths).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--backbone resnet18|densenet18]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- cnn_linear / ResNet-18 training step on synthetic
256 x 20 x 1 x 224 batches per GPU, bf16 storage + tcgen05 convolutions, fp32 statistics / gradients / weights.
One "step" = forward + BCEWithLogits + backward + (N>1: NCCL gradient all-reduce) + clamp + SGD-Nesterov update,
i.e. everything `run_train_epoch` does per batch (deepards/train_ards_detector.py:139-173) except the host ETL.
N>1 (torchrun): weak scaling, 256 sequences per rank, sequences are independent so there is no other collective.

Printed JSON (rank 0, one line): see the contract in the task statement.  `value` = device-timed throughput with
the inputs already resident in HBM; `e2e` = the same step driven from pinned HOST buffers (H2D of the batch and
D2H of the loss inside the timed region).  `roofline` is measured live with CUDA events around every kernel call
of a few extra steps; `cpu_baseline` times the CPU oracle port on this box's host cores.

--impl reference: times the reference algorithm's CPU implementation (the oracle port of the reference's module
graph; the Python reference itself cannot travel to the GPU box) with all host threads, same metric and config.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark leaves the tree as build() left it: without this its imports that build() does not make
# (deepards_b200.data_parallel, deepards_b200.synthetic, the CPU oracle) would write __pycache__ files there
sys.dont_write_bytecode = True

SEQ_PER_GPU = 256
SUB_BATCH = 20
FLOP_PER_SEQ = {"resnet18": 4.5733e9, "densenet18": 0.66809e9}      # fwd+bwd, SURVEY.md section 8d
FLOP_FWD_PER_SEQ = {"resnet18": 1.5251e9, "densenet18": 0.22337e9}
BYTES_PER_SEQ_BF16 = {"resnet18": 17.29e6, "densenet18": 12.43e6}     # fwd+bwd activation traffic, bf16


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md).  One long-running
    `nvidia-smi -lms 25` process streams a line every 25 ms (starting a new process per sample takes ~100 ms, about as
    long as a short timed region); one process per sample runs next to it in case the stream is block-buffered.
    `mark()` brackets the timed regions: the summary uses the samples taken inside them (all samples if none fell inside)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc, self.windows = index, [], False, None, []

    def _parse(self, line):
        parts = [s.strip() for s in line.strip().split(",")]
        if len(parts) >= 7:
            self.rows.append((time.perf_counter(), parts))

    def _stream(self, cmd):
        try:
            self.proc = subprocess.Popen(cmd + ["-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
                                         bufsize=1)
            for line in self.proc.stdout:
                self._parse(line)
                if self.stop_flag:
                    break
        except Exception:
            pass

    def run(self):
        cmd = ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"]
        threading.Thread(target=self._stream, args=(cmd,), daemon=True).start()   # dense samples, if its output is unbuffered
        while not self.stop_flag:      # and one process per sample (~100 ms each), which always works
            try:
                self._parse(subprocess.run(cmd, capture_output=True, text=True, timeout=5).stdout)
            except Exception:
                pass
            time.sleep(0.05)

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        self.stop_flag = True
        try:
            if self.proc is not None:
                self.proc.terminate()
        except Exception:
            pass
        self.join(timeout=3)

    def window_summary(self, windows):
        """median SM clock and peak power over the samples that fell inside the given (t0, t1) windows"""
        rows = [r for t, r in self.rows if any(a <= t <= b for a, b in windows)]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(r[col].lower().startswith("active") for r in rows):
                reasons.append(name)
        return {"sm_mhz_median": statistics.median(sm) if sm else None, "power_w_max": max(pw) if pw else None,
                "reasons": reasons, "samples": len(rows)}

    def summary(self):
        inside = [r for t, r in self.rows if any(a <= t <= b for a, b in self.windows)]
        rows = inside or [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(r[col].lower().startswith("active") for r in rows):
                reasons.append(name)
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None,
                "reasons": reasons, "samples": len(rows), "samples_in_timed_region": len(inside)}


# ------------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port), also used for cpu_baseline
# ------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(backbone, n_seq, steps, warmup, threads=None):
    """Times `steps` CPU training steps (forward + BCE + backward + SGD update) of the reference algorithm on
    n_seq sequences.  Returns (seq_per_s, ms_per_step, threads)."""
    import torch
    from oracle import cnn_linear_oracle as O
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = O.cnn_linear_state(backbone, seed=0)
    x = O.synthetic_breaths(n_seq, seed=1234)
    t = O.synthetic_targets(n_seq, seed=1234)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, _, grads = O.forward_backward(sd, x, t, clip_val=0.01, running_update=backbone.startswith("resnet"))
        with torch.no_grad():
            for k, g in grads.items():
                sd[k].add_(g + 1e-4 * sd[k], alpha=-1e-3)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return n_seq * len(times) / tot, 1e3 * tot / len(times), threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_seq = 16  # bounded sample of the 256-sequence batch (BASELINE configs[0] shape); ~1 s per step on 8 cores
    v, ms, threads = cpu_reference_steps(args.backbone, n_seq, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "train sequences/sec (20x224 breaths)", "value": v, "unit": "sequences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cpu_sample=n_seq),
        "cpu_baseline": {"value": v, "unit": "sequences/s", "cores": threads, "kind": "port",
                         "sample": "%d of the %d sequences of one batch per step (oracle port of the reference's "
                                   "per-sequence loop, torch CPU fp32)" % (n_seq, SEQ_PER_GPU)},
        "e2e": {"value": v, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args, cpu_sample=None):
    per_gpu = getattr(args, "seq_per_gpu", SEQ_PER_GPU)
    c = {"workload": "cnn_linear %s training step (fwd + BCEWithLogits + bwd + grad all-reduce + clamp + SGD-Nesterov), "
                     "%d x %d x 1 x 224 synthetic breaths per GPU (BASELINE.json configs[1]%s)" %
                     (args.backbone, per_gpu, SUB_BATCH, "; strong scaling: the 256-sequence batch split over the GPUs"
                      if getattr(args, "scaling", "weak") == "strong" else ""),
         "backbone": args.backbone, "sequences_per_gpu": per_gpu, "sub_batch": SUB_BATCH, "precision": "bf16 storage / "
         "tcgen05 convolutions, fp32 statistics, gradients and weights", "parallelism": "dp%d" % args.gpus,
         "wgrad": os.environ.get("DEEPARDS_B200_WGRAD", "accumulate"),
         "cuda_graph": (not args.no_graph) and ("whole step" if args.gpus == 1 else getattr(args, "dp_graph_desc", "per segment, NCCL between")),
         "l2": "working set per step (>1 GB of activations) exceeds the 126 MB L2; 4 resident input batches are rotated"}
    if cpu_sample:
        c["cpu_sample_sequences"] = cpu_sample
    return c


# ------------------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import deepards_b200 as D
    from deepards_b200 import _lib
    from deepards_b200.data_parallel import DataParallelTrainer
    from deepards_b200 import synthetic as O   # workload generator (the CPU checker is only used by cpu_reference_steps)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # the all-reduces overlap the backward pass: keep NCCL to a few CTAs (the trainer sizes the persistent kernels'
        # grids for the SMs that are left, DEEPARDS_B200_DP_SM_RESERVE)
        if os.environ.get("DEEPARDS_B200_NCCL_CHANNELS"):
            os.environ["NCCL_MAX_NCHANNELS"] = os.environ["DEEPARDS_B200_NCCL_CHANNELS"]
        # NCCL prints its version banner on stdout at init; the contract is ONE JSON line there
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()
    strong = args.scaling == "strong"
    seq_per_gpu = SEQ_PER_GPU // world if strong else SEQ_PER_GPU
    if strong and SEQ_PER_GPU % world:
        raise SystemExit("--scaling strong needs %d %% n_gpus == 0" % SEQ_PER_GPU)
    args.seq_per_gpu = seq_per_gpu

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()            # started before the warm-up so that it is streaming by the time the clock starts

    def timed(fn, steps, window=None):
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        t1 = time.perf_counter()
        if sampler is not None:
            sampler.mark(t0, t1)
            if window is not None:
                window.append((t0, t1))
        ms = e0.elapsed_time(e1)
        if world > 1:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms)
        return ms

    def measure(backbone, steps, want_roofline, want_sustained):
        """One backbone: device-timed throughput (resident inputs), e2e (pinned host batches, loss read back), optionally
        a >= 2 s sustained leg and the per-kernel roofline.  Returns (dict, trainer, xs, ts)."""
        torch.manual_seed(0)
        bb = D.resnet18() if backbone == "resnet18" else D.densenet18()
        net = D.CNNLinearNetwork(bb, SUB_BATCH, 0).to(dev)
        net.precision = args.precision
        net.train()
        trainer = DataParallelTrainer(net, lr=1e-3, optimizer="sgd", weight_decay=1e-4, clip_val=0.01,
                                      use_graph=not args.no_graph)
        n_in = 4
        xs_host = [O.synthetic_breaths(seq_per_gpu, seed=1234 + rank * 17 + i).pin_memory() for i in range(n_in)]
        ts_host = [O.synthetic_targets(seq_per_gpu, seed=1234 + rank * 17 + i).pin_memory() for i in range(n_in)]
        xs = [x.to(dev) for x in xs_host]
        ts = [t.to(dev) for t in ts_host]

        def resident_step(i):
            trainer.train_step(xs[i % n_in], ts[i % n_in])

        # e2e: the batch starts in pinned HOST memory.  Like a DataLoader with pin_memory + non_blocking copies
        # (train_ards_detector.py:324-337, 150-152), the copy of batch i+1 is issued on a copy stream while step i runs;
        # the loss of EVERY step is read back to the host (the reference's Meter does, metrics.py:142-153), so each step
        # ends with a stream synchronisation.  H2D and D2H are inside the timed region.
        copy_stream = torch.cuda.Stream(device=dev)
        x_stage = [torch.empty_like(xs[0]) for _ in range(2)]
        t_stage = [torch.empty_like(ts[0]) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        loss_host = torch.zeros(1).pin_memory()

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                x_stage[i % 2].copy_(xs_host[i % n_in], non_blocking=True)
                t_stage[i % 2].copy_(ts_host[i % n_in], non_blocking=True)
                ready[i % 2].record(copy_stream)

        def e2e_step(i):
            cur = torch.cuda.current_stream()
            cur.wait_event(ready[i % 2])
            loss = trainer.train_step(x_stage[i % 2], t_stage[i % 2])
            loss_host.copy_(loss, non_blocking=True)
            prefetch(i + 1)      # overlaps this step's kernels; buffer (i+1)%2 was consumed by step i-1, which is complete
            cur.synchronize()    # the trainer reads the loss every step

        for i in range(max(args.warmup, 3)):
            resident_step(i)
        l0, g0 = lib.dards_launch_count(), trainer.graph_launches
        ms = timed(resident_step, steps)
        launches = (lib.dards_launch_count() - l0) + (trainer.graph_launches - g0)
        if args.dump_outputs and backbone == args.backbone and rank == 0:
            dump_outputs(args.dump_outputs, trainer, trainer.plan_for(xs[0]))
        prefetch(0)
        for i in range(2):
            e2e_step(i)
        ms_e2e = timed(lambda i: e2e_step(2 + i), steps)
        seqs = seq_per_gpu * world * steps
        out = {"value": seqs / (ms / 1e3), "ms_per_step": ms / steps,
               "e2e": {"value": seqs / (ms_e2e / 1e3), "unit": "sequences/s", "ms_per_step": ms_e2e / steps,
                       "h2d_bytes_per_step": int(xs_host[0].numel() * 4 + ts_host[0].numel() * 4), "d2h_bytes_per_step": 4},
               "gpu_launches": int(launches), "final_loss": float(trainer.loss_buf)}
        if want_sustained:
            # >= 2 s of back-to-back steps: the clocks settle under the power cap (the short leg above runs at boost clocks)
            n_sus = max(steps, int(args.sustained_s * 1e3 / (ms / steps)) + 1)
            win = []
            ms_sus = timed(resident_step, n_sus, window=win)
            sus = {"value": seq_per_gpu * world * n_sus / (ms_sus / 1e3), "unit": "sequences/s", "steps": n_sus,
                   "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus}
            if sampler is not None:
                sus.update(sampler.window_summary(win))
            out["sustained"] = sus
        if want_roofline and rank == 0:
            out["roofline"] = kernel_roofline(trainer, xs[0], ts[0], args, backbone)
            ceil = min(out["roofline"]["step_ceiling_seq_per_s"].values())
            out["frac_of_step_ceiling"] = out["value"] / world / ceil
        return out, trainer, xs, ts

    main_bb = args.backbone
    res, trainer, xs, ts = measure(main_bb, args.steps, True, not args.no_extra)
    dp_par = dp_parity(trainer, xs[0], ts[0], args, D, main_bb) if world > 1 and not args.no_extra else None
    other = None
    if not args.no_extra and main_bb == "resnet18":
        # BASELINE.json configs[2]'s backbone (the reference's default, deepards/defaults.yml:18) in the same record
        trainer.close()
        o, tr2, _, _ = measure("densenet18", args.steps, True, False)
        tr2.close()
        other = {"metric": "train sequences/sec (20x224 breaths)", "unit": "sequences/s", "value": o["value"],
                 "ms_per_step": o["ms_per_step"], "e2e": o["e2e"], "gpu_launches": o["gpu_launches"]}
        if "roofline" in o:
            r = o["roofline"]
            other["roofline"] = {k: r[k] for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "share_of_step",
                                                   "step_ceiling_seq_per_s", "breakdown_ms_per_step") if k in r}
            other["frac_of_step_ceiling"] = o.get("frac_of_step_ceiling")
    module_path = module_path_rates(args, D, O, dev) if world == 1 and not args.no_extra else None
    if sampler:
        sampler.stop()
    if world > 1:
        trainer.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world > 1:
        args.dp_graph_desc = ("whole step incl. the bucketed NCCL all-reduces (captured on the communication stream)"
                              if trainer.dp_graph == "whole" else
                              "one graph per backward segment; NCCL all-reduce + optimizer per bucket on the communication stream")
    cpu_v, cpu_ms, cpu_threads = cpu_reference_steps(main_bb, 16, 3, 1) if world == 1 and not args.no_cpu else (None, None, None)
    line = {
        "metric": "train sequences/sec (20x224 breaths)", "value": res["value"], "unit": "sequences/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
        "data": "synthetic", "config": workload_config(args),
        "e2e": res["e2e"], "gpu_launches": res["gpu_launches"],
        "clocks": sampler.summary() if sampler else None,
        "roofline": res.get("roofline"),
        "final_loss": res["final_loss"],
    }
    if "frac_of_step_ceiling" in res:
        line["frac_of_step_ceiling"] = res["frac_of_step_ceiling"]
    if "sustained" in res:
        line["sustained"] = res["sustained"]
    if other is not None:
        line["densenet18"] = other
    if module_path is not None:
        line["module_path"] = module_path
    if dp_par is not None:
        line["dp_parity"] = dp_par
    if cpu_v is not None:
        line["cpu_baseline"] = {"value": cpu_v, "unit": "sequences/s", "cores": cpu_threads, "kind": "port",
                                "sample": "3 steps of 16 sequences (BASELINE configs[0] shape) of the same training step, "
                                          "oracle port of the reference loop, torch CPU fp32, %.0f ms/step" % cpu_ms}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dp_parity(trainer, x, t, args, D, backbone):
    """Data-parallel correctness inside the benchmark record (every rank calls this):
      * max_param_divergence: after all the timed steps, the largest |difference| between any rank's parameters and
        rank 0's (replicas must stay bit-identical: same reduced gradients, same update);
      * grad_vs_single_rank: one more step's REDUCED gradient (sum over ranks / world, before the clamp) against rank 0
        recomputing the gathered global batch in one process with the same weights -- relative error per the whole flat
        buffer and the worst per-tensor cosine."""
    import torch
    import torch.distributed as dist
    from deepards_b200 import engine
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = x.device
    torch.cuda.synchronize()
    ref = trainer.param_flat.clone()
    dist.broadcast(ref, src=0)
    div = (trainer.param_flat - ref).abs().max().reshape(1)
    dist.all_reduce(div, op=dist.ReduceOp.MAX)
    # gradient of one more batch: distributed vs single process
    xs = [torch.empty_like(x) for _ in range(world)]
    tg = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(xs, x)
    dist.all_gather(tg, t)
    plan = trainer.plan_for(x)
    plan.load_input(x)
    plan.run_forward()
    st = plan._stream()
    from deepards_b200 import _lib
    t_flat = t.reshape(-1).contiguous()
    loss = torch.zeros(1, device=dev)
    _lib.call("dards_bce_with_logits", plan.logits.data_ptr(), t_flat.data_ptr(), loss.data_ptr(), plan.dlogits.data_ptr(),
              plan.logits.numel(), 1.0, st)
    plan.run_backward()
    g = plan.grad_flat.clone()
    dist.all_reduce(g, op=dist.ReduceOp.SUM)
    g /= world
    out = {"max_param_divergence": float(div), "ranks": world}
    if rank == 0:
        net = trainer.net
        xg, tgc = torch.cat(xs, 0), torch.cat(tg, 0)
        from deepards_b200.autograd import module_precision
        from deepards_b200.torch_cnn_linear_network import _drop_key
        bb = net.breath_block
        big = engine.Plan(net, bb, net.linear_final, xg.numel() // engine.SEQ_LEN, xg.shape[1], module_precision(net),
                          "cnn_linear", dropout=(), update_running=False)
        # dropout off in both for a deterministic comparison?  The timed plan keeps the network's dropout setting, so
        # compare only when the backbone has none (ResNet); DenseNet reports the divergence check alone
        if not _drop_key(bb):
            big.load_input(xg)
            big.run_forward()
            tf = tgc.reshape(-1).contiguous()
            _lib.call("dards_bce_with_logits", big.logits.data_ptr(), tf.data_ptr(), loss.data_ptr(), big.dlogits.data_ptr(),
                      big.logits.numel(), 1.0, st)
            big.run_backward()
            torch.cuda.synchronize()
            gb = big.grad_flat
            err = float((g - gb).abs().max() / gb.abs().max())
            worst = 1.0
            for n, p in net.named_parameters():
                if id(p) in plan.grad_written and p.numel() >= 64:
                    off = plan.goff[id(p)]
                    a, b = g[off:off + p.numel()].double(), gb[off:off + p.numel()].double()
                    c = float((a @ b) / (a.norm() * b.norm() + 1e-300))
                    worst = min(worst, c)
            out["grad_vs_single_rank"] = {"rel_err": err, "min_tensor_cosine": worst, "global_batch": int(xg.shape[0])}
        del big
    return out


def module_path_rates(args, D, O, dev):
    """The drop-in path as train_ards_detector.py drives it (:139-173, 416-422): net(x) -> BCEWithLogits -> backward ->
    torch.optim.SGD.step(), through the autograd bridge, at fp32 (parity precision) and bf16."""
    import torch
    out = {"unit": "sequences/s", "what": "net(x, None) -> BCEWithLogitsLoss -> backward -> torch.optim.SGD.step() on "
           "256 x 20 x 1 x 224 (the reference trainer's loop over the B200 modules)"}
    x = O.synthetic_breaths(SEQ_PER_GPU, seed=4321).to(dev)
    t = O.synthetic_targets(SEQ_PER_GPU, seed=4321).to(dev)
    for prec in ("bf16", "fp32"):
        torch.manual_seed(0)
        net = D.CNNLinearNetwork(D.resnet18() if args.backbone == "resnet18" else D.densenet18(), SUB_BATCH, 0).to(dev)
        net.precision = prec
        net.train()
        opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
        crit = torch.nn.BCEWithLogitsLoss()
        for p in net.parameters():
            p.register_hook(lambda g: torch.clamp(g, -0.01, 0.01))   # train_ards_detector.py:474-476

        def one():
            opt.zero_grad()
            loss = crit(net(x, None), t)
            loss.backward()
            opt.step()

        n = 10 if prec == "bf16" else 4
        for _ in range(3):
            one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            one()
        e1.record()
        torch.cuda.synchronize()
        out[prec] = SEQ_PER_GPU * n / (e0.elapsed_time(e1) / 1e3)
        del net, opt
    return out


def kernel_roofline(trainer, x, t, args, backbone, steps=3):
    """CUDA-event time of every recorded kernel call over a few steps, grouped by entry point.  Returns the
    roofline object of the dominant kernel class plus the per-class breakdown."""
    import torch
    plan = trainer.plan_for(x)
    P = peaks()
    st = torch.cuda.current_stream()
    agg = {}
    for _ in range(steps):
        plan.load_input(x)
        for rec in (plan.pack, plan.fwd, plan.bwd):
            evs = []
            for name, f, a in rec.calls:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                rc = f(*a, st.cuda_stream)
                e1.record(st)
                if rc != 0:
                    raise RuntimeError(name)
                evs.append((name, a, e0, e1))
            torch.cuda.synchronize()
            for name, a, e0, e1 in evs:
                key = name
                if name in ("dards_conv1d_fwd", "dards_conv1d_dgrad", "dards_conv1d_wgrad"):
                    key = name + (":tcgen05" if (a[-1] & 0xff) == 1 else ":simt")
                d = agg.setdefault(key, {"ms": 0.0, "launches": 0, "flops": 0.0, "bytes": 0.0})
                d["ms"] += e0.elapsed_time(e1)
                d["launches"] += 1
                esz = 2 if args.precision == "bf16" else 4
                if name == "dards_conv1d_fwd" or name == "dards_conv1d_dgrad":
                    n, l_in, l_out, cin, cout, k = a[4], a[5], a[6], a[7], a[8], a[12]
                    d["flops"] += 2.0 * n * l_out * cin * cout * k
                    d["bytes"] += esz * n * (l_in * cin + l_out * cout)
                elif name == "dards_conv1d_wgrad":
                    n, l_in, l_out, cin, cout, k = a[6], a[7], a[8], a[9], a[10], a[13]
                    d["flops"] += 2.0 * n * l_out * cin * cout * k
                    d["bytes"] += esz * n * (l_in * cin + l_out * cout)
                elif name == "dards_conv1d_wgrad_accum":
                    n, l_in, l_out, cin, cout, k = a[3], a[4], a[5], a[6], a[7], a[10]
                    d["flops"] += 2.0 * n * l_out * cin * cout * k
                    d["bytes"] += esz * n * (l_in * cin + l_out * cout)
                elif name == "dards_conv1d_bn_fwd":
                    # convolution + BatchNorm in one kernel: reads the input, writes y (kept for the backward) and, when the
                    # whole normalisation runs in the epilogue, the activation (+ reads the residual)
                    n, l_in, l_out, cin, cout, k = a[10], a[12], a[13], a[14], a[15], a[20]
                    d["flops"] += 2.0 * n * l_out * cin * cout * k
                    d["bytes"] += esz * n * (l_in * cin + l_out * cout * (1 + (1 if a[3] else 0) + (1 if a[4] else 0)))
                elif name == "dards_gbn_apply_fwd":
                    g, rows, c = a[16], a[17], a[18]
                    d["bytes"] += esz * g * rows * c * (2 + (1 if a[2] else 0) + (1 if a[9] else 0))
                elif name == "dards_gbn_fwd":
                    # algorithmic traffic: x read once, out written once (+ the residual read)
                    g, rows, c = a[7], a[8], a[9]
                    d["bytes"] += esz * g * rows * c * (2 + (1 if a[2] else 0))
                elif name == "dards_gbn_bwd":
                    # dout and x read once, dx written once (+ mask read, + residual-gradient write, + dx read when accumulating)
                    g, rows, c = a[12], a[13], a[14]
                    d["bytes"] += esz * g * rows * c * (3 + (1 if a[2] else 0) + (1 if a[9] else 0) + (1 if a[8] else 0))
        plan.fwd_serial += 1
        plan.bwd_serial = plan.fwd_serial
    total_ms = sum(d["ms"] for d in agg.values())
    top = max(agg.items(), key=lambda kv: kv[1]["ms"])
    name, d = top
    out = {"kernel": name, "share_of_step": d["ms"] / total_ms, "launches_per_step": d["launches"] / steps,
           "avg_launch_ms": d["ms"] / d["launches"], "traffic": None,
           "breakdown_ms_per_step": {k: round(v["ms"] / steps, 4) for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}}
    if d["flops"] > 0:
        ach = d["flops"] / (d["ms"] / 1e3) / 1e12
        out.update({"bound": "tensor", "achieved": ach, "peak": P["tf_sustained"], "unit": "TFLOP/s",
                    "frac": ach / P["tf_sustained"], "peak_source": P["src"] + " bf16 sustained (kernel timed inside a long step)"})
    else:
        ach = d["bytes"] / (d["ms"] / 1e3) / 1e9 if d["bytes"] > 0 else None
        out.update({"bound": "hbm", "achieved": ach, "peak": P["hbm"], "unit": "GB/s",
                    "frac": ach / P["hbm"] if ach else None, "peak_source": P["src"] + " copy bandwidth"})
    # measured DRAM traffic per launch of that kernel from the committed `ncu --set full` capture, if there is one
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        out["traffic"] = json.load(open(tpath)).get(backbone, {}).get(name)
    out["per_kernel"] = {}
    for k, v in agg.items():
        e = {"ms_per_step": round(v["ms"] / steps, 4), "launches_per_step": v["launches"] / steps}
        if v["flops"] > 0:
            e["tflops"] = round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1)
            e["frac_of_tensor_peak"] = round(e["tflops"] / P["tf_sustained"], 3)
        if v["bytes"] > 0:
            e["algorithmic_gbs"] = round(v["bytes"] / (v["ms"] / 1e3) / 1e9, 1)
            e["frac_of_hbm_peak"] = round(e["algorithmic_gbs"] / P["hbm"], 3)
        out["per_kernel"][k] = e
    # whole-step view against the algorithmic ceilings of SURVEY.md section 8d
    conv_ms = sum(v["ms"] for k, v in agg.items() if k.startswith("dards_conv1d")) / steps
    conv_fl = sum(v["flops"] for k, v in agg.items() if k.startswith("dards_conv1d")) / steps
    out["conv_tflops_all"] = conv_fl / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else None
    out["conv_share_of_step"] = conv_ms / (total_ms / steps)
    out["step_ceiling_seq_per_s"] = {"tensor": P["tf_sustained"] * 1e12 / FLOP_PER_SEQ[backbone],
                                     "hbm": P["hbm"] * 1e9 / BYTES_PER_SEQ_BF16[backbone]}
    return out


def dump_outputs(outdir, trainer, plan):
    """--dump-outputs: what the last timed step computed, as float32 DIR/<name>.npy, so that two builds can be compared
    output for output on the same seeded inputs: the loss it returned, the logits of its forward pass and, concatenated
    in named_parameters() order, its gradients (before the clamp) and the parameters after its update (31 MB for
    ResNet-18).  Unless DEEPARDS_B200_WGRAD is set, main() runs such a benchmark with the fixed-order weight-gradient
    reduction, so the files are the same bit for bit from run to run."""
    import numpy as np
    import torch
    params = [p for _, p in trainer.net.named_parameters()]
    arrays = {"loss": trainer.loss_buf, "logits": plan.logits,
              "grads": torch.cat([plan.grad_view(p).reshape(-1) for p in params]),
              "params": torch.cat([p.detach().reshape(-1) for p in params])}
    assert sum(a.numel() for a in arrays.values()) * 4 <= 64 << 20
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--backbone", default="resnet18", choices=["resnet18", "densenet18"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="issue every kernel from Python instead of one CUDA graph")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 256 sequences per GPU; strong: the 256-sequence batch split over the GPUs (SURVEY 8d C3)")
    ap.add_argument("--no-extra", action="store_true",
                    help="only the headline legs: no sustained leg, no densenet18 / module_path / dp_parity sub-objects")
    ap.add_argument("--sustained-s", type=float, default=2.5, help="length of the sustained leg in seconds")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, logits, gradients and updated parameters of the last timed step as DIR/<name>.npy; "
                         "unless DEEPARDS_B200_WGRAD is set, the run then sums weight gradients in a fixed order "
                         "(DEEPARDS_B200_WGRAD=deterministic), so that repeated runs write identical files.  With the "
                         "default arrival-order sums (DEEPARDS_B200_WGRAD=accumulate) two runs drift apart over the "
                         "warm-up and timed steps")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.dump_outputs:
        # Outputs that can be compared need a step that computes the same thing every run.  The default weight-gradient
        # kernels add their fp32 tiles in the L2 in arrival order; one step is reproducible to rounding, but the warm-up
        # and timed steps of bf16 training can amplify those differences far beyond it (pairs of --warmup 5 --steps 20
        # runs with DEEPARDS_B200_WGRAD=accumulate on a B200 at 1000 W: some agreed to 2e-8, one ended with logits 7 %
        # of their largest value apart).  The
        # fixed-order split-K reduction is bit-reproducible and slower (INTEGRATION.md, DEEPARDS_B200_WGRAD); the
        # timings of the run are of the reduction config.wgrad names.
        os.environ.setdefault("DEEPARDS_B200_WGRAD", "deterministic")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

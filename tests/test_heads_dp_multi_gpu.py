"""GPU (needs 2 devices; skipped on a 1-GPU box): the generic data-parallel step of the torch heads over NCCL, a 3 + 2
ragged split, eager and per-segment CUDA graphs, against a single process on the whole batch.  The sequence heads'
BatchNorm statistics are per sequence, so sharding is exact.  The regressor normalises each rank's flat shard as one
BatchNorm group, as each nn.DataParallel replica does: its reference is the module path run on the two shards one after
the other, with the loss as the global mean."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, kind, use_graph, q):
    import torch.distributed as dist
    from deepards_b200.data_parallel import DataParallelTrainer, shard_bounds
    from tests.test_heads_trainer_gpu import _batch, _clamp_hooks, _criterion, _make, _out
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    solo = dist.new_group([0])          # collective call on every rank; only rank 0 is a member
    crit = _criterion(kind)
    batches = [_batch(kind, 5, 800 + i) for i in range(4)]
    unit = 20 if kind == "regressor" else 1      # rows of x per sequence
    tr = DataParallelTrainer(_make(kind, seed=21), lr=1e-2, clip_val=0.01, use_graph=use_graph, criterion=crit)
    losses = []
    b, e = shard_bounds(5, world, rank)          # 3 + 2 sequences
    for i in range(5):
        x, t = batches[i % 4]
        losses.append(float(tr.train_step(x[b * unit:e * unit], t[b * unit:e * unit], global_batch=5 * unit)))
    res = {"rank": rank, "params": tr.param_flat.cpu(), "losses": losses, "n": e - b}
    if rank == 0:
        if kind == "regressor":
            net = _make(kind, seed=21)
            _clamp_hooks(net)
            opt = torch.optim.SGD(net.parameters(), lr=1e-2, momentum=0.9, weight_decay=1e-4, nesterov=True)
            ref_losses = []
            for i in range(5):
                x, t = batches[i % 4]
                opt.zero_grad()
                loss = 0.0
                for r in range(world):
                    lo, hi = shard_bounds(5, world, r)
                    loss = loss + crit(_out(net(x[lo * unit:hi * unit], None)), t[lo * unit:hi * unit]) * (hi - lo) / 5.0
                loss.backward()
                opt.step()
                ref_losses.append(float(loss))
            ref_params = torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu()
            res["params"] = torch.cat([p.detach().reshape(-1) for p in tr.net.parameters()]).cpu()
        else:
            ref = DataParallelTrainer(_make(kind, seed=21), lr=1e-2, clip_val=0.01, group=solo, use_graph=False,
                                      criterion=crit)
            assert ref.world == 1
            ref_losses = [float(ref.train_step(*batches[i % 4])) for i in range(5)]
            ref_params = ref.param_flat.cpu()
        res["ref_params"], res["ref_losses"] = ref_params, ref_losses
    else:
        if kind == "regressor":
            res["params"] = torch.cat([p.detach().reshape(-1) for p in tr.net.parameters()]).cpu()
    q.put(res)
    dist.barrier()
    tr.close()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind,use_graph", [("transformer", False), ("transformer", True), ("lstm", False),
                                            ("lstm", True), ("to_mean", True), ("regressor", False),
                                            ("regressor", True)])
def test_two_rank_head_step_equals_single_process_step(kind, use_graph):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, use_graph, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=600) for _ in procs), key=lambda r: r["rank"])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    r0, r1 = res
    assert torch.equal(r0["params"], r1["params"])                    # replicas stay identical
    combined = [(l0 * r0["n"] + l1 * r1["n"]) / 5 for l0, l1 in zip(r0["losses"], r1["losses"])]
    diffs = [abs(lc - lr) for lc, lr in zip(combined, r0["ref_losses"])]
    # as in test_dp_multi_gpu.py: step 1 runs on identical weights, later steps compare two fp32 trajectories whose
    # gradients differ in summation order
    assert diffs[0] <= 1e-6 * max(1.0, abs(r0["ref_losses"][0])), diffs
    assert max(diffs) <= 1e-4 * max(1.0, max(abs(v) for v in r0["ref_losses"])), (diffs, combined, r0["ref_losses"])
    ref = r0["ref_params"]
    err = float((r0["params"] - ref).abs().max() / ref.abs().max())
    assert err <= 1e-4, err
    print("%s graph=%s: 2-rank vs single-process: loss |diff| per step %s, parameters after 5 steps rel err %.2e" %
          (kind, use_graph, " ".join("%.1e" % d for d in diffs), err))

"""Data-parallel training step: one process per GPU, NCCL all-reduce of the flat gradient buffer.

Replaces `nn.DataParallel(model).cuda()` (deepards/train_ards_detector.py:93-96), which the reference's author
notes is effectively unusable (:198-203).  Semantics kept from that path (SURVEY.md section 8e):

  * the batch is split on dim 0; every sequence's forward/backward (incl. its BatchNorm statistics) is independent
    of every other sequence, so sharding is exact and the ONLY collective is the gradient all-reduce;
  * the loss is the mean over the GLOBAL batch: each rank back-propagates its local mean and the reduced gradient
    is scaled by 1/world_size;
  * the reference's gradient clamp (`p.register_hook(clamp)`, :474-476) acts on the REDUCED gradient under
    DataParallel, so here it is applied after the all-reduce, fused with the optimizer update
    (SGD-Nesterov momentum 0.9 / Adam, :416-422) in one kernel over the flat buffers;
  * parameters that never receive a gradient (ResNet's conv1_alt/conv2/bn2; frozen parameters) are left out of
    the update, exactly like torch.optim skipping `p.grad is None`.

Every head of the package trains here.  CNNLinearNetwork and CNNSingleBreathLinearNetwork with the default
BCEWithLogits loss run the fused plan (linear head and loss in the recorded kernels).  Every other head, and those two
with a caller-supplied `criterion`, run the generic step: the backbone plan forward, the head's own torch arithmetic
(`net._head`, the code its forward() runs) and the criterion under autograd, their gradients written into the flat
gradient buffer, then the backbone plan backward and the same reduction and update.  CNNRegressor takes a flat batch of
breaths (N, 1, 224); its BatchNorm group is the rank's whole flat batch, i.e. each rank normalises its own shard, as
each nn.DataParallel replica normalises its own chunk.

The gradient buffer is reduced in buckets, last layers first, on a communication stream that waits on events
recorded inside the backward pass, so the reduction of layer4's 11.5 MB overlaps the backward of layers 1-3.
"""
import os

import torch
import torch.distributed as dist

from . import _lib, engine


def param_layout(net):
    """[(name, param, offset)] and total length of the flat fp32 buffers (16-byte aligned slots)."""
    out, off = [], 0
    for n, p in net.named_parameters():
        out.append((n, p, off))
        off += (p.numel() + 3) // 4 * 4
    return out, off


def shard_bounds(batch, world, rank):
    """[begin, end) of this rank's sequences: contiguous, remainder to the first ranks."""
    base, rem = divmod(batch, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def sharded_map(fn, x, group=None):
    """Inference / GradCAM over several GPUs (SURVEY.md 8e: replicas only, no data-path collective): this rank runs
    `fn` on its contiguous shard of the sequences in `x` (dim 0), and the per-sequence results of all ranks are
    gathered in order.  `fn(x_shard)` returns a tensor, or a tuple of tensors, with one leading row per sequence;
    every rank gets the full result(s).  Shards may be ragged or empty (B < world)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return fn(x)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    b, e = shard_bounds(x.shape[0], world, rank)
    out = fn(x[b:e])
    single = not isinstance(out, (tuple, list))
    outs = [out] if single else list(out)
    sizes = [shard_bounds(x.shape[0], world, r) for r in range(world)]
    gathered = []
    rows = max(hi - lo for lo, hi in sizes)
    for t in outs:
        # ragged shards: pad to the largest shard (at most one extra row), gather equal-sized parts, trim
        mine = torch.zeros((rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        mine[:t.shape[0]].copy_(t)
        parts = [torch.empty_like(mine) for _ in sizes]
        dist.all_gather(parts, mine, group=group)
        gathered.append(torch.cat([p[:hi - lo] for p, (lo, hi) in zip(parts, sizes)], 0))
    return gathered[0] if single else tuple(gathered)


def live_ranges(layout, live_ids):
    """Merge the flat slots of the parameters in `live_ids` into maximal contiguous [begin, end) ranges."""
    ranges = []
    for _, p, off in layout:
        if id(p) not in live_ids:
            continue
        end = off + (p.numel() + 3) // 4 * 4
        if ranges and ranges[-1][1] == off:
            ranges[-1][1] = end
        else:
            ranges.append([off, end])
    return [tuple(r) for r in ranges]


def make_buckets(total, cut_points, min_elems):
    """Split [0, total) at the given candidate offsets (descending readiness order: a suffix of the buffer is
    complete first) into buckets of at least `min_elems`, returned last-first."""
    cuts = sorted(set(c for c in cut_points if 0 < c < total), reverse=True)
    buckets, end = [], total
    for c in cuts:
        if end - c >= min_elems:
            buckets.append((c, end))
            end = c
    if end > 0:
        buckets.append((0, end))
    return buckets


class BucketedAllReduce(object):
    """Sum-all-reduce of slices of one flat tensor, issued asynchronously per bucket."""

    def __init__(self, group=None):
        self.group = group
        self.handles = []

    def reduce(self, flat, begin, end):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            self.handles.append(dist.all_reduce(flat[begin:end], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def reduce_now(self, flat, begin, end):
        """All-reduce ordered on the CURRENT stream: work issued to it afterwards (the bucket's optimizer update) sees the
        reduced values; the host does not block."""
        if os.environ.get("DEEPARDS_B200_DP_NO_ALLREDUCE") == "1":
            return   # measurement only: the step's structure without the collective (replicas diverge)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            dist.all_reduce(flat[begin:end], op=dist.ReduceOp.SUM, group=self.group)

    def wait(self):
        for h in self.handles:
            h.wait()
        self.handles = []


def head_backbone_plan(net, x, bn_rule, update_running, input_grad=False):
    """The "backbone" plan that runs a head's backbone when the head's own arithmetic (`net._head`) stays in torch: the
    trainer's generic step and saliency.input_gradients.  Its owner is the head module, so its grad_flat has the slot table
    of param_layout(net), the head's parameters included.  BatchNorm group: the sequence (x.shape[1]), or for CNNRegressor
    the whole flat batch.  bn_rule(backbone) -> the plan's bn ('train' / 'frozen'); dropout follows the backbone's
    training flag."""
    bb = net.breath_block
    from .torch_cnn_linear_network import CNNDoubleLinearNetwork, CNNLinearNetwork, CNNRegressor, _drop_key
    from .autograd import module_precision
    if x.shape[-1] != engine.SEQ_LEN:
        raise Exception('input breaths must have sequence length of 224')
    n = x.numel() // engine.SEQ_LEN
    group = n if isinstance(net, CNNRegressor) else x.shape[1]
    want = {CNNLinearNetwork: group * bb.n_out_filters, CNNDoubleLinearNetwork: 2 * group}.get(type(net))
    if want is not None and net.linear_final.in_features != want:
        raise NotImplementedError("deepards_b200: metadata_features > 0 is not implemented (linear_final expects %d "
                                  "features, the head provides %d)" % (net.linear_final.in_features, want))
    training = bb.training
    bn = bn_rule(bb)
    return engine.get_plan(net, bb, None, n, group, module_precision(net), "backbone",
                           dropout=_drop_key(bb) if training else (), update_running=update_running, bn=bn,
                           input_grad=input_grad)


class _HeadCall(torch.nn.Module):
    """forward(feat) = net._head(feat): lets torch.func.functional_call run the head on substitute parameters."""

    def __init__(self, net):
        super(_HeadCall, self).__init__()
        self.net = net

    def forward(self, feat):
        return self.net._head(feat)


class DataParallelTrainer(object):
    """criterion: any callable (outputs, target) -> scalar tensor, given what the module's forward returns ((B, 2),
    (B, S, 2), the LSTM's per-step outputs without its state, the regressor's (N, n_final_features)).  None means
    nn.BCEWithLogitsLoss(), the reference's default; on CNNLinearNetwork / CNNSingleBreathLinearNetwork it keeps the
    fused plan with the loss kernel."""

    def __init__(self, net, lr=1e-3, optimizer="sgd", momentum=0.9, weight_decay=1e-4, clip_val=0.01, group=None,
                 bucket_mb=1.0, use_graph=False, criterion=None):
        if optimizer not in ("sgd", "adam"):
            raise ValueError("optimizer must be 'sgd' or 'adam'")
        from .torch_cnn_linear_network import CNNLinearNetwork, CNNRegressor, CNNSingleBreathLinearNetwork, _HeadBase
        if not isinstance(net, _HeadBase) or not hasattr(net, "_head"):
            raise TypeError("DataParallelTrainer trains the heads of deepards_b200 (registry.network_heads), not %s"
                            % type(net).__name__)
        self.fused = criterion is None and isinstance(net, (CNNLinearNetwork, CNNSingleBreathLinearNetwork))
        self.criterion = torch.nn.BCEWithLogitsLoss() if criterion is None else criterion
        self.flat_batch = isinstance(net, CNNRegressor)     # (N, 1, 224) breaths, one BatchNorm group per rank
        self.use_graph = use_graph
        # world > 1: "segments" (default) replays one graph per backward segment with the NCCL calls issued from the host
        # in between.  "whole" (opt-in, experimental) captures the entire step INCLUDING the bucketed NCCL all-reduces
        # (issued on the communication stream, which joins the capture through the same events that order it in eager
        # mode) in one CUDA graph: measured no faster at 2 GPUs (164.6 k vs ~165 k seq/s) and the processes hang in
        # destroy_process_group() at exit with torch 2.11 / NCCL 2.28, so it is not the default.
        self.dp_graph = os.environ.get("DEEPARDS_B200_DP_GRAPH", "segments")
        self.graph_launches = 0  # kernels launched through CUDA-graph replays (not seen by dards_launch_count)
        self.net, self.lr, self.optimizer = net, lr, optimizer
        self.momentum, self.weight_decay = momentum, weight_decay
        self.clip = float(clip_val) if clip_val else 0.0
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.bucket_elems = int(bucket_mb * (1 << 20) / 4)
        self.step_count = 0
        self._flatten()
        self.comm_stream = torch.cuda.Stream(device=self.device) if self.world > 1 else None
        self.reducer = BucketedAllReduce(group)
        if self.world > 1:
            # With an OVERLAPPED schedule (several buckets, DEEPARDS_B200_DP_BUCKET_ELEMS) leave a few SMs to the NCCL kernels
            # that run next to the backward pass: every persistent kernel here launches one CTA per SM, and with some SMs
            # held by NCCL its last CTAs would run as a second wave (8 x B200: 3.006 ms without, 2.964 ms with 8 reserved).
            # The default single-bucket schedule reduces after the backward and needs no reservation.
            reserve = int(os.environ.get("DEEPARDS_B200_DP_SM_RESERVE", "0"))
            sms = torch.cuda.get_device_properties(self.device).multi_processor_count
            if 0 < reserve < sms:
                _lib.call("dards_set_sm_limit", sms - reserve)
        self.loss_buf = torch.zeros(1, dtype=torch.float32, device=self.device)
        backbone = set(id(p) for p in net.breath_block.parameters())
        self.head_named = [("net." + n, p) for n, p, _ in self.layout if id(p) not in backbone and p.requires_grad]
        self.head_params = [p for _, p in self.head_named]
        self._head_call = _HeadCall(net)

    # ---- flat parameter / optimizer-state buffers (same slot table as Plan.grad_flat) ----------------------
    def _flatten(self):
        layout, total = param_layout(self.net)
        p0 = layout[0][1]
        self.device = p0.device
        if self.device.type != "cuda":
            raise RuntimeError("DataParallelTrainer needs the network on a CUDA device")
        flat = torch.zeros(max(total, 4), dtype=torch.float32, device=self.device)
        for _, p, off in layout:
            flat[off:off + p.numel()].copy_(p.data.reshape(-1))
            p.data = flat[off:off + p.numel()].view(p.shape)
        self.layout, self.total, self.param_flat = layout, total, flat
        self.state1 = torch.zeros_like(flat)
        self.state2 = torch.zeros_like(flat) if self.optimizer == "adam" else None
        if self.world > 1:
            dist.broadcast(self.param_flat, src=0, group=self.group)  # DataParallel broadcasts device-0 weights

    def plan_for(self, x):
        if not self.fused:
            return self._generic_plan(x)
        net = self.net
        bb = net.breath_block
        from .torch_cnn_linear_network import CNNSingleBreathLinearNetwork, _drop_key
        mode = "per_breath" if isinstance(net, CNNSingleBreathLinearNetwork) else "cnn_linear"
        n = x.numel() // engine.SEQ_LEN
        training = bb.training
        bn = self._bn_mode(bb)
        from .autograd import module_precision
        plan = engine.get_plan(net, bb, net.linear_final, n, x.shape[1], module_precision(net), mode,
                               dropout=_drop_key(bb) if training else (), update_running=training, bn=bn)
        if getattr(plan, "_dp_ranges", None) is None:
            live = set(i for i in plan.grad_written
                       if any(id(p) == i and p.requires_grad for _, p, _ in self.layout))
            plan._dp_ranges = live_ranges(self.layout, live)
            plan._dp_buckets = make_buckets(self.total, [off for off, _ in plan.bwd_marks], self.bucket_elems)
        return plan

    @staticmethod
    def _bn_mode(bb):
        # the same rule as the autograd path (autograd.run_plan, engine.bn_mode): batch statistics, or frozen running
        # statistics when every BatchNorm layer of a ResNet in train() is in eval(); mixed states raise
        bn = engine.bn_mode(bb)
        if bn == "eval":
            # a ResNet in eval() is inference only (its backward raises on the autograd path as well)
            raise NotImplementedError("deepards_b200: DataParallelTrainer trains a ResNet in train() mode only (BatchNorm "
                                      "layers all in train(), or all in eval() to fine-tune with frozen statistics); "
                                      "this one is in eval()")
        return bn

    def _generic_plan(self, x):
        """The backbone plan of the generic step (head_backbone_plan)."""
        plan = head_backbone_plan(self.net, x, self._bn_mode, self.net.breath_block.training)
        if getattr(plan, "_dp_buckets", None) is None:
            # the head's slots come last in named_parameters() order: they are in the first (suffix) bucket, which is
            # complete before the backbone backward starts
            plan._dp_buckets = make_buckets(self.total, [off for off, _ in plan.bwd_marks], self.bucket_elems)
        # _dp_ranges: set by the first _head_step, which sees which head parameters get a gradient
        return plan

    def _static_target(self, plan, target):
        """The generic step's target, copied into a per-plan device buffer (captured CUDA graphs read it there).  A
        target of another shape or dtype gets a new buffer and drops the graphs that read the old one."""
        t = plan.__dict__.get("_dp_target")
        if t is None or t.shape != target.shape or t.dtype != target.dtype:
            plan.__dict__.pop("_dp_graph", None)
            plan.__dict__.pop("_dp_seg", None)
            t = plan._dp_target = torch.empty(target.shape, dtype=target.dtype, device=self.device)
        t.copy_(target, non_blocking=True)
        return t

    def _head_step(self, plan, target):
        """Generic step, between the backbone forward and backward: the head's torch arithmetic on the pooled features,
        the criterion, and their backward.  The feature gradient goes to plan.dfeat, each head parameter's gradient to
        its slot of plan.grad_flat; the loss is back-propagated with the weight gs = world * B_local / global_batch, as
        dards_bce_with_logits scales dlogits on the fused path."""
        feat = plan.feat.detach()          # (N, F)
        if not self.flat_batch:
            feat = feat.view(plan.G, plan.group, -1)
        feat.requires_grad_(True)
        # fresh leaves over the parameters' storage every step: a head that keeps part of its last autograd graph alive
        # (the transformer's attention map) would otherwise hand a parameter's AccumulateGrad node, created on the stream
        # of an eager step, to the CUDA-graph capture of a later one, and the capture fails
        leaves = dict((n, p.detach().requires_grad_(True)) for n, p in self.head_named)
        params = list(leaves.values())
        with torch.enable_grad():
            out = torch.func.functional_call(self._head_call, leaves, (feat,), strict=False, tie_weights=False)
            if isinstance(out, tuple):      # CNNLSTMNetwork: (per-step outputs, (hx, cx))
                out = out[0]
            loss = self.criterion(out, target)
            if loss.numel() != 1:
                raise ValueError("criterion must return a scalar loss, got shape %s" % (tuple(loss.shape),))
            gs = plan.__dict__.get("_dp_grad_scale", 1.0)
            grads = torch.autograd.grad(loss, [feat] + params, grad_outputs=torch.full_like(loss, gs), allow_unused=True)
        self.loss_buf.copy_(loss.detach().reshape(1))
        plan.dfeat.copy_(grads[0].reshape(plan.dfeat.shape))
        for (_, p), g in zip(self.head_named, grads[1:]):
            if g is not None:
                plan.grad_view(p).copy_(g)
        if plan.__dict__.get("_dp_ranges") is None:
            live = set(i for i in plan.grad_written if any(id(p) == i and p.requires_grad for _, p, _ in self.layout))
            live.update(id(p) for (_, p), g in zip(self.head_named, grads[1:]) if g is not None)
            plan._dp_ranges = live_ranges(self.layout, live)

    def train_step(self, x, target, global_batch=None):
        """x: this rank's (B_local, 20, 1, 224) on the device (CNNRegressor: (N_local, 1, 224) breaths), target what the
        criterion takes ((B_local, 2) for the default loss of the sequence-level heads).  Returns the device tensor
        holding the local mean loss (no host synchronisation).
        global_batch: total number of sequences over all ranks.  The reference's DataParallel computes ONE mean loss over
        the gathered outputs (train_ards_detector.py:153-163); with equal shards that is the mean of the ranks' local means
        (the default), with a ragged split (last batch of an epoch) pass the global size and every rank's gradient is
        weighted by its share, B_local / global_batch."""
        return self._train_step(x, target, None, global_batch)

    def train_step_raw(self, raw, target, mu, std, padded=False, global_batch=None):
        """The same step fed with RAW float64 / float32 windows on the device: the dataset's `(data - mu) / std` +
        `.float()` (dataset.py:1375-1379) runs as the plan's input load, so the host pipeline only has to hand over
        the stored windows (SURVEY.md 8f-2)."""
        return self._train_step(raw, target, (mu, std, padded), global_batch)

    def _train_step(self, x, target, scaling, global_batch=None):
        with engine.nvtx_range("deepards_b200.train_step"):
            return self._train_step_impl(x, target, scaling, global_batch)

    def _train_step_impl(self, x, target, scaling, global_batch=None):
        plan = self.plan_for(x)
        # dlogits carries world * B_local / B_global, the update 1 / world: together the global-mean weighting
        gs = 1.0 if global_batch is None else self.world * x.shape[0] / float(global_batch)
        # lr / momentum / weight decay / clip are kernel arguments, i.e. constants of a captured CUDA graph: when the caller
        # changes one (lr decay, warm-up) the captured graphs are dropped and re-captured with the new values
        hp = (self.lr, self.momentum, self.weight_decay, self.clip)
        if plan.__dict__.setdefault("_dp_hp", hp) != hp:
            plan.__dict__.pop("_dp_graph", None)
            plan.__dict__.pop("_dp_seg", None)
            plan._dp_hp = hp
        if plan.__dict__.setdefault("_dp_grad_scale", gs) != gs:
            raise RuntimeError("deepards_b200: this plan (%d sequences per rank) was first used with a different global "
                               "batch size; the loss scale is part of its captured CUDA graphs" % x.shape[0])
        if plan.dropout and self.world > 1:
            # dropout masks are keyed by the global sequence index: same masks whatever the number of ranks
            first = shard_bounds(int(global_batch), self.world, self.rank)[0] if global_batch is not None else self.rank * x.shape[0]
            plan.set_sequence_offset(first)
        if scaling is None:
            plan.load_input(x)
        else:
            plan.load_raw(x, *scaling)
        if self.fused:
            t_static = plan.__dict__.get("_dp_target")
            if t_static is None:
                t_static = plan._dp_target = torch.empty((plan.logits.numel(),), dtype=torch.float32, device=self.device)
            t_static.copy_(target.reshape(-1), non_blocking=True)
        else:
            t_static = self._static_target(plan, target)
        if self.use_graph and self.world == 1 and self.optimizer == "sgd":
            return self._graphed_step(plan, t_static)
        if self.use_graph and self.world > 1 and self.optimizer == "sgd":
            if self.dp_graph == "whole" and self.fused:
                try:
                    return self._graphed_step(plan, t_static)
                except RuntimeError as e:       # NCCL under stream capture refused: replay per segment instead
                    import warnings
                    warnings.warn("deepards_b200: whole-step CUDA graph with NCCL failed (%s); using per-segment graphs" % e)
                    self.dp_graph = "segments"
                    plan.__dict__.pop("_dp_graph", None)
                    torch.cuda.synchronize(self.device)
            return self._segment_graphed_step(plan, t_static)
        self._step_body(plan, t_static)
        return self.loss_buf

    def _step_body(self, plan, t_static):
        st = plan._stream()
        plan.run_forward()
        if self.fused:
            _lib.call("dards_bce_with_logits", plan.logits.data_ptr(), t_static.data_ptr(), self.loss_buf.data_ptr(),
                      plan.dlogits.data_ptr(), plan.logits.numel(), plan.__dict__.get("_dp_grad_scale", 1.0), st)
        else:
            self._head_step(plan, t_static)
        if self.world > 1:
            self.step_count += 1
            self._backward_overlapped(plan)   # all-reduce + optimizer per bucket, on the communication stream
            plan._packed_version = None
        else:
            plan.run_backward()
            self._update(plan, st)

    def _graphed_step(self, plan, t_static):
        """The SGD step as ONE CUDA-graph launch (weight packing, forward, loss, backward, update: ~200 kernel
        launches otherwise issued from Python; with more than one rank also the overlapped NCCL all-reduces, captured
        on the communication stream).  Captured lazily on the third call for a plan, after the eager warm-up
        steps have initialised every lazily-set function attribute, the momentum buffers and the NCCL communicator."""
        st = plan.__dict__.setdefault("_dp_graph", {"calls": 0, "graph": None, "launches": 0})
        if st["graph"] is not None:
            st["graph"].replay()
            self.step_count += 1
            plan.fwd_serial += 1
            plan.bwd_serial = plan.fwd_serial
            self.graph_launches += st["launches"]
            return self.loss_buf
        st["calls"] += 1
        if st["calls"] < 3 or self.step_count < 1:
            self._step_body(plan, t_static)
            return self.loss_buf
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        l0 = _lib.load().dards_launch_count()
        with torch.cuda.graph(g):
            plan._packed_version = None
            self._step_body(plan, t_static)
        st["launches"] = int(_lib.load().dards_launch_count() - l0)
        st["graph"] = g
        # capture does not execute: undo its bookkeeping, then run the step for real
        self.step_count -= 1
        g.replay()
        self.step_count += 1
        self.graph_launches += st["launches"]
        return self.loss_buf

    # ---- multi-GPU: CUDA graphs per segment, NCCL between them --------------------------------------------
    def _segment_graphed_step(self, plan, t_static):
        """world > 1: the step is replayed as a handful of CUDA graphs -- [pack + forward + loss], one graph per
        backward segment between two all-reduce marks, [clamp + SGD] -- with the bucketed NCCL all-reduces issued
        between them on the communication stream.  ~12 graph launches instead of ~140 kernel launches from Python,
        so the host never limits the step and the reduce of the last layers still overlaps the backward of the first."""
        st = plan.__dict__.setdefault("_dp_seg", {"calls": 0, "graphs": None})
        if st["graphs"] is None:
            st["calls"] += 1
            if st["calls"] < 3 or self.step_count < 1:
                self._step_body(plan, t_static)
                return self.loss_buf
            st["graphs"] = self._capture_segments(plan, t_static)
        g = st["graphs"]
        cur = torch.cuda.current_stream(self.device)
        if self.step_count > 0:
            cur.wait_stream(self.comm_stream)   # the previous step's last parameter updates ran on the communication stream
        self.step_count += 1
        g["fwd"].replay()
        plan.fwd_serial += 1
        pending = list(plan._dp_buckets)
        for seg_graph, done_from in g["bwd"]:
            seg_graph.replay()
            ready = []
            while done_from is not None and pending and pending[0][0] >= done_from:
                ready.append(pending.pop(0))
            if ready:
                self._reduce_and_update(plan, ready, cur)
        if pending:
            self._reduce_and_update(plan, pending, cur)
        plan.bwd_serial = plan.fwd_serial
        plan._packed_version = None
        self.graph_launches += g["launches"]
        # the loss is read by the caller on the current stream: nothing of this step is left on it but the backward; the
        # next step (or a reader of the parameters) waits for the communication stream
        cur.wait_stream(self.comm_stream)
        return self.loss_buf

    def _capture_segments(self, plan, t_static):
        lib = _lib.load()
        torch.cuda.synchronize(self.device)
        l0 = lib.dards_launch_count()
        out = {"bwd": []}

        def capture(fn):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                fn()
            return gr

        def fwd():
            st = plan._stream()
            plan.pack.run(st)
            if plan.dropout:
                plan.seed_dev[0:1].add_(1)
            plan.fwd.run(st)
            if self.fused:
                _lib.call("dards_bce_with_logits", plan.logits.data_ptr(), t_static.data_ptr(), self.loss_buf.data_ptr(),
                          plan.dlogits.data_ptr(), plan.logits.numel(), plan.__dict__.get("_dp_grad_scale", 1.0), st)
            else:
                self._head_step(plan, t_static)

        out["fwd"] = capture(fwd)
        # backward segments: cut after every call index that carries a mark
        marks = sorted((idx, off) for off, idx in plan.bwd_marks)
        calls = plan.bwd.calls
        begin = 0
        cuts = [(idx, off) for idx, off in marks if 0 < idx <= len(calls)]
        if not cuts or cuts[-1][0] != len(calls):
            cuts.append((len(calls), None))
        for idx, off in cuts:
            if idx <= begin:
                continue
            seg = calls[begin:idx]

            def run_seg(seg=seg):
                st = plan._stream()
                for name, f, args in seg:
                    rc = f(*args, st)
                    if rc != 0:
                        _lib.check(rc, name)

            out["bwd"].append((capture(run_seg), off))
            begin = idx

        # launches per replayed step: the captured kernels + the per-bucket optimizer launches issued behind the all-reduces
        n_upd = sum(1 for lo, hi in plan._dp_buckets for b, e in plan._dp_ranges if max(b, lo) < min(e, hi))
        out["launches"] = int(lib.dards_launch_count() - l0) + n_upd
        return out

    def _backward_overlapped(self, plan):
        """Replay the backward in segments; after each segment the comm stream reduces the buckets that became
        complete and updates their parameters.  Buckets are suffixes of the flat buffer (backward finishes the last
        layers first)."""
        if plan.bwd_serial == plan.fwd_serial:
            raise RuntimeError("backward() without a new forward()")
        cur = torch.cuda.current_stream(self.device)
        st = cur.cuda_stream
        marks = dict((idx, off) for off, idx in plan.bwd_marks)  # call index -> offset complete from there on
        pending = list(plan._dp_buckets)
        calls = plan.bwd.calls
        for i, (name, f, args) in enumerate(calls):
            rc = f(*args, st)
            if rc != 0:
                _lib.check(rc, name)
            done_from = marks.get(i + 1)
            ready = []
            while done_from is not None and pending and pending[0][0] >= done_from:
                ready.append(pending.pop(0))
            if ready:
                self._reduce_and_update(plan, ready, cur)
        if pending:
            self._reduce_and_update(plan, pending, cur)
        plan.bwd_serial = plan.fwd_serial
        cur.wait_stream(self.comm_stream)

    def _update_bucket(self, plan, lo, hi, st):
        """The optimizer step for the live parameter ranges inside the flat slice [lo, hi) -- issued right behind that
        bucket's all-reduce on the communication stream, so only the LAST (small) bucket's update is on the step's tail."""
        for b, e in plan._dp_ranges:
            b, e = max(b, lo), min(e, hi)
            if b < e:
                self._update_range(plan, b, e, st)

    def _update_range(self, plan, b, e, st):
        scale = 1.0 / self.world
        g, p = plan.grad_flat.data_ptr(), self.param_flat.data_ptr()
        if self.optimizer == "sgd":
            _lib.call("dards_clamp_sgd_nesterov", p + 4 * b, g + 4 * b, self.state1.data_ptr() + 4 * b, e - b, self.lr,
                      self.momentum, self.weight_decay, self.clip, scale, 1 if self.step_count == 1 else 0, st)
        else:
            _lib.call("dards_clamp_adam", p + 4 * b, g + 4 * b, self.state1.data_ptr() + 4 * b,
                      self.state2.data_ptr() + 4 * b, e - b, self.lr, 0.9, 0.999, 1e-8, self.clip, scale,
                      self.step_count, st)

    def _reduce_and_update(self, plan, buckets, cur):
        """comm stream: wait for the backward work recorded so far, all-reduce the given buckets, update their parameters."""
        ev = torch.cuda.Event()
        ev.record(cur)
        self.comm_stream.wait_event(ev)
        with torch.cuda.stream(self.comm_stream):
            for b, e in buckets:
                self.reducer.reduce_now(plan.grad_flat, b, e)
                self._update_bucket(plan, b, e, self.comm_stream.cuda_stream)

    def close(self):
        """Drop the captured CUDA graphs (they hold NCCL work when the whole step is captured: destroy them before
        torch.distributed.destroy_process_group())."""
        torch.cuda.synchronize(self.device)
        for plan in list(getattr(self.net, "_dards_plans", {}).values()):
            plan.__dict__.pop("_dp_graph", None)
            plan.__dict__.pop("_dp_seg", None)

    def _update(self, plan, st):
        self.step_count += 1
        scale = 1.0 / self.world
        g, p = plan.grad_flat.data_ptr(), self.param_flat.data_ptr()
        for b, e in plan._dp_ranges:
            if self.optimizer == "sgd":
                _lib.call("dards_clamp_sgd_nesterov", p + 4 * b, g + 4 * b, self.state1.data_ptr() + 4 * b, e - b, self.lr,
                          self.momentum, self.weight_decay, self.clip, scale, 1 if self.step_count == 1 else 0, st)
            else:
                _lib.call("dards_clamp_adam", p + 4 * b, g + 4 * b, self.state1.data_ptr() + 4 * b,
                          self.state2.data_ptr() + 4 * b, e - b, self.lr, 0.9, 0.999, 1e-8, self.clip, scale,
                          self.step_count, st)
        plan._packed_version = None  # weights changed behind autograd's back: repack before the next forward

"""Execution plans: the host-side scheduling of the C-ABI kernels for one network and one batch shape.

A `Plan` is built once per (network, number of breaths N, BatchNorm group size, precision, head mode).  Building
it allocates every activation / statistics / gradient buffer once (PyTorch's caching allocator owns the
memory) and RECORDS the forward and the backward as flat lists of (C function, argument tuple).  Running a step
replays the lists on the current CUDA stream: no tensor allocation, no shape logic and no synchronisation in
the hot loop, which also makes the whole step capturable in a CUDA graph (`Plan.capture()`).

Layout: activations are channels-last (N, L, C) in the plan's storage dtype (fp32 or bf16); parameters and
parameter gradients are fp32.  Gradients land in one flat fp32 buffer (`Plan.grad_flat`, ordered like
`named_parameters()`), which is what the data-parallel all-reduce and the fused optimizer operate on.

Reference semantics implemented here (file:line in /root/reference/deepards):
  models/resnet.py:24-40, 43-78, 141-163   BasicBlock / Bottleneck / ResNet forward
  models/densenet.py:18-43, 68-80, 179-193   dense layer / transition / DenseNet forward
  models/torch_cnn_linear_network.py:57-67, 104-113   per-breath and per-sequence linear heads
"""
import os
from collections import namedtuple

import torch

from . import _lib

BN_EPS = 1e-5
STEM_FUSED_GROUP = 226   # stem.cu: larger BatchNorm groups run through the chunked stem (two passes, a workspace)
BN_MOMENTUM = 0.1
SEQ_LEN = 224

_DTYPES = {"fp32": (torch.float32, _lib.F32), "bf16": (torch.bfloat16, _lib.BF16)}

# Smallest gradient suffix (fp32 elements) worth an all-reduce bucket of its own.  Default: effectively infinite, i.e. ONE
# bucket reduced after the backward pass.  Measured on 8 x B200 (profiles/r02_bench8_*): overlapping the reduction with the
# backward in 5 buckets costs MORE than it hides -- every mark is a flush of the pending partial-sum / weight-gradient
# launches plus a CUDA-graph boundary (+0.13 ms per step at 2 GPUs with the collective switched off), the NCCL kernels
# take SMs from persistent kernels that were sized for all of them, and the whole 15.5 MB all-reduce is only ~0.1 ms
# over NVSwitch: 2.850 ms (5 buckets, 8 SMs reserved) vs 2.728 ms (one bucket) per ResNet-18 step.  Set
# DEEPARDS_B200_DP_BUCKET_ELEMS=262144 to get the overlapped schedule (layer4.1 | layer4.0 | layer3.1 | layer3.0 | rest).
DP_MARK_ELEMS = int(os.environ.get("DEEPARDS_B200_DP_BUCKET_ELEMS", 1 << 30))


def _multi_rank():
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def default_precision():
    """Storage / arithmetic of a network whose `.precision` was not set.  "bf16" (the default): bf16 activations,
    tcgen05 convolutions, fp32 statistics / gradients / weights -- the path bench.py measures; logits within 5e-2 and a
    200-step loss trajectory within 1.3e-2 of the fp32 reference (tests/test_model_parity_gpu.py).  "fp32"
    (DEEPARDS_B200_PRECISION=fp32 or `net.precision = "fp32"`): the 1e-4 parity path on the CUDA cores, ~14x slower."""
    return os.environ.get("DEEPARDS_B200_PRECISION", "bf16")


def _conv_impl_override():
    return os.environ.get("DEEPARDS_B200_CONV_IMPL", "")  # "simt" forces the CUDA-core kernels everywhere


NVTX = int(os.environ.get("DEEPARDS_B200_NVTX", "0"))   # 1: a range per phase (forward / backward / update); 2: + per call


class nvtx_range(object):
    """`with nvtx_range("forward"):` -- an NVTX range when DEEPARDS_B200_NVTX is set, nothing otherwise (SURVEY.md section
    5: tracing; the ranges show up in Nsight Systems / Compute timelines around the recorded kernel lists)."""

    def __init__(self, name, level=1):
        self.on = NVTX >= level
        self.name = name

    def __enter__(self):
        if self.on:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *a):
        if self.on:
            torch.cuda.nvtx.range_pop()


def resnet_bn_layers(backbone):
    """(name, module) of the BatchNorm layers a ResNet's forward uses (resnet.py:141-163): the stem's bn1, its bn2 with
    double_conv_first=True (the default stem builds bn2 and never calls it), and every block's bn1 / bn2 / bn3 (Bottleneck) /
    downsample BatchNorm."""
    out = [("bn1", backbone.bn1)]
    if backbone.double_conv_first:
        out.append(("bn2", backbone.bn2))
    for li, layer in enumerate((backbone.layer1, backbone.layer2, backbone.layer3, backbone.layer4), 1):
        for bi, blk in enumerate(layer):
            pre = "layer%d.%d." % (li, bi)
            out += [(pre + "bn1", blk.bn1), (pre + "bn2", blk.bn2)]
            if isinstance(getattr(blk, "bn3", None), torch.nn.BatchNorm1d):
                out.append((pre + "bn3", blk.bn3))
            if blk.downsample is not None:
                out.append((pre + "downsample.1", blk.downsample[1]))
    return out


def bn_mode(backbone):
    """Which BatchNorm a plan for `backbone` implements, from the module's own training flags, as nn.BatchNorm1d would:
      'train'  -- batch statistics, running statistics updated (every DenseNet; a ResNet in train() with its BatchNorm
                  layers in train());
      'frozen' -- a ResNet in train() with every BatchNorm layer in eval(): normalised with the running statistics, which
                  stay untouched, and still back-propagated into gamma, beta and the convolutions (fine-tuning with frozen
                  BatchNorm);
      'eval'   -- a ResNet in eval(): inference with the running statistics, whatever its BatchNorm layers say.
    A ResNet in train() with some BatchNorm layers in train() and others in eval() raises NotImplementedError.
    DenseNet's BatchNorm layers keep no running statistics, so torch normalises with batch statistics in either state."""
    if not backbone.network_name.startswith("resnet"):
        return "train"
    if not backbone.training:
        return "eval"
    layers = resnet_bn_layers(backbone)
    frozen = [n for n, m in layers if not m.training]
    if not frozen:
        return "train"
    if len(frozen) == len(layers):
        return "frozen"
    training = [n for n, m in layers if m.training]
    raise NotImplementedError("deepards_b200: a ResNet in train() needs its BatchNorm layers all in train() (batch "
                              "statistics) or all in eval() (frozen running statistics); in train(): %s; in eval(): %s"
                              % (", ".join(training), ", ".join(frozen)))


class Recorder(object):
    """A replayable list of C-ABI calls."""

    def __init__(self):
        self.calls = []

    def add(self, name, *args):
        self.calls.append((name, _lib.fn(name), args))

    def run(self, stream):
        if NVTX >= 2:
            for name, f, args in self.calls:
                with nvtx_range(name, 2):
                    rc = f(*args, stream)
                if rc != 0:
                    _lib.check(rc, name)
            return
        for name, f, args in self.calls:
            rc = f(*args, stream)
            if rc != 0:
                _lib.check(rc, name)

    def __len__(self):
        return len(self.calls)


class _ConvRec(object):
    __slots__ = ("mod", "cin", "cout", "k", "stride", "pad", "kio", "koi", "goff", "dwt")


# A BatchNorm layer applied with its running statistics (Plan._eval_coeffs): pointers to its fp32 scale and shift, and, for
# frozen plans, whose backward needs them, to rstd = 1/sqrt(running_var + eps) and running_mean (None in eval plans).
Coef = namedtuple("Coef", "scale shift rstd mean")


class Plan(object):
    """See module docstring.  mode: 'backbone' (-> feat (N,F)), 'cnn_linear' (-> logits (B,2)),
    'per_breath' (-> logits (B,group,2)), 'features' (DenseNet only, -> norm5 output (N,F,7)).
    bn: 'train' (batch statistics; forward and backward), 'eval' (ResNet only: BatchNorm with the running statistics,
    applied in the convolution epilogues; a forward only, see _build_resnet_eval) or 'frozen' (ResNet only: BatchNorm with
    the running statistics, forward and backward, no running-statistics update; see bn_mode and _build_resnet).
    input_grad (train and frozen plans): the backward also writes the gradient w.r.t. the input, `dx` (N, 224) fp32, with the
    stem's dgrad kernel recorded right after the stem's weight-gradient backward (saliency.input_gradients)."""

    def __init__(self, net, backbone, linear, n_breaths, group, precision, mode, dropout, update_running, bn="train",
                 input_grad=False):
        if precision not in _DTYPES:
            raise ValueError("precision must be 'fp32' or 'bf16', got %r" % (precision,))
        if n_breaths % group != 0:
            raise ValueError("number of breaths (%d) is not a multiple of the BatchNorm group (%d)" % (n_breaths, group))
        if bn not in ("train", "eval", "frozen"):
            raise ValueError("bn must be 'train', 'eval' or 'frozen', got %r" % (bn,))
        if input_grad and bn == "eval":
            raise ValueError("an eval plan has no backward: input_grad needs bn='train' or 'frozen'")
        self.bn = bn
        self.input_grad = input_grad
        self.net, self.backbone, self.linear = net, backbone, linear
        self.N, self.group, self.G = n_breaths, group, n_breaths // group
        self.precision, self.mode = precision, mode
        self.tdtype, self.dt = _DTYPES[precision]
        self.dropout, self.update_running = dropout, update_running
        p0 = next(backbone.parameters())
        if p0.device.type != "cuda":
            raise RuntimeError("deepards_b200 runs on CUDA devices only (parameters are on %s); there is no CPU "
                               "fallback" % p0.device)
        self.device = p0.device
        self.simt_only = _conv_impl_override() == "simt" or precision != "bf16"
        # conv + BatchNorm in one kernel: "0" never, "2" only where the whole normalisation runs in the epilogue,
        # "1" also with statistics partials + the streaming normalisation (long sequences)
        self.fuse_bn = os.environ.get("DEEPARDS_B200_FUSE_BN", "2")
        self.bufs = []  # keeps every tensor referenced by a recorded pointer alive
        self.pack = Recorder()
        self.fwd = Recorder()
        self.bwd = Recorder()
        self.convs = []
        self.sites = {}  # ReLU site name -> post-activation buffer (N, L, C); the parity tests read the decisions here
        self.bwd_marks = []  # (flat-gradient offset that is complete from there to the end, #bwd calls issued)
        self._scratch = {}
        self._packed_version = None
        self.graph = None
        self.fwd_serial = 0
        self.bwd_serial = 0

        # ---- parameter table: flat gradient buffer in named_parameters() order ------------------------------
        self.params = [(n, p) for n, p in net.named_parameters()]
        self.goff = {}
        off = 0
        for n, p in self.params:
            self.goff[id(p)] = off
            off += (p.numel() + 3) // 4 * 4  # keep every slot 16-byte aligned
        self.grad_numel = off
        # an eval plan has no backward: no gradient buffer
        self.grad_flat = self.new((max(off, 4),), torch.float32, zero=True) if bn != "eval" else None
        self.grad_written = set()
        self.eval_reads = set()  # eval plans: the parameters the forward reads (the autograd inputs)
        self.param_sig = self._param_signature()

        # ---- I/O buffers ------------------------------------------------------------------------------------
        self.x_buf = self.new((n_breaths, SEQ_LEN), torch.float32)
        self.dx = self.new((n_breaths, SEQ_LEN), torch.float32) if input_grad else None
        # [0] forward counter (fresh dropout masks per step), [1] global index of this rank's first sequence
        self.seed_dev = self.new((2,), torch.int64, zero=True)
        self._seq_offset = 0
        # tcgen05 weight gradients: "accumulate" (default) adds every CTA's fp32 tile into a tap-major buffer at the L2 (no
        # split-K partials, no reduce kernels; fp32 summation order = arrival order), "deterministic" keeps the split-K
        # partials + fixed-order reduce kernels (bit-reproducible)
        self.wgrad_mode = os.environ.get("DEEPARDS_B200_WGRAD", "accumulate")
        self._dwt_arena = None
        self._dwt_used = 0
        self._pending_unpack = []
        if not self.simt_only and self.wgrad_mode == "accumulate" and bn != "eval":
            import torch.nn as nn
            total = sum((m.weight.numel() + 3) // 4 * 4 for m in backbone.modules() if isinstance(m, nn.Conv1d))
            self._dwt_arena = self.new((max(total, 4),), torch.float32, zero=True)
        self._running = []   # (mean, rstd, bn, rows, c): running-statistics updates, one batched launch per forward
        self._pending_red = []  # (partial table, rows, c, destination pointer): flushed as one batched launch
        kind = backbone.network_name
        if bn != "train" and not kind.startswith("resnet"):
            raise NotImplementedError("running-statistics BatchNorm plans exist for ResNet backbones only (DenseNet's "
                                      "BatchNorm layers keep no running statistics)")
        if bn == "eval":
            self._build_resnet_eval()
        elif kind.startswith("resnet"):
            self._build_resnet()
        elif kind.startswith("densenet"):
            self._build_densenet()
        else:
            raise NotImplementedError(kind)
        self._flush_running()
        self._flush_reductions()
        if self._dwt_arena is not None and self._dwt_used:
            # zeroed at the end of every forward: the backward's weight-gradient kernels add into it
            self.fwd.add("dards_memset_zero", self._dwt_arena.data_ptr(), 4 * self._dwt_used)
        self._build_pack_table()

    # ------------------------------------------------------------------------------------------------------
    # helpers
    # ------------------------------------------------------------------------------------------------------
    def new(self, shape, dtype=None, zero=False):
        t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype or self.tdtype, device=self.device)
        self.bufs.append(t)
        return t

    def scratch(self, key, shape, dtype=None):
        k = (key, tuple(shape), dtype or self.tdtype)
        if k not in self._scratch:
            self._scratch[k] = self.new(shape, dtype)
        return self._scratch[k]

    def _param_signature(self):
        sig = tuple(p.data_ptr() for _, p in self.params)
        if self.bn != "train":  # the recorded coefficient launch reads the running buffers through their pointers
            sig += tuple(b.data_ptr() for _, b in self.backbone.named_buffers() if b is not None)
        return sig

    def valid(self):
        return self.param_sig == self._param_signature()

    def gptr(self, p):
        self.grad_written.add(id(p))
        return self.grad_flat.data_ptr() + 4 * self.goff[id(p)]

    def mark(self, first_param):
        """Backward bookkeeping for the overlapped all-reduce: every gradient slot at or after `first_param`'s
        is final once the calls recorded so far have run (backward visits the layers last to first).
        With more than one rank the pending partial-sum reductions are flushed here, so that the bucket behind the mark
        can go to the all-reduce; a single rank reduces everything in ONE launch at the end of the backward.
        A mark is only set once at least DP_MARK_ELEMS gradient elements have become final since the previous one:
        every mark costs a reduction launch and a CUDA-graph boundary in the multi-GPU step, and a smaller bucket
        would be merged by the trainer anyway (DenseNet-18's 0.86 MB of gradients are ONE bucket and ONE backward graph)."""
        off = self.goff[id(first_param)]
        last = self.bwd_marks[-1][0] if self.bwd_marks else self.grad_numel
        if last - off < DP_MARK_ELEMS:
            return
        if _multi_rank():
            self._flush_reductions()
        self.bwd_marks.append((off, len(self.bwd.calls)))

    def grad_view(self, p):
        off = self.goff[id(p)]
        return self.grad_flat[off:off + p.numel()].view(p.shape)

    # ---- op recorders -------------------------------------------------------------------------------------
    def conv(self, mod):
        c = _ConvRec()
        c.mod = mod
        c.cout, c.cin, c.k = mod.weight.shape
        c.stride, c.pad = mod.stride[0], mod.padding[0]
        c.kio = self.new((c.k, c.cin, c.cout))
        c.koi = self.new((c.k, c.cout, c.cin))
        c.dwt = None
        self.convs.append(c)
        return c

    def _tc_ok(self, c, direction):
        """tcgen05 path for this conv?  (bf16 plans only; everything else runs the CUDA-core kernels)"""
        if self.simt_only or c.stride not in (1, 2):
            return False
        if direction == "wgrad":
            if "wgrad" in _conv_impl_override():
                return False
            # k7 / stride 2 / pad 3 (the two-convolution stem's conv2): seven 64-column TMEM accumulators, c_in <= 64
            k7 = c.k == 7 and c.pad == 3 and c.stride == 2 and c.cin <= 64
            return ((c.k == 3 and c.pad == 1) or (c.k == 1 and c.pad == 0) or k7) and c.cin % 16 == 0 and c.cout % 8 == 0
        return c.cin % 8 == 0 and c.cout % 8 == 0

    def conv_fwd(self, c, src, src_stride, dst, dst_stride, l_in, dst_ptr_off=0, src_last_use=False):
        """src_last_use: no later kernel of the forward pass reads `src` (L2 eviction hint, DARDS_HINT_LAST_USE)."""
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        tc = self._tc_ok(c, "fwd")
        w = c.koi if tc else c.kio
        self.fwd.add("dards_conv1d_fwd", src, w.data_ptr(), dst + dst_ptr_off, None, self.N, l_in, l_out, c.cin, c.cout,
                     src_stride, dst_stride, 0, c.k, c.stride, c.pad, self.dt,
                     (1 if tc else 0) | (_lib.HINT_LAST_USE if src_last_use else 0))
        return l_out

    def conv_dgrad(self, c, dout, dout_stride, din, din_stride, l_in, addend=None, addend_stride=0, src_last_use=True):
        """src_last_use: the weight gradient of the same layer has already consumed `dout` (every plan records wgrad
        before dgrad), so this is its last reader."""
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        tc = self._tc_ok(c, "dgrad")
        w = c.kio if tc else c.koi
        self.bwd.add("dards_conv1d_dgrad", dout, w.data_ptr(), din, addend, self.N, l_in, l_out, c.cin, c.cout,
                     dout_stride, din_stride, addend_stride, c.k, c.stride, c.pad, self.dt,
                     (1 if tc else 0) | (_lib.HINT_LAST_USE if src_last_use else 0))

    def conv_wgrad(self, c, src, src_stride, dout, dout_stride, l_in):
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        tc = self._tc_ok(c, "wgrad")
        if tc and self._dwt_arena is not None and c.cin % 32 == 0:
            if c.dwt is None:
                n = c.k * c.cout * c.cin
                c.dwt = self._dwt_arena[self._dwt_used:self._dwt_used + n]
                self._dwt_used += (n + 3) // 4 * 4
            self.bwd.add("dards_conv1d_wgrad_accum", src, dout, c.dwt.data_ptr(), self.N, l_in, l_out, c.cin, c.cout,
                         src_stride, dout_stride, c.k, c.stride, c.pad, self.dt)
            self._pending_unpack.append((c, self.gptr(c.mod.weight)))
            return
        impl = 1 if tc else 0
        need = _lib.fn("dards_conv1d_wgrad_workspace_bytes")(self.N, l_out, c.cin, c.cout, c.k, impl)
        ws = self._wgrad_ws(need)
        self.bwd.add("dards_conv1d_wgrad", src, dout, self.gptr(c.mod.weight), 0, ws.data_ptr(), ws.numel() * 4, self.N,
                     l_in, l_out, c.cin, c.cout, src_stride, dout_stride, c.k, c.stride, c.pad, self.dt, impl)

    def _wgrad_ws(self, nbytes):
        cur = getattr(self, "_ws", None)
        n = (int(nbytes) + 3) // 4
        if cur is None or cur.numel() < n:
            # recorded pointers of earlier convs must stay valid: never shrink/free, only add
            self._ws = self.new((max(n, 1),), torch.float32)
        return self._ws

    def stats(self, c):
        return self.new((self.G, c), torch.float32), self.new((self.G, c), torch.float32)

    def gbn_fwd(self, bn, x, x_stride, out, out_stride, rows, c, relu, res=None, res_stride=0, x_last_use=True):
        """x_last_use: x is a convolution output that nothing else reads before the backward pass (False for DenseNet's
        concatenation buffer, which the following layers read again).
        Frozen plans: the affine map of the running statistics over all G * rows rows; returns the layer's coefficients."""
        if self.bn == "frozen":
            return self.bn_affine_apply(bn, x, x_stride, out, out_stride, self.G * rows, c, relu, res, res_stride)
        mean, rstd = self.stats(c)
        self.fwd.add("dards_gbn_fwd", x, out, res, bn.weight.data_ptr(), bn.bias.data_ptr(), mean.data_ptr(),
                     rstd.data_ptr(), self.G, rows, c, x_stride, out_stride, res_stride, BN_EPS,
                     (1 if relu else 0) | (_lib.HINT_LAST_USE if x_last_use else 0), self.dt)
        self._note_running(bn, mean, rstd, rows, c)
        return mean, rstd

    # ---- convolution + BatchNorm in one kernel (conv_bn_tc.cu) -----------------------------------------------
    def _cb_shape(self, c, l_in):
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        return (self.N, self.group, l_in, l_out, c.cin, c.cout, c.k, c.stride, c.pad)

    def cb_mode(self, c, l_in, merged_branch=False):
        """0: separate conv + BatchNorm kernels; 1: statistics in the convolution epilogue + one elementwise pass;
        2: BatchNorm (+ residual, + ReLU) entirely in the convolution epilogue.
        merged_branch: the layer is one of the two branches of a downsample block, whose two BatchNorms + add + ReLU
        become ONE elementwise pass in mode 1 (fuse_bn "3" enables mode 1 for those only)."""
        if self.simt_only or self.fuse_bn == "0" or self.bn == "frozen" or not self._tc_ok(c, "fwd"):
            return 0  # (the fused kernel takes batch statistics)
        mode = _lib.fn("dards_conv1d_bn_mode")(*self._cb_shape(c, l_in), self.dt)
        if mode == 1 and not (self.fuse_bn == "1" or (merged_branch and self.fuse_bn == "3")):
            return 0
        return mode

    def _cb_conv(self, c, bn, src, src_stride, l_in, y, y_stride, out, out_stride, relu, res, res_stride, st, part,
                 src_last_use):
        shape = self._cb_shape(c, l_in)
        mean, rstd = st
        flags = (1 if relu else 0) | (_lib.HINT_LAST_USE if src_last_use else 0)
        self.fwd.add("dards_conv1d_bn_fwd", src, c.koi.data_ptr(), y, out, res, bn.weight.data_ptr(), bn.bias.data_ptr(),
                     mean.data_ptr(), rstd.data_ptr(), part, shape[0], shape[1], shape[2], shape[3], c.cin, c.cout,
                     src_stride, y_stride, out_stride, res_stride, c.k, c.stride, c.pad, BN_EPS, flags, self.dt)

    def conv_bn_fwd(self, c, bn, src, src_stride, l_in, y, out, relu, res=None, src_last_use=False, ds=None,
                    part_key="cb_part", merged_branch=False):
        """y = conv(src) and out = [relu](bn(y) [+ res] [+ bn_d(conv_d(src_d))]) with the BatchNorm statistics taken in
        the convolution epilogue.  `y` / `out` are (N, l_out, cout) plan buffers, `res` a same-shape buffer;
        ds = (conv record, bn module, source pointer, source stride, source length, y_d buffer): the downsample branch
        of a ResNet block.  Returns (statistics of bn, statistics of the downsample bn or None).  Both convolutions
        must report the same mode (cb_mode)."""
        mode = self.cb_mode(c, l_in, merged_branch)
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        cout = c.cout
        rows = self.group * l_out
        st = self.stats(cout)
        std = None
        res_ptr = res.data_ptr() if res is not None else None
        if mode == 2:
            if ds is not None:
                cd, bnd, dsrc, dstride, dl, yd = ds
                std = self.stats(cout)
                resd = self.scratch("ds_res", (self.N, l_out, cout))
                self._cb_conv(cd, bnd, dsrc, dstride, dl, yd.data_ptr(), cout, resd.data_ptr(), cout, False, None, 0, std,
                              None, False)
                self._note_running(bnd, std[0], std[1], rows, cout)
                res_ptr = resd.data_ptr()
            self._cb_conv(c, bn, src, src_stride, l_in, y.data_ptr(), cout, out.data_ptr(), cout, relu, res_ptr, cout, st,
                          None, src_last_use)
        elif mode == 1:
            shape = self._cb_shape(c, l_in)
            entries = _lib.fn("dards_conv1d_bn_part_entries")(*shape)
            part = self.scratch(part_key, (self.G * entries * 3 * cout,), torch.float32)
            self._cb_conv(c, bn, src, src_stride, l_in, y.data_ptr(), cout, None, 0, relu, None, 0, st, part.data_ptr(),
                          src_last_use)
            x2 = [None, None, None, None, 0, None, None]
            if ds is not None:
                cd, bnd, dsrc, dstride, dl, yd = ds
                std = self.stats(cout)
                shaped = self._cb_shape(cd, dl)
                entd = _lib.fn("dards_conv1d_bn_part_entries")(*shaped)
                partd = self.scratch(part_key + "_d", (self.G * entd * 3 * cout,), torch.float32)
                self._cb_conv(cd, bnd, dsrc, dstride, dl, yd.data_ptr(), cout, None, 0, False, None, 0, std,
                              partd.data_ptr(), False)
                self._note_running(bnd, std[0], std[1], rows, cout)
                x2 = [yd.data_ptr(), bnd.weight.data_ptr(), bnd.bias.data_ptr(), partd.data_ptr(), entd,
                      std[0].data_ptr(), std[1].data_ptr()]
            self.fwd.add("dards_gbn_apply_fwd", y.data_ptr(), out.data_ptr(), res_ptr, bn.weight.data_ptr(),
                         bn.bias.data_ptr(), part.data_ptr(), entries, st[0].data_ptr(), st[1].data_ptr(), *x2, self.G, rows,
                         cout, cout, cout, cout if res is not None else 0, cout if ds is not None else 0, BN_EPS,
                         1 if relu else 0, self.dt)
        else:
            raise RuntimeError("conv_bn_fwd called for a shape the fused kernel does not support")
        self._note_running(bn, st[0], st[1], rows, cout)
        return st, std

    # ---- frozen BatchNorm (running statistics under train()) -------------------------------------------------
    def bn_affine_apply(self, bn, y, y_stride, out, out_stride, rows, c, relu, res=None, res_stride=0, second=None):
        """out = [relu](bn(y) [+ res] [+ bn_d(y_d)]) with the running statistics; second = (bn_d, y_d pointer, stride)."""
        co = self._coef[id(bn)]
        y2, s2, h2, y2s = None, None, None, 0
        if second is not None:
            bnd, y2, y2s = second
            s2, h2 = self._coef[id(bnd)].scale, self._coef[id(bnd)].shift
        self.fwd.add("dards_bn_affine_apply", y, out, res, co.scale, co.shift, y2, s2, h2, rows, c, y_stride, out_stride,
                     res_stride if res is not None else 0, y2s, 1 if relu else 0, self.dt)
        return co

    @staticmethod
    def _frozen_tile_rows(total, c):
        """Rows per tile of a frozen BatchNorm backward: the largest divisor of `total` up to the tile of the training
        kernels (rows * C = 71680, at most 1120 rows), so that the whole tile fits the cached kernel."""
        target = min(1120, max(8, 71680 // c), total)
        for d in range(target, 0, -1):
            if total % d == 0:
                return d
        return 1

    def _frozen_bwd(self, bn, co, dout, dout_stride, y, y_stride, dx, dx_stride, rows, c, relu_mode, mask, mask_stride,
                    accumulate, dres, dres_stride):
        total = self.G * rows
        tile = self._frozen_tile_rows(total, c)
        n_tiles = total // tile
        dg = self.new((n_tiles, c), torch.float32)
        db = self.new((n_tiles, c), torch.float32)
        self.bwd.add("dards_bn_frozen_bwd", dout, y, mask, co.scale, co.shift, co.mean, co.rstd, dx, 1 if accumulate else 0,
                     dres, dg.data_ptr(), db.data_ptr(), n_tiles, tile, c, dout_stride, y_stride, mask_stride, dx_stride,
                     dres_stride, relu_mode, self.dt)
        self._pending_red.append((dg, n_tiles, c, self.gptr(bn.weight)))
        self._pending_red.append((db, n_tiles, c, self.gptr(bn.bias)))

    def _note_running(self, bn, mean, rstd, rows, c):
        if self.update_running and getattr(bn, "running_mean", None) is not None:
            self._running.append((mean, rstd, bn, rows, c))

    def _flush_running(self):
        """nn.BatchNorm1d running statistics of EVERY layer in one launch at the end of the forward (nothing in the
        step reads them)."""
        if not self._running:
            return
        descs = [(mean.data_ptr(), rstd.data_ptr(), bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                  bn.num_batches_tracked.data_ptr() if bn.num_batches_tracked is not None else None, self.G, rows, c,
                  BN_MOMENTUM if bn.momentum is None else bn.momentum) for mean, rstd, bn, rows, c in self._running]
        t, total = _lib.desc_table(_lib.RunningDesc, descs, self.device)
        self.bufs.append(t)
        self.fwd.add("dards_bn_running_update_batched", t.data_ptr(), len(descs), total, BN_EPS)
        self._running = []

    def _flush_unpack(self):
        """Tap-major accumulation buffers of the weight gradients computed since the last flush -> the parameters'
        (Cout, Cin, K) gradient slots, in one launch."""
        if not self._pending_unpack:
            return
        descs = [(c.dwt.data_ptr(), dst, c.cout, c.cin, c.k) for c, dst in self._pending_unpack]
        t, total = _lib.desc_table(_lib.UnpackDesc, descs, self.device)
        self.bufs.append(t)
        self.bwd.add("dards_unpack_wgrad_batched", t.data_ptr(), len(descs), total)
        self._pending_unpack = []

    def _flush_reductions(self):
        """Per-group partial sums (BatchNorm dgamma/dbeta, stem dW) accumulated since the last flush -> their gradient
        slots, in one launch."""
        self._flush_unpack()
        if not self._pending_red:
            return
        descs = [(part.data_ptr(), dst, rows, c, 0) for part, rows, c, dst in self._pending_red]
        t, total = _lib.desc_table(_lib.ReduceDesc, descs, self.device)
        self.bufs.append(t)
        self.bwd.add("dards_reduce_rows_batched", t.data_ptr(), len(descs), total)
        self._pending_red = []

    def gbn_bwd(self, bn, st, dout, dout_stride, x, x_stride, dx, dx_stride, rows, c, relu_mode, mask=None,
                mask_stride=0, accumulate=False, dres=None, dres_stride=0):
        if self.bn == "frozen":
            return self._frozen_bwd(bn, st, dout, dout_stride, x, x_stride, dx, dx_stride, rows, c, relu_mode, mask,
                                    mask_stride, accumulate, dres, dres_stride)
        mean, rstd = st
        dg = self.new((self.G, c), torch.float32)   # per layer: they live until the next flush
        db = self.new((self.G, c), torch.float32)
        self.bwd.add("dards_gbn_bwd", dout, x, mask, bn.weight.data_ptr(), bn.bias.data_ptr(), mean.data_ptr(),
                     rstd.data_ptr(), dx, 1 if accumulate else 0, dres, dg.data_ptr(), db.data_ptr(), self.G, rows, c,
                     dout_stride, x_stride, mask_stride, dx_stride, dres_stride, relu_mode, self.dt)
        self._pending_red.append((dg, self.G, c, self.gptr(bn.weight)))
        self._pending_red.append((db, self.G, c, self.gptr(bn.bias)))

    # ------------------------------------------------------------------------------------------------------
    # stem (shared by both backbones)
    # ------------------------------------------------------------------------------------------------------
    def _stem(self, conv, bn, pool, out, out_stride):
        c0 = conv.out_channels
        if conv.in_channels != 1 or conv.kernel_size[0] != 7 or conv.stride[0] != 2 or conv.padding[0] != 3:
            raise NotImplementedError("stem must be Conv1d(1, C0, 7, stride 2, padding 3)")
        if self.bn != "train":  # frozen and eval plans: the running statistics' affine map, every breath on its own
            co = self._coef[id(bn)]
            self.eval_reads.add(id(conv.weight))
            self.fwd.add("dards_stem_eval_fwd", self.x_buf.data_ptr(), conv.weight.data_ptr(), co.scale, co.shift, out,
                         self.N, c0, out_stride, pool, self.dt)
            return co
        mean, rstd = self.stats(c0)
        # a BatchNorm group that does not fit the fused stem's shared memory (a flat batch of more than 226 breaths is ONE
        # group) runs in chunks and needs a workspace for the chunk records (stem.cu)
        ws, ws_bytes = self._stem_ws(c0, 0)
        self.fwd.add("dards_stem_fwd", self.x_buf.data_ptr(), conv.weight.data_ptr(), bn.weight.data_ptr(),
                     bn.bias.data_ptr(), out, mean.data_ptr(), rstd.data_ptr(), self.G, self.group, c0, out_stride,
                     BN_EPS, pool, ws, ws_bytes, self.dt)
        self._note_running(bn, mean, rstd, self.group * 112, c0)
        return mean, rstd

    def _stem_ws(self, c0, backward):
        nbytes = _lib.fn("dards_stem_workspace_bytes")(self.G, self.group, c0, backward)
        if not nbytes:
            return None, 0
        t = self.new(((nbytes + 3) // 4,), torch.float32)
        return t.data_ptr(), t.numel() * 4

    def _stem_bwd(self, conv, bn, pool, st, dout, dout_stride):
        c0 = conv.out_channels
        if self.bn == "frozen":
            nc = _lib.fn("dards_stem_frozen_chunks")(self.N)
            dwp = self.new((nc, c0 * 7), torch.float32)
            dgp = self.new((nc, c0), torch.float32)
            dbp = self.new((nc, c0), torch.float32)
            self.bwd.add("dards_stem_frozen_bwd", dout, self.x_buf.data_ptr(), conv.weight.data_ptr(), st.scale, st.shift,
                         st.mean, st.rstd, dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), self.N, c0, dout_stride, pool,
                         self.dt)
            if self.input_grad:
                self.bwd.add("dards_stem_frozen_dgrad", dout, self.x_buf.data_ptr(), conv.weight.data_ptr(), st.scale,
                             st.shift, self.dx.data_ptr(), self.N, c0, dout_stride, pool, self.dt)
            self._pending_red.append((dwp, nc, c0 * 7, self.gptr(conv.weight)))
            self._pending_red.append((dgp, nc, c0, self.gptr(bn.weight)))
            self._pending_red.append((dbp, nc, c0, self.gptr(bn.bias)))
            self._flush_reductions()
            return
        mean, rstd = st
        dwp = self.new((self.G, c0 * 7), torch.float32)
        dgp = self.new((self.G, c0), torch.float32)
        dbp = self.new((self.G, c0), torch.float32)
        ws, ws_bytes = self._stem_ws(c0, 1)
        self.bwd.add("dards_stem_bwd", dout, self.x_buf.data_ptr(), conv.weight.data_ptr(), bn.weight.data_ptr(),
                     bn.bias.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(),
                     self.G, self.group, c0, dout_stride, pool, ws, ws_bytes, self.dt)
        if self.input_grad:  # reads the group totals dgp / dbp that the backward just wrote
            self.bwd.add("dards_stem_dgrad", dout, self.x_buf.data_ptr(), conv.weight.data_ptr(), bn.weight.data_ptr(),
                         bn.bias.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dgp.data_ptr(), dbp.data_ptr(),
                         self.dx.data_ptr(), self.G, self.group, c0, dout_stride, pool, self.dt)
        self._pending_red.append((dwp, self.G, c0 * 7, self.gptr(conv.weight)))
        self._pending_red.append((dgp, self.G, c0, self.gptr(bn.weight)))
        self._pending_red.append((dbp, self.G, c0, self.gptr(bn.bias)))
        self._flush_reductions()

    # ------------------------------------------------------------------------------------------------------
    # head
    # ------------------------------------------------------------------------------------------------------
    def _head_fwd(self, act, act_stride, l, f):
        """act: (N, l, f) post-ReLU activations -> feat (N, f) -> [linear] ; records forward."""
        self.feat = self.new((self.N, f), torch.float32)
        self.fwd.add("dards_avgpool_full_fwd", act, self.feat.data_ptr(), self.N, l, f, act_stride, self.dt)
        self.out_features = f
        if self.mode in ("cnn_linear", "per_breath"):
            lin = self.linear
            rows, k = (self.G, self.group * f) if self.mode == "cnn_linear" else (self.N, f)
            if lin.in_features != k:
                raise RuntimeError("linear_final expects %d features but the backbone provides %d (metadata features "
                                   "are not supported)" % (lin.in_features, k))
            n_out = lin.out_features
            self.logits = self.new((rows, n_out), torch.float32)
            self.dlogits = self.new((rows, n_out), torch.float32)
            self.fwd.add("dards_linear_fwd", self.feat.data_ptr(), lin.weight.data_ptr(), lin.bias.data_ptr(),
                         self.logits.data_ptr(), rows, k, n_out)
            self.head_rows, self.head_k, self.head_out = rows, k, n_out

    def _head_bwd(self, dact, dact_stride, l, f):
        self.dfeat = self.new((self.N, f), torch.float32)
        if self.mode in ("cnn_linear", "per_breath"):
            lin = self.linear
            self.bwd.add("dards_linear_bwd", self.dlogits.data_ptr(), self.feat.data_ptr(), lin.weight.data_ptr(),
                         self.dfeat.data_ptr(), self.gptr(lin.weight), self.gptr(lin.bias), 0, self.head_rows,
                         self.head_k, self.head_out)
        self.bwd.add("dards_avgpool_full_bwd", self.dfeat.data_ptr(), dact, self.N, l, f, dact_stride, self.dt)

    # ------------------------------------------------------------------------------------------------------
    # ResNet (BasicBlock and Bottleneck)
    # ------------------------------------------------------------------------------------------------------
    @staticmethod
    def _block_stages(blk):
        """The main branch of a block as (conv, bn) in order: conv1 / conv2 for BasicBlock (resnet.py:24-40), conv1 (1x1) /
        conv2 (k3, the block's stride) / conv3 (1x1, x4) for Bottleneck (resnet.py:43-78).  Every stage but the last is
        followed by a ReLU; the last one's BatchNorm is added to the identity or downsample branch before the ReLU."""
        stages = [(blk.conv1, blk.bn1), (blk.conv2, blk.bn2)]
        if getattr(blk, "conv3", None) is not None:
            stages.append((blk.conv3, blk.bn3))
        return stages

    def _resnet_blocks(self):
        """The checks every ResNet plan shares, run before anything is recorded (the stem's shape is checked by _stem).
        Returns (stem pool type, c0, [(block, site prefix 'layer{li}.{bi}', l_in, l_out, cin, cout)]), cin / cout being the
        block's input and output channels."""
        m = self.backbone
        if m.double_conv_first and self.bn == "frozen":
            raise NotImplementedError("resnet double_conv_first=True with frozen BatchNorm (train() with the BatchNorm "
                                      "layers in eval()) is not implemented on the B200 backend")
        if self.mode == "features":
            raise NotImplementedError("'features' mode exists for DenseNet only (gradcam.py:45 needs .features)")
        blocks, L = [], 56
        for li, layer in enumerate((m.layer1, m.layer2, m.layer3, m.layer4), 1):
            for bi, blk in enumerate(layer):
                stages = self._block_stages(blk)
                cin, cout = stages[0][0].in_channels, stages[-1][0].out_channels
                lo = L
                for conv, _ in stages:
                    lo = (lo + 2 * conv.padding[0] - conv.kernel_size[0]) // conv.stride[0] + 1
                if blk.downsample is None and (cin != cout or lo != L):
                    raise RuntimeError("%s without downsample must keep the shape" % type(blk).__name__)
                blocks.append((blk, "layer%d.%d" % (li, bi), L, lo, cin, cout))
                L = lo
        if L != 7:
            raise RuntimeError("unexpected final length %d" % L)
        return (0 if m.first_pool_type == "max" else 1), m.conv1.out_channels, blocks

    def _build_resnet(self):
        m = self.backbone
        pool, c0, blocks = self._resnet_blocks()
        N = self.N
        if self.bn == "frozen":
            # scale / shift / rstd of every layer from the running buffers, computed at the start of every forward
            self._coef = self._eval_coeffs(with_rstd=True)
        a = self.new((N, 56, c0))
        if m.double_conv_first:
            stem_st = self._double_stem_fwd(pool, c0, a.data_ptr())
        else:
            stem_st = self._stem(m.conv1, m.bn1, pool, a.data_ptr(), c0)
        recs = []
        for blk, site, L, lo, cin, cout in blocks:
            r = {"a_in": a}
            # the main branch: every stage but the last -> conv + BatchNorm + ReLU (sites relu1, relu2)
            convs = [self.conv(conv) for conv, _ in self._block_stages(blk)]
            bns = [bn for _, bn in self._block_stages(blk)]
            h, lh, ch = a, L, cin
            stages = []
            for i, (c, bn) in enumerate(zip(convs[:-1], bns[:-1])):
                lc = (lh + 2 * c.pad - c.k) // c.stride + 1
                y = self.new((N, lc, c.cout))
                act = self.new((N, lc, c.cout))
                if self.cb_mode(c, lh):
                    st, _ = self.conv_bn_fwd(c, bn, h.data_ptr(), ch, lh, y, act, True, src_last_use=i > 0)
                else:
                    self.conv_fwd(c, h.data_ptr(), ch, y.data_ptr(), c.cout, lh, src_last_use=i > 0)
                    st = self.gbn_fwd(bn, y.data_ptr(), c.cout, act.data_ptr(), c.cout, self.group * lc, c.cout, True)
                stages.append(dict(c=c, bn=bn, src=h, cin=ch, l_in=lh, y=y, act=act, st=st))
                self.sites[site + ".relu%d" % (i + 1)] = act
                h, lh, ch = act, lc, c.cout
            # the last stage: out = relu(bn(conv(h)) + identity or downsample branch)
            cl, bnl = convs[-1], bns[-1]
            yl = self.new((N, lo, cout))
            out = self.new((N, lo, cout))
            ml = self.cb_mode(cl, lh, blk.downsample is not None)
            if blk.downsample is not None:
                cd = self.conv(blk.downsample[0])
                yd = self.new((N, lo, cout))
                if ml and self.cb_mode(cd, L, True) == ml:
                    stl, std = self.conv_bn_fwd(cl, bnl, h.data_ptr(), ch, lh, yl, out, True, src_last_use=True,
                                                ds=(cd, blk.downsample[1], a.data_ptr(), cin, L, yd), merged_branch=True)
                elif self.bn == "frozen":
                    # out = relu(bn(y) + bn_d(y_d)): one pass over both branches
                    self.conv_fwd(cl, h.data_ptr(), ch, yl.data_ptr(), cout, lh, src_last_use=True)
                    self.conv_fwd(cd, a.data_ptr(), cin, yd.data_ptr(), cout, L)
                    stl = self.bn_affine_apply(bnl, yl.data_ptr(), cout, out.data_ptr(), cout, N * lo, cout, True,
                                               second=(blk.downsample[1], yd.data_ptr(), cout))
                    std = self._coef[id(blk.downsample[1])]
                else:
                    self.conv_fwd(cl, h.data_ptr(), ch, yl.data_ptr(), cout, lh, src_last_use=True)
                    self.conv_fwd(cd, a.data_ptr(), cin, yd.data_ptr(), cout, L)
                    res = self.scratch("ds_res", (N, lo, cout))
                    std = self.gbn_fwd(blk.downsample[1], yd.data_ptr(), cout, res.data_ptr(), cout, self.group * lo,
                                       cout, False)
                    stl = self.gbn_fwd(bnl, yl.data_ptr(), cout, out.data_ptr(), cout, self.group * lo, cout, True,
                                       res=res.data_ptr(), res_stride=cout)
                r.update(cd=cd, yd=yd, std=std)
            elif ml:
                stl, _ = self.conv_bn_fwd(cl, bnl, h.data_ptr(), ch, lh, yl, out, True, res=a, src_last_use=True)
            else:
                self.conv_fwd(cl, h.data_ptr(), ch, yl.data_ptr(), cout, lh, src_last_use=True)
                stl = self.gbn_fwd(bnl, yl.data_ptr(), cout, out.data_ptr(), cout, self.group * lo, cout, True,
                                   res=a.data_ptr(), res_stride=cout)
            stages.append(dict(c=cl, bn=bnl, src=h, cin=ch, l_in=lh, y=yl, act=out, st=stl))
            r.update(stages=stages, out=out)
            self.sites[site + ".relu%d" % len(stages)] = out
            recs.append(r)
            a = out
        L, f = blocks[-1][3], blocks[-1][5]
        self._head_fwd(a.data_ptr(), f, L, f)

        # ---------------- backward ----------------
        d_out = self.scratch("gA", (N, L, f))
        self._head_bwd(d_out.data_ptr(), f, L, f)
        for (blk, _, l_in, lo, cin, cout), r in zip(reversed(blocks), reversed(recs)):
            stages = r["stages"]
            last = stages[-1]
            # out = relu(bn(y) + res):  g = d_out * (out > 0) written over d_out; dy = the last BatchNorm's backward
            dy = self.scratch("gB", (N, lo, cout))
            self.gbn_bwd(last["bn"], last["st"], d_out.data_ptr(), cout, last["y"].data_ptr(), cout, dy.data_ptr(), cout,
                         self.group * lo, cout, 2, mask=r["out"].data_ptr(), mask_stride=cout, dres=d_out.data_ptr(),
                         dres_stride=cout)
            # back through the main branch to the first stage's output gradient
            for k in range(len(stages) - 1, 0, -1):
                s, prev = stages[k], stages[k - 1]
                cp = prev["c"].cout
                # wgrad before dgrad: measured 1 % faster per step than the other order (the BatchNorm backward that
                # follows finds dgrad's output still in L2)
                self.conv_wgrad(s["c"], s["src"].data_ptr(), s["cin"], dy.data_ptr(), s["c"].cout, s["l_in"])
                da = self.scratch("gC" if k == len(stages) - 1 else "gD", (N, s["l_in"], cp))
                self.conv_dgrad(s["c"], dy.data_ptr(), s["c"].cout, da.data_ptr(), cp, s["l_in"])
                # prev's output = relu(bn(y)): its y gradient in place over da
                self.gbn_bwd(prev["bn"], prev["st"], da.data_ptr(), cp, prev["y"].data_ptr(), cp, da.data_ptr(), cp,
                             self.group * s["l_in"], cp, 1)
                dy = da
            c1, p1 = stages[0]["c"], stages[0]["c"].cout
            self.conv_wgrad(c1, r["a_in"].data_ptr(), cin, dy.data_ptr(), p1, l_in)
            if blk.downsample is not None:
                # residual branch: g -> BN(ds) backward in place -> conv1x1 backward
                self.gbn_bwd(blk.downsample[1], r["std"], d_out.data_ptr(), cout, r["yd"].data_ptr(), cout,
                             d_out.data_ptr(), cout, self.group * lo, cout, 0)
                self.conv_wgrad(r["cd"], r["a_in"].data_ptr(), cin, d_out.data_ptr(), cout, l_in)
                d_in = self.scratch("gA", (N, l_in, cin))
                # main branch first (writes every position), then the 1x1 downsample branch accumulates in place
                self.conv_dgrad(c1, dy.data_ptr(), p1, d_in.data_ptr(), cin, l_in)
                self.conv_dgrad(r["cd"], d_out.data_ptr(), cout, d_in.data_ptr(), cin, l_in, addend=d_in.data_ptr(),
                                addend_stride=cin)
            else:
                d_in = d_out  # g is the identity-branch gradient: accumulate conv1's dgrad onto it in place
                self.conv_dgrad(c1, dy.data_ptr(), p1, d_in.data_ptr(), cin, l_in, addend=d_out.data_ptr(),
                                addend_stride=cout)
            d_out = d_in
            self.mark(blk.conv1.weight)
        if m.double_conv_first:
            self._double_stem_bwd(pool, c0, stem_st, d_out.data_ptr())
        else:
            self._stem_bwd(m.conv1, m.bn1, pool, stem_st, d_out.data_ptr(), c0)

    # ------------------------------------------------------------------------------------------------------
    # two-convolution stem (double_conv_first=True, resnet.py:145-150):
    #   a0 = bn1(conv1_alt(x))  (N,224,C0)   stage 1, stem.cu (no ReLU)
    #   r2 = relu(bn2(conv2(a0)))  (N,112,C0)   the generic convolution (k7, s2, p3) + BatchNorm, site "relu0"
    #   a  = first_pool(r2)  (N,56,C0)   dards_pool3s2
    # conv2 zero-pads a0, the BatchNorm output, so the two convolutions are not one 9-tap convolution of x.
    # ------------------------------------------------------------------------------------------------------
    def _double_stem_fwd(self, pool, c0, a_ptr):
        m, N = self.backbone, self.N
        self._check_double_stem(c0)
        c2 = self.conv(m.conv2)
        a0 = self.new((N, SEQ_LEN, c0))
        y2 = self.new((N, 112, c0))
        r2 = self.new((N, 112, c0))
        mean1, rstd1 = self.stats(c0)
        ws, ws_bytes = self._stem_alt_ws(c0, 0)
        self.fwd.add("dards_stem_alt_fwd", self.x_buf.data_ptr(), m.conv1_alt.weight.data_ptr(), m.bn1.weight.data_ptr(),
                     m.bn1.bias.data_ptr(), a0.data_ptr(), mean1.data_ptr(), rstd1.data_ptr(), self.G, self.group, c0, c0,
                     BN_EPS, ws, ws_bytes, self.dt)
        self._note_running(m.bn1, mean1, rstd1, self.group * SEQ_LEN, c0)
        if self.cb_mode(c2, SEQ_LEN):
            st2, _ = self.conv_bn_fwd(c2, m.bn2, a0.data_ptr(), c0, SEQ_LEN, y2, r2, True)
        else:
            self.conv_fwd(c2, a0.data_ptr(), c0, y2.data_ptr(), c0, SEQ_LEN)
            st2 = self.gbn_fwd(m.bn2, y2.data_ptr(), c0, r2.data_ptr(), c0, self.group * 112, c0, True)
        self.fwd.add("dards_pool3s2_fwd", r2.data_ptr(), a_ptr, N, 112, c0, c0, c0, pool, self.dt)
        self.sites["relu0"] = r2
        return dict(c2=c2, a0=a0, y2=y2, r2=r2, st1=(mean1, rstd1), st2=st2)

    def _double_stem_bwd(self, pool, c0, r, d_a):
        """d_a: gradient of the pooled stem output (N,56,C0)."""
        m, N = self.backbone, self.N
        dr2 = self.scratch("gB", (N, 112, c0))
        self.bwd.add("dards_pool3s2_bwd", d_a, r["r2"].data_ptr(), dr2.data_ptr(), N, 112, c0, c0, c0, c0, pool, self.dt)
        dy2 = self.scratch("gC", (N, 112, c0))
        self.gbn_bwd(m.bn2, r["st2"], dr2.data_ptr(), c0, r["y2"].data_ptr(), c0, dy2.data_ptr(), c0, self.group * 112, c0, 2,
                     mask=r["r2"].data_ptr(), mask_stride=c0)
        self.conv_wgrad(r["c2"], r["a0"].data_ptr(), c0, dy2.data_ptr(), c0, SEQ_LEN)
        da0 = self.scratch("gD", (N, SEQ_LEN, c0))
        self.conv_dgrad(r["c2"], dy2.data_ptr(), c0, da0.data_ptr(), c0, SEQ_LEN)
        mean1, rstd1 = r["st1"]
        dwp = self.new((self.G, c0 * 3), torch.float32)
        dgp = self.new((self.G, c0), torch.float32)
        dbp = self.new((self.G, c0), torch.float32)
        ws, ws_bytes = self._stem_alt_ws(c0, 1)
        self.bwd.add("dards_stem_alt_bwd", da0.data_ptr(), self.x_buf.data_ptr(), m.conv1_alt.weight.data_ptr(),
                     m.bn1.weight.data_ptr(), mean1.data_ptr(), rstd1.data_ptr(), dwp.data_ptr(), dgp.data_ptr(),
                     dbp.data_ptr(), self.G, self.group, c0, c0, ws, ws_bytes, self.dt)
        if self.input_grad:
            self.bwd.add("dards_stem_alt_dgrad", da0.data_ptr(), self.x_buf.data_ptr(), m.conv1_alt.weight.data_ptr(),
                         m.bn1.weight.data_ptr(), mean1.data_ptr(), rstd1.data_ptr(), dgp.data_ptr(), dbp.data_ptr(),
                         self.dx.data_ptr(), self.G, self.group, c0, c0, self.dt)
        self._pending_red.append((dwp, self.G, c0 * 3, self.gptr(m.conv1_alt.weight)))
        self._pending_red.append((dgp, self.G, c0, self.gptr(m.bn1.weight)))
        self._pending_red.append((dbp, self.G, c0, self.gptr(m.bn1.bias)))
        self._flush_reductions()

    def _double_stem_eval(self, pool, c0, a_ptr):
        """Eval plans: stage 1 with bn1's running-statistics affine map, then conv2 with bn2 + ReLU in its epilogue, then
        the pool.  a0 and r2 get buffers of their own (a0 is four times the largest block activation)."""
        m, N = self.backbone, self.N
        self._check_double_stem(c0)
        co = self._coef[id(m.bn1)]
        a0 = self.new((N, SEQ_LEN, c0))
        r2 = self.new((N, 112, c0))
        self.act_bytes += (a0.numel() + r2.numel()) * a0.element_size()
        self.eval_reads.add(id(m.conv1_alt.weight))
        self.fwd.add("dards_stem_alt_eval_fwd", self.x_buf.data_ptr(), m.conv1_alt.weight.data_ptr(), co.scale, co.shift,
                     a0.data_ptr(), N, c0, c0, self.dt)
        self.conv_affine_fwd(self.conv(m.conv2), m.bn2, a0.data_ptr(), c0, SEQ_LEN, r2.data_ptr(), True, src_last_use=True)
        self.fwd.add("dards_pool3s2_fwd", r2.data_ptr(), a_ptr, N, 112, c0, c0, c0, pool, self.dt)

    def _check_double_stem(self, c0):
        m = self.backbone
        shapes = ((m.conv1_alt, 1, 3, 1, 1), (m.conv2, c0, 7, 2, 3))
        for conv, cin, k, s, p in shapes:
            if (conv.in_channels, conv.out_channels, conv.kernel_size[0], conv.stride[0], conv.padding[0]) != (cin, c0, k, s, p):
                raise NotImplementedError("double_conv_first stem must be Conv1d(1, C0, 3, 1, 1) then Conv1d(C0, C0, 7, 2, 3)")
        if c0 % 16:
            raise NotImplementedError("double_conv_first stem: initial planes must be a multiple of 16 (got %d)" % c0)

    def _stem_alt_ws(self, c0, backward):
        nbytes = _lib.fn("dards_stem_alt_workspace_bytes")(self.G, self.group, c0, backward)
        if not nbytes:
            return None, 0
        t = self.new(((nbytes + 3) // 4,), torch.float32)
        return t.data_ptr(), t.numel() * 4

    # ------------------------------------------------------------------------------------------------------
    # ResNet in eval(): BatchNorm with the running statistics, a fixed per-channel affine map per layer
    # ------------------------------------------------------------------------------------------------------
    def _eval_coeffs(self, with_rstd=False):
        """Coef of every BatchNorm layer of the ResNet's forward (resnet_bn_layers): scale / shift in fp32, 16-byte aligned
        slots, computed by ONE launch at the start of every forward: load_state_dict() and `.data` edits change the running
        buffers in place, so values taken when the plan is built would go stale.  Returns {id(bn): Coef}.
        with_rstd (frozen plans, whose backward needs the normalised input): the same launch also evaluates every layer with
        gamma = 1, beta = 0, i.e. rstd = 1/sqrt(running_var + eps), in descriptors after the scale / shift ones."""
        bns = [bn for _, bn in resnet_bn_layers(self.backbone)]
        for bn in bns:
            if getattr(bn, "running_mean", None) is None or getattr(bn, "running_var", None) is None:
                raise NotImplementedError("eval() with a BatchNorm layer that keeps no running statistics "
                                          "(track_running_stats=False) is not implemented on the B200 backend")
        slots = [(bn.num_features + 3) // 4 * 4 for bn in bns]
        coef = self.new((4 if with_rstd else 2, max(sum(slots), 4)), torch.float32)
        if with_rstd:
            unit = self.new((2, max(bn.num_features for bn in bns)), torch.float32)
            unit[0].fill_(1.0)
            unit[1].zero_()
        descs, rstd_descs, out, off = [], [], {}, 0
        for bn, slot in zip(bns, slots):
            rm, rv, c = bn.running_mean.data_ptr(), bn.running_var.data_ptr(), bn.num_features
            sc, sh = coef[0].data_ptr() + 4 * off, coef[1].data_ptr() + 4 * off
            descs.append((bn.weight.data_ptr(), bn.bias.data_ptr(), rm, rv, sc, sh, c))
            out[id(bn)] = Coef(sc, sh, None, None)
            if with_rstd:
                rs = coef[2].data_ptr() + 4 * off
                rstd_descs.append((unit[0].data_ptr(), unit[1].data_ptr(), rm, rv, rs, coef[3].data_ptr() + 4 * off, c))
                out[id(bn)] = Coef(sc, sh, rs, rm)
            self.eval_reads.update((id(bn.weight), id(bn.bias)))
            off += slot
        t, total = _lib.desc_table(_lib.EvalCoeffDesc, descs + rstd_descs, self.device)
        self.bufs.append(t)
        self.fwd.add("dards_bn_eval_coeffs_batched", t.data_ptr(), len(descs) + len(rstd_descs), total, BN_EPS)
        return out

    def conv_affine_fwd(self, c, bn, src, src_stride, l_in, dst, relu, res=None, src_last_use=False):
        """dst = [relu](bn_eval(conv(src)) [+ res]): one launch, BatchNorm / residual / ReLU in the convolution epilogue.
        `dst` and `res` are (N, l_out, cout) pointers."""
        l_out = (l_in + 2 * c.pad - c.k) // c.stride + 1
        tc = self._tc_ok(c, "fwd")
        w = c.koi if tc else c.kio
        co = self._coef[id(bn)]
        self.eval_reads.add(id(c.mod.weight))
        self.fwd.add("dards_conv1d_affine_fwd", src, w.data_ptr(), dst, res, co.scale, co.shift, self.N, l_in, l_out, c.cin,
                     c.cout, src_stride, c.cout, c.cout if res is not None else 0, c.k, c.stride, c.pad,
                     (1 if relu else 0) | (_lib.HINT_LAST_USE if src_last_use else 0), self.dt, 1 if tc else 0)

    def _build_resnet_eval(self):
        """Forward only: pack, coefficients, eval stem, then per block conv1 -> affine + ReLU and conv2 -> affine + residual +
        ReLU (the downsample branch -> affine into a scratch buffer first), avgpool, head.  No statistics, no running-statistics
        update, no gradient buffers.  Activations rotate through four buffers, each the size of the largest (N, L, C)
        activation: block input (= identity residual), the main branch's inner activation, downsample output, block output.
        A Bottleneck's two inner activations take turns in the same two buffers: conv2 reads a1 and writes a2, and nothing
        reads a1 after that, so its buffer takes the downsample output."""
        m = self.backbone
        pool, c0, blocks = self._resnet_blocks()
        N = self.N
        self._coef = self._eval_coeffs()
        largest = max([56 * c0] + [lo * cout for _, _, _, lo, _, cout in blocks])
        pool_bufs = [self.new((N * largest,)) for _ in range(4)]
        self.act_bytes = sum(t.numel() * t.element_size() for t in pool_bufs)

        def free(*busy):
            return next(t for t in pool_bufs if all(t is not b for b in busy))

        a = pool_bufs[0]
        if m.double_conv_first:
            self._double_stem_eval(pool, c0, a.data_ptr())
        else:
            self._stem(m.conv1, m.bn1, pool, a.data_ptr(), c0)
        for blk, _, L, lo, cin, cout in blocks:
            stages = self._block_stages(blk)
            convs = [self.conv(conv) for conv, _ in stages]
            h, lh = a, L
            for i, (c, (_, bn)) in enumerate(zip(convs[:-1], stages[:-1])):
                # the main branch's inner stages: affine + ReLU; a Bottleneck's a1 is free again once a2 is written
                nxt = free(a, h)
                self.conv_affine_fwd(c, bn, h.data_ptr(), c.cin, lh, nxt.data_ptr(), True, src_last_use=i > 0)
                h, lh = nxt, (lh + 2 * c.pad - c.k) // c.stride + 1
            if blk.downsample is not None:
                cd = self.conv(blk.downsample[0])
                res = free(a, h)
                self.conv_affine_fwd(cd, blk.downsample[1], a.data_ptr(), cin, L, res.data_ptr(), False, src_last_use=True)
            else:
                res = a
            out = free(a, h, res)
            self.conv_affine_fwd(convs[-1], stages[-1][1], h.data_ptr(), convs[-1].cin, lh, out.data_ptr(), True,
                                 res=res.data_ptr(), src_last_use=True)
            a = out
        L, f = blocks[-1][3], blocks[-1][5]
        self._head_fwd(a.data_ptr(), f, L, f)
        if self.linear is not None and self.mode in ("cnn_linear", "per_breath"):
            self.eval_reads.update((id(self.linear.weight), id(self.linear.bias)))

    # ------------------------------------------------------------------------------------------------------
    # DenseNet
    # ------------------------------------------------------------------------------------------------------
    def _build_densenet(self):
        m = self.backbone
        feats = getattr(m, "features", m)  # `m` may be the DenseNet or its `.features` container
        N = self.N
        if feats.conv0.in_channels != 1:
            raise NotImplementedError("densenet with_fft / only_fft inputs are not implemented on the B200 backend")
        blocks = [(n, mod) for n, mod in feats.named_children() if n.startswith("denseblock")]
        trans = dict((n, mod) for n, mod in feats.named_children() if n.startswith("transition"))
        c0 = feats.conv0.out_channels
        L = 56
        # concat buffer of block 1: stem output goes to channels [0, c0)
        layers0 = list(blocks[0][1].children())
        growth = layers0[0].conv2.out_channels
        ctot = c0 + growth * len(layers0)
        cat = self.new((N, L, ctot), zero=True)
        stem_st = self._stem(feats.conv0, feats.norm0, 0, cat.data_ptr(), ctot)
        esz = cat.element_size()
        brecs = []
        cin0 = c0
        drop_id = 0
        for bi, (bname, block) in enumerate(blocks):
            lrecs = []
            cin = cin0
            for lname, layer in block.named_children():
                c1, c2 = self.conv(layer.conv1), self.conv(layer.conv2)
                mid, g = c1.cout, c2.cout
                rows = self.group * L
                a = self.new((N, L, cin))
                st1 = self.gbn_fwd(layer.norm1, cat.data_ptr(), ctot, a.data_ptr(), cin, rows, cin, True, x_last_use=False)
                y1 = self.new((N, L, mid))
                b = self.new((N, L, mid))
                if self.cb_mode(c1, L):
                    st2, _ = self.conv_bn_fwd(c1, layer.norm2, a.data_ptr(), cin, L, y1, b, True, src_last_use=True)
                else:
                    self.conv_fwd(c1, a.data_ptr(), cin, y1.data_ptr(), mid, L, src_last_use=True)
                    st2 = self.gbn_fwd(layer.norm2, y1.data_ptr(), mid, b.data_ptr(), mid, rows, mid, True)
                self.conv_fwd(c2, b.data_ptr(), mid, cat.data_ptr(), ctot, L, dst_ptr_off=cin * esz, src_last_use=True)
                seed = None
                drop_p = float(getattr(layer, "drop_rate", 0.0)) if self.dropout else 0.0
                if drop_p > 0.0:
                    drop_id += 1
                    seed = 0x5DEECE66D * drop_id + 11
                    self.fwd.add("dards_dropout", cat.data_ptr() + cin * esz, N * L, g, ctot, drop_p, seed,
                                 self.seed_dev.data_ptr(), self.group * L, self.dt)
                self.sites["%s.%s.relu1" % (bname, lname)] = a
                self.sites["%s.%s.relu2" % (bname, lname)] = b
                lrecs.append(dict(layer=layer, c1=c1, c2=c2, a=a, st1=st1, y1=y1, b=b, st2=st2, cin=cin, mid=mid, g=g,
                                  seed=seed, drop_p=drop_p))
                cin += g
            if cin != ctot:
                raise RuntimeError("dense block channel bookkeeping is off")
            br = dict(layers=lrecs, cat=cat, ctot=ctot, L=L, cin0=cin0)
            tname = "transition%d" % (bi + 1)
            if tname in trans:
                t = trans[tname]
                ct = self.conv(t.conv)
                rows = self.group * L
                a = self.new((N, L, ctot))
                stt = self.gbn_fwd(t.norm, cat.data_ptr(), ctot, a.data_ptr(), ctot, rows, ctot, True, x_last_use=False)
                y = self.new((N, L, ct.cout))
                self.conv_fwd(ct, a.data_ptr(), ctot, y.data_ptr(), ct.cout, L, src_last_use=True)
                nxt_layers = list(blocks[bi + 1][1].children())
                ntot = ct.cout + nxt_layers[0].conv2.out_channels * len(nxt_layers)
                ncat = self.new((N, L // 2, ntot), zero=True)
                self.fwd.add("dards_avgpool2_fwd", y.data_ptr(), ncat.data_ptr(), N, L, ct.cout, ct.cout, ntot, self.dt)
                br.update(trans=t, ct=ct, ta=a, tst=stt, ty=y)
                self.sites["%s.relu" % tname] = a
                brecs.append(br)
                cat, ctot, L, cin0 = ncat, ntot, L // 2, ct.cout
            else:
                brecs.append(br)
        f = ctot
        if L != 7:
            raise RuntimeError("unexpected final length %d" % L)
        # norm5 (+ ReLU for the pooled head; the raw map for 'features' / GradCAM)
        rows = self.group * L
        if self.mode == "features":
            self.feat_map = self.new((N, L, f))
            st5 = self.gbn_fwd(feats.norm5, cat.data_ptr(), ctot, self.feat_map.data_ptr(), f, rows, f, False,
                               x_last_use=False)
            self.dfeat_map = self.new((N, L, f))
            d_act, relu5 = self.dfeat_map, 0
            self.out_features = f
        else:
            act = self.new((N, L, f))
            st5 = self.gbn_fwd(feats.norm5, cat.data_ptr(), ctot, act.data_ptr(), f, rows, f, True, x_last_use=False)
            self._head_fwd(act.data_ptr(), f, L, f)
            self.sites["relu5"] = act
            d_act, relu5 = self.scratch("d_act", (N, L, f)), 1
            self._head_bwd(d_act.data_ptr(), f, L, f)

        # ---------------- backward ----------------
        d_cat = self.scratch("d_cat%d" % L, (N, L, ctot))
        self.gbn_bwd(feats.norm5, st5, d_act.data_ptr(), f, cat.data_ptr(), ctot, d_cat.data_ptr(), ctot, rows, f, relu5)
        for bi in range(len(brecs) - 1, -1, -1):
            br = brecs[bi]
            cat, ctot, L = br["cat"], br["ctot"], br["L"]
            rows = self.group * L
            for lr in reversed(br["layers"]):
                layer, cin, mid, g = lr["layer"], lr["cin"], lr["mid"], lr["g"]
                dnew = d_cat.data_ptr() + cin * esz  # (N, L, g) slice, row stride ctot
                if lr["seed"] is not None:
                    self.bwd.add("dards_dropout", dnew, N * L, g, ctot, lr["drop_p"], lr["seed"], self.seed_dev.data_ptr(),
                                 self.group * L, self.dt)
                self.conv_wgrad(lr["c2"], lr["b"].data_ptr(), mid, dnew, ctot, L)
                db = self.scratch("d_mid", (N, L, mid))
                self.conv_dgrad(lr["c2"], dnew, ctot, db.data_ptr(), mid, L)
                self.gbn_bwd(layer.norm2, lr["st2"], db.data_ptr(), mid, lr["y1"].data_ptr(), mid, db.data_ptr(), mid, rows,
                             mid, 1)
                self.conv_wgrad(lr["c1"], lr["a"].data_ptr(), cin, db.data_ptr(), mid, L)
                da = self.scratch("d_a", (N, L, cin))
                self.conv_dgrad(lr["c1"], db.data_ptr(), mid, da.data_ptr(), cin, L)
                self.gbn_bwd(layer.norm1, lr["st1"], da.data_ptr(), cin, cat.data_ptr(), ctot, d_cat.data_ptr(), ctot,
                             rows, cin, 1, accumulate=True)
                self.mark(layer.norm1.weight)
            if bi > 0:
                pr = brecs[bi - 1]
                pL, pct, ct = pr["L"], pr["ctot"], pr["ct"]
                dy = self.scratch("d_ty", (N, pL, ct.cout))
                self.bwd.add("dards_avgpool2_bwd", d_cat.data_ptr(), dy.data_ptr(), N, pL, ct.cout, ctot, ct.cout, self.dt)
                self.conv_wgrad(ct, pr["ta"].data_ptr(), pct, dy.data_ptr(), ct.cout, pL)
                dta = self.scratch("d_ta", (N, pL, pct))
                self.conv_dgrad(ct, dy.data_ptr(), ct.cout, dta.data_ptr(), pct, pL)
                d_prev = self.scratch("d_cat%d" % pL, (N, pL, pct))
                self.gbn_bwd(pr["trans"].norm, pr["tst"], dta.data_ptr(), pct, pr["cat"].data_ptr(), pct, d_prev.data_ptr(),
                             pct, self.group * pL, pct, 1)
                self.mark(pr["trans"].norm.weight)
                d_cat = d_prev
            else:
                self._stem_bwd(feats.conv0, feats.norm0, 0, stem_st, d_cat.data_ptr(), ctot)

    # ------------------------------------------------------------------------------------------------------
    # execution
    # ------------------------------------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _build_pack_table(self):
        """One `dards_pack_desc` per convolution, uploaded once: the whole network's weights are re-packed by a
        single launch whenever they change."""
        descs = [(c.mod.weight.data_ptr(), c.kio.data_ptr(), c.koi.data_ptr(), c.cout, c.cin, c.k) for c in self.convs]
        self.pack_table, total = _lib.desc_table(_lib.PackDesc, descs, self.device)
        self.bufs.append(self.pack_table)
        self.pack.add("dards_pack_conv_weights_batched", self.pack_table.data_ptr(), len(descs), total, self.dt)

    def _pack_if_needed(self, st):
        ver = 0
        for c in self.convs:
            ver += c.mod.weight._version
        if ver != self._packed_version:
            self.pack.run(st)
            self._packed_version = ver

    def load_input(self, x):
        """x: (..., 1, 224) or (N, 224) float tensor on the plan's device -> static input buffer."""
        if x.shape[-1] != SEQ_LEN or x.numel() != self.N * SEQ_LEN:
            raise RuntimeError("plan was built for %d breaths of %d samples, got %s" % (self.N, SEQ_LEN, tuple(x.shape)))
        self.x_buf.copy_(x.reshape(self.N, SEQ_LEN), non_blocking=True)

    def load_raw(self, raw, mu, std, padded=False):
        """The dataset's scaling step fused into the input load (dataset.py:1375-1379, train_ards_detector.py:150-151):
        raw float64 / float32 windows on the device -> (raw - mu) / std as float32, straight into the static input
        buffer (float64 arithmetic, one rounding: bit-exact with the reference's numpy + .float())."""
        if raw.shape[-1] != SEQ_LEN or raw.numel() != self.N * SEQ_LEN:
            raise RuntimeError("plan was built for %d breaths of %d samples, got %s" % (self.N, SEQ_LEN, tuple(raw.shape)))
        if raw.device != self.device or raw.dtype not in (torch.float64, torch.float32):
            raise RuntimeError("raw windows must be float64 / float32 tensors on %s" % (self.device,))
        raw = raw.contiguous()
        _lib.call("dards_scale_windows", raw.data_ptr(), 1 if raw.dtype == torch.float64 else 0, self.x_buf.data_ptr(),
                  raw.numel(), float(mu), float(std), 1 if padded else 0, self._stream())

    # The autograd path (`net(x)` -> loss.backward(), what train_ards_detector.py drives) replays the recorded forward and
    # backward as two CUDA graphs after two eager calls: ~260 launches issued one by one from Python through ctypes
    # otherwise.  The weight re-packing launch is part of the forward graph, i.e. it runs on EVERY forward: the packed
    # copies can then never be stale, whatever edits the parameters between two calls (optimizer.step(), `.data` edits,
    # weight averaging, ...).  DEEPARDS_B200_PLAN_GRAPH=0 keeps everything eager.
    def _graph_for(self, which, run):
        if os.environ.get("DEEPARDS_B200_PLAN_GRAPH", "1") == "0" or torch.cuda.is_current_stream_capturing():
            return None     # inside somebody else's capture (the trainer's whole-step graph): just record the launches
        st = self.__dict__.setdefault("_graphs", {})
        ent = st.setdefault(which, {"calls": 0, "graph": None})
        if ent["graph"] is None:
            ent["calls"] += 1
            if ent["calls"] <= 2:
                return None
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                run(self._stream())
            ent["graph"] = g
        return ent["graph"]

    def drop_graphs(self):
        self.__dict__.pop("_graphs", None)

    def set_sequence_offset(self, first_sequence):
        """Index of this call's first sequence in the global (all-ranks) batch: the dropout masks are keyed by the global
        sequence index, so a sharded step draws the masks of the unsharded one."""
        first_sequence = int(first_sequence)
        if first_sequence != self._seq_offset:
            self.seed_dev[1] = first_sequence
            self._seq_offset = first_sequence

    def run_forward(self):
        if self.dropout:
            self.seed_dev[0:1].add_(1)

        def run(st):
            self.pack.run(st)
            self.fwd.run(st)

        with nvtx_range("deepards_b200.forward"):
            g = self._graph_for("fwd", run)
            if g is not None:
                g.replay()
            else:
                run(self._stream())
        self.fwd_serial += 1

    def run_backward(self):
        if self.bwd_serial == self.fwd_serial:
            raise RuntimeError("backward() without a new forward(): forward #%d has already been back-propagated "
                               "(in-place backward kernels consumed its buffers)" % self.fwd_serial)
        with nvtx_range("deepards_b200.backward"):
            g = self._graph_for("bwd", self.bwd.run)
            if g is not None:
                g.replay()
            else:
                self.bwd.run(self._stream())
        self.bwd_serial = self.fwd_serial

    def mark_no_backward(self):
        """forward-only use (no_grad): keep the serial numbers consistent."""
        self.bwd_serial = self.fwd_serial

    def autograd_params(self):
        """The parameters that receive a gradient from this plan's backward, in named_parameters() order.  An eval plan has
        no backward: there they are the parameters its forward reads, so that an output computed with grad enabled stays
        attached to a node whose backward says so."""
        ids = self.eval_reads if self.bn == "eval" else self.grad_written
        return [p for _, p in self.params if id(p) in ids]

    def grads(self):
        """{param: gradient view} for every parameter the backward writes (fresh copy of the flat buffer)."""
        flat = self.grad_flat.clone()
        out = {}
        for n, p in self.params:
            if id(p) in self.grad_written:
                off = self.goff[id(p)]
                out[id(p)] = flat[off:off + p.numel()].view(p.shape)
        return out


def get_plan(net, backbone, linear, n_breaths, group, precision, mode, dropout, update_running, bn="train",
             input_grad=False):
    """Plan cache on the owning module (invalidated when a parameter's storage moves)."""
    cache = net.__dict__.setdefault("_dards_plans", {})
    # multi-rank plans flush their pending partial-sum reductions at every all-reduce mark: a plan built before
    # init_process_group() must not be reused afterwards
    key = (n_breaths, group, precision, mode, tuple(dropout), bool(update_running), _multi_rank())
    if bn != "train":
        key += (bn,)
    if input_grad:
        key += ("input_grad",)
    plan = cache.get(key)
    if plan is None or not plan.valid():
        plan = Plan(net, backbone, linear, n_breaths, group, precision, mode, dropout, update_running, bn, input_grad)
        cache[key] = plan
    return plan

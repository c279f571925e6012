"""Tensor-level wrappers of the C ABI (one Python function per entry point).

These allocate outputs with torch and call the library immediately on the current stream.  The networks do
not use them (they replay recorded plans, engine.py); the per-kernel parity tests and ad-hoc users do.
All activation tensors are channels-last: (N, L, C), contiguous or a channel slice of a wider buffer.
"""
import torch

from . import _lib

_DT = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _st(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _dt(t):
    return _DT[t.dtype]


def _rowstride(t):
    assert t.dim() == 3 and t.stride(2) == 1 and t.stride(0) == t.shape[1] * t.stride(1), "need (N, L, C) rows"
    return t.stride(1)


def pack_conv_weight(w, dtype):
    cout, cin, k = w.shape
    kio = torch.empty((k, cin, cout), dtype=dtype, device=w.device)
    koi = torch.empty((k, cout, cin), dtype=dtype, device=w.device)
    _lib.call("dards_pack_conv_weight", w.data_ptr(), kio.data_ptr(), koi.data_ptr(), cout, cin, k, _DT[dtype], _st(w))
    return kio, koi


def conv1d_fwd(x, w, stride, pad, impl=0, out=None, addend=None):
    """x (N, L, Cin) channels-last; w (Cout, Cin, K) fp32 -> (N, Lout, Cout)."""
    n, l, cin = x.shape
    cout, _, k = w.shape
    lo = (l + 2 * pad - k) // stride + 1
    kio, koi = pack_conv_weight(w, x.dtype)
    if out is None:
        out = torch.empty((n, lo, cout), dtype=x.dtype, device=x.device)
    _lib.call("dards_conv1d_fwd", x.data_ptr(), (koi if impl == 1 else kio).data_ptr(), out.data_ptr(),
              addend.data_ptr() if addend is not None else None, n, l, lo, cin, cout, _rowstride(x), _rowstride(out),
              _rowstride(addend) if addend is not None else 0, k, stride, pad, _dt(x), impl, _st(x))
    return out


def conv1d_affine_fwd(x, w, scale, shift, stride, pad, impl=0, res=None, relu=True, out=None):
    """out = [relu](conv(x) * scale + shift [+ res]): eval-mode BatchNorm in the convolution epilogue."""
    n, l, cin = x.shape
    cout, _, k = w.shape
    lo = (l + 2 * pad - k) // stride + 1
    kio, koi = pack_conv_weight(w, x.dtype)
    if out is None:
        out = torch.empty((n, lo, cout), dtype=x.dtype, device=x.device)
    _lib.call("dards_conv1d_affine_fwd", x.data_ptr(), (koi if impl == 1 else kio).data_ptr(), out.data_ptr(),
              res.data_ptr() if res is not None else None, scale.data_ptr(), shift.data_ptr(), n, l, lo, cin, cout,
              _rowstride(x), _rowstride(out), _rowstride(res) if res is not None else 0, k, stride, pad, 1 if relu else 0,
              _dt(x), impl, _st(x))
    return out


def bn_eval_coeffs(layers, eps=1e-5):
    """layers: [(gamma, beta, running_mean, running_var)] fp32 -> [(scale, shift)], one batched launch."""
    outs = [(torch.empty_like(g), torch.empty_like(g)) for g, _, _, _ in layers]
    descs = [(g.data_ptr(), b.data_ptr(), rm.data_ptr(), rv.data_ptr(), sc.data_ptr(), sh.data_ptr(), g.numel())
             for (g, b, rm, rv), (sc, sh) in zip(layers, outs)]
    t, total = _lib.desc_table(_lib.EvalCoeffDesc, descs, layers[0][0].device)
    _lib.call("dards_bn_eval_coeffs_batched", t.data_ptr(), len(layers), total, eps, _st(t))
    torch.cuda.current_stream(t.device).synchronize()  # the table is freed on return
    return outs


def stem_eval_fwd(x, w, scale, shift, pool, dtype):
    """x (N, 224) fp32 -> (N, 56, C0): conv -> y*scale + shift -> ReLU -> pool (eval-mode BatchNorm)."""
    n, c0 = x.shape[0], w.shape[0]
    out = torch.empty((n, 56, c0), dtype=dtype, device=x.device)
    _lib.call("dards_stem_eval_fwd", x.data_ptr(), w.data_ptr(), scale.data_ptr(), shift.data_ptr(), out.data_ptr(), n, c0,
              c0, pool, _DT[dtype], _st(x))
    return out


def _reduce_rows(part):
    """(rows, c) fp32 partials -> (c,) sums in a fixed order."""
    rows, c = part.shape
    out = torch.empty((c,), dtype=torch.float32, device=part.device)
    _lib.call("dards_reduce_rows", part.data_ptr(), out.data_ptr(), rows, c, 0, _st(part))
    return out


def bn_affine_apply(y, scale, shift, res=None, relu=True, second=None, out=None):
    """out = [relu](y * scale + shift [+ res] [+ y2 * scale2 + shift2]) over (N, L, C) rows (BatchNorm with the running
    statistics); second = (y2, scale2, shift2)."""
    n, l, c = y.shape
    if out is None:
        out = torch.empty((n, l, c), dtype=y.dtype, device=y.device)
    y2, s2, h2 = second if second is not None else (None, None, None)
    _lib.call("dards_bn_affine_apply", y.data_ptr(), out.data_ptr(), res.data_ptr() if res is not None else None,
              scale.data_ptr(), shift.data_ptr(), y2.data_ptr() if y2 is not None else None,
              s2.data_ptr() if s2 is not None else None, h2.data_ptr() if h2 is not None else None, n * l, c, _rowstride(y),
              _rowstride(out), _rowstride(res) if res is not None else 0, _rowstride(y2) if y2 is not None else 0,
              1 if relu else 0, _dt(y), _st(y))
    return out


def bn_frozen_bwd(dout, y, scale, shift, running_mean, rstd, relu_mode, mask_src=None, want_dres=False, dx=None,
                  accumulate=False, tile_rows=None):
    """Backward of bn_affine_apply with constant statistics: -> (dx, dgamma, dbeta, dres or None).  `dx` may be given
    (and accumulated into); tile_rows splits the N*L rows into tiles for the partial sums (default: one tile per breath)."""
    n, l, c = y.shape
    rows = n * l
    tile = tile_rows or l
    assert rows % tile == 0
    tiles = rows // tile
    if dx is None:
        dx = torch.empty_like(y)
    dres = torch.empty_like(dout) if want_dres else None
    dg = torch.empty((tiles, c), dtype=torch.float32, device=y.device)
    db = torch.empty((tiles, c), dtype=torch.float32, device=y.device)
    _lib.call("dards_bn_frozen_bwd", dout.data_ptr(), y.data_ptr(), mask_src.data_ptr() if mask_src is not None else None,
              scale.data_ptr(), shift.data_ptr(), running_mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(),
              1 if accumulate else 0, dres.data_ptr() if dres is not None else None, dg.data_ptr(), db.data_ptr(), tiles, tile,
              c, _rowstride(dout), _rowstride(y), _rowstride(mask_src) if mask_src is not None else 0, _rowstride(dx),
              _rowstride(dres) if dres is not None else 0, relu_mode, _dt(y), _st(y))
    return dx, _reduce_rows(dg), _reduce_rows(db), dres


def stem_frozen_bwd(dout, x, w, scale, shift, running_mean, rstd, pool):
    """dout (N, 56, C0) of stem_eval_fwd -> (dW (C0, 1, 7), dgamma, dbeta) with constant statistics."""
    n, c0 = x.shape[0], w.shape[0]
    nc = _lib.fn("dards_stem_frozen_chunks")(n)
    dwp = torch.empty((nc, c0 * 7), dtype=torch.float32, device=x.device)
    dgp = torch.empty((nc, c0), dtype=torch.float32, device=x.device)
    dbp = torch.empty((nc, c0), dtype=torch.float32, device=x.device)
    _lib.call("dards_stem_frozen_bwd", dout.data_ptr(), x.data_ptr(), w.data_ptr(), scale.data_ptr(), shift.data_ptr(),
              running_mean.data_ptr(), rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), n, c0, _rowstride(dout),
              pool, _dt(dout), _st(x))
    return _reduce_rows(dwp).view(c0, 1, 7), _reduce_rows(dgp), _reduce_rows(dbp)


def conv1d_dgrad(dout, w, l_in, stride, pad, impl=0, out=None, addend=None):
    n, lo, cout = dout.shape
    _, cin, k = w.shape
    kio, koi = pack_conv_weight(w, dout.dtype)
    if impl == 1 and addend is not None:
        # the tcgen05 path accumulates in place (TMA reduce-add): out must BE the addend
        out = addend.clone() if out is None else out.copy_(addend)
        addend = out
    if out is None:
        out = torch.empty((n, l_in, cin), dtype=dout.dtype, device=dout.device)
    _lib.call("dards_conv1d_dgrad", dout.data_ptr(), (kio if impl == 1 else koi).data_ptr(), out.data_ptr(),
              addend.data_ptr() if addend is not None else None, n, l_in, lo, cin, cout, _rowstride(dout),
              _rowstride(out), _rowstride(addend) if addend is not None else 0, k, stride, pad, _dt(dout), impl,
              _st(dout))
    return out


def conv1d_wgrad(x, dout, k, stride, pad, impl=0):
    n, l, cin = x.shape
    _, lo, cout = dout.shape
    dw = torch.empty((cout, cin, k), dtype=torch.float32, device=x.device)
    nbytes = _lib.fn("dards_conv1d_wgrad_workspace_bytes")(n, lo, cin, cout, k, impl)
    ws = torch.empty((max(nbytes // 4, 1),), dtype=torch.float32, device=x.device)
    _lib.call("dards_conv1d_wgrad", x.data_ptr(), dout.data_ptr(), dw.data_ptr(), 0, ws.data_ptr(), ws.numel() * 4, n, l,
              lo, cin, cout, _rowstride(x), _rowstride(dout), k, stride, pad, _dt(x), impl, _st(x))
    return dw


def conv1d_wgrad_accum(x, dout, k, stride, pad):
    """tcgen05 weight gradient through the accumulate path: zeroed tap-major buffer, L2 reduce-adds, one unpack launch."""
    n, l, cin = x.shape
    _, lo, cout = dout.shape
    dwt = torch.zeros((k, cout, cin), dtype=torch.float32, device=x.device)
    dw = torch.empty((cout, cin, k), dtype=torch.float32, device=x.device)
    _lib.call("dards_memset_zero", dwt.data_ptr(), dwt.numel() * 4, _st(x))
    _lib.call("dards_conv1d_wgrad_accum", x.data_ptr(), dout.data_ptr(), dwt.data_ptr(), n, l, lo, cin, cout, _rowstride(x),
              _rowstride(dout), k, stride, pad, _dt(x), _st(x))
    t, total = _lib.desc_table(_lib.UnpackDesc, [(dwt.data_ptr(), dw.data_ptr(), cout, cin, k)], x.device)
    _lib.call("dards_unpack_wgrad_batched", t.data_ptr(), 1, total, _st(x))
    torch.cuda.synchronize()
    return dw


def conv1d_bn_fwd(x, w, gamma, beta, group, stride, pad, relu, res=None, eps=1e-5, ds=None):
    """conv -> grouped BatchNorm (+ res) (+ ReLU) through the fused tcgen05 kernel (bf16 only).
    x (N, L, Cin) channels-last bf16; returns (mode, y, out, mean, rstd, extra).  mode 2: one kernel; mode 1: convolution with
    statistics partials + the streaming normalisation.  ds = (x_d, w_d, gamma_d, beta_d, stride_d, pad_d): a second
    convolution + BatchNorm branch added before the ReLU (the downsample branch of a ResNet block; mode 1 only merges
    it into the same elementwise pass, mode 2 runs it as its own fused call and passes the result as `res`)."""
    n, l, cin = x.shape
    cout, _, k = w.shape
    lo = (l + 2 * pad - k) // stride + 1
    dev = x.device
    g = n // group
    shape = (n, group, l, lo, cin, cout, k, stride, pad)
    mode = _lib.fn("dards_conv1d_bn_mode")(*shape, _dt(x))
    if mode == 0:
        raise RuntimeError("conv1d_bn_fwd: unsupported shape %r" % (shape,))
    _, koi = pack_conv_weight(w, x.dtype)
    y = torch.empty((n, lo, cout), dtype=x.dtype, device=dev)
    out = torch.empty((n, lo, cout), dtype=x.dtype, device=dev)
    mean = torch.empty((g, cout), dtype=torch.float32, device=dev)
    rstd = torch.empty((g, cout), dtype=torch.float32, device=dev)
    extra = {}
    if ds is not None:
        xd, wd, gd, bd, sd, pd = ds
        if mode == 2:
            _, _, res, md, rd, _ = conv1d_bn_fwd(xd, wd, gd, bd, group, sd, pd, False, eps=eps)
            extra = dict(mean_d=md, rstd_d=rd)
            ds = None
    entries = _lib.fn("dards_conv1d_bn_part_entries")(*shape) if mode == 1 else 0
    part = torch.empty((max(g * entries * 3 * cout, 1),), dtype=torch.float32, device=dev)
    _lib.call("dards_conv1d_bn_fwd", x.data_ptr(), koi.data_ptr(), y.data_ptr(), out.data_ptr(),
              res.data_ptr() if res is not None else None, gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(),
              rstd.data_ptr(), part.data_ptr(), n, group, l, lo, cin, cout, _rowstride(x), _rowstride(y), _rowstride(out),
              _rowstride(res) if res is not None else 0, k, stride, pad, eps, 1 if relu else 0, _dt(x), _st(x))
    if mode == 1:
        a2 = [None, None, None, None, 0, None, None]
        x2s = 0
        if ds is not None:
            xd, wd, gd, bd, sd, pd = ds
            nd, ld, cind = xd.shape
            kd = wd.shape[2]
            shape_d = (nd, group, ld, lo, cind, cout, kd, sd, pd)
            if _lib.fn("dards_conv1d_bn_mode")(*shape_d, _dt(x)) != 1:
                raise RuntimeError("conv1d_bn_fwd: the downsample branch does not run in partial-statistics mode")
            _, koid = pack_conv_weight(wd, x.dtype)
            yd = torch.empty((n, lo, cout), dtype=x.dtype, device=dev)
            ed = _lib.fn("dards_conv1d_bn_part_entries")(*shape_d)
            partd = torch.empty((g * ed * 3 * cout,), dtype=torch.float32, device=dev)
            md = torch.empty((g, cout), dtype=torch.float32, device=dev)
            rd = torch.empty((g, cout), dtype=torch.float32, device=dev)
            _lib.call("dards_conv1d_bn_fwd", xd.data_ptr(), koid.data_ptr(), yd.data_ptr(), None, None, None, None, None,
                      None, partd.data_ptr(), n, group, ld, lo, cind, cout, _rowstride(xd), _rowstride(yd), 0, 0, kd, sd, pd,
                      eps, 0, _dt(x), _st(x))
            a2 = [yd.data_ptr(), gd.data_ptr(), bd.data_ptr(), partd.data_ptr(), ed, md.data_ptr(), rd.data_ptr()]
            x2s = _rowstride(yd)
            extra = dict(mean_d=md, rstd_d=rd, y_d=yd)
        _lib.call("dards_gbn_apply_fwd", y.data_ptr(), out.data_ptr(), res.data_ptr() if res is not None else None,
                  gamma.data_ptr(), beta.data_ptr(), part.data_ptr(), entries, mean.data_ptr(), rstd.data_ptr(), *a2, g,
                  group * lo, cout, _rowstride(y), _rowstride(out), _rowstride(res) if res is not None else 0, x2s, eps,
                  1 if relu else 0, _dt(x), _st(x))
    return mode, y, out, mean, rstd, extra


def gbn_fwd(x, gamma, beta, group_rows, relu, res=None, eps=1e-5):
    """x (N, L, C); statistics over `group_rows` consecutive rows of the flattened (N*L, C) view."""
    n, l, c = x.shape
    g = (n * l) // group_rows
    out = torch.empty((n, l, c), dtype=x.dtype, device=x.device)
    mean = torch.empty((g, c), dtype=torch.float32, device=x.device)
    rstd = torch.empty((g, c), dtype=torch.float32, device=x.device)
    _lib.call("dards_gbn_fwd", x.data_ptr(), out.data_ptr(), res.data_ptr() if res is not None else None,
              gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(), rstd.data_ptr(), g, group_rows, c, _rowstride(x),
              _rowstride(out), _rowstride(res) if res is not None else 0, eps, 1 if relu else 0, _dt(x), _st(x))
    return out, mean, rstd


def gbn_bwd(dout, x, gamma, beta, mean, rstd, group_rows, relu_mode, mask_src=None, want_dres=False):
    n, l, c = x.shape
    g = (n * l) // group_rows
    dx = torch.empty((n, l, c), dtype=x.dtype, device=x.device)
    dres = torch.empty_like(dx) if want_dres else None
    dgp = torch.empty((g, c), dtype=torch.float32, device=x.device)
    dbp = torch.empty((g, c), dtype=torch.float32, device=x.device)
    _lib.call("dards_gbn_bwd", dout.data_ptr(), x.data_ptr(), mask_src.data_ptr() if mask_src is not None else None,
              gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(), 0,
              dres.data_ptr() if dres is not None else None, dgp.data_ptr(), dbp.data_ptr(), g, group_rows, c,
              _rowstride(dout), _rowstride(x), _rowstride(mask_src) if mask_src is not None else 0, _rowstride(dx),
              _rowstride(dres) if dres is not None else 0, relu_mode, _dt(x), _st(x))
    dgamma = torch.empty((c,), dtype=torch.float32, device=x.device)
    dbeta = torch.empty((c,), dtype=torch.float32, device=x.device)
    _lib.call("dards_reduce_rows", dgp.data_ptr(), dgamma.data_ptr(), g, c, 0, _st(x))
    _lib.call("dards_reduce_rows", dbp.data_ptr(), dbeta.data_ptr(), g, c, 0, _st(x))
    return dx, dgamma, dbeta, dres


def stem_fwd(x, w, gamma, beta, group, pool, dtype, eps=1e-5):
    """x (N, 224) fp32 -> (N, 56, C0) in `dtype`, plus per-group mean / rstd."""
    n = x.shape[0]
    c0 = w.shape[0]
    g = n // group
    out = torch.empty((n, 56, c0), dtype=dtype, device=x.device)
    mean = torch.empty((g, c0), dtype=torch.float32, device=x.device)
    rstd = torch.empty((g, c0), dtype=torch.float32, device=x.device)
    ws = _stem_workspace(g, group, c0, 0, x.device)
    _lib.call("dards_stem_fwd", x.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
              mean.data_ptr(), rstd.data_ptr(), g, group, c0, c0, eps, pool, ws.data_ptr() if ws is not None else None,
              ws.numel() * 4 if ws is not None else 0, _DT[dtype], _st(x))
    return out, mean, rstd


def _stem_workspace(n_groups, group, c0, backward, device):
    """Chunk records of the stem's large-group path (None when the group fits the one-kernel path)."""
    nbytes = _lib.fn("dards_stem_workspace_bytes")(n_groups, group, c0, backward)
    return torch.empty(((nbytes + 3) // 4,), dtype=torch.float32, device=device) if nbytes else None


def stem_bwd(dout, x, w, gamma, beta, mean, rstd, group, pool):
    n = x.shape[0]
    c0 = w.shape[0]
    g = n // group
    dev = x.device
    dwp = torch.empty((g, c0 * 7), dtype=torch.float32, device=dev)
    dgp = torch.empty((g, c0), dtype=torch.float32, device=dev)
    dbp = torch.empty((g, c0), dtype=torch.float32, device=dev)
    ws = _stem_workspace(g, group, c0, 1, dev)
    _lib.call("dards_stem_bwd", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
              mean.data_ptr(), rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), g, group, c0,
              _rowstride(dout), pool, ws.data_ptr() if ws is not None else None, ws.numel() * 4 if ws is not None else 0,
              _dt(dout), _st(x))
    return dwp.sum(0).view(c0, 1, 7), dgp.sum(0), dbp.sum(0)


def _stem_alt_workspace(n_groups, group, c0, backward, device):
    nbytes = _lib.fn("dards_stem_alt_workspace_bytes")(n_groups, group, c0, backward)
    return torch.empty(((nbytes + 3) // 4,), dtype=torch.float32, device=device) if nbytes else None


def stem_alt_fwd(x, w, gamma, beta, group, dtype, eps=1e-5):
    """Stage 1 of the two-convolution stem: x (N, 224) fp32, w (C0, 1, 3) -> a0 = bn1(conv1_alt(x)) (N, 224, C0) in `dtype`,
    plus per-group mean / rstd."""
    n, c0 = x.shape[0], w.shape[0]
    g = n // group
    out = torch.empty((n, 224, c0), dtype=dtype, device=x.device)
    mean = torch.empty((g, c0), dtype=torch.float32, device=x.device)
    rstd = torch.empty((g, c0), dtype=torch.float32, device=x.device)
    ws = _stem_alt_workspace(g, group, c0, 0, x.device)
    _lib.call("dards_stem_alt_fwd", x.data_ptr(), w.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
              mean.data_ptr(), rstd.data_ptr(), g, group, c0, c0, eps, ws.data_ptr() if ws is not None else None,
              ws.numel() * 4 if ws is not None else 0, _DT[dtype], _st(x))
    return out, mean, rstd


def stem_alt_eval_fwd(x, w, scale, shift, dtype):
    n, c0 = x.shape[0], w.shape[0]
    out = torch.empty((n, 224, c0), dtype=dtype, device=x.device)
    _lib.call("dards_stem_alt_eval_fwd", x.data_ptr(), w.data_ptr(), scale.data_ptr(), shift.data_ptr(), out.data_ptr(), n,
              c0, c0, _DT[dtype], _st(x))
    return out


def stem_alt_bwd(dout, x, w, gamma, mean, rstd, group):
    """dout (N, 224, C0) -> dW (C0, 1, 3), dgamma, dbeta (summed over the groups)."""
    n, c0 = x.shape[0], w.shape[0]
    g = n // group
    dev = x.device
    dwp = torch.empty((g, c0 * 3), dtype=torch.float32, device=dev)
    dgp = torch.empty((g, c0), dtype=torch.float32, device=dev)
    dbp = torch.empty((g, c0), dtype=torch.float32, device=dev)
    ws = _stem_alt_workspace(g, group, c0, 1, dev)
    _lib.call("dards_stem_alt_bwd", dout.data_ptr(), x.data_ptr(), w.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
              rstd.data_ptr(), dwp.data_ptr(), dgp.data_ptr(), dbp.data_ptr(), g, group, c0, _rowstride(dout),
              ws.data_ptr() if ws is not None else None, ws.numel() * 4 if ws is not None else 0, _dt(dout), _st(x))
    return dwp.sum(0).view(c0, 1, 3), dgp.sum(0), dbp.sum(0)


def pool3s2(x, pool):
    """Max (pool 0) / Avg (pool 1) Pool1d(3, 2, 1): (N, L, C) -> (N, (L - 1) // 2 + 1, C)."""
    n, l, c = x.shape
    out = torch.empty((n, (l - 1) // 2 + 1, c), dtype=x.dtype, device=x.device)
    _lib.call("dards_pool3s2_fwd", x.data_ptr(), out.data_ptr(), n, l, c, _rowstride(x), _rowstride(out), pool, _dt(x),
              _st(x))
    return out


def pool3s2_bwd(dout, x, pool):
    n, l, c = x.shape
    din = torch.empty_like(x)
    _lib.call("dards_pool3s2_bwd", dout.data_ptr(), x.data_ptr(), din.data_ptr(), n, l, c, _rowstride(dout), _rowstride(x),
              _rowstride(din), pool, _dt(x), _st(x))
    return din


def avgpool2(x, backward=False):
    n, l, c = x.shape
    if not backward:
        out = torch.empty((n, l // 2, c), dtype=x.dtype, device=x.device)
        _lib.call("dards_avgpool2_fwd", x.data_ptr(), out.data_ptr(), n, l, c, _rowstride(x), _rowstride(out), _dt(x),
                  _st(x))
    else:  # x is dout (N, L/2, C)
        out = torch.empty((n, l * 2, c), dtype=x.dtype, device=x.device)
        _lib.call("dards_avgpool2_bwd", x.data_ptr(), out.data_ptr(), n, l * 2, c, _rowstride(x), _rowstride(out),
                  _dt(x), _st(x))
    return out


def avgpool_full(x):
    n, l, c = x.shape
    feat = torch.empty((n, c), dtype=torch.float32, device=x.device)
    _lib.call("dards_avgpool_full_fwd", x.data_ptr(), feat.data_ptr(), n, l, c, _rowstride(x), _dt(x), _st(x))
    return feat


def avgpool_full_bwd(dfeat, l, dtype):
    n, c = dfeat.shape
    din = torch.empty((n, l, c), dtype=dtype, device=dfeat.device)
    _lib.call("dards_avgpool_full_bwd", dfeat.data_ptr(), din.data_ptr(), n, l, c, c, _DT[dtype], _st(dfeat))
    return din


def dropout_(x, p, seed, seed_dev=None, rows_per_seq=0):
    n, l, c = x.shape
    _lib.call("dards_dropout", x.data_ptr(), n * l, c, _rowstride(x), p, seed,
              seed_dev.data_ptr() if seed_dev is not None else None, rows_per_seq, _dt(x), _st(x))
    return x


def linear_fwd(feat, w, b):
    rows, k = feat.shape
    out = torch.empty((rows, w.shape[0]), dtype=torch.float32, device=feat.device)
    _lib.call("dards_linear_fwd", feat.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), rows, k, w.shape[0],
              _st(feat))
    return out


def linear_bwd(dlogits, feat, w):
    rows, k = feat.shape
    dfeat = torch.empty_like(feat)
    dw = torch.empty_like(w)
    db = torch.empty((w.shape[0],), dtype=torch.float32, device=w.device)
    _lib.call("dards_linear_bwd", dlogits.data_ptr(), feat.data_ptr(), w.data_ptr(), dfeat.data_ptr(), dw.data_ptr(),
              db.data_ptr(), 0, rows, k, w.shape[0], _st(feat))
    return dfeat, dw, db


def bce_with_logits(logits, target, grad_scale=1.0):
    loss = torch.empty((1,), dtype=torch.float32, device=logits.device)
    dl = torch.empty_like(logits)
    _lib.call("dards_bce_with_logits", logits.data_ptr(), target.data_ptr(), loss.data_ptr(), dl.data_ptr(),
              logits.numel(), grad_scale, _st(logits))
    return loss, dl

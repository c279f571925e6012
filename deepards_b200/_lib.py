"""ctypes binding of the C ABI in include/deepards_b200.h.

The product path has no CPU or PyTorch fallback: if the shared library is missing, or a call returns an
error, a RuntimeError is raised.
"""
import ctypes
import os
from ctypes import c_double, c_float, c_int, c_longlong, c_ulonglong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdeepards_b200.so")

F32, BF16 = 0, 1
HINT_LAST_USE = 0x100   # DARDS_HINT_LAST_USE: OR-ed into `impl` (conv fwd / dgrad) or `relu` (gbn_fwd)
ABI_VERSION = 8

P, I, LL, ULL, F, D = c_void_p, c_int, c_longlong, c_ulonglong, c_float, c_double


class GradcamDesc(ctypes.Structure):
    """dards_gradcam_desc (include/deepards_b200.h)."""
    _fields_ = [(n, c_void_p) for n in ("a", "w", "bias", "target_dev", "logits", "target_used", "read_raw", "read_u8",
                                        "seq_raw", "seq_u8", "read_resized", "seq_resized", "conv_out", "grad_out")] + \
               [(n, c_int) for n in ("a_stride", "target", "n_groups", "group", "l", "f", "n_out", "resized_len", "dtype",
                                     "reserved")]


# Descriptors of the batched entry points, read from a DEVICE array (desc_table).  Each kernel gives descriptor j the
# blocks [first_block_j, first_block_j + blocks()).
class _ChannelBlocks(ctypes.Structure):
    def blocks(self):  # one per 64 channels
        return (self.c + 63) // 64


class _TileBlocks(ctypes.Structure):
    def blocks(self):  # one per 32 x 32 tile of the (c_out, c_in) weight plane
        return ((self.c_out + 31) // 32) * ((self.c_in + 31) // 32)


class PackDesc(_TileBlocks):
    """dards_pack_desc."""
    _fields_ = [("w", P), ("w_kio", P), ("w_koi", P), ("c_out", I), ("c_in", I), ("ktaps", I), ("first_block", I)]


class UnpackDesc(_TileBlocks):
    """dards_unpack_desc."""
    _fields_ = [("dw_t", P), ("dw", P), ("c_out", I), ("c_in", I), ("ktaps", I), ("first_block", I)]


class ReduceDesc(_ChannelBlocks):
    """dards_reduce_desc."""
    _fields_ = [("part", P), ("out", P), ("rows", I), ("c", I), ("accumulate", I), ("first_block", I)]


class RunningDesc(_ChannelBlocks):
    """dards_running_desc."""
    _fields_ = [("save_mean", P), ("save_rstd", P), ("running_mean", P), ("running_var", P), ("num_batches_tracked", P),
                ("n_groups", I), ("rows_per_group", I), ("c", I), ("momentum", F), ("first_block", I), ("reserved", I)]


class EvalCoeffDesc(_ChannelBlocks):
    """dards_eval_coeff_desc."""
    _fields_ = [("gamma", P), ("beta", P), ("running_mean", P), ("running_var", P), ("scale", P), ("shift", P),
                ("c", I), ("first_block", I)]


def desc_table(layout, rows, device):
    """rows -> (uint8 tensor on `device` holding one `layout` descriptor per row, total_blocks).  A row gives the fields
    before first_block in declaration order (pointers as ints, None for NULL); first_block is the running sum of the
    blocks of the rows before it, and fields after it are 0."""
    tab = (layout * len(rows))(*[layout(*r) for r in rows])
    total = 0
    for d in tab:
        d.first_block = total
        total += d.blocks()
    return torch.frombuffer(bytearray(tab), dtype=torch.uint8).to(device), total


# name -> argtypes (all functions return int unless listed in _RESTYPES)
_SIGNATURES = {
    "dards_version": [],
    "dards_last_error": [],
    "dards_device_supported": [],
    "dards_launch_count": [],
    "dards_pack_conv_weight": [P, P, P, I, I, I, I, P],
    "dards_pack_conv_weights_batched": [P, I, I, I, P],
    "dards_conv1d_fwd": [P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "dards_conv1d_dgrad": [P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "dards_conv1d_wgrad": [P, P, P, I, P, LL, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "dards_conv1d_wgrad_workspace_bytes": [I, I, I, I, I, I],
    "dards_conv1d_wgrad_accum": [P, P, P, I, I, I, I, I, I, I, I, I, I, I, P],
    "dards_unpack_wgrad_batched": [P, I, I, P],
    "dards_memset_zero": [P, LL, P],
    "dards_conv1d_bn_mode": [I, I, I, I, I, I, I, I, I, I],
    "dards_conv1d_bn_part_entries": [I, I, I, I, I, I, I, I, I],
    "dards_conv1d_bn_fwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, F, I, I, P],
    "dards_gbn_apply_fwd": [P, P, P, P, P, P, I, P, P, P, P, P, P, I, P, P, I, I, I, I, I, I, I, F, I, I, P],
    "dards_gbn_fwd": [P, P, P, P, P, P, P, I, I, I, I, I, I, F, I, I, P],
    "dards_gbn_bwd": [P, P, P, P, P, P, P, P, I, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    "dards_reduce_rows": [P, P, I, I, I, P],
    "dards_reduce_rows_batched": [P, I, I, P],
    "dards_bn_running_update_batched": [P, I, I, F, P],
    "dards_bn_running_update": [P, P, P, P, P, I, I, I, F, F, P],
    "dards_bn_eval_coeffs_batched": [P, I, I, F, P],
    "dards_conv1d_affine_fwd": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, I, I, I, I, P],
    "dards_stem_workspace_bytes": [I, I, I, I],
    "dards_stem_fwd": [P, P, P, P, P, P, P, I, I, I, I, F, I, P, LL, I, P],
    "dards_stem_eval_fwd": [P, P, P, P, P, I, I, I, I, I, P],
    "dards_stem_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, P, LL, I, P],
    "dards_bn_affine_apply": [P, P, P, P, P, P, P, P, I, I, I, I, I, I, I, I, P],
    "dards_bn_frozen_bwd": [P, P, P, P, P, P, P, P, I, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    "dards_stem_frozen_chunks": [I],
    "dards_stem_frozen_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, P],
    "dards_stem_alt_workspace_bytes": [I, I, I, I],
    "dards_stem_alt_fwd": [P, P, P, P, P, P, P, I, I, I, I, F, P, LL, I, P],
    "dards_stem_alt_eval_fwd": [P, P, P, P, P, I, I, I, I, P],
    "dards_stem_alt_bwd": [P, P, P, P, P, P, P, P, P, I, I, I, I, P, LL, I, P],
    "dards_stem_dgrad": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, I, I, P],
    "dards_stem_frozen_dgrad": [P, P, P, P, P, P, I, I, I, I, I, P],
    "dards_stem_alt_dgrad": [P, P, P, P, P, P, P, P, P, I, I, I, I, I, P],
    "dards_pool3s2_fwd": [P, P, I, I, I, I, I, I, I, P],
    "dards_pool3s2_bwd": [P, P, P, I, I, I, I, I, I, I, I, P],
    "dards_avgpool2_fwd": [P, P, I, I, I, I, I, I, P],
    "dards_avgpool2_bwd": [P, P, I, I, I, I, I, I, P],
    "dards_avgpool_full_fwd": [P, P, I, I, I, I, I, P],
    "dards_avgpool_full_bwd": [P, P, I, I, I, I, I, P],
    "dards_dropout": [P, I, I, I, F, ULL, P, I, I, P],
    "dards_linear_fwd": [P, P, P, P, I, I, I, P],
    "dards_linear_bwd": [P, P, P, P, P, P, I, I, I, I, P],
    "dards_bce_with_logits": [P, P, P, P, I, F, P],
    "dards_clamp_sgd_nesterov": [P, P, P, LL, F, F, F, F, F, I, P],
    "dards_clamp_adam": [P, P, P, P, LL, F, F, F, F, F, F, I, P],
    "dards_scale_windows": [P, I, P, LL, D, D, I, P],
    "dards_gradcam": [ctypes.POINTER(GradcamDesc), P],
    "dards_tc_debug_set": [I, I],
    "dards_set_sm_limit": [I],
}
_RESTYPES = {"dards_last_error": ctypes.c_char_p, "dards_launch_count": c_longlong, "dards_conv1d_wgrad_workspace_bytes": c_longlong,
             "dards_stem_workspace_bytes": c_longlong, "dards_stem_alt_workspace_bytes": c_longlong}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))

_lib = None


def load():
    """Load (once) and return the ctypes library with argtypes set."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "deepards_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, c_int)
    if lib.dards_version() != ABI_VERSION:
        raise RuntimeError("deepards_b200: ABI version mismatch (library %d, binding %d)" % (lib.dards_version(), ABI_VERSION))
    _lib = lib
    # DEEPARDS_B200_TC_DEBUG="key=value,key=value": kernel-variant switches of dards_tc_debug_set (A/B measurements)
    for item in filter(None, os.environ.get("DEEPARDS_B200_TC_DEBUG", "").split(",")):
        k, v = item.split("=")
        check(lib.dards_tc_debug_set(int(k), int(v)), "dards_tc_debug_set")
    return lib


def last_error():
    return load().dards_last_error().decode("utf-8", "replace")


def check(rc, name="call"):
    if rc != 0:
        raise RuntimeError("deepards_b200.%s failed (%d): %s" % (name, rc, last_error()))


def fn(name):
    return getattr(load(), name)


def call(name, *args):
    """Immediate checked call (used by the unit tests and one-off setup work)."""
    rc = getattr(load(), name)(*args)
    check(rc, name)

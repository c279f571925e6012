"""CPU: the ctypes binding (deepards_b200/_lib.py) against include/deepards_b200.h -- the descriptor structs' fields,
offsets and sizes, the argument and return types of every prototype -- and the descriptor tables built from those
layouts.  The library is neither loaded nor called."""
import ctypes
import os
import re

import torch

from deepards_b200 import _lib

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "deepards_b200.h")

_SCALARS = {"int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double, "long long": ctypes.c_longlong,
            "unsigned long long": ctypes.c_ulonglong}


def _header():
    src = open(HEADER).read()
    return re.sub(r"//[^\n]*", " ", re.sub(r"/\*.*?\*/", " ", src, flags=re.S))


def _ctype(c_type):
    """A C type as the header writes it -> the ctypes type the binding must use for it."""
    t = " ".join(c_type.replace("*", " * ").replace("const", " ").split())
    if t == "char *":
        return ctypes.c_char_p
    if t == "dards_gradcam_desc *":       # a HOST struct, read during the call
        return ctypes.POINTER(_lib.GradcamDesc)
    if t.endswith("*"):                   # device buffers, device descriptor arrays, the stream
        return ctypes.c_void_p
    return _SCALARS[t]


def _split(decl):
    """'const float* w' -> ('const float*', 'w')"""
    return re.match(r"(.*?)\s*\b(\w+)$", decl.strip()).groups()


def _structs():
    """{struct name: [(field, ctypes type)]} of every `typedef struct` in the header."""
    out = {}
    for name, body in re.findall(r"typedef struct (\w+) \{(.*?)\} \1;", _header(), flags=re.S):
        fields = []
        for decl in filter(None, (d.strip() for d in body.split(";"))):
            head, *more = [s.strip() for s in decl.split(",")]
            c_type, first = _split(head)
            fields += [(n, _ctype(c_type)) for n in [first] + more]
        out[name] = fields
    return out


def _prototypes():
    """{function: (return ctypes type, [argument ctypes types])} of every dards_* prototype in the header."""
    out = {}
    for ret, name, args in re.findall(r"^([A-Za-z_][\w \*]*?)\s*\b(dards_\w+)\s*\(([^)]*)\)\s*;", _header(), flags=re.M):
        args = [a.strip() for a in args.split(",") if a.strip() not in ("", "void")]
        out[name] = (_ctype(ret), [_ctype(_split(a)[0]) for a in args])
    return out


def test_descriptor_layouts_match_the_header_structs():
    """Natural alignment (x86-64 / aarch64 Linux): every field at a multiple of its size, the struct padded to its widest
    field.  A _lib layout named after each struct (dards_eval_coeff_desc -> EvalCoeffDesc)."""
    structs = _structs()
    assert {"dards_pack_desc", "dards_unpack_desc", "dards_reduce_desc", "dards_running_desc", "dards_eval_coeff_desc",
            "dards_gradcam_desc"} <= set(structs)
    for name, fields in structs.items():
        layout = getattr(_lib, "".join(w.capitalize() for w in name[len("dards_"):].split("_")))
        offsets, off = [], 0
        for _, t in fields:
            size = ctypes.sizeof(t)
            off = (off + size - 1) // size * size
            offsets.append(off)
            off += size
        widest = max(ctypes.sizeof(t) for _, t in fields)
        assert layout._fields_ == fields, name
        assert [getattr(layout, n).offset for n, _ in fields] == offsets, name
        assert ctypes.sizeof(layout) == (off + widest - 1) // widest * widest, name


def test_bindings_match_the_header_prototypes():
    protos = _prototypes()
    assert len(protos) >= 47
    assert sorted(protos) == sorted(_lib._SIGNATURES)
    for name, (ret, args) in protos.items():
        assert _lib._SIGNATURES[name] == args, name
        assert _lib._RESTYPES.get(name, ctypes.c_int) is ret, name


def _decode(layout, tab):
    raw = bytes(tab.numpy())
    assert tab.dtype == torch.uint8 and len(raw) % ctypes.sizeof(layout) == 0
    return list((layout * (len(raw) // ctypes.sizeof(layout))).from_buffer_copy(raw))


def test_desc_table_first_block_is_the_running_block_count():
    # ceil(c / 64) blocks per row
    tab, total = _lib.desc_table(_lib.ReduceDesc, [(16 + 16 * i, 4096 + 16 * i, 7, c, i % 2)
                                                   for i, c in enumerate((64, 65, 4, 512))], "cpu")
    rows = _decode(_lib.ReduceDesc, tab)
    assert [d.first_block for d in rows] == [0, 1, 3, 4] and total == 12
    assert [(d.part, d.out, d.rows, d.c, d.accumulate) for d in rows] == \
        [(16, 4096, 7, 64, 0), (32, 4112, 7, 65, 1), (48, 4128, 7, 4, 0), (64, 4144, 7, 512, 1)]
    # ceil(c_out / 32) * ceil(c_in / 32) blocks per row
    tab, total = _lib.desc_table(_lib.PackDesc, [(8, 16, 24, co, ci, k) for co, ci, k in
                                                 ((64, 64, 3), (40, 24, 5), (512, 256, 3), (1, 1, 1))], "cpu")
    rows = _decode(_lib.PackDesc, tab)
    assert [d.first_block for d in rows] == [0, 4, 6, 134] and total == 135
    assert [(d.c_out, d.c_in, d.ktaps) for d in rows] == [(64, 64, 3), (40, 24, 5), (512, 256, 3), (1, 1, 1)]
    tab, total = _lib.desc_table(_lib.UnpackDesc, [(8, 16, 33, 65, 3)], "cpu")
    assert [d.first_block for d in _decode(_lib.UnpackDesc, tab)] == [0] and total == 6
    # a field after first_block stays 0; a None pointer is NULL
    tab, total = _lib.desc_table(_lib.RunningDesc, [(8, 16, 24, 32, None, 13, 1120, 96, 0.1),
                                                    (40, 48, 56, 64, 72, 1, 56, 512, 0.3)], "cpu")
    rows = _decode(_lib.RunningDesc, tab)
    assert [(d.first_block, d.reserved) for d in rows] == [(0, 0), (2, 0)] and total == 10
    assert rows[0].num_batches_tracked is None and rows[1].num_batches_tracked == 72
    assert rows[0].momentum == ctypes.c_float(0.1).value and (rows[1].n_groups, rows[1].rows_per_group) == (1, 56)
    # a frozen plan's coefficient table: the rstd rows continue the prefix of the scale / shift rows
    cs = (64, 64, 128)
    tab, total = _lib.desc_table(_lib.EvalCoeffDesc, [(8, 16, 24, 32, 40, 48, c) for c in cs + cs], "cpu")
    assert [d.first_block for d in _decode(_lib.EvalCoeffDesc, tab)] == [0, 1, 2, 4, 5, 6] and total == 8

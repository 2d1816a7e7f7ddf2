"""ctypes binding of libtwowl_b200.so - the C ABI declared in include/twowl.h.

The prototypes are read from the header itself, so the binding cannot drift from it. There
is no CPU fallback: if the library is missing, importing this module raises with the build
command, and every op raises on a non-CUDA tensor.
"""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtwowl_b200.so")
HEADER_PATH = os.path.normpath(os.path.join(_HERE, "..", "..", "include", "twowl.h"))

_CTYPES = {
    "int": ctypes.c_int32, "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64,
    "uint64_t": ctypes.c_uint64, "size_t": ctypes.c_size_t, "float": ctypes.c_float, "double": ctypes.c_double,
}


class SegArgs(ctypes.Structure):
    """``twowl_seg_args`` of include/twowl.h (field order must match)."""
    _fields_ = [
        ("ptr", ctypes.c_void_p), ("col", ctypes.c_void_p), ("M", ctypes.c_int64),
        ("X", ctypes.c_void_p), ("C", ctypes.c_int32), ("flip", ctypes.c_int32),
        ("row_flip", ctypes.c_int32), ("src_scale", ctypes.c_void_p),
        ("skip_mask", ctypes.c_void_p), ("row_skip_mask", ctypes.c_void_p),
        ("skip_self", ctypes.c_int32), ("self_mode", ctypes.c_int32),
        ("dst_scale", ctypes.c_void_p), ("bias", ctypes.c_void_p), ("X2", ctypes.c_void_p),
        ("mul_idx", ctypes.c_void_p), ("out", ctypes.c_void_p), ("accumulate", ctypes.c_int32),
        ("plan_counts", ctypes.c_void_p), ("long_row", ctypes.c_void_p), ("long_base", ctypes.c_void_p),
        ("chunk_owner", ctypes.c_void_p), ("partial", ctypes.c_void_p), ("chunk_cap", ctypes.c_int64),
        ("long_cap", ctypes.c_int64), ("pair_sum", ctypes.c_int32), ("entry_mask", ctypes.c_void_p),
        ("src_scale2", ctypes.c_void_p), ("out2", ctypes.c_void_p), ("partial2", ctypes.c_void_p),
        ("row_begin", ctypes.c_int64), ("row_end", ctypes.c_int64), ("X_mate", ctypes.c_void_p),
    ]


class ConvArgs(ctypes.Structure):
    """``twowl_conv_args`` of include/twowl.h (field order must match)."""
    _fields_ = [
        ("nsrc", ctypes.c_int32), ("ngather", ctypes.c_int32), ("Kd", ctypes.c_int32), ("Nd", ctypes.c_int32),
        ("M", ctypes.c_int64), ("A", ctypes.c_void_p * 2), ("row_scale", ctypes.c_void_p * 2),
        ("W", ctypes.c_void_p * 2), ("w_kn", ctypes.c_int32 * 2), ("T", ctypes.c_void_p * 2),
        ("tidx", ctypes.c_void_p * 2), ("tcoef", ctypes.c_void_p * 2), ("bias", ctypes.c_void_p),
        ("out", ctypes.c_void_p), ("stats", ctypes.c_void_p), ("mean_scale", ctypes.c_void_p), ("eps", ctypes.c_float),
        ("moments", ctypes.c_void_p), ("pair_sum_out", ctypes.c_int32), ("a_pairs", ctypes.c_int32),
    ]


def parse_header(path: str = HEADER_PATH):
    """-> {name: (restype_str, [argtype_str, ...])} for every function the header declares."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"typedef struct.*?\}\s*\w+;", " ", text, flags=re.S)
    text = re.sub(r"#.*", " ", text)
    protos = {}
    for m in re.finditer(r"(const char\*|size_t|int64_t|int)\s+(twowl_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3).strip()
        argl = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                argl.append("ptr" if "*" in a else a.replace("const ", "").split()[0])
        protos[name] = (ret, argl)
    return protos


def _bind(lib, protos):
    for name, (ret, args) in protos.items():
        fn = getattr(lib, name)  # AttributeError here = header declares a symbol the .so lacks
        fn.restype = ctypes.c_char_p if ret == "const char*" else _CTYPES[ret]
        fn.argtypes = [ctypes.c_void_p if a == "ptr" else _CTYPES[a] for a in args]


if not os.path.isfile(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python link-prediction-gnn_b200/build.py` "
        "(nvcc, sm_100a). There is no CPU fallback for the TwoWL hot path.")

lib = ctypes.CDLL(LIB_PATH)
PROTOS = parse_header()
_bind(lib, PROTOS)
for _name, _cls in (("twowl_sizeof_seg_args", SegArgs), ("twowl_sizeof_conv_args", ConvArgs)):
    if getattr(lib, _name)() != ctypes.sizeof(_cls):
        raise ImportError(f"{_cls.__name__} (ctypes) is {ctypes.sizeof(_cls)} bytes but the library's struct is "
                          f"{getattr(lib, _name)()}: twowl_b200/_lib.py and include/twowl.h disagree")


def check(rc: int, op: str = "") -> None:
    if rc != 0:
        msg = lib.twowl_last_error()
        raise RuntimeError(f"twowl {op} failed (code {rc}): {msg.decode() if msg else ''}")

"""ctypes binding of libeavsr_b200.so (the C ABI declared in include/eavsr_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or a
call fails, the error is raised -- loudly -- to the caller.
"""
from __future__ import annotations

import ctypes
import functools
import os
import re
from ctypes import c_char_p, c_float, c_int, c_int64, c_longlong, c_size_t, c_uint, c_uint64, c_void_p, POINTER
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "libeavsr_b200.so"
_lib = None

F32, BF16 = 0, 1
FLOW_N2HW, FLOW_NHW2 = 0, 1
PAD_ZEROS, PAD_BORDER = 0, 1
DCN_FORCE_GENERIC = 1
DCN_FORCE_V1 = 2
DCN_FORCE_WS = 4
DCN_BLEND_FP32 = 8
DCN_WS_PACKED = 16
DCN_BWD_GENERIC_DATA = 32
DCN_BWD_GENERIC_WEIGHT = 64
DCN_FORCE_WIN1 = 128
DCN_FORCE_WIN2 = 256
CONV_SUMS_PREZEROED = 1
CORR_TF32 = 2

Strides = c_int64 * 4


class EavsrError(RuntimeError):
    pass


class FlowTerm(ctypes.Structure):
    """EavsrFlowTerm of include/eavsr_b200.h (one term of a pyramid flow)."""
    _fields_ = [("flow", c_void_p), ("scaled_out", c_void_p), ("h", c_int), ("w", c_int), ("scale", c_float)]


class ConvLayer(ctypes.Structure):
    """EavsrConvLayer of include/eavsr_b200.h (one convolution of eavsr_conv3x3_chain_forward)."""
    _fields_ = [("x", c_void_p), ("packed_weight", c_void_p), ("bias", c_void_p), ("out", c_void_p),
                ("channel_sums", c_void_p), ("res", c_void_p), ("res_sums", c_void_p), ("w1", c_void_p),
                ("b1", c_void_p), ("w2", c_void_p), ("b2", c_void_p), ("y_out", c_void_p),
                ("negative_slope", c_float)]


_HEADER = Path(__file__).resolve().parents[1] / "include" / "eavsr_b200.h"
# ctypes type of each spelling the header uses; any other pointer is passed as a raw address (c_void_p)
_CTYPES = {"const char*": c_char_p, "const int64_t[4]": POINTER(c_int64), "const EavsrFlowTerm*": POINTER(FlowTerm),
           "const EavsrConvLayer*": POINTER(ConvLayer), "int": c_int, "unsigned": c_uint, "size_t": c_size_t,
           "long long": c_longlong, "float": c_float, "uint64_t": c_uint64}


def _ctype(spelling: str, name: str):
    if spelling in _CTYPES:
        return _CTYPES[spelling]
    if spelling.endswith("*"):
        return c_void_p
    raise EavsrError(f"{_HEADER}: {name} uses `{spelling}`, which has no ctypes type in eavsr_b200._lib")


def _arg_type(decl: str, name: str):
    """ctypes type of one declared parameter: "const int64_t x_strides[4]" -> POINTER(c_int64)."""
    m = re.fullmatch(r"(.*?\S)\s*\b\w+(\[4\])?", " ".join(decl.split()))
    if m is None:
        raise EavsrError(f"{_HEADER}: cannot read parameter `{decl.strip()}` of {name}")
    return _ctype(m[1] + (m[2] or ""), name)


@functools.cache
def _signatures() -> dict:
    """{name: (restype, argtypes)} of every eavsr_* prototype in include/eavsr_b200.h."""
    if not _HEADER.exists():
        raise EavsrError(f"{_HEADER} not found: the ctypes signatures are read from the C header")
    text = re.sub(r"/\*.*?\*/", "", _HEADER.read_text(), flags=re.S)
    sigs = {}
    for ret, name, params in re.findall(r"^(\w[\w ]*?\**)\s*\b(eavsr_\w+)\(([^)]*)\);", text, flags=re.M):
        args = [] if params.strip() == "void" else [_arg_type(p, name) for p in params.split(",")]
        sigs[name] = (_ctype(ret, name), args)
    return sigs


def __getattr__(attr):
    if attr == "EXPORTED_SYMBOLS":      # every entry point the header declares (and load() binds)
        return tuple(_signatures())
    raise AttributeError(f"module {__name__!r} has no attribute {attr!r}")


def lib_path() -> Path:
    return Path(os.environ.get("EAVSR_B200_LIB", _LIB_PATH))


def load():
    """Load (once) and return the ctypes handle; raises EavsrError if the .so is not built."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not path.exists():
            raise EavsrError(
                f"{path} not found: build it with `python -m eavsr_b200.build` "
                "(eavsr_b200 has no CPU or PyTorch fallback)")
        sigs = _signatures()
        lib = ctypes.CDLL(str(path))
        for name, (res, args) in sigs.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().eavsr_last_error().decode("utf-8", "replace")
        raise EavsrError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().eavsr_launch_count())

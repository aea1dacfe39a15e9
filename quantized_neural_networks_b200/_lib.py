"""ctypes binding of libgpfq.so (include/gpfq.h).  No CPU fallback: if the CUDA library is missing
or no sm_100 GPU is present, every compute entry point raises."""
from __future__ import annotations

import ctypes
import os
import subprocess
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgpfq.so")
CSRC = os.path.join(_HERE, "csrc")

# flags (include/gpfq.h)
X_DEVICE, W_DEVICE, Q_DEVICE = 1, 2, 4
ALL_DEVICE = 7
METHOD_AUTO, METHOD_STREAM, METHOD_GRAM, METHOD_STREAM_FAST = 0 << 4, 1 << 4, 2 << 4, 3 << 4
NO_SYNC = 1 << 8
MAX_K = 64
ROUND_NEAREST, ROUND_STOCHASTIC = 0, 1

ERRORS = {1: "GPFQ_ERR_ARG", 2: "GPFQ_ERR_CUDA", 3: "GPFQ_ERR_OOM", 4: "GPFQ_ERR_UNSUPPORTED"}


class GpfqStats(ctypes.Structure):
    _fields_ = [
        ("method", c_int32), ("kernel_launches", c_int32),
        ("ms_total", c_float), ("ms_h2d", c_float), ("ms_d2h", c_float),
        ("ms_gram", c_float), ("ms_sweep", c_float), ("ms_stream", c_float),
        ("weights", c_int64), ("bytes_algorithmic", c_int64), ("flops_algorithmic", c_int64),
        ("gram_kernel", c_int32), ("reserved", c_int32),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class GpfqError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"{ERRORS.get(code, code)}: {message}")
        self.code = code


EXPORTS = {
    # name: (restype, argtypes) -- one entry per symbol declared in include/gpfq.h
    "gpfq_version": (c_int, []),
    "gpfq_create": (c_int, [c_int, POINTER(c_void_p)]),
    "gpfq_destroy": (None, [c_void_p]),
    "gpfq_last_error": (c_char_p, [c_void_p]),
    "gpfq_set_stream": (c_int, [c_void_p, c_void_p]),
    "gpfq_set_option": (c_int, [c_void_p, c_char_p, c_int64]),
    "gpfq_set_rounding": (c_int, [c_void_p, c_int32, POINTER(c_uint64), c_int32]),
    "gpfq_set_l1_penalty": (c_int, [c_void_p, POINTER(c_double), c_int32]),
    "gpfq_trim": (c_int, [c_void_p]),
    "gpfq_conv_partial_bytes": (c_int64, [c_void_p]),
    "gpfq_query_stats": (c_int, [c_void_p, c_int32, POINTER(GpfqStats)]),
    "gpfq_dense_layer": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                 c_int64, c_int64, c_int64, POINTER(c_double), POINTER(c_int32), c_int32,
                                 c_void_p, c_int64, c_uint32, POINTER(GpfqStats)]),
    "gpfq_dense_layer_from_gram": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                           c_int64, POINTER(c_double), POINTER(c_int32), c_int32, c_void_p, c_int64,
                                           c_uint32, POINTER(GpfqStats)]),
    "gpfq_conv_channels": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_int64, c_int32, c_void_p,
                                   c_int64, c_int64, c_int64, c_int64, POINTER(c_double), POINTER(c_int32),
                                   c_int32, c_void_p, c_uint32, POINTER(GpfqStats)]),
    "gpfq_conv_layer_nhwc": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int32,
                                     c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64,
                                     c_int64, c_int64, POINTER(c_double), POINTER(c_int32), c_int32, c_void_p,
                                     c_uint32, POINTER(GpfqStats)]),
    "gpfq_conv_gram_nhwc": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int32, c_int32,
                                    c_int32, c_int32, c_int32, c_int32, c_int32, c_int64, c_int64, c_void_p, c_uint32]),
    "gpfq_conv_layer_from_gram": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                          POINTER(c_double), POINTER(c_int32), c_int32, c_void_p, c_uint32,
                                          POINTER(GpfqStats)]),
    "gpfq_conv_layer_nhwc_grouped": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int32,
                                             c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64,
                                             c_int64, c_int64, POINTER(c_double), POINTER(c_int32), c_int32, c_void_p,
                                             c_uint32, POINTER(GpfqStats), c_int32]),
    "gpfq_conv_layer_from_gram_grouped": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                                  POINTER(c_double), POINTER(c_int32), c_int32, c_void_p, c_uint32,
                                                  POINTER(GpfqStats), c_int32]),
    "gpfq_dense_layer_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64,
                                        c_int64, c_int64, c_int64, POINTER(c_double), POINTER(c_int32), c_int32,
                                        c_void_p, c_int64, c_uint32, POINTER(GpfqStats), POINTER(c_double)]),
    "gpfq_dense_layer_from_gram_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64,
                                                  c_int64, POINTER(c_double), POINTER(c_int32), c_int32, c_void_p, c_int64,
                                                  c_uint32, POINTER(GpfqStats), POINTER(c_double)]),
    "gpfq_conv_channels_scaled": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_int64, c_int32, c_void_p,
                                          c_int64, c_int64, c_int64, c_int64, POINTER(c_double), POINTER(c_int32),
                                          c_int32, c_void_p, c_uint32, POINTER(GpfqStats), POINTER(c_double)]),
    "gpfq_conv_layer_nhwc_scaled": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int32,
                                            c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64,
                                            c_int64, c_int64, POINTER(c_double), POINTER(c_int32), c_int32, c_void_p,
                                            c_uint32, POINTER(GpfqStats), c_int32, POINTER(c_double)]),
    "gpfq_conv_layer_from_gram_scaled": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_int64, c_int64, c_int64, c_int64,
                                                 POINTER(c_double), POINTER(c_int32), c_int32, c_void_p, c_uint32,
                                                 POINTER(GpfqStats), c_int32, POINTER(c_double)]),
    "gpfq_msq": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_double), c_int32, c_void_p, c_uint32]),
    "gpfq_msq_scaled": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_double), c_int32, POINTER(c_double), c_int64, c_void_p,
                                c_uint32]),
    "gpfq_bit_round": (c_int, [c_void_p, c_void_p, c_int64, POINTER(c_double), c_int32, c_void_p, c_uint32]),
    "gpfq_gram_matrices": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p,
                                   c_uint32]),
    "gpfq_debug_slgemm": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_int32, c_void_p]),
}

_lib = None


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libgpfq.so (in-tree).  nvcc cross-compiles without a GPU."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    srcs.append(os.path.join(_HERE, "..", "include", "gpfq.h"))
    stale = (not os.path.exists(LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC, "-j4"] + (["-B"] if force else [])
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if verbose or res.returncode:
            print(res.stdout)
        if res.returncode:
            raise RuntimeError("building libgpfq.so failed")
    return LIB_PATH


def lib():
    """Load libgpfq.so and declare every exported prototype.  Raises if the library is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib

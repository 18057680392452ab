"""TEST INFRASTRUCTURE: ctypes binding of tests/soft_ref.c, the restatement's frame layer with the equalized data
symbols handed out.  Compiled on first use with the oracle's flags into a temporary directory, linked against
oracle/libsc_oracle.so (whose primitives it calls)."""
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile
import threading

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    po.Oracle()                                                  # builds oracle/libsc_oracle.so if it is missing
    tmp = tempfile.mkdtemp(prefix="sc_soft_ref_")
    out = os.path.join(tmp, "libsc_soft_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", out,
                        os.path.join(HERE, "soft_ref.c"), po.ORACLE_SO, "-lm"], check=True)
        L = C.CDLL(out)                                          # needs oracle/libsc_oracle.so by its full path
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    L.scs_run_stream_soft.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.scs_run_stream_soft.restype = None
    return L


def _lib():
    with _lock:                                                  # the GPU tests call in from a thread pool
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run_stream_soft(samples: np.ndarray, wide: bool = False, foffset: float = 0.0):
    """Oracle.run_stream plus the equalizer output of every data step, valid call or not:
    (bits[nf, 62] (255 = invalid row), stats[nf], symbols complex64 [nf, 31])."""
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // po.FRAME_SIZE
    bits = np.full((nf, po.BITS_PER_CALL), 255, np.uint8)
    stats = np.zeros(nf, po.STATS_DTYPE)
    sym = np.zeros((nf, po.DATA_SYMBOLS), np.complex64)
    _lib().scs_run_stream_soft(_p(x), nf, int(wide), float(foffset), _p(bits), _p(stats), _p(sym))
    return bits, stats, sym

"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_soft_ref.c, the packet-mode specification with the equalized
data symbols of every packet handed out.  Compiled on first use with the oracle's flags into a temporary directory,
linked against oracle/libsc_oracle.so (whose primitives it calls)."""
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
PACKET_DATA_SYMBOLS = 8 * po.DATA_SYMBOLS                        # 248

_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    po.Oracle()                                                  # builds oracle/libsc_oracle.so if it is missing
    tmp = tempfile.mkdtemp(prefix="sc_packet_soft_ref_")
    out = os.path.join(tmp, "libsc_packet_soft_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", out,
                        os.path.join(HERE, "packet_soft_ref.c"), po.ORACLE_SO, "-lm"], check=True)
        L = C.CDLL(out)                                          # needs oracle/libsc_oracle.so by its full path
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    L.scs_ext_run_stream_soft.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int]
    L.scs_ext_run_stream_soft.restype = C.c_int
    return L


def _lib():
    with _lock:                                                  # the GPU tests call in from a thread pool
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def ext_run_stream_soft(samples: np.ndarray, wide: bool = False, foffset: float = 0.0):
    """pyoracle.ext_run_stream plus the equalizer output of the 248 data steps of every packet:
    (bits[nf, 62], stats[nf], packets[EXT_PACKET_DTYPE], packet symbols complex64 [n, 248])."""
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // po.FRAME_SIZE
    max_packets = max(nf, 1)                                     # at most one per call
    bits = np.full((nf, po.BITS_PER_CALL), 255, np.uint8)
    stats = np.zeros(nf, po.STATS_DTYPE)
    pk = np.zeros(max_packets, po.EXT_PACKET_DTYPE)
    psym = np.zeros((max_packets, PACKET_DATA_SYMBOLS), np.complex64)
    n = _lib().scs_ext_run_stream_soft(_p(x), nf, int(wide), float(foffset), _p(bits), _p(stats), _p(pk), _p(psym),
                                       max_packets)
    return bits, stats, pk[:n], psym[:n]

"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_acq_ref.c, the specification of packet-mode acquisition
(SC_FLAG_PACKET_ACQ), and its float64 model.  Compiled on first use with the oracle's flags into a temporary
directory, linked against oracle/libsc_oracle.so (whose primitives it calls)."""
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
PACKET_SYMS = po.PREAMBLE_LENGTH + PACKET_DATA_SYMBOLS + 4       # 380
FRAME = po.FRAME_SIZE

ACQ_PACKET_DTYPE = np.dtype([("grid_sample", "<i8"), ("call", "<i4"), ("max_index", "<i4"), ("matches", "<i4"),
                             ("frame", "<i4"), ("cost", "<f4"), ("metric", "<f4"), ("freq_hz", "<f4"), ("nu0", "<f4"),
                             ("bits", "u1", (2 * PACKET_DATA_SYMBOLS,))])
assert ACQ_PACKET_DTYPE.itemsize == 536

_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    po.Oracle()                                                  # builds oracle/libsc_oracle.so if it is missing
    tmp = tempfile.mkdtemp(prefix="sc_packet_acq_ref_")
    out = os.path.join(tmp, "libsc_packet_acq_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", out,
                        os.path.join(HERE, "packet_acq_ref.c"), po.ORACLE_SO, "-lm"], check=True)
        L = C.CDLL(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    L.scd_acq_params.argtypes = [C.c_void_p]
    L.scd_acq_params.restype = None
    L.scd_acq_filt.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p]
    L.scd_acq_filt.restype = None
    L.scd_acq_metric.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_void_p]
    L.scd_acq_metric.restype = C.c_float
    L.scd_acq_rho_lags.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_int, C.c_void_p]
    L.scd_acq_rho_lags.restype = None
    L.scd_dd_packet_seeded.argtypes = [C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.scd_dd_packet_seeded.restype = C.c_float
    L.scd_acq_run_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int]
    L.scd_acq_run_stream.restype = C.c_int
    return L


def _lib():
    with _lock:                                                  # the GPU tests call in from a thread pool
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def acq_params():
    """(tau, W, hz_per_rad): tau and hz_per_rad as the spec's float32 constants, W an int"""
    out = np.zeros(3, np.float32)
    _lib().scd_acq_params(_p(out))
    return np.float32(out[0]), int(out[1]), np.float32(out[2])


def acq_filt(samples: np.ndarray, wide: bool = False, foffset: float = 0.0) -> np.ndarray:
    """filt[q] of one stream, complex64 [n_frames * 1880]"""
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // FRAME
    out = np.zeros(nf * FRAME, np.complex64)
    if nf:
        _lib().scd_acq_filt(_p(x), nf, int(wide), float(foffset), _p(out))
    return out


def acq_metric(filt: np.ndarray, g0: int):
    """(rho float32, D complex64) on the grid filt[g0 + 5 i], i < 128 (zero outside filt)"""
    f = np.ascontiguousarray(filt, np.complex64)
    D = np.zeros(1, np.complex64)
    r = _lib().scd_acq_metric(_p(f), f.size, int(g0), _p(D))
    return np.float32(r), D[0]


def acq_rho_lags(filt: np.ndarray, k0: int, n: int) -> np.ndarray:
    """rho(k) on g0 = 5 k, k = k0 .. k0 + n - 1, float32 [n]"""
    f = np.ascontiguousarray(filt, np.complex64)
    out = np.zeros(n, np.float32)
    _lib().scd_acq_rho_lags(_p(f), f.size, int(k0), int(n), _p(out))
    return out


def dd_packet_seeded(S: np.ndarray, nu0: float):
    """-> (bits uint8 [496], cost float32, symbols complex64 [248], matches int)"""
    s = np.ascontiguousarray(S, np.complex64)
    assert s.shape == (PACKET_SYMS,)
    bits = np.zeros(2 * PACKET_DATA_SYMBOLS, np.uint8)
    z = np.zeros(PACKET_DATA_SYMBOLS, np.complex64)
    m = np.zeros(1, np.int32)
    cost = _lib().scd_dd_packet_seeded(_p(s), float(nu0), _p(bits), _p(z), _p(m))
    return bits, np.float32(cost), z, int(m[0])


def acq_run_stream(samples: np.ndarray, wide: bool = False, foffset: float = 0.0, seed_nu: bool = True):
    """The spec over one stream -> (packets[ACQ_PACKET_DTYPE], symbols complex64 [n, 248], grids complex64 [n, 380])"""
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // FRAME
    cap = max(nf, 1)                                             # at most one per frame
    pk = np.zeros(cap, ACQ_PACKET_DTYPE)
    psym = np.zeros((cap, PACKET_DATA_SYMBOLS), np.complex64)
    grids = np.zeros((cap, PACKET_SYMS), np.complex64)
    n = _lib().scd_acq_run_stream(_p(x), nf, int(wide), float(foffset), int(seed_nu), _p(pk), _p(psym), _p(grids),
                                  cap)
    return pk[:n], psym[:n], grids[:n]


# ---- float64 model ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _pre():
    return np.array((C.c_int8 * po.PREAMBLE_LENGTH).in_dll(po.Oracle().lib, "sco_preamblevalues"), np.float64)


def filt64(x: np.ndarray, foffset: float = 0.0, wide: bool = False) -> np.ndarray:
    """filt in float64 from int16 samples: mixer at -1100 + foffset Hz, RRC, gain 2.2 -> complex128"""
    taps = np.array((C.c_float * po.NTAPS).in_dll(po.Oracle().lib, "sco_alpha50_root" if wide else "sco_alpha35_root"),
                    np.float64)
    i = np.arange(x.size)
    m = np.exp(2j * np.pi * (-1100.0 + foffset) * (i + 1) / 8000.0) * (x.astype(np.float64) / 16384.0)
    return np.convolve(m, taps)[: x.size] * 2.2


def metric64(filt: np.ndarray, g0: int):
    """(rho, nu0) of the grid filt[g0 + 5 i] in float64"""
    idx = g0 + 5 * np.arange(po.PREAMBLE_LENGTH)
    u = np.where((idx >= 0) & (idx < filt.size), filt[np.clip(idx, 0, filt.size - 1)], 0).astype(np.complex128)
    pre = _pre()
    D = np.sum(pre[1:] * pre[:-1] * u[1:] * np.conj(u[:-1]))
    E = np.sum(np.abs(u) ** 2)
    elo = np.sum(np.abs(u[:64]) ** 2)
    rho = 0.0 if E == 0 or not (0.25 * E <= elo <= 0.75 * E) else abs(D) ** 2 / E ** 2
    return rho, (D.imag / D.real if D.real > 0 else 0.0)

"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_dd_ref.c, the specification of packet mode's decision-directed
equalizer (SC_FLAG_PACKET_DD), and helpers shared by its CPU and GPU tests.  Compiled on first use with the oracle's
flags into a temporary directory, linked against oracle/libsc_oracle.so (whose primitives it calls)."""
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

_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    po.Oracle()                                                  # builds oracle/libsc_oracle.so if it is missing
    tmp = tempfile.mkdtemp(prefix="sc_packet_dd_ref_")
    out = os.path.join(tmp, "libsc_packet_dd_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-I", os.path.join(ROOT, "oracle"), "-o", out,
                        os.path.join(HERE, "packet_dd_ref.c"), po.ORACLE_SO, "-lm"], check=True)
        L = C.CDLL(out)                                          # needs oracle/libsc_oracle.so by its full path
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    L.scd_ext_run_stream_dd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_int]
    L.scd_ext_run_stream_dd.restype = C.c_int
    L.scd_dd_packet.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.scd_dd_packet.restype = C.c_float
    L.scd_dd_params.argtypes = [C.c_void_p]
    L.scd_dd_params.restype = None
    L.scd_kalman_packet.argtypes = [C.c_void_p, C.c_void_p]
    L.scd_kalman_packet.restype = C.c_float
    return L


def _lib():
    with _lock:                                                  # the GPU tests call in from a thread pool
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def dd_params():
    """(mu, alpha, beta, eps, train_amp, phase_eps) as the spec's float32 constants"""
    out = np.zeros(6, np.float32)
    _lib().scd_dd_params(_p(out))
    return tuple(np.float32(v) for v in out)


def dd_packet(S: np.ndarray):
    """One packet's grid complex64 [380] -> (bits uint8 [496], cost float32, symbols complex64 [248])"""
    s = np.ascontiguousarray(S, np.complex64)
    assert s.shape == (PACKET_SYMS,)
    bits = np.zeros(2 * PACKET_DATA_SYMBOLS, np.uint8)
    z = np.zeros(PACKET_DATA_SYMBOLS, np.complex64)
    cost = _lib().scd_dd_packet(_p(s), _p(bits), _p(z))
    return bits, np.float32(cost), z


def kalman_packet(S: np.ndarray):
    """The reference's equalizer (packet mode without the flag) on one grid -> bits uint8 [496]"""
    s = np.ascontiguousarray(S, np.complex64)
    assert s.shape == (PACKET_SYMS,)
    bits = np.zeros(2 * PACKET_DATA_SYMBOLS, np.uint8)
    _lib().scd_kalman_packet(_p(s), _p(bits))
    return bits


def ext_run_stream_dd(samples: np.ndarray, wide: bool = False, foffset: float = 0.0):
    """pyoracle.ext_run_stream with the packets decoded by the decision-directed equalizer:
    (bits[nf, 62], stats[nf], packets[EXT_PACKET_DTYPE], packet symbols complex64 [n, 248], grids complex64 [n, 380])"""
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // po.FRAME_SIZE
    max_packets = max(nf, 1)                                     # at most one per call
    bits = np.full((nf, po.BITS_PER_CALL), 255, np.uint8)
    stats = np.zeros(nf, po.STATS_DTYPE)
    pk = np.zeros(max_packets, po.EXT_PACKET_DTYPE)
    psym = np.zeros((max_packets, PACKET_DATA_SYMBOLS), np.complex64)
    grids = np.zeros((max_packets, PACKET_SYMS), np.complex64)
    n = _lib().scd_ext_run_stream_dd(_p(x), nf, int(wide), float(foffset), _p(bits), _p(stats), _p(pk), _p(psym),
                                     _p(grids), max_packets)
    return bits, stats, pk[:n], psym[:n], grids[:n]


# ---- float64 model of the same algorithm ---------------------------------------------------------------------------
def dd_model64(S: np.ndarray):
    """scd_dd_packet in float64 (complex128): -> (raw decisions bI, bQ [248], derotated outputs complex128 [248])"""
    mu, alpha, beta, eps, amp, peps = (float(v) for v in dd_params())
    pre = po_preamble()
    S = np.asarray(S, np.complex128)
    w = np.zeros(5, np.complex128)
    p, nu = 1.0 + 0.0j, 0.0
    ys = np.zeros(PACKET_DATA_SYMBOLS, np.complex128)
    for i in range(po.PREAMBLE_LENGTH + PACKET_DATA_SYMBOLS):
        x = S[i:i + 5]
        y = np.sum(np.conj(w) * x) * np.conj(p)
        if i < po.PREAMBLE_LENGTH:
            d = amp * pre[i] * (1 + 1j)
        else:
            d = complex(-1.0 if y.real < 0 else 1.0, -1.0 if y.imag < 0 else 1.0)
            ys[i - po.PREAMBLE_LENGTH] = y
        e = d - y
        q = y * np.conj(d)
        pe = q.imag / (abs(q) + peps)
        w = w + x * np.conj(e * p) * (mu / (eps + np.sum(np.abs(x) ** 2)))
        nu += beta * pe
        p = p * (1 + 1j * (alpha * pe + nu))
        p /= abs(p)
    return (ys.real < 0).astype(np.uint8), (ys.imag < 0).astype(np.uint8), ys


@functools.lru_cache(maxsize=None)
def po_preamble():
    return np.array((C.c_int8 * po.PREAMBLE_LENGTH).in_dll(po.Oracle().lib, "sco_preamblevalues"), np.float64)


def grids64(x: np.ndarray, pk, foffset: float = 0.0, wide: bool = False) -> np.ndarray:
    """The 380-symbol grids of the records pk rebuilt in float64 from int16 samples x, with the receiver's mixer at
    -1100 + foffset Hz (a carrier offset of foffset Hz) on grids whose positions (call, max_index, timing) were found
    without it -> complex64 [len(pk), 380]"""
    taps = np.array((C.c_float * po.NTAPS).in_dll(po.Oracle().lib, "sco_alpha50_root" if wide else "sco_alpha35_root"),
                    np.float64)
    i = np.arange(x.size)
    m = np.exp(2j * np.pi * (-1100.0 + foffset) * (i + 1) / 8000.0) * (x.astype(np.float64) / 16384.0)
    filt = np.convolve(m, taps)[: x.size] * 2.2
    idx = ((pk["call"].astype(np.int64) - 2) * po.FRAME_SIZE + pk["timing"].astype(np.int64))[:, None] \
        + 5 * (pk["max_index"].astype(np.int64)[:, None] + np.arange(PACKET_SYMS)[None, :])
    return filt[idx].astype(np.complex64)


# ---- loop-back streams with known bits ----------------------------------------------------------------------------
def loop_streams(oracle, rng, n_streams, n_packets, sigma=0.0, gap=903, lead_max=2000):
    """Loop-back streams from the spec's packet-mode transmitter (pyoracle.ext_tx_packet, scrambled): random lead-in
    of 0 .. lead_max - 1 samples, gap zeros after every packet, AWGN of sigma LSB -> (int16 [n, n_frames * 1880],
    tx bits uint8 [n, n_packets, 496], packet starts int [n, n_packets])"""
    total = ((n_packets * (1880 + gap) + 2000 + 2 * 1880) // 1880) * 1880
    out = np.zeros((n_streams, total), np.int16)
    txb = np.zeros((n_streams, n_packets, 496), np.uint8)
    starts = np.zeros((n_streams, n_packets), np.int64)
    for s in range(n_streams):
        st = oracle.new_state()
        lead = int(rng.integers(0, lead_max))
        parts = [np.zeros(lead, np.int16)]
        for j in range(n_packets):
            txb[s, j] = rng.integers(0, 2, 496).astype(np.uint8)
            starts[s, j] = lead + j * (1880 + gap)
            parts.append(po.ext_tx_packet(oracle, st, txb[s, j]))
            parts.append(np.zeros(gap, np.int16))
        x = np.concatenate(parts).astype(np.float64)
        x = np.concatenate([x, np.zeros(max(0, total - x.size))])[:total]
        if sigma > 0:
            x = x + rng.normal(0, sigma, total)
        out[s] = np.clip(x, -32767, 32767).round().astype(np.int16)
    return out, txb, starts


def aligned(pk, starts, tol=10):
    """index of the transmitted packet each record's grid starts at (|pos - start| <= tol), or -1;
    pos = 1880 (call - 2) + 5 max_index + timing - 48 (the two filters' delays)"""
    pos = (pk["call"].astype(np.int64) - 2) * 1880 + 5 * pk["max_index"].astype(np.int64) + pk["timing"] - 48
    d = np.abs(pos[:, None] - np.asarray(starts)[None, :])
    j = d.argmin(axis=1) if len(starts) else np.zeros(len(pos), np.int64)
    return np.where(d[np.arange(len(pos)), j] <= tol, j, -1) if len(pos) else j

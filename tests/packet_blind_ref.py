"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_blind_ref.c, the specification of blind code detection
(sc_packet_decode_blind_dev), a numpy model of its selection over the three decode_code records, and loop-back streams
whose code changes packet by packet.  The candidates' decoder and the code-rate pieces are packet_code_ref's.  The C
file is compiled on first use with the oracle's flags into a temporary directory."""
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile
import threading

import numpy as np

from packet_code_ref import CODE_BYTES, CODE_CODED, PAYLOAD_EX_DTYPE, PAYLOAD_MAX, encode_code
from packet_fec_ref import PACKET_BITS

HERE = os.path.dirname(os.path.abspath(__file__))
_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    tmp = tempfile.mkdtemp(prefix="sc_packet_blind_ref_")
    out = os.path.join(tmp, "libsc_packet_blind_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-o", out, os.path.join(HERE, "packet_blind_ref.c"), "-lm"],
                       check=True)
        L = C.CDLL(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    vp = C.c_void_p
    L.scf_decode_blind_batch.argtypes, L.scf_decode_blind_batch.restype = [C.c_uint, vp, C.c_long, vp], None
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def decode_blind(mask: int, llrs: np.ndarray) -> np.ndarray:
    """mask (1..7), LLRs float32 [n, 496] -> PAYLOAD_EX_DTYPE [n]"""
    L = np.ascontiguousarray(llrs, np.float32).reshape(-1, PACKET_BITS)
    out = np.zeros(L.shape[0], PAYLOAD_EX_DTYPE)
    with _lock:
        lib = _build()
    lib.scf_decode_blind_batch(int(mask), _p(L), L.shape[0], _p(out))
    return out


def select_np(mask: int, records) -> np.ndarray:
    """numpy model of the selection: records[c] = decode_code(c, llrs) for c = 0, 1, 2 (PAYLOAD_EX_DTYPE [n] each) ->
    the chosen record per row.  Candidates are ordered by (crc_ok descending, flipped / N ascending, code ascending);
    the ratio is exact as flipped times the product of the other two N (flipped / N over a common denominator), and
    the three keys go into one int64 whose minimum is chosen."""
    cands = [c for c in range(3) if (mask >> c) & 1]
    n = records[0].shape[0]
    den = int(np.prod(np.asarray(CODE_CODED, np.int64)))
    keys = []
    for c in cands:
        ratio = records[c]["flipped"].astype(np.int64) * (den // CODE_CODED[c])       # < 2^27
        keys.append(((1 - records[c]["crc_ok"].astype(np.int64)) << 32) + (ratio << 2) + c)
    best = np.asarray(cands)[np.argmin(np.stack(keys), axis=0)]
    out = np.zeros(n, PAYLOAD_EX_DTYPE)
    for c in cands:
        out[best == c] = records[c][best == c]
    return out


def coded_streams_packet_code(oracle, rng, codes, sigma=0.0, gap=903):
    """loop-back streams of coded packets, packet j of stream s at code codes[s, j] (uint8 [n_streams, n_packets]) ->
    (int16 [n, n_frames * 1880], payloads uint8 [n, n_packets, 41] with the bytes past each packet's B zero, packet
    starts int [n, n_packets])"""
    from oracle import pyoracle as po
    codes = np.asarray(codes, np.uint8)
    n_streams, n_packets = codes.shape
    total = ((n_packets * (1880 + gap) + 2000 + 2 * 1880) // 1880) * 1880
    out = np.zeros((n_streams, total), np.int16)
    pay = rng.integers(0, 256, (n_streams, n_packets, PAYLOAD_MAX)).astype(np.uint8)
    pay[np.arange(PAYLOAD_MAX) >= np.asarray(CODE_BYTES)[codes][..., None]] = 0
    bits = encode_code(codes.reshape(-1), pay.reshape(-1, PAYLOAD_MAX)).reshape(n_streams, n_packets, PACKET_BITS)
    starts = np.zeros((n_streams, n_packets), np.int64)
    for s in range(n_streams):
        st = oracle.new_state()
        lead = int(rng.integers(0, 2000))
        parts = [np.zeros(lead, np.int16)]
        for j in range(n_packets):
            starts[s, j] = lead + j * (1880 + gap)
            parts.append(po.ext_tx_packet(oracle, st, bits[s, j]))
            parts.append(np.zeros(gap, np.int16))
        x = np.concatenate(parts).astype(np.float64)
        x = np.concatenate([x, np.zeros(max(0, total - x.size))])[:total]
        if sigma > 0:
            x = x + rng.normal(0, sigma, total)
        out[s] = np.clip(x, -32767, 32767).round().astype(np.int16)
    return out, pay, starts

"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_code_ref.c, the specification of the code rates of packet
mode's coded payload (sc_packet_encode_ex_dev, sc_packet_decode_ex_dev), an independent numpy model of the punctured
code (integer encoder, float64 Viterbi), its free distance, and loop-back streams at one code.  The rate-1/2 pieces (CRC,
interleaver, LLRs, the numpy parity table) are packet_fec_ref's.  The C file is compiled on first use with the oracle's
flags into a temporary directory."""
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile
import threading

import numpy as np

from packet_fec_ref import G0, G1, PACKET_BITS, PARITY, PERM64, crc16_np

HERE = os.path.dirname(os.path.abspath(__file__))
_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    tmp = tempfile.mkdtemp(prefix="sc_packet_code_ref_")
    out = os.path.join(tmp, "libsc_packet_code_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-o", out, os.path.join(HERE, "packet_code_ref.c"), "-lm"],
                       check=True)
        L = C.CDLL(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    vp = C.c_void_p
    for name in ("scf_code_bytes", "scf_code_steps", "scf_code_coded"):
        getattr(L, name).argtypes, getattr(L, name).restype = [C.c_int], C.c_int
    L.scf_mother.argtypes, L.scf_mother.restype = [C.c_int, C.c_int], C.c_int
    L.scf_encode_code_batch.argtypes, L.scf_encode_code_batch.restype = [vp, vp, C.c_long, vp], None
    L.scf_decode_code_batch.argtypes, L.scf_decode_code_batch.restype = [vp, vp, C.c_long, vp, vp, vp], None
    return L


def _code_lib():
    with _lock:
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


PAYLOAD_MAX, STEPS_MAX = 41, 350
CODE_BYTES, CODE_CODED = (27, 36, 41), (476, 465, 467)
CODE_STEPS = tuple(8 * b + 22 for b in CODE_BYTES)
PAYLOAD_EX_DTYPE = np.dtype([("data", "u1", (41,)), ("code", "u1"), ("crc_ok", "u1"), ("reserved0", "u1"),
                             ("flipped", "<u2"), ("reserved1", "<u2")])
assert PAYLOAD_EX_DTYPE.itemsize == 48
PATTERNS = {0: ((1, 1),), 1: ((1, 1), (1, 0)), 2: ((1, 1), (1, 0), (0, 1))}   # mother bits (c0, c1) kept per step


def code_sizes(code: int):
    """(B, T, N) of the spec"""
    L = _code_lib()
    return L.scf_code_bytes(code), L.scf_code_steps(code), L.scf_code_coded(code)


def mother_map(code: int) -> np.ndarray:
    """m(n), n < N"""
    return np.array([_code_lib().scf_mother(code, n) for n in range(code_sizes(code)[2])], np.int64)


def _codes(code, n):
    """a scalar code or one per record -> uint8 [n]"""
    return np.ascontiguousarray(np.broadcast_to(np.asarray(code, np.uint8), (n,)))


def encode_code(code, payload: np.ndarray) -> np.ndarray:
    """code (scalar or uint8 [n]), payload uint8 [n, 41] -> bits uint8 [n, 496]"""
    p = np.ascontiguousarray(payload, np.uint8).reshape(-1, PAYLOAD_MAX)
    out = np.zeros((p.shape[0], PACKET_BITS), np.uint8)
    c = _codes(code, p.shape[0])
    _code_lib().scf_encode_code_batch(_p(c), _p(p), p.shape[0], _p(out))
    return out


def decode_code(code, llrs: np.ndarray, path: bool = False):
    """code (scalar or uint8 [n]), LLRs float32 [n, 496] -> PAYLOAD_EX_DTYPE [n]; with path also the decoded info bits
    uint8 [n, 350] (the first T valid) and the final path metrics float32 [n, 64]"""
    L = np.ascontiguousarray(llrs, np.float32).reshape(-1, PACKET_BITS)
    out = np.zeros(L.shape[0], PAYLOAD_EX_DTYPE)
    pm = np.zeros((L.shape[0], 64), np.float32)
    u = np.zeros((L.shape[0], STEPS_MAX), np.uint8)
    c = _codes(code, L.shape[0])
    _code_lib().scf_decode_code_batch(_p(c), _p(L), L.shape[0], _p(out), _p(pm), _p(u))
    return (out, u, pm) if path else out


# numpy model of the punctured code (integer encoder, float64 Viterbi), written from the patterns, not from scf_mother
def mother_map_np(code: int) -> np.ndarray:
    pat = PATTERNS[code]
    T = CODE_STEPS[code]
    return np.array([2 * t + i for t in range(T) for i in (0, 1) if pat[t % len(pat)][i]], np.int64)


def info_bits_code(code: int, payload: np.ndarray) -> np.ndarray:
    """uint8 [n, >= B] -> u uint8 [n, T]"""
    B, T = CODE_BYTES[code], CODE_STEPS[code]
    p = np.asarray(payload, np.uint8).reshape(payload.shape[0], -1)[:, :B]
    crc = np.array([crc16_np(row.tobytes()) for row in p], np.int64)
    by = np.concatenate([p, (crc >> 8).astype(np.uint8)[:, None], (crc & 255).astype(np.uint8)[:, None]], axis=1)
    return np.concatenate([np.unpackbits(by, axis=1), np.zeros((p.shape[0], T - 8 * B - 16), np.uint8)], axis=1)


def mother_bits(u: np.ndarray) -> np.ndarray:
    """info bits [n, T] -> mother bits [n, 2T] (integer shift register)"""
    u = np.asarray(u, np.int64)
    c = np.zeros((u.shape[0], 2 * u.shape[1]), np.uint8)
    s = np.zeros(u.shape[0], np.int64)
    for t in range(u.shape[1]):
        r = (u[:, t] << 6) | s
        c[:, 2 * t] = PARITY[r & G0]
        c[:, 2 * t + 1] = PARITY[r & G1]
        s = r >> 1
    return c


def encode_code_np(code: int, payload: np.ndarray) -> np.ndarray:
    c = mother_bits(info_bits_code(code, payload))[:, mother_map_np(code)]
    bits = np.zeros((c.shape[0], PACKET_BITS), np.uint8)
    bits[:, PERM64[:c.shape[1]]] = c
    return bits


def mother_llrs64(code: int, llrs: np.ndarray) -> np.ndarray:
    """sanitised LLRs [n, 496] -> L' float64 [n, 2T] in mother order, 0 where punctured"""
    L = np.clip(np.nan_to_num(np.asarray(llrs, np.float64), nan=0.0, posinf=0.0, neginf=0.0), -2.0 ** 24, 2.0 ** 24)
    m = mother_map_np(code)
    out = np.zeros((L.shape[0], 2 * CODE_STEPS[code]))
    out[:, m] = L[:, PERM64[:m.size]]
    return out


def viterbi64_code(code: int, llrs: np.ndarray):
    """float64 Viterbi of the punctured code -> (info bits [n, T], final metrics float64 [n, 64])"""
    Lm = mother_llrs64(code, llrs)
    n, T = Lm.shape[0], CODE_STEPS[code]
    pm = np.full((n, 64), -np.inf)
    pm[:, 0] = 0.0
    dec = np.zeros((T, n, 64), np.uint8)
    sp = np.arange(64)
    for t in range(T):
        l0, l1 = Lm[:, 2 * t][:, None], Lm[:, 2 * t + 1][:, None]
        cand = []
        for b in (0, 1):
            q = ((sp << 1) & 63) | b
            r = ((sp >> 5) << 6) | q
            cand.append(pm[:, q] + np.where(PARITY[r & G0], -l0, l0) + np.where(PARITY[r & G1], -l1, l1))
        take = cand[1] > cand[0]
        dec[t] = take
        pm = np.where(take, cand[1], cand[0])
    s = np.zeros(n, np.int64)
    u = np.zeros((n, T), np.uint8)
    for t in range(T - 1, -1, -1):
        u[:, t] = s >> 5
        s = ((s << 1) & 63) | dec[t, np.arange(n), s]
    return u, pm


def correlation64_code(code: int, llrs: np.ndarray, c: np.ndarray) -> np.ndarray:
    """sum_m (1 - 2 c_m) L'[m] in float64 over the mother bits c [n, 2T]"""
    return ((1.0 - 2.0 * c.astype(np.float64)) * mother_llrs64(code, llrs)).sum(axis=1)


def free_distance(code: int) -> int:
    """minimum Hamming weight of a nonzero codeword of the terminated, punctured code: a search over the trellis from
    every divergence step (a path leaves state 0 at t0 with input 1 and is followed until it returns to state 0;
    inputs of the last 6 steps are 0)"""
    pat, T = PATTERNS[code], CODE_STEPS[code]

    def w(t, r):
        k = pat[t % len(pat)]
        return (int(PARITY[r & G0]) if k[0] else 0) + (int(PARITY[r & G1]) if k[1] else 0)

    best = 1 << 30
    for t0 in range(T - 6):
        cur = {(1 << 6) >> 1: w(t0, 1 << 6)}
        t = t0 + 1
        while t < T and cur:
            nxt = {}
            for s, ws in cur.items():
                for u in ((0, 1) if t < T - 6 else (0,)):
                    r = (u << 6) | s
                    ww = ws + w(t, r)
                    if r >> 1 == 0:
                        best = min(best, ww)
                    elif ww < best and ww < nxt.get(r >> 1, 1 << 30):
                        nxt[r >> 1] = ww
            cur, t = nxt, t + 1
    return best


def coded_streams_code(oracle, rng, n_streams, n_packets, code, sigma=0.0, gap=903):
    """coded_streams at one code for every stream -> (int16 [n, n_frames * 1880], payloads uint8 [n, n_packets, 41]
    with the bytes past B zero, packet starts int [n, n_packets])"""
    from oracle import pyoracle as po
    B = CODE_BYTES[code]
    total = ((n_packets * (1880 + gap) + 2000 + 2 * 1880) // 1880) * 1880
    out = np.zeros((n_streams, total), np.int16)
    pay = np.zeros((n_streams, n_packets, PAYLOAD_MAX), np.uint8)
    pay[:, :, :B] = rng.integers(0, 256, (n_streams, n_packets, B))
    bits = encode_code(code, pay.reshape(-1, PAYLOAD_MAX)).reshape(n_streams, n_packets, PACKET_BITS)
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

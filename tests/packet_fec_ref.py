"""TEST INFRASTRUCTURE: ctypes binding of tests/packet_fec_ref.c, the specification of packet mode's coded payload
(sc_packet_encode_dev, sc_packet_llr_dev, sc_packet_decode_dev), an independent numpy model of the same code (integer
encoder, float64 Viterbi) and loop-back streams that carry chosen payloads.  The C file is compiled on first use with
the oracle's flags into a temporary directory."""
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile
import threading

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PAYLOAD_BYTES, CODED_BITS, PACKET_BITS, STEPS = 27, 476, 496, 238
PAYLOAD_DTYPE = np.dtype([("data", "u1", (27,)), ("crc_ok", "u1"), ("flipped", "<u2"), ("reserved", "<u2")])
assert PAYLOAD_DTYPE.itemsize == 32

_lock = threading.Lock()


@functools.lru_cache(maxsize=None)
def _build():
    tmp = tempfile.mkdtemp(prefix="sc_packet_fec_ref_")
    out = os.path.join(tmp, "libsc_packet_fec_ref.so")
    try:
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-ffp-contract=off", "-fPIC", "-fno-strict-aliasing", "-Wall",
                        "-Wextra", "-Werror", "-shared", "-o", out, os.path.join(HERE, "packet_fec_ref.c"), "-lm"],
                       check=True)
        L = C.CDLL(out)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    vp = C.c_void_p
    L.scf_crc16.argtypes, L.scf_crc16.restype = [vp, C.c_int], C.c_uint16
    L.scf_perm.argtypes, L.scf_perm.restype = [C.c_int], C.c_int
    L.scf_keystream.argtypes, L.scf_keystream.restype = [vp], None
    L.scf_encode_batch.argtypes, L.scf_encode_batch.restype = [vp, C.c_long, vp], None
    L.scf_llr_batch.argtypes, L.scf_llr_batch.restype = [vp, C.c_long, vp], None
    L.scf_decode_batch.argtypes, L.scf_decode_batch.restype = [vp, C.c_long, vp, vp, vp], None
    return L


def _lib():
    with _lock:
        return _build()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def crc16(data) -> int:
    b = np.frombuffer(bytes(data), np.uint8).copy()
    return int(_lib().scf_crc16(_p(b), b.size))


def perm() -> np.ndarray:
    """pi(n), n < 476: the packet bit position of coded bit n"""
    return np.array([_lib().scf_perm(n) for n in range(CODED_BITS)], np.int64)


def keystream() -> np.ndarray:
    ks = np.zeros(8, np.uint64)
    _lib().scf_keystream(_p(ks))
    return ks


def encode(payload: np.ndarray) -> np.ndarray:
    """uint8 [..., 27] -> bits uint8 [..., 496]"""
    p = np.ascontiguousarray(payload, np.uint8)
    n = p.size // PAYLOAD_BYTES
    out = np.zeros((n, PACKET_BITS), np.uint8)
    _lib().scf_encode_batch(_p(p), n, _p(out))
    return out.reshape(p.shape[:-1] + (PACKET_BITS,))


def llr(blocks: np.ndarray) -> np.ndarray:
    """packet symbols complex64 [n, 248] (or float32 [n, 496]) -> LLRs float32 [n, 496]"""
    y = np.ascontiguousarray(blocks).view(np.float32).reshape(-1, PACKET_BITS)
    out = np.zeros_like(y)
    _lib().scf_llr_batch(_p(y), y.shape[0], _p(out))
    return out


def decode(llrs: np.ndarray, path: bool = False):
    """LLRs float32 [n, 496] -> PAYLOAD_DTYPE [n]; with path also the decoded info bits uint8 [n, 238] and the final
    path metrics float32 [n, 64]"""
    L = np.ascontiguousarray(llrs, np.float32).reshape(-1, PACKET_BITS)
    out = np.zeros(L.shape[0], PAYLOAD_DTYPE)
    pm = np.zeros((L.shape[0], 64), np.float32)
    u = np.zeros((L.shape[0], STEPS), np.uint8)
    _lib().scf_decode_batch(_p(L), L.shape[0], _p(out), _p(pm), _p(u))
    return (out, u, pm) if path else out


# ---- independent numpy model ---------------------------------------------------------------------------------------
G0, G1 = 0o133, 0o171
PARITY = np.array([bin(i).count("1") & 1 for i in range(128)], np.uint8)
PERM64 = np.array([17 * (n % 28) + n // 28 for n in range(CODED_BITS)], np.int64)


def crc16_np(data) -> int:
    c = 0xFFFF
    for x in bytes(data):
        c ^= x << 8
        for _ in range(8):
            c = ((c << 1) ^ 0x1021) & 0xFFFF if c & 0x8000 else (c << 1) & 0xFFFF
    return c


def info_bits(payload: np.ndarray) -> np.ndarray:
    """uint8 [n, 27] -> u uint8 [n, 238] (payload, CRC high byte first, 6 tail zeros)"""
    p = np.asarray(payload, np.uint8).reshape(-1, PAYLOAD_BYTES)
    crc = np.array([crc16_np(row.tobytes()) for row in p], np.int64)
    by = np.concatenate([p, (crc >> 8).astype(np.uint8)[:, None], (crc & 255).astype(np.uint8)[:, None]], axis=1)
    u = np.unpackbits(by, axis=1)
    return np.concatenate([u, np.zeros((p.shape[0], STEPS - 232), np.uint8)], axis=1)


def code_bits(u: np.ndarray) -> np.ndarray:
    """info bits [n, 238] -> coded bits [n, 476] (integer shift register)"""
    u = np.asarray(u, np.int64)
    c = np.zeros((u.shape[0], CODED_BITS), np.uint8)
    s = np.zeros(u.shape[0], np.int64)
    for t in range(STEPS):
        r = (u[:, t] << 6) | s
        c[:, 2 * t] = PARITY[r & G0]
        c[:, 2 * t + 1] = PARITY[r & G1]
        s = r >> 1
    return c


def encode_np(payload: np.ndarray) -> np.ndarray:
    c = code_bits(info_bits(payload))
    bits = np.zeros((c.shape[0], PACKET_BITS), np.uint8)
    bits[:, PERM64] = c
    return bits


def viterbi64(llrs: np.ndarray):
    """float64 Viterbi on sanitised LLRs [n, 496] -> (info bits [n, 238], final metrics float64 [n, 64])"""
    L = np.nan_to_num(np.asarray(llrs, np.float64), nan=0.0, posinf=0.0, neginf=0.0)
    L = np.clip(L, -2.0 ** 24, 2.0 ** 24)[:, PERM64]
    n = L.shape[0]
    pm = np.full((n, 64), -np.inf)
    pm[:, 0] = 0.0
    dec = np.zeros((STEPS, n, 64), np.uint8)
    sp = np.arange(64)
    for t in range(STEPS):
        l0, l1 = L[:, 2 * t][:, None], L[:, 2 * t + 1][:, None]
        cand = []
        for b in (0, 1):
            q = ((sp << 1) & 63) | b
            r = ((sp >> 5) << 6) | q
            m = np.where(PARITY[r & G0], -l0, l0) + np.where(PARITY[r & G1], -l1, l1)
            cand.append(pm[:, q] + m)
        take = cand[1] > cand[0]
        dec[t] = take
        pm = np.where(take, cand[1], cand[0])
    s = np.zeros(n, np.int64)
    u = np.zeros((n, STEPS), np.uint8)
    for t in range(STEPS - 1, -1, -1):
        u[:, t] = s >> 5
        s = ((s << 1) & 63) | dec[t, np.arange(n), s]
    return u, pm


def correlation64(llrs: np.ndarray, c: np.ndarray) -> np.ndarray:
    """sum_n (1 - 2 c_n) L'[pi(n)] in float64: the metric the decoder maximises"""
    L = np.clip(np.nan_to_num(np.asarray(llrs, np.float64), nan=0.0, posinf=0.0, neginf=0.0), -2.0 ** 24, 2.0 ** 24)
    return ((1.0 - 2.0 * c.astype(np.float64)) * L[:, PERM64]).sum(axis=1)


# ---- loop-back streams with chosen payloads -------------------------------------------------------------------------
def coded_streams(oracle, rng, n_streams, n_packets, sigma=0.0, gap=903):
    """Loop-back streams from the spec's packet-mode transmitter (pyoracle.ext_tx_packet, scrambled) carrying random
    payloads through the packet code: random lead-in, gap zeros after every packet, AWGN of sigma LSB ->
    (int16 [n, n_frames * 1880], payloads uint8 [n, n_packets, 27], packet starts int [n, n_packets])"""
    from oracle import pyoracle as po
    total = ((n_packets * (1880 + gap) + 2000 + 2 * 1880) // 1880) * 1880
    out = np.zeros((n_streams, total), np.int16)
    pay = rng.integers(0, 256, (n_streams, n_packets, PAYLOAD_BYTES)).astype(np.uint8)
    bits = encode(pay)
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

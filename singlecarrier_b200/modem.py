"""Host mirror of the reference's modem interface, batched over a bank of streams.

``ModemBank.rx_frames`` is N lock-step copies of the reference's ``while(1) { fread;
qpsk_rx_frame(); fwrite }`` loop (/root/reference/src/qpsk.c:436-458); ``ModemBank.tx_packets`` is
N copies of its transmit loop (qpsk.c:380-413).  Everything is computed by the CUDA kernels behind
``libsinglecarrier_b200.so``; this file only moves pointers.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from ._lib import SC_FLAG_DEBUG_EQ, SC_FLAG_PACKET, SC_FLAG_PACKET_ACQ, SC_FLAG_PACKET_DD, SC_FLAG_WIDE, Channel, check, lib

FRAME_SIZE = 1880
SYMBOLS_PER_FRAME = 376
BITS_PER_CALL = 62
DATA_SYMBOLS = 31          # data steps per call: bits 2i (Q) and 2i+1 (I) are sliced from symbol i
PACKET_FRAMES = 8          # data frames per packet (packet mode)
PACKET_DATA_SYMBOLS = PACKET_FRAMES * DATA_SYMBOLS   # 248 data steps per packet record
PACKET_SAMPLES = 1880
OPT_SLAB_PARTS, OPT_PROFILE, OPT_H2D_MODE, OPT_FE_SEARCH, OPT_TRACKER, OPT_OVERLAP = 1, 2, 3, 4, 5, 6
OVERLAP_AUTO, OVERLAP_OFF, OVERLAP_ON, OVERLAP_MAX = 0, 1, 2, 32768
TRACKER_AUTO, TRACKER_THREAD, TRACKER_COOP, TRACKER_COOP_MAX = 0, 1, 2, 1024
FE_SEARCH_DIRECT, FE_SEARCH_MMA, FE_SEARCH_TCGEN05 = 0, 1, 2
H2D_COLUMNS, H2D_ROWS, H2D_FULL, H2D_COLUMNS_3D = 0, 1, 2, 3
N_COUNTERS, N_BER_COUNTERS, N_PACKET_BER_COUNTERS = 16, 8, 32
REFERENCE_GAP = 903         # dead air between packets in the reference's main(), qpsk.c:410-412

# sc_frame_result, include/singlecarrier_b200.h
RESULT_DTYPE = np.dtype([("bits", "<u8"), ("max_value", "<f4"), ("cost", "<f4"), ("max_index", "<i2"),
                         ("matches", "<i2"), ("rx_timing", "<i2"), ("valid", "u1"), ("reserved0", "u1"),
                         ("call_index", "<u4"), ("reserved1", "<u4")])
assert RESULT_DTYPE.itemsize == 32
# sc_packet_result (packet mode, an extension without a counterpart in the reference)
PACKET_DTYPE = np.dtype([("bits", "<u8", (8,)), ("stream", "<i4"), ("call_index", "<u4"), ("max_index", "<i2"),
                         ("matches", "<i2"), ("cost", "<f4"), ("acq_metric", "<f4"), ("acq_freq_hz", "<f4"),
                         ("grid_sample", "<i8")])
assert PACKET_DTYPE.itemsize == 96
# sc_packet_payload: one decoded packet of the coded payload (DESIGN.md section 8c)
PAYLOAD_BYTES, PACKET_CODED_BITS, PACKET_BITS = 27, 476, 496
PAYLOAD_DTYPE = np.dtype([("data", "u1", (PAYLOAD_BYTES,)), ("crc_ok", "u1"), ("flipped", "<u2"), ("reserved", "<u2")])
assert PAYLOAD_DTYPE.itemsize == 32
# code rates (DESIGN.md section 8c, "Code rates"): one code per stream; sc_packet_payload_ex records
CODE_R12, CODE_R23, CODE_R34 = 0, 1, 2
PAYLOAD_MAX = 41
PAYLOAD_EX_DTYPE = np.dtype([("data", "u1", (PAYLOAD_MAX,)), ("code", "u1"), ("crc_ok", "u1"), ("reserved0", "u1"),
                             ("flipped", "<u2"), ("reserved1", "<u2")])
assert PAYLOAD_EX_DTYPE.itemsize == 48


def payload_bytes(code: int) -> int:
    """Payload bytes of a packet at code rate ``code`` (27, 36, 41; 0 for any other value)."""
    return int(lib.sc_packet_payload_bytes(int(code)))


def keystream_word(call_index: int) -> int:
    return int(lib.sc_keystream_word(call_index))


def soft_bits(results: np.ndarray, symbols: np.ndarray) -> np.ndarray:
    """Soft decisions in the order of ``bits``: float32 [..., 62] with soft[2i] = +-Im and soft[2i+1] = +-Re of
    symbol i, negated where the call's keystream bit is 1, so that bit k == (soft[k] < 0) wherever the component
    is non-zero.  ``results`` RESULT_DTYPE [...], ``symbols`` complex64 [..., 31] from rx_frames_soft_*."""
    r = np.asarray(results)
    assert r.dtype == RESULT_DTYPE
    sym = np.asarray(symbols, np.complex64)
    assert sym.shape == r.shape + (DATA_SYMBOLS,)
    soft = np.empty(r.shape + (BITS_PER_CALL,), np.float32)
    soft[..., 0::2] = sym.imag
    soft[..., 1::2] = sym.real
    calls = r["call_index"].ravel()
    uniq, inv = np.unique(calls, return_inverse=True)
    words = np.array([keystream_word(int(c)) for c in uniq], np.uint64)[inv].reshape(r.shape)
    flip = ((words[..., None] >> np.arange(BITS_PER_CALL, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    soft[flip] = -soft[flip]
    return soft


def packet_keystream_word(frame: int) -> int:
    """Descrambler word of data frame ``frame`` (0..7) of every packet (the register is seeded per packet)."""
    return int(lib.sc_packet_keystream_word(frame))


def packet_soft_bits(packets: np.ndarray, packet_symbols: np.ndarray) -> np.ndarray:
    """The packet counterpart of soft_bits: float32 [n, 8, 62] in the order of the packets' bits (frame f, bit k),
    soft[f, 2i] = +-Im and soft[f, 2i+1] = +-Re of symbol 31 f + i, negated where the packet keystream bit is 1, so
    that bit == (soft < 0) wherever the component is non-zero.  ``packets`` PACKET_DTYPE [n], ``packet_symbols``
    complex64 [n, 248] from rx_packets_soft_*."""
    p = np.asarray(packets)
    assert p.dtype == PACKET_DTYPE and p.ndim == 1
    sym = np.asarray(packet_symbols, np.complex64).reshape(p.shape[0], PACKET_FRAMES, DATA_SYMBOLS)
    soft = np.empty((p.shape[0], PACKET_FRAMES, BITS_PER_CALL), np.float32)
    soft[..., 0::2] = sym.imag
    soft[..., 1::2] = sym.real
    words = np.array([packet_keystream_word(f) for f in range(PACKET_FRAMES)], np.uint64)
    flip = ((words[:, None] >> np.arange(BITS_PER_CALL, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    soft[:, flip] = -soft[:, flip]
    return soft


def launch_count() -> int:
    return int(lib.sc_launch_count())


def unpack_packet_bits(packets: np.ndarray) -> np.ndarray:
    """PACKET_DTYPE records -> payload bits [n, 8, 62] (bit-per-byte, the layout of sc_tx_*_dev's bits_out)."""
    w = packets["bits"].astype(np.uint64)                                       # [n, 8]
    return ((w[:, :, None] >> np.arange(62, dtype=np.uint64)[None, None, :]) & np.uint64(1)).astype(np.uint8)


def unpack_bits(results: np.ndarray, rows: Optional[np.ndarray] = None) -> np.ndarray:
    """Results -> the reference's bit-per-byte rows (62 per VALID call); invalid rows stay 255."""
    r = np.ascontiguousarray(results)
    assert r.dtype == RESULT_DTYPE
    if rows is None:
        rows = np.full(r.shape + (BITS_PER_CALL,), 255, np.uint8)
    lib.sc_unpack_bits(r.ctypes.data, r.size, rows.ctypes.data)
    return rows


class PinnedBuffer:
    """Page-locked host memory on the NUMA node of ``device`` (sc_host_alloc); ``array(dtype, shape)``
    gives numpy views.  Freed by ``close()`` / garbage collection."""

    def __init__(self, nbytes: int, device: int = 0):
        self._p = C.c_void_p()
        node = C.c_int(-1)
        check(lib.sc_host_alloc(C.byref(self._p), nbytes, device, C.byref(node)))
        self.nbytes, self.numa_node = nbytes, node.value

    def array(self, dtype, shape, offset: int = 0) -> np.ndarray:
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        assert offset + count * dtype.itemsize <= self.nbytes
        buf = (C.c_char * (count * dtype.itemsize)).from_address(self._p.value + offset)
        a = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)
        a.flags.writeable = True
        return a

    def close(self) -> None:
        if self._p:
            lib.sc_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def h2d_probe(device: int, buffer_bytes: int, row_bytes: int = 0, src_pitch_bytes: int = 0, min_seconds: float = 0.5,
              d2h: bool = False) -> float:
    """GB/s of plain pinned-host <-> device copies (sc_h2d_probe): the platform ceiling of the host entry point."""
    out = C.c_double(0.0)
    check(lib.sc_h2d_probe(device, buffer_bytes, row_bytes, src_pitch_bytes, min_seconds, int(d2h), C.byref(out)))
    return out.value


class NcclComm:
    """A ncclComm_t created through the library's NCCL bridge (sc_comm_*)."""

    def __init__(self, handle):
        self._c = handle

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        check(lib.sc_comm_unique_id(buf))
        return buf.raw

    @classmethod
    def init_rank(cls, n_ranks: int, rank: int, unique_id: bytes, device: int) -> "NcclComm":
        h = C.c_void_p()
        check(lib.sc_comm_init_rank(C.byref(h), n_ranks, rank, unique_id, device))
        return cls(h)

    @classmethod
    def init_all(cls, devices) -> list:
        n = len(devices)
        arr = (C.c_void_p * n)()
        devs = (C.c_int * n)(*devices)
        check(lib.sc_comm_init_all(arr, n, devs))
        return [cls(C.c_void_p(arr[i])) for i in range(n)]

    def all_reduce_counters(self, counters, stream: int = 0) -> None:
        """In-place sum of a CUDA int64/uint64 tensor over the communicator (sc_reduce_stats)."""
        check(lib.sc_reduce_stats(counters.data_ptr(), counters.numel(), self._c, stream))

    def close(self) -> None:
        if self._c:
            lib.sc_comm_destroy(self._c)
            self._c = C.c_void_p()


def _ptr(t) -> int:
    """Device/host pointer of a torch tensor or numpy array (0 for None)."""
    if t is None:
        return 0
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


class ModemBank:
    """A bank of ``n_streams`` synchronized modems on one GPU (sc_modem handle)."""

    def __init__(self, n_streams: int, device: int = 0, wide: bool = False, foffset_hz: float = 0.0,
                 debug_eq: bool = False, packet: bool = False, dd: bool = False, acq: bool = False):
        """packet: packet mode (SC_FLAG_PACKET); dd: its packets decoded by the decision-directed equalizer
        (SC_FLAG_PACKET_DD, needs packet=True); acq: packets found by acquisition on the samples (SC_FLAG_PACKET_ACQ,
        needs packet=True and dd=True)."""
        self._h = C.c_void_p()
        flags = (SC_FLAG_WIDE if wide else 0) | (SC_FLAG_DEBUG_EQ if debug_eq else 0) | (SC_FLAG_PACKET if packet else 0) \
            | (SC_FLAG_PACKET_DD if dd else 0) | (SC_FLAG_PACKET_ACQ if acq else 0)
        self.packet = packet
        self.dd = dd
        self.acq = acq
        check(lib.sc_create(C.byref(self._h), device, n_streams, flags, foffset_hz))
        self.n_streams = n_streams
        self.device = device
        self.debug_eq = debug_eq

    @staticmethod
    def result_dtype() -> np.dtype:
        return RESULT_DTYPE

    def close(self) -> None:
        if self._h:
            lib.sc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self) -> None:
        check(lib.sc_reset(self._h))

    @property
    def call_index(self) -> int:
        return int(lib.sc_call_index(self._h))

    def set_option(self, option: int, value: int) -> None:
        check(lib.sc_set_option(self._h, option, value))

    def profile_read(self) -> dict:
        out = (C.c_double * 4)()
        check(lib.sc_profile_read(self._h, out))
        return {"frontend_ms": out[0], "frontend_launches": int(out[1]), "track_ms": out[2], "track_launches": int(out[3])}

    def lock_stats(self, results, n_frames: int, counters, stream: int = 0) -> None:
        """Accumulate the 16 lock/bit counters of results (CUDA uint8 [n, >= n_frames*32]) into counters (CUDA int64[16])."""
        check(lib.sc_lock_stats_dev(self.device, results.data_ptr(), self.n_streams, results.stride(0) // 32, n_frames,
                                    counters.data_ptr(), stream))

    def ber_stats(self, results, n_frames: int, tx_bits, lead_in, gap: int, counters, group=None, n_groups: int = 1,
                  stream: int = 0) -> None:
        """Accumulate the bit-error counters (sc_ber_stats_dev) of a cold-started batch into counters
        (CUDA int64 [n_groups, 8]): calls, valid, aligned, bits, errors."""
        n_packets = tx_bits.shape[1]
        check(lib.sc_ber_stats_dev(self.device, results.data_ptr(), self.n_streams, results.stride(0) // 32, n_frames,
                                   tx_bits.data_ptr(), n_packets, _ptr(lead_in), gap, _ptr(group), n_groups,
                                   counters.data_ptr(), stream))

    def packet_ber_stats(self, packets, n_found, results, n_frames: int, tx_bits, lead_in, gap: int, counters,
                         group=None, n_groups: int = 1, stream: int = 0) -> None:
        """Accumulate the bit-error counters of packet records (sc_packet_ber_stats_dev) into counters (CUDA int64
        [n_groups, 32]).  packets = CUDA uint8 [capacity * 96] and n_found = CUDA int64[1] as rx_packets_dev filled
        them (n_found is read on the device); results, tx_bits, lead_in, gap, group as for ber_stats."""
        check(lib.sc_packet_ber_stats_dev(self.device, packets.data_ptr(), packets.numel() // 96, n_found.data_ptr(),
                                          results.data_ptr(), self.n_streams, results.stride(0) // 32, n_frames,
                                          tx_bits.data_ptr(), tx_bits.shape[1], _ptr(lead_in), gap, _ptr(group),
                                          n_groups, counters.data_ptr(), stream))

    def packet_encode(self, payload, bits, stream: int = 0) -> None:
        """Encode payloads (CUDA uint8 [..., 27]) into packet bits (CUDA uint8 [..., 8, 62], e.g. [n, n_packets, 8, 62]),
        the bits tx_packets_dev takes (sc_packet_encode_dev)."""
        n = payload.numel() // PAYLOAD_BYTES
        assert payload.is_contiguous() and bits.is_contiguous() and bits.numel() == n * PACKET_BITS
        check(lib.sc_packet_encode_dev(self.device, payload.data_ptr(), n, bits.data_ptr(), stream))

    def packet_llr(self, packet_symbols, n_found, llr, stream: int = 0) -> None:
        """LLRs (L > 0: bit 0) of the 496 bits of every record rx_packets_soft_dev left (sc_packet_llr_dev):
        packet_symbols as filled (496 floats per record, its size sets the capacity), n_found = CUDA int64[1] (read on
        the device), llr a CUDA float32 tensor of the same number of floats."""
        capacity = packet_symbols.numel() * packet_symbols.element_size() // (PACKET_BITS * 4)
        assert llr.numel() * llr.element_size() >= capacity * PACKET_BITS * 4, "capacity"
        check(lib.sc_packet_llr_dev(self.device, packet_symbols.data_ptr(), capacity, n_found.data_ptr(),
                                    llr.data_ptr(), stream))

    def packet_decode(self, llr, n_found, out, stream: int = 0) -> None:
        """Viterbi-decode the records' LLRs (CUDA float32, 496 per record, its size sets the capacity) into out (CUDA
        uint8 [capacity * 32], viewable as PAYLOAD_DTYPE) for the first min(n_found, capacity) records
        (sc_packet_decode_dev)."""
        capacity = llr.numel() * llr.element_size() // (PACKET_BITS * 4)
        assert out.numel() * out.element_size() >= capacity * PAYLOAD_DTYPE.itemsize, "capacity"
        check(lib.sc_packet_decode_dev(self.device, llr.data_ptr(), capacity, n_found.data_ptr(), out.data_ptr(),
                                       stream))

    def packet_encode_ex(self, payload, stream_code, bits, stream: int = 0) -> None:
        """Encode payloads (CUDA uint8 [n_streams, n_packets, 41]; bytes past the stream's payload_bytes are ignored)
        at each stream's code (stream_code: CUDA uint8 [n_streams]) into packet bits (CUDA uint8
        [n_streams, n_packets, 8, 62]) (sc_packet_encode_ex_dev).  A stream whose code is not 0..2 gets zero bits."""
        n_streams, n_packets = payload.shape[0], payload.shape[1]
        assert payload.is_contiguous() and bits.is_contiguous() and stream_code.is_contiguous()
        assert payload.numel() == n_streams * n_packets * PAYLOAD_MAX and stream_code.numel() == n_streams
        assert bits.numel() == n_streams * n_packets * PACKET_BITS
        check(lib.sc_packet_encode_ex_dev(self.device, payload.data_ptr(), n_streams, n_packets,
                                          stream_code.data_ptr(), bits.data_ptr(), stream))

    def packet_decode_ex(self, llr, packets, n_found, stream_code, out, stream: int = 0) -> None:
        """Viterbi-decode the records' LLRs (CUDA float32, 496 per record, its size sets the capacity) at the code of
        each record's stream (stream_code: CUDA uint8 [n_streams], packets: the records as rx_packets_soft_dev left
        them) into out (CUDA uint8 [capacity * 48], viewable as PAYLOAD_EX_DTYPE) for the first min(n_found, capacity)
        records (sc_packet_decode_ex_dev)."""
        capacity = llr.numel() * llr.element_size() // (PACKET_BITS * 4)
        assert packets.numel() * packets.element_size() >= capacity * PACKET_DTYPE.itemsize, "capacity"
        assert out.numel() * out.element_size() >= capacity * PAYLOAD_EX_DTYPE.itemsize, "capacity"
        assert stream_code.is_contiguous()
        check(lib.sc_packet_decode_ex_dev(self.device, llr.data_ptr(), packets.data_ptr(), capacity, n_found.data_ptr(),
                                          stream_code.data_ptr(), stream_code.numel(), out.data_ptr(), stream))

    def packet_decode_blind(self, llr, n_found, out, code_mask: int = 7, stream: int = 0) -> None:
        """Viterbi-decode the records' LLRs (CUDA float32, 496 per record, its size sets the capacity) at every code of
        code_mask (bit c for code c) and keep, per record, the best whose CRC passes (fewest flipped bits per
        transmitted bit, then the lower code), or the best of all when none passes, into out (CUDA uint8
        [capacity * 48], viewable as PAYLOAD_EX_DTYPE) for the first min(n_found, capacity) records
        (sc_packet_decode_blind_dev).  No code table is needed: each record's code field says which code it is."""
        capacity = llr.numel() * llr.element_size() // (PACKET_BITS * 4)
        assert out.numel() * out.element_size() >= capacity * PAYLOAD_EX_DTYPE.itemsize, "capacity"
        check(lib.sc_packet_decode_blind_dev(self.device, llr.data_ptr(), capacity, n_found.data_ptr(), int(code_mask),
                                             out.data_ptr(), stream))

    def transfer_bytes(self):
        out = (C.c_uint64 * 2)()
        check(lib.sc_transfer_bytes(self._h, out))
        return int(out[0]), int(out[1])

    def state_export(self) -> np.ndarray:
        """Checkpoint of the whole bank (sc_state_export) as a uint8 array."""
        n = int(lib.sc_state_size(self._h))
        buf = np.empty(n, np.uint8)
        check(lib.sc_state_export(self._h, buf.ctypes.data, n))
        return buf

    def state_import(self, image: np.ndarray) -> None:
        image = np.ascontiguousarray(image, np.uint8)
        check(lib.sc_state_import(self._h, image.ctypes.data, image.size))

    # ---- RX ------------------------------------------------------------------------------------
    def rx_frames_host(self, samples: np.ndarray, n_frames: Optional[int] = None, results: Optional[np.ndarray] = None):
        """samples: host int16 [n_streams, >= n_frames*1880] (numpy, or a pinned torch tensor's
        numpy view).  Returns (results[n_streams, n_frames], eq_coeff or None)."""
        assert samples.dtype == np.int16 and samples.ndim == 2 and samples.shape[0] == self.n_streams
        assert samples.strides[1] == 2
        stride = samples.strides[0] // 2
        if n_frames is None:
            n_frames = samples.shape[1] // FRAME_SIZE
        if results is None:
            results = np.zeros((self.n_streams, n_frames), RESULT_DTYPE)
        eq = np.zeros((self.n_streams, n_frames, 10), np.float32) if self.debug_eq else None
        check(lib.sc_rx_frames_host(self._h, samples.ctypes.data, stride, n_frames, results.ctypes.data,
                                    results.strides[0] // 32, _ptr(eq)))
        return results, eq

    def rx_frames_soft_host(self, samples: np.ndarray, n_frames: Optional[int] = None):
        """rx_frames_host plus the equalizer output of every data step (sc_rx_frames_soft_host).  Returns
        (results[n_streams, n_frames], symbols complex64 [n_streams, n_frames, 31]); see soft_bits()."""
        assert samples.dtype == np.int16 and samples.ndim == 2 and samples.shape[0] == self.n_streams
        assert samples.strides[1] == 2
        stride = samples.strides[0] // 2
        if n_frames is None:
            n_frames = samples.shape[1] // FRAME_SIZE
        results = np.zeros((self.n_streams, n_frames), RESULT_DTYPE)
        symbols = np.zeros((self.n_streams, n_frames, DATA_SYMBOLS), np.complex64)
        check(lib.sc_rx_frames_soft_host(self._h, samples.ctypes.data, stride, n_frames, results.ctypes.data,
                                         n_frames, symbols.ctypes.data))
        return results, symbols

    def rx_packets_host(self, samples: np.ndarray, n_frames: Optional[int] = None, capacity: Optional[int] = None):
        """Packet mode (extension): the ordinary results plus one PACKET_DTYPE record per valid call n >= 2 with all
        8 x 62 bits of the packet, sorted by (stream, call).  Returns (results, packets, n_found)."""
        assert samples.dtype == np.int16 and samples.ndim == 2 and samples.shape[0] == self.n_streams
        stride = samples.strides[0] // 2
        if n_frames is None:
            n_frames = samples.shape[1] // FRAME_SIZE
        results = np.zeros((self.n_streams, n_frames), RESULT_DTYPE)
        if capacity is None:
            capacity = self.n_streams * n_frames
        packets = np.zeros(max(capacity, 1), PACKET_DTYPE)
        n = C.c_uint64(0)
        check(lib.sc_rx_packets_host(self._h, samples.ctypes.data, stride, n_frames, results.ctypes.data,
                                     results.strides[0] // 32, packets.ctypes.data, capacity, C.byref(n)))
        got = packets[: min(int(n.value), capacity)]
        got = got[np.lexsort((got["call_index"], got["stream"]))]
        return results, got, int(n.value)

    def rx_packets_soft_host(self, samples: np.ndarray, n_frames: Optional[int] = None, capacity: Optional[int] = None,
                             call_symbols: bool = False):
        """rx_packets_host plus the equalizer output of the 248 data steps of every packet (sc_rx_packets_soft_host)
        and, with call_symbols, of the 31 of every call.  Returns (results, call symbols complex64
        [n_streams, n_frames, 31] or None, packets sorted by (stream, call), packet symbols complex64 [n, 248] in the
        same order, n_found); see packet_soft_bits()."""
        assert samples.dtype == np.int16 and samples.ndim == 2 and samples.shape[0] == self.n_streams
        assert samples.strides[1] == 2
        stride = samples.strides[0] // 2
        if n_frames is None:
            n_frames = samples.shape[1] // FRAME_SIZE
        results = np.zeros((self.n_streams, n_frames), RESULT_DTYPE)
        symbols = np.zeros((self.n_streams, n_frames, DATA_SYMBOLS), np.complex64) if call_symbols else None
        if capacity is None:
            capacity = self.n_streams * n_frames
        packets = np.zeros(max(capacity, 1), PACKET_DTYPE)
        psym = np.zeros((max(capacity, 1), PACKET_DATA_SYMBOLS), np.complex64)
        n = C.c_uint64(0)
        check(lib.sc_rx_packets_soft_host(self._h, samples.ctypes.data, stride, n_frames, results.ctypes.data, n_frames,
                                          _ptr(symbols), packets.ctypes.data, capacity, C.byref(n), psym.ctypes.data))
        kept = min(int(n.value), capacity)
        got = packets[:kept]
        order = np.lexsort((got["call_index"], got["stream"]))
        return results, symbols, got[order], psym[:kept][order], int(n.value)

    def rx_packets_dev(self, samples, n_frames: int, results, packets, n_packets, stream: int = 0) -> None:
        """Device form: packets = CUDA uint8 [capacity * 96], n_packets = CUDA int64[1] (accumulated into)."""
        check(lib.sc_rx_packets_dev(self._h, samples.data_ptr(), samples.stride(0), n_frames, results.data_ptr(),
                                    results.stride(0) // 32, packets.data_ptr(), packets.numel() // 96,
                                    n_packets.data_ptr(), stream))

    def rx_packets_soft_dev(self, samples, n_frames: int, results, packets, n_packets, packet_symbols,
                            symbols=None, stream: int = 0) -> None:
        """Device form of rx_packets_soft_host: as rx_packets_dev, plus packet_symbols, a CUDA tensor with 496 floats
        (248 complex) per record of packets (e.g. complex64 [capacity, 248]), and symbols (None, or as for
        rx_frames_soft_dev)."""
        result_stride = results.stride(0) // 32
        capacity = packets.numel() // 96
        assert packet_symbols.numel() * packet_symbols.element_size() >= capacity * PACKET_DATA_SYMBOLS * 8, "capacity"
        if symbols is not None:
            assert symbols.stride(0) * symbols.element_size() == result_stride * DATA_SYMBOLS * 8, "records' stride"
        check(lib.sc_rx_packets_soft_dev(self._h, samples.data_ptr(), samples.stride(0), n_frames, results.data_ptr(),
                                         result_stride, _ptr(symbols), packets.data_ptr(), capacity,
                                         n_packets.data_ptr(), packet_symbols.data_ptr(), stream))

    def rx_frames_dev(self, samples, n_frames: int, results, eq_dbg=None, stream: int = 0) -> None:
        """samples: CUDA int16 tensor [n_streams, stride]; results: CUDA uint8 tensor
        [n_streams, n_frames*32] (view as RESULT_DTYPE after copying back)."""
        check(lib.sc_rx_frames_dev(self._h, samples.data_ptr(), samples.stride(0), n_frames,
                                   results.data_ptr(), results.stride(0) // 32, _ptr(eq_dbg), stream))

    def rx_frames_soft_dev(self, samples, n_frames: int, results, symbols, stream: int = 0) -> None:
        """rx_frames_dev plus the equalizer outputs: symbols is a CUDA tensor with 62 floats (31 complex) per record,
        records indexed like results (e.g. float32 [n_streams, n_frames*62] or complex64 [n_streams, n_frames, 31])."""
        result_stride = results.stride(0) // 32
        assert symbols.stride(0) * symbols.element_size() == result_stride * DATA_SYMBOLS * 8, "records' stride"
        check(lib.sc_rx_frames_soft_dev(self._h, samples.data_ptr(), samples.stride(0), n_frames, results.data_ptr(),
                                        result_stride, symbols.data_ptr(), stream))

    # ---- TX ------------------------------------------------------------------------------------
    def tx_packets_dev(self, out, n_packets: int, gap_samples: int = REFERENCE_GAP, bits=None, bits_out=None,
                       seed: int = 0, lead_in=None, channel: Optional[dict] = None, stream: int = 0) -> None:
        """out: CUDA int16 tensor [n_streams, samples_per_stream]."""
        if channel is None:
            check(lib.sc_tx_packets_dev(self._h, _ptr(bits), _ptr(bits_out), seed, n_packets, gap_samples,
                                        _ptr(lead_in), out.data_ptr(), out.stride(0), out.shape[1], stream))
        else:
            ch = Channel(*[_ptr(channel.get(k)) for k in ("df_hz", "phi_rad", "drift_hz_s", "sigma_lsb",
                                                           "echo_amp", "echo_theta", "echo_delay")])
            check(lib.sc_tx_channel_dev(self._h, _ptr(bits), _ptr(bits_out), seed, n_packets, gap_samples,
                                        _ptr(lead_in), C.byref(ch), out.data_ptr(), out.stride(0), out.shape[1],
                                        stream))

    def nco_table(self, first_call: int, n_calls: int, tx: bool = False) -> np.ndarray:
        out = np.zeros((n_calls, FRAME_SIZE), np.complex64)
        check(lib.sc_nco_table_host(self._h, int(tx), first_call, n_calls, out.ctypes.data))
        return out

"""ctypes bindings for the CPU oracle -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` leg may import this module.  The product package
(``singlecarrier_b200``) never does.

Two libraries:

* ``libsc_oracle.so``   -- the restatement (``oracle/sc_oracle.c``), buildable anywhere gcc is.
* ``_ref/libsc_ref.so`` -- the reference's own sources compiled from ``/root/reference`` (only
  buildable in the build container; travels to the GPU box as a prebuilt file).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "libsc_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libsc_ref.so")

FRAME_SIZE = 1880
BITS_PER_CALL = 62
PREAMBLE_LENGTH = 128
DATA_SYMBOLS = 31
NTAPS = 49


def build(quiet: bool = True) -> None:
    """(Re)build the oracle, and the reference library when /root/reference is present."""
    subprocess.run(["make", "-C", HERE, "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


class FrameStats(C.Structure):
    """sco_frame_stats (oracle/sc_oracle.h)."""
    _fields_ = [("valid", C.c_int32), ("max_index", C.c_int32), ("matches", C.c_int32),
                ("rx_timing", C.c_int32), ("max_value", C.c_float), ("cost", C.c_float),
                ("eq_coeff", C.c_float * 10)]


STATS_DTYPE = np.dtype([("valid", "<i4"), ("max_index", "<i4"), ("matches", "<i4"),
                        ("rx_timing", "<i4"), ("max_value", "<f4"), ("cost", "<f4"),
                        ("eq_coeff", "<f4", (10,))])
assert STATS_DTYPE.itemsize == C.sizeof(FrameStats)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Oracle:
    """The restatement library."""

    def __init__(self, path: str = ORACLE_SO):
        if not os.path.exists(path):
            build()
        self.lib = L = C.CDLL(path)
        L.sco_sizeof_state.restype = C.c_ulong
        L.sco_run_streams.restype = C.c_long
        L.sco_run_streams.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.sco_run_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
        L.sco_init.argtypes = [C.c_void_p, C.c_int, C.c_float]
        L.sco_rx_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sco_tx_preamble.argtypes = [C.c_void_p, C.c_void_p]
        L.sco_tx_data.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sco_tx_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.sco_tx_preamble_analytic.argtypes = [C.c_void_p, C.c_void_p]
        L.sco_tx_data_analytic.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sco_fir.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.sco_correlate.restype = C.c_float
        L.sco_correlate.argtypes = [C.c_void_p, C.c_int]
        L.sco_search.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.sco_kalman_init.argtypes = [C.c_void_p]
        L.sco_kalman_reset.argtypes = [C.c_void_p]
        L.sco_kalman_calculate.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.sco_train_eq.restype = C.c_float
        L.sco_train_eq.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float]
        L.sco_data_eq.restype = C.c_float
        L.sco_data_eq.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.sco_scramble2.argtypes = [C.c_void_p, C.c_void_p]
        L.sco_nco_rect.argtypes = [C.c_float, C.c_void_p]
        self.state_size = int(L.sco_sizeof_state())

    # ---- whole streams -------------------------------------------------------------------
    def run_stream(self, samples: np.ndarray, wide: bool = False, foffset: float = 0.0):
        """Cold-start one stream through sco_rx_frame; returns (bits[nf,62] (255 = invalid row), stats[nf])."""
        x = np.ascontiguousarray(samples, dtype="<i2")
        nf = x.size // FRAME_SIZE
        bits = np.full((nf, BITS_PER_CALL), 255, np.uint8)
        stats = np.zeros(nf, STATS_DTYPE)
        self.lib.sco_run_stream(_p(x), nf, int(wide), float(foffset), _p(bits), _p(stats))
        return bits, stats

    def run_streams(self, samples: np.ndarray, n_frames: int, wide: bool = False):
        """samples[n_streams, >= n_frames*1880] -> (bits[ns,nf,62], valid[ns,nf])."""
        x = np.ascontiguousarray(samples, dtype="<i2")
        ns, stride = x.shape
        bits = np.full((ns, n_frames, BITS_PER_CALL), 255, np.uint8)
        valid = np.zeros((ns, n_frames), np.int32)
        self.lib.sco_run_streams(_p(x), ns, stride, n_frames, int(wide), _p(bits), _p(valid))
        return bits, valid

    # ---- stateful single-stream object ---------------------------------------------------
    def new_state(self, wide: bool = False, foffset: float = 0.0):
        buf = np.zeros(self.state_size + 64, np.uint8)
        self.lib.sco_init(_p(buf), int(wide), float(foffset))
        return buf

    def rx_frame(self, state, frame: np.ndarray):
        x = np.ascontiguousarray(frame, dtype="<i2")
        assert x.size == FRAME_SIZE
        bits = np.full(BITS_PER_CALL, 255, np.uint8)
        st = np.zeros(1, STATS_DTYPE)
        self.lib.sco_rx_frame(_p(state), _p(x), _p(bits), _p(st))
        return bits, st[0]

    def tx_preamble(self, state) -> np.ndarray:
        out = np.zeros(PREAMBLE_LENGTH * 5, "<i2")
        self.lib.sco_tx_preamble(_p(state), _p(out))
        return out

    def tx_data(self, state, bits: np.ndarray) -> np.ndarray:
        b = np.ascontiguousarray(bits, np.uint8)
        nsym = b.size // 2
        out = np.zeros(nsym * 5, "<i2")
        self.lib.sco_tx_data(_p(state), _p(out), _p(b), nsym)
        return out

    def tx_preamble_analytic(self, state) -> np.ndarray:
        """tx_preamble() before the real part is taken: the scaled complex signal (complex64)."""
        out = np.zeros(PREAMBLE_LENGTH * 5, np.complex64)
        self.lib.sco_tx_preamble_analytic(_p(state), _p(out))
        return out

    def tx_data_analytic(self, state, bits: np.ndarray) -> np.ndarray:
        """tx_data() before the real part is taken: the scaled complex signal (complex64)."""
        b = np.ascontiguousarray(bits, np.uint8)
        nsym = b.size // 2
        out = np.zeros(nsym * 5, np.complex64)
        self.lib.sco_tx_data_analytic(_p(state), _p(out), _p(b), nsym)
        return out

    # ---- stage primitives ----------------------------------------------------------------
    def fir(self, memory: np.ndarray, wide: bool, sample: np.ndarray):
        """In place on complex64 arrays (memory[49], sample[n])."""
        assert memory.dtype == np.complex64 and sample.dtype == np.complex64
        self.lib.sco_fir(_p(memory), int(wide), _p(sample), sample.size)

    def search(self, symbols: np.ndarray):
        s = np.ascontiguousarray(symbols, np.complex64)
        assert s.size >= 255
        idx = C.c_int32(0)
        val = C.c_float(0)
        self.lib.sco_search(_p(s), C.byref(idx), C.byref(val))
        return idx.value, np.float32(val.value)

    def correlate(self, symbols: np.ndarray, lag: int) -> np.float32:
        s = np.ascontiguousarray(symbols, np.complex64)
        return np.float32(self.lib.sco_correlate(_p(s), lag))

    def nco_rect(self, freq_hz: float) -> np.complex64:
        out = np.zeros(1, np.complex64)
        self.lib.sco_nco_rect(float(freq_hz), _p(out))
        return out[0]


EXT_PACKET_DTYPE = np.dtype([("call", "<i4"), ("max_index", "<i4"), ("matches", "<i4"), ("timing", "<i4"),
                             ("cost", "<f4"), ("bits", "u1", (496,))])


def ext_run_stream(oracle, samples: np.ndarray, max_packets: int = 64, wide: bool = False, foffset: float = 0.0):
    """Packet-mode extension (oracle/sc_oracle_ext.c, NO reference counterpart): the ordinary receiver plus the
    full 8 x 31 symbol decode of every valid call.  Returns (bits[nf,62], stats[nf], packets[EXT_PACKET_DTYPE])."""
    L = oracle.lib
    L.sco_ext_run_stream.restype = C.c_int
    L.sco_ext_run_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.sco_ext_sizeof_packet.restype = C.c_ulong
    assert int(L.sco_ext_sizeof_packet()) == EXT_PACKET_DTYPE.itemsize
    x = np.ascontiguousarray(samples, dtype="<i2")
    nf = x.size // FRAME_SIZE
    bits = np.full((nf, BITS_PER_CALL), 255, np.uint8)
    stats = np.zeros(nf, STATS_DTYPE)
    pk = np.zeros(max_packets, EXT_PACKET_DTYPE)
    n = L.sco_ext_run_stream(_p(x), nf, int(wide), float(foffset), _p(bits), _p(stats), _p(pk), max_packets)
    return bits, stats, pk[:n]


def ext_tx_packet(oracle, state, bits: np.ndarray) -> np.ndarray:
    """One packet with TX scrambling enabled (qpsk.c:386,397 un-commented): 1880 int16 samples."""
    L = oracle.lib
    L.sco_ext_tx_packet.restype = C.c_int
    L.sco_ext_tx_packet.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    b = np.ascontiguousarray(bits, np.uint8)
    assert b.size == 496
    out = np.zeros(FRAME_SIZE, "<i2")
    n = L.sco_ext_tx_packet(_p(state), _p(out), _p(b))
    assert n == FRAME_SIZE
    return out


def synth_streams(oracle, rng, n_streams, n_frames, noise_levels=(0.0, 30.0, 300.0, 1500.0, 4000.0),
                  max_lead=2000, gaps=(903, 0, 500, 1880)):
    """Oracle-TX loop-back streams with random lead-in, dead air and additive noise -> int16[n, n_frames*1880]."""
    total = n_frames * FRAME_SIZE
    out = np.zeros((n_streams, total), np.int16)
    for s in range(n_streams):
        st = oracle.new_state()
        lead = int(rng.integers(0, max_lead))
        gap = int(gaps[s % len(gaps)])
        parts = [np.zeros(lead, np.int16)]
        n = lead
        while n < total:
            parts.append(oracle.tx_preamble(st))
            for _ in range(8):
                parts.append(oracle.tx_data(st, rng.integers(0, 2, 62).astype(np.uint8)))
            parts.append(np.zeros(gap, np.int16))
            n += 1880 + gap
        x = np.concatenate(parts)[:total].astype(np.float64)
        noise = noise_levels[s % len(noise_levels)]
        if noise > 0:
            x = x + rng.normal(0, noise, total)
        out[s] = np.clip(x, -32767, 32767).round().astype(np.int16)
    return out



class RefStats(C.Structure):
    """ref_frame_stats (oracle/ref_harness_post.c)."""
    _fields_ = [("valid", C.c_int32), ("max_index", C.c_int32), ("matches", C.c_int32),
                ("rx_timing", C.c_int32), ("max_value", C.c_float), ("mean", C.c_float),
                ("eq_coeff", C.c_float * 10)]


REF_STATS_DTYPE = np.dtype([("valid", "<i4"), ("max_index", "<i4"), ("matches", "<i4"),
                            ("rx_timing", "<i4"), ("max_value", "<f4"), ("mean", "<f4"),
                            ("eq_coeff", "<f4", (10,))])


def have_ref() -> bool:
    return os.path.exists(REF_SO)


class Reference:
    """The reference's own object code (process-global state: one stream at a time)."""

    def __init__(self, path: str = REF_SO):
        self.lib = L = C.CDLL(path)
        L.ref_reset.argtypes = [C.c_int]
        L.ref_rx_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.ref_run_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.ref_run_streams.restype = C.c_long
        L.ref_run_streams.argtypes = [C.c_void_p, C.c_long, C.c_long, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.ref_tx_preamble.argtypes = [C.c_void_p]
        L.ref_tx_data.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.ref_get_filtered.argtypes = [C.c_void_p, C.c_int]
        L.ref_get_decimated.argtypes = [C.c_void_p, C.c_int]
        L.fir.argtypes = [C.c_void_p, C.c_bool, C.c_void_p, C.c_int]
        L.train_eq.restype = C.c_float
        L.train_eq.argtypes = [C.c_void_p, C.c_int, C.c_float]
        L.data_eq.restype = C.c_float
        L.data_eq.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.kalman_calculate.argtypes = [C.c_void_p, C.c_int]
        L.scramble_init.argtypes = [C.c_int]
        L.scramble.argtypes = [C.c_void_p, C.c_int]

    def reset(self, wide: bool = False):
        self.lib.ref_reset(int(wide))

    def run_stream(self, samples: np.ndarray, wide: bool = False):
        x = np.ascontiguousarray(samples, dtype="<i2")
        nf = x.size // FRAME_SIZE
        bits = np.full((nf, BITS_PER_CALL), 255, np.uint8)
        stats = np.zeros(nf, REF_STATS_DTYPE)
        self.lib.ref_run_stream(_p(x), nf, int(wide), _p(bits), _p(stats))
        return bits, stats

    def run_streams(self, samples: np.ndarray, n_frames: int, wide: bool = False):
        x = np.ascontiguousarray(samples, dtype="<i2")
        ns, stride = x.shape
        bits = np.full((ns, n_frames, BITS_PER_CALL), 255, np.uint8)
        valid = np.zeros((ns, n_frames), np.int32)
        self.lib.ref_run_streams(_p(x), ns, stride, n_frames, int(wide), _p(bits), _p(valid))
        return bits, valid

    def rx_frame(self, frame: np.ndarray):
        x = np.ascontiguousarray(frame, dtype="<i2")
        bits = np.full(496, 255, np.uint8)
        st = np.zeros(1, REF_STATS_DTYPE)
        self.lib.ref_rx_frame(_p(x), _p(bits), _p(st))
        return bits[:BITS_PER_CALL], st[0]

    def filtered(self, n: int = FRAME_SIZE) -> np.ndarray:
        out = np.zeros(n, np.complex64)
        self.lib.ref_get_filtered(_p(out), n)
        return out

    def decimated(self, n: int = 752) -> np.ndarray:
        out = np.zeros(n, np.complex64)
        self.lib.ref_get_decimated(_p(out), n)
        return out

    def tx_preamble(self) -> np.ndarray:
        out = np.zeros(PREAMBLE_LENGTH * 5, "<i2")
        self.lib.ref_tx_preamble(_p(out))
        return out

    def tx_data(self, bits: np.ndarray) -> np.ndarray:
        b = np.ascontiguousarray(bits, np.uint8).copy()
        nsym = b.size // 2
        out = np.zeros(nsym * 5, "<i2")
        self.lib.ref_tx_data(_p(out), _p(b), nsym)
        return out

    def global_c32(self, name: str, n: int) -> np.ndarray:
        arr = (C.c_float * (2 * n)).in_dll(self.lib, name)
        return np.frombuffer(arr, np.float32).view(np.complex64)

    def global_f32(self, name: str) -> C.c_float:
        return C.c_float.in_dll(self.lib, name)


REF_REPLAY = os.path.join(os.path.dirname(HERE), "tests", "golden", "ref_replay.npz")


def _digest(a) -> str:
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


class RecordingReference:
    """Wraps an engine with the Reference interface and records every output under a key made of the call and a
    digest of its input (the key RecordedReference looks up); ``save()`` writes them (tools/make_golden.py)."""

    def __init__(self, engine):
        self.engine, self.out, self.n = engine, {}, 0

    def _put(self, key, **arrays):
        for k, v in arrays.items():
            self.out[f"{key}/{k}"] = np.asarray(v)

    def reset(self, wide: bool = False):
        self.engine.reset(wide)
        self.n = 0

    def run_stream(self, samples, wide: bool = False):
        bits, st = self.engine.run_stream(samples, wide)
        self._put(f"run_stream/{_digest(samples)}/{int(wide)}", bits=bits, stats=st)
        return bits, st

    def rx_frame(self, frame):
        bits, st = self.engine.rx_frame(frame)
        self._put(f"rx_frame/{self.n}/{_digest(frame)}", bits=bits, stats=st, filtered=self.engine.filtered(),
                  decimated=self.engine.decimated())
        self.n += 1
        return bits, st

    def tx_preamble(self):
        out = self.engine.tx_preamble()
        self._put(f"tx_preamble/{self.n}", out=out)
        self.n += 1
        return out

    def tx_data(self, bits):
        out = self.engine.tx_data(bits)
        self._put(f"tx_data/{self.n}/{_digest(np.ascontiguousarray(bits, np.uint8))}", out=out)
        self.n += 1
        return out

    def save(self, path: str = REF_REPLAY, **meta):
        np.savez_compressed(path, **self.out, **{f"meta/{k}": np.asarray(v) for k, v in meta.items()})


class RecordedReference:
    """The reference's outputs replayed from tests/golden/ref_replay.npz, for machines without oracle/_ref: the same
    calls as Reference, answered from what the reference returned for the same input (and, for the stateful
    calls, the same position since reset()).  An input that was not recorded is an error, never a skip."""

    def __init__(self, path: str = REF_REPLAY):
        self.g = dict(np.load(path))
        self.n = 0
        self._last = None

    def _get(self, key):
        if f"{key}/bits" not in self.g and f"{key}/out" not in self.g:
            raise KeyError(f"no recorded reference output for {key} in {os.path.basename(REF_REPLAY)} "
                           "(inputs changed? re-record with tools/make_golden.py)")
        return key

    def reset(self, wide: bool = False):
        self.n = 0

    def run_stream(self, samples, wide: bool = False):
        k = self._get(f"run_stream/{_digest(samples)}/{int(wide)}")
        return self.g[k + "/bits"].copy(), self.g[k + "/stats"].copy()

    def rx_frame(self, frame):
        k = self._last = self._get(f"rx_frame/{self.n}/{_digest(frame)}")
        self.n += 1
        return self.g[k + "/bits"].copy(), self.g[k + "/stats"].copy()

    def filtered(self, n: int = FRAME_SIZE) -> np.ndarray:
        return self.g[self._last + "/filtered"][:n].copy()

    def decimated(self, n: int = 752) -> np.ndarray:
        return self.g[self._last + "/decimated"][:n].copy()

    def tx_preamble(self) -> np.ndarray:
        k = self._get(f"tx_preamble/{self.n}")
        self.n += 1
        return self.g[k + "/out"].copy()

    def tx_data(self, bits: np.ndarray) -> np.ndarray:
        k = self._get(f"tx_data/{self.n}/{_digest(np.ascontiguousarray(bits, np.uint8))}")
        self.n += 1
        return self.g[k + "/out"].copy()


def synth_bench_stream(oracle, seed: int, stream_id: int, n_samples: int) -> np.ndarray:
    """One stream of bench.py's workload made entirely on the CPU (no GPU, no product code): the reference's
    packet structure from the oracle's TX (640 preamble + 8 x 155 data + 903 dead air, random lead-in), then the
    same channel model as the device generator -- rotation of the analytic signal by exp(j(2 pi df t + phi)),
    df ~ U(-20, 20) Hz, and real AWGN at Eb/N0 = stream_id mod 13 dB -- saturated to int16.  Deterministic in
    (seed, stream_id); used by ``bench.py --impl reference`` so that arm never loads the CUDA library."""
    rng = np.random.default_rng([seed & 0x7fffffff, stream_id])
    st = oracle.new_state()
    period = FRAME_SIZE + 903
    lead = int(rng.integers(0, period))
    parts, n = [np.zeros(lead, np.int16)], lead
    while n < n_samples:
        parts.append(oracle.tx_preamble(st))
        for _ in range(8):
            parts.append(oracle.tx_data(st, rng.integers(0, 2, 62).astype(np.uint8)))
        parts.append(np.zeros(903, np.int16))
        n += period
    x = np.concatenate(parts)[:n_samples].astype(np.float64)
    # analytic signal by the FFT (Hilbert) method, then the frequency / phase offset
    spec = np.fft.fft(x)
    h = np.zeros(n_samples)
    h[0] = 1.0
    h[1:(n_samples + 1) // 2] = 2.0
    if n_samples % 2 == 0:
        h[n_samples // 2] = 1.0
    xa = np.fft.ifft(spec * h)
    df, phi = rng.uniform(-20.0, 20.0), rng.uniform(0.0, 2 * np.pi)
    t = np.arange(n_samples) / 8000.0
    y = (xa * np.exp(1j * (2 * np.pi * df * t + phi))).real
    ebn0_db = float(stream_id % 13)
    # bench.py's P_sig, kept so that both arms run the same workload.  The data section's true RMS is
    # harness.DATA_RMS_LSB (7,207 LSB, not 16384 * 0.48 = 7,864), so the real Eb/N0 is the label minus 0.76 dB.
    p_sig = (16384.0 * 0.48) ** 2
    sigma = np.sqrt(p_sig * 8000.0 / (2.0 * 1600.0 * 2.0 * 10.0 ** (ebn0_db / 10.0)))
    y = y + rng.normal(0.0, sigma, n_samples)
    return np.clip(np.rint(y), -32767, 32767).astype(np.int16)

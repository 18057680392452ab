#!/usr/bin/env python
"""Generate the committed golden vectors under tests/golden/ from the REFERENCE's own object code.

Needs the reference's sources, compiled by oracle/Makefile into oracle/_ref/libsc_ref.so.  The fixtures let
the oracle restatement -- and through it the CUDA path -- be pinned on machines where the reference does not
exist.  Re-run: ``python tools/make_golden.py``.

Fixtures
  preamble_qpsk_8k.raw   the reference's shipped sample file (data, copied verbatim; SURVEY section 2)
  rx_shipped.npz         qpsk_rx_frame() outputs for the 14 calls over that file
  rx_synth.npz           8 synthetic streams (reference TX + lead-in + noise) and their RX outputs
  tx_golden.npz          reference TX output for seeded bits (3 packets)
  stage_golden.npz       fir(), train_eq()/data_eq() trajectories, scrambler keystream
  fft_golden.npz         fft()/encode_fftr()/encode_fftri() outputs of src/fft.c
  ref_replay.npz         what the reference returned to the tests that compare with it directly
                         (tests/test_oracle_vs_ref.py, test_round2_gpu.py::test_cuda_path_vs_reference_objects_directly),
                         keyed by call and input digest; replayed by pyoracle.RecordedReference where oracle/_ref is absent
  dropin_interleave_ref.jsonl  tests/dropin_interleave.py's lines on the reference's objects

``python tools/make_golden.py --replay-from-restatement`` writes only the last two where the reference is not
available: ref_replay.npz from the oracle restatement (bit-identical to the reference on these inputs wherever
both ran, tests/test_oracle_vs_ref.py) and the drop-in lines from libsinglecarrier_b200.so (equal to the
reference's line for line, test_dropin_gpu.py::test_interleaved_globals_match_reference; needs a GPU).  The
committed files were made this way; ref_replay.npz names its source in "meta/source".  A run with the
reference overwrites both.
"""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
REF_RAW = "/root/reference/preamble_qpsk_8k.raw"


def ref_outputs(R, x):
    bits, st = R.run_stream(x)
    return dict(bits=bits, valid=st["valid"], max_index=st["max_index"], matches=st["matches"],
                rx_timing=st["rx_timing"], max_value=st["max_value"], mean=st["mean"], eq_coeff=st["eq_coeff"])


def synth_stream(R, rng, n_packets, lead, gap, noise, total):
    """Reference TX (cold) -> int16 stream with lead-in zeros, dead air and additive noise."""
    R.reset()
    parts = [np.zeros(lead, np.int16)]
    allbits = []
    for _ in range(n_packets):
        parts.append(R.tx_preamble())
        for _ in range(8):
            b = rng.integers(0, 2, 62).astype(np.uint8)
            allbits.append(b)
            parts.append(R.tx_data(b))
        parts.append(np.zeros(gap, np.int16))
    x = np.concatenate(parts)[:total]
    x = np.concatenate([x, np.zeros(total - x.size, np.int16)])
    if noise > 0:
        x = np.clip(x.astype(np.float64) + rng.normal(0, noise, x.size), -32767, 32767).round().astype(np.int16)
    return x, np.array(allbits)


class RestatementAsReference:
    """The oracle restatement behind the Reference interface (stats with the reference's "mean" field)."""

    def __init__(self):
        self.o = po.Oracle()
        self.reset()

    def reset(self, wide=False):
        self.st = self.o.new_state(wide)

    def _stats(self, s):
        out = np.zeros(s.shape, po.REF_STATS_DTYPE)
        for f in ("valid", "max_index", "matches", "rx_timing", "max_value", "eq_coeff"):
            out[f] = s[f]
        out["mean"] = s["cost"]
        return out

    def run_stream(self, x, wide=False):
        bits, s = self.o.run_stream(x, wide=wide)
        return bits, self._stats(s)

    def rx_frame(self, frame):
        bits, s = self.o.rx_frame(self.st, frame)
        return bits, self._stats(np.array([s]))[0]

    def filtered(self, n=po.FRAME_SIZE):
        return np.frombuffer(self.st, np.float32, count=2 * 3760).view(np.complex64)[:n].copy()

    def decimated(self, n=752):
        return np.frombuffer(self.st, np.float32, count=2 * 752, offset=3760 * 8).view(np.complex64)[:n].copy()

    def tx_preamble(self):
        return self.o.tx_preamble(self.st)

    def tx_data(self, bits):
        return self.o.tx_data(self.st, bits)


def record_ref_replay(engine, source):
    """The reference calls of the tests that compare with it directly, on their seeded inputs (kept in step with
    the tests: an input that differs is not found at replay and fails the test)."""
    o = po.Oracle()
    R = po.RecordingReference(engine)
    rng = np.random.default_rng(99)                                # test_oracle_vs_ref.py::test_rx_random_streams
    samples = po.synth_streams(o, rng, 24, 10)
    noise = [rng.integers(-a, a + 1, 1880 * 8).astype(np.int16) for a in (3, 100, 3000, 32767)]
    for x in list(samples) + noise:
        R.run_stream(x)
    x = po.synth_streams(o, np.random.default_rng(5), 3, 8)        # ::test_wide_filter
    for s in range(3):
        R.run_stream(x[s], wide=True)
    x = po.synth_streams(o, np.random.default_rng(6), 1, 6)[0]     # ::test_stage_taps_filtered_and_decimated
    R.reset()
    for n in range(6):
        R.rx_frame(x[n * 1880:(n + 1) * 1880])
    rng = np.random.default_rng(7)                                 # ::test_tx_random
    R.reset()
    for _ in range(5):
        R.tx_preamble()
        for _ in range(8):
            R.tx_data(rng.integers(0, 2, 62).astype(np.uint8))
    shipped = np.fromfile(os.path.join(GOLD, "preamble_qpsk_8k.raw"), dtype="<i2")[: 14 * 1880]
    noisy = po.synth_streams(o, np.random.default_rng(2024), 64, 14)   # test_round2_gpu.py::test_cuda_path_vs_...
    for x in [shipped] + list(noisy):
        R.run_stream(x)
    R.save(source=source)


def interleave_lines(lib, kind):
    raw = os.path.join(GOLD, "preamble_qpsk_8k.raw")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "dropin_interleave.py"), lib, raw, kind],
                         check=True, capture_output=True, text=True).stdout
    with open(os.path.join(GOLD, "dropin_interleave_ref.jsonl"), "w") as f:
        f.write(out)


def replay_from_restatement():
    po.build(quiet=False)
    record_ref_replay(RestatementAsReference(), "oracle restatement (oracle/sc_oracle.c)")
    interleave_lines(os.path.join(ROOT, "singlecarrier_b200", "libsinglecarrier_b200.so"), "ours")


def main():
    po.build(quiet=False)
    assert po.have_ref(), "needs the reference's objects (oracle/_ref/libsc_ref.so)"
    R = po.Reference()
    os.makedirs(GOLD, exist_ok=True)
    shutil.copyfile(REF_RAW, os.path.join(GOLD, "preamble_qpsk_8k.raw"))

    x = np.fromfile(REF_RAW, dtype="<i2")
    np.savez_compressed(os.path.join(GOLD, "rx_shipped.npz"), **ref_outputs(R, x))

    rng = np.random.default_rng(20261018)
    nfr = 10
    streams, outs = [], []
    cfg = [(80, 903, 0.0), (80 + 5 * 37, 903, 0.0), (1234, 0, 0.0), (80 + 5 * 100, 903, 300.0),
           (17, 500, 1500.0), (80, 903, 4000.0), (0, 0, 30.0), (333, 1880, 0.0)]
    for lead, gap, noise in cfg:
        xs, _ = synth_stream(R, rng, 8, lead, gap, noise, nfr * 1880)
        streams.append(xs)
        outs.append(ref_outputs(R, xs))
    np.savez_compressed(os.path.join(GOLD, "rx_synth.npz"), samples=np.stack(streams),
                        **{k: np.stack([o[k] for o in outs]) for k in outs[0]})

    # TX known answers
    R.reset()
    txbits = rng.integers(0, 2, (3, 8, 62)).astype(np.uint8)
    tx = []
    for p in range(3):
        tx.append(R.tx_preamble())
        for j in range(8):
            tx.append(R.tx_data(txbits[p, j]))
    np.savez_compressed(os.path.join(GOLD, "tx_golden.npz"), bits=txbits, samples=np.concatenate(tx))

    # stage primitives
    g = {}
    for wide in (0, 1):
        mem = (rng.normal(size=49) + 1j * rng.normal(size=49)).astype(np.complex64)
        sam = (rng.normal(size=700) + 1j * rng.normal(size=700)).astype(np.complex64)
        g[f"fir_mem_in_{wide}"], g[f"fir_x_{wide}"] = mem.copy(), sam.copy()
        R.lib.fir(mem.ctypes.data, bool(wide), sam.ctypes.data, sam.size)
        g[f"fir_mem_out_{wide}"], g[f"fir_y_{wide}"] = mem, sam
    sym = (rng.normal(size=200) + 1j * rng.normal(size=200)).astype(np.complex64)
    pre = np.array([1 if v else -1 for v in rng.integers(0, 2, 128)], np.float32)
    R.reset()
    R.lib.kalman_reset()
    traj, rets = [], []
    for i in range(128):
        rets.append(R.lib.train_eq(sym.ctypes.data, i, float(pre[i])))
        traj.append(R.global_c32("eq_coeff", 5).copy())
    dibits = []
    for i in range(31):
        d = C.c_uint8(0)
        rets.append(R.lib.data_eq(C.byref(d), sym.ctypes.data, 128 + i))
        dibits.append(d.value)
        traj.append(R.global_c32("eq_coeff", 5).copy())
    g.update(eq_sym=sym, eq_ref=pre, eq_traj=np.stack(traj), eq_ret=np.array(rets, np.float32),
             eq_dibits=np.array(dibits, np.uint8),
             eq_gain=R.global_c32("kalman_gain", 5).copy(), eq_y=np.float32(R.global_f32("kalman_y").value))
    R.lib.scramble_init(2)
    ks = []
    for _ in range(62 * 4 // 2):
        d = C.c_uint8(0)
        R.lib.scramble(C.byref(d), 1)
        ks += [d.value & 1, d.value >> 1]
    g["keystream"] = np.array(ks, np.uint8)
    np.savez_compressed(os.path.join(GOLD, "stage_golden.npz"), **g)

    # fft.c
    L = R.lib
    L.fft_alloc.restype = C.c_void_p
    L.fft_alloc.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.fft.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fftr_alloc.restype = C.c_void_p
    L.fftr_alloc.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.encode_fftr.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.encode_fftri.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    f = {}
    for n in (2, 3, 4, 5, 6, 7, 8, 11, 16, 30, 49, 60, 64, 100, 125, 128, 243, 256, 512, 1024, 2048):
        xin = (rng.normal(size=n) + 1j * rng.normal(size=n)).astype(np.complex64)
        for inv in (0, 1):
            cfg_ = L.fft_alloc(n, inv, None, None)
            out = np.zeros(n, np.complex64)
            L.fft(cfg_, xin.ctypes.data, out.ctypes.data)
            f[f"c{n}_{inv}"] = out
        f[f"c{n}_in"] = xin
    for n in (6, 20, 64, 250, 256):
        xr = rng.normal(size=n).astype(np.float32)
        cf = L.fftr_alloc(n, 0, None, None)
        spec = np.zeros(n // 2 + 1, np.complex64)
        L.encode_fftr(cf, xr.ctypes.data, spec.ctypes.data)
        ci = L.fftr_alloc(n, 1, None, None)
        back = np.zeros(n, np.float32)
        L.encode_fftri(ci, spec.ctypes.data, back.ctypes.data)
        f[f"r{n}_in"], f[f"r{n}_spec"], f[f"r{n}_back"] = xr, spec, back
    np.savez_compressed(os.path.join(GOLD, "fft_golden.npz"), **f)
    record_ref_replay(R, "reference objects (oracle/_ref/libsc_ref.so)")
    interleave_lines(po.REF_SO, "ref")
    for fn in sorted(os.listdir(GOLD)):
        print(fn, os.path.getsize(os.path.join(GOLD, fn)))


if __name__ == "__main__":
    replay_from_restatement() if "--replay-from-restatement" in sys.argv[1:] else main()

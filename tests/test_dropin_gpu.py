"""Drop-in boundary on the GPU: a C program written against the reference's headers, compiled against
include/sc_compat and linked with libsinglecarrier_b200.so, must print what the reference prints."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dropin_output(tmp_path_factory):
    exe = tmp_path_factory.mktemp("dropin") / "dropin_main"
    libdir = os.path.join(ROOT, "singlecarrier_b200")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-I", os.path.join(ROOT, "include", "sc_compat"),
                    os.path.join(ROOT, "tests", "dropin_main.c"), "-o", str(exe), "-L", libdir,
                    "-lsinglecarrier_b200", "-lm", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe), os.path.join(ROOT, "tests", "golden", "preamble_qpsk_8k.raw")],
                         check=True, capture_output=True, text=True, timeout=300).stdout
    return out.strip().splitlines()


def test_dropin_program_matches_reference(dropin_output, gold, oracle):
    lines = dropin_output
    txp = lines[0].split()
    assert txp[0] == "TXP" and txp[1] == "640"
    assert [int(v) for v in txp[2:]] == [0, -45, -72, -20, -6, -74, -112, -13, -22, -158, -111, -3, -251, -462, -160,
                                         7, -628, -972, -99, 397, -885, -1602, 1044, 4959]
    # data frame right after the preamble: oracle TX with the same bits
    st = oracle.new_state()
    oracle.tx_preamble(st)
    obits = np.array([(i * 7 + 3) % 5 < 2 for i in range(62)], np.uint8)
    frame = oracle.tx_data(st, obits)
    acc = 0
    for v in frame.tolist():
        acc = (acc * 31 + v)
        acc = (acc + 2 ** 63) % 2 ** 64 - 2 ** 63                            # C long wrap-around
    assert lines[1].split() == ["TXD", "155", str(acc)]
    g = gold("rx_shipped.npz")
    rx = [ln.split() for ln in lines if ln.startswith("RX ")]
    assert len(rx) == 14
    for n, f in enumerate(rx):
        assert int(f[2]) == g["valid"][n]
        if g["valid"][n]:
            assert f[3] == "".join(map(str, g["bits"][n]))
        assert np.float32(float(f[-2])) == g["eq_coeff"][n][0] and np.float32(float(f[-1])) == g["eq_coeff"][n][9]
    ks = [ln for ln in lines if ln.startswith("KS ")][0].split()
    assert ks[1] == "".join(map(str, gold("stage_golden.npz")["keystream"][:62])) and ks[2] == "-1"
    assert ks[1].startswith("000000111111011000001000001101")                # DVB PRBS, SURVEY section 4 pin 3
    misc = [ln for ln in lines if ln.startswith("MISC ")][0].split()
    assert float(misc[1]) == 25.0 and misc[2] == "01"                        # bits[0] = Q (im<0), bits[1] = I (re<0)
    fir_line = [ln for ln in lines if ln.startswith("FIR ")][0].split()
    m = np.zeros(49, np.complex64)
    x = np.array([1, 0, 0, 0, 0, 1j, 0, 0], np.complex64)
    oracle.fir(m, False, x)
    assert [np.float32(float(v)) for v in fir_line[1:]] == [x[0].real, x[4].real, x[7].imag]


def test_legacy_l1_symbols_via_ctypes(gold):
    """train_eq / data_eq / kalman_* / exported globals against the reference trajectory."""
    import singlecarrier_b200 as sc
    L = sc.lib
    g = gold("stage_golden.npz")
    L.train_eq.restype = C.c_float
    L.train_eq.argtypes = [C.c_void_p, C.c_int, C.c_float]
    L.data_eq.restype = C.c_float
    L.data_eq.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.scramble_init.argtypes = [C.c_int]
    eq = np.frombuffer((C.c_float * 10).in_dll(L, "eq_coeff"), np.float32)
    gain = np.frombuffer((C.c_float * 10).in_dll(L, "kalman_gain"), np.float32)
    ky = C.c_float.in_dll(L, "kalman_y")
    sym = g["eq_sym"].copy()
    L.kalman_init()
    L.scramble_init(2)
    L.scramble_init(1)
    rets = []
    for i in range(128):
        rets.append(L.train_eq(sym.ctypes.data, i, float(g["eq_ref"][i])))
        assert np.array_equal(eq.view(np.uint32), g["eq_traj"][i].view(np.float32).view(np.uint32)), i
    dibits = []
    for i in range(31):
        d = C.c_uint8(0)
        rets.append(L.data_eq(C.byref(d), sym.ctypes.data, 128 + i))
        dibits.append(d.value)
        assert np.array_equal(eq.view(np.uint32), g["eq_traj"][128 + i].view(np.float32).view(np.uint32)), i
    assert np.array_equal(np.array(rets, np.float32).view(np.uint32), g["eq_ret"].view(np.uint32))
    assert dibits == g["eq_dibits"].tolist()
    assert np.array_equal(gain.view(np.uint32), g["eq_gain"].view(np.float32).view(np.uint32))
    assert np.float32(ky.value).view(np.uint32) == g["eq_y"].view(np.uint32)
    # fft.h through the legacy symbols
    f = gold("fft_golden.npz")
    L.fft_alloc.restype = C.c_void_p
    L.fft_alloc.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.fft.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    for n in (64, 60):
        cfg = L.fft_alloc(n, 0, None, None)
        out = np.zeros(n, np.complex64)
        L.fft(cfg, f[f"c{n}_in"].ctypes.data, out.ctypes.data)
        assert np.array_equal(out.view(np.uint32), f[f"c{n}_0"].view(np.uint32))
    L.fftr_alloc.restype = C.c_void_p
    L.fftr_alloc.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    assert L.fftr_alloc(63, 0, None, None) is None                           # odd length -> NULL (src/fft.c:89-91)
    cf = L.fftr_alloc(64, 0, None, None)
    spec = np.zeros(33, np.complex64)
    L.fftr.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.fftr(cf, f["r64_in"].ctypes.data, spec.ctypes.data)
    assert np.array_equal(spec.view(np.uint32), f["r64_spec"].view(np.uint32))


def test_interleaved_globals_match_reference(ref):
    """qpsk_rx_frame() shares RXMemory with scramble()/scramble_init()/data_eq() and leaves eq_coeff,
    kalman_gain, kalman_y and the internal u/d behind (src/scramble.c:41-42, src/equalizer.c:87,
    src/kalman.c:19-35): a caller that interleaves them sees exactly what the reference's objects give."""
    from oracle import pyoracle as po
    raw = os.path.join(ROOT, "tests", "golden", "preamble_qpsk_8k.raw")
    drv = os.path.join(ROOT, "tests", "dropin_interleave.py")
    ours = os.path.join(ROOT, "singlecarrier_b200", "libsinglecarrier_b200.so")
    if po.have_ref():
        a = subprocess.run([sys.executable, drv, po.REF_SO, raw, "ref"], check=True, capture_output=True, text=True,
                           timeout=300)
        la = a.stdout.strip().splitlines()
    else:                                                                    # the reference's lines, recorded
        la = open(os.path.join(ROOT, "tests", "golden", "dropin_interleave_ref.jsonl")).read().strip().splitlines()
    b = subprocess.run([sys.executable, drv, ours, raw, "ours"], check=True, capture_output=True, text=True, timeout=300)
    lb = b.stdout.strip().splitlines()
    assert len(la) == len(lb) == 14 + 4
    for x, y in zip(la, lb):
        assert x == y
    assert '"valid": 1' in la[15] and '"call": 12' in la[15]     # the locked frame is part of the sequence


def test_legacy_tx_frame_arbitrary_symbols(oracle):
    """qpsk_tx_frame() with symbols that are not +-1 (general 49-tap path, filter memory and phasor carried
    across calls) against the oracle's restatement."""
    import singlecarrier_b200 as sc
    L = sc.lib
    L.qpsk_tx_frame.restype = C.c_int
    L.qpsk_tx_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_bool]
    rng = np.random.default_rng(17)
    st = oracle.new_state()
    # the legacy TX state is process-global and earlier tests in this process may have used it, so both sides
    # are first flushed with the same long call history only if untouched; instead compare deltas: run the
    # library in a fresh interpreter
    code = (
        "import ctypes as C, numpy as np, sys; sys.path.insert(0, %r); import singlecarrier_b200 as sc; L = sc.lib;"
        "L.qpsk_tx_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_bool];"
        "rng = np.random.default_rng(17); out = [];\n"
        "for n, pre in ((17, True), (31, False), (1, False), (128, True), (250, False)):\n"
        "    sym = (rng.normal(size=n) + 1j * rng.normal(size=n)).astype(np.complex64) * np.float32(0.4)\n"
        "    y = np.zeros(n * 5, np.int16); L.qpsk_tx_frame(y.ctypes.data, sym.ctypes.data, n, pre); out.append(y)\n"
        "np.concatenate(out).tofile(sys.argv[1])" % ROOT)
    import tempfile
    path = tempfile.mktemp(suffix=".i16")
    subprocess.run([sys.executable, "-c", code, path], check=True, cwd=ROOT, timeout=300)
    got = np.fromfile(path, np.int16)
    os.unlink(path)
    want = []
    for n, pre in ((17, True), (31, False), (1, False), (128, True), (250, False)):
        sym = (rng.normal(size=n) + 1j * rng.normal(size=n)).astype(np.complex64) * np.float32(0.4)
        y = np.zeros(n * 5, np.int16)
        oracle.lib.sco_tx_frame(st.ctypes.data, y.ctypes.data, sym.ctypes.data, n, int(pre))
        want.append(y)
    assert np.array_equal(got, np.concatenate(want))


def test_batched_c_example(tmp_path, oracle, gold):
    """examples/batched_demo.c: the batched C ABI driven from plain C (no Python in the loop)."""
    exe = tmp_path / "batched_demo"
    libdir = os.path.join(ROOT, "singlecarrier_b200")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "batched_demo.c"), "-o", str(exe), "-L", libdir,
                    "-lsinglecarrier_b200", f"-Wl,-rpath,{libdir}"], check=True)
    out = subprocess.run([str(exe), os.path.join(ROOT, "tests", "golden", "preamble_qpsk_8k.raw"), "3"], check=True,
                         capture_output=True, text=True, timeout=300).stdout.strip().splitlines()
    x = gold("preamble_qpsk_8k.raw")
    nf = (x.size + 3) // 1880 + 2
    want = []
    for k in range(3):
        s = np.zeros(nf * 1880, np.int16)
        s[k:k + x.size] = x
        bits, st = oracle.run_stream(s)
        for n in range(nf):
            if st["valid"][n]:
                want.append(f"stream {k} call {n} matches {st['matches'][n]} max_index {st['max_index'][n]} "
                            f"max_value {st['max_value'][n]:.2f} bits " + "".join(map(str, bits[n])))
    assert out[:-1] == want and out[-1].startswith(f"3 streams x {nf} calls")


def test_reduce_c_example(tmp_path, oracle, gold):
    """examples/reduce_2gpu.c: shard -> demodulate -> count on the device -> ONE NCCL all-reduce, all through the C ABI
    from plain C (no CUDA headers).  Uses min(2, visible GPUs) ranks; every rank must print the job's totals."""
    exe = tmp_path / "reduce_2gpu"
    libdir = os.path.join(ROOT, "singlecarrier_b200")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", "reduce_2gpu.c"), "-o", str(exe), "-L", libdir,
                    "-lsinglecarrier_b200", f"-Wl,-rpath,{libdir}"], check=True)
    ns = 6
    out = subprocess.run([str(exe), os.path.join(ROOT, "tests", "golden", "preamble_qpsk_8k.raw"), str(ns)], check=True,
                         capture_output=True, text=True, timeout=300).stdout.strip().splitlines()
    out = [ln for ln in out if ln.startswith("rank ")]                        # NCCL may print its version line
    x = gold("preamble_qpsk_8k.raw")
    nf = (x.size + 3 * ns) // 1880 + 2
    calls = valid = matches = 0
    for k in range(ns):
        s = np.zeros(nf * 1880, np.int16)
        s[3 * k:3 * k + x.size] = x
        _, st = oracle.run_stream(s)
        calls += nf
        valid += int(st["valid"].sum())
        matches += int(st["matches"].sum())
    assert 1 <= len(out) <= 2
    for ln in out:
        assert f"calls {calls} valid {valid} sum_matches {matches} " in ln, (ln, calls, valid, matches)

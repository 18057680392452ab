"""CPU: the C-ABI library loads without a GPU, exports every symbol the headers declare, and fails
loudly (no CPU fallback) when asked to compute without a CUDA device."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "singlecarrier_b200", "libsinglecarrier_b200.so")


def exported():
    out = subprocess.run(["nm", "-D", "--defined-only", LIB], check=True, capture_output=True, text=True).stdout
    return {ln.split()[-1] for ln in out.splitlines() if ln.strip()}


def declared(header, pattern):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(pattern, src))


def test_library_exports_every_declared_symbol():
    assert os.path.exists(LIB), "build with `make -C singlecarrier_b200/csrc`"
    syms = exported()
    batched = declared("singlecarrier_b200.h", r"\b(sc_[a-z0-9_]+)\s*\(")
    assert len(batched) >= 20
    assert batched <= syms, sorted(batched - syms)
    compat_fns = declared("sc_compat/singlecarrier_compat.h",
                          r"\b(fir|kalman_init|kalman_reset|kalman_calculate|train_eq|data_eq|scramble_init|scramble|"
                          r"cnormf|qpsk_mod|qpsk_demod|qpsk_rx_frame|qpsk_tx_frame|fft_alloc|fft|fftr_alloc|fftr|fftri|"
                          r"encode_fftr|encode_fftri)\s*\(")
    assert len(compat_fns) == 20 and compat_fns <= syms, sorted(compat_fns - syms)
    data = {"eq_coeff", "kalman_gain", "kalman_y", "preamble_frames_detected", "constellation", "preamblevalues",
            "alpha50_root", "alpha35_root"}
    assert data <= syms, sorted(data - syms)


def test_compat_headers_compile_as_c_and_cxx(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "qpsk_internal.h"\n#include "fir.h"\n#include "fft.h"\n#include "equalizer.h"\n'
                   '#include "kalman.h"\n#include "scramble.h"\n#include "../singlecarrier_b200.h"\n'
                   'int f(void){ return NTAPS + EQ_LENGTH + FRAME_SIZE + (int) sizeof(sc_frame_result) + CYCLES; }\n')
    inc = os.path.join(ROOT, "include", "sc_compat")
    subprocess.run(["gcc", "-std=gnu11", "-Wall", "-Werror", "-I", inc, "-c", str(src), "-o", str(tmp_path / "t.o")], check=True)
    cxx = tmp_path / "t.cpp"
    cxx.write_text('#include "singlecarrier_b200.h"\nstatic_assert(sizeof(sc_frame_result) == 32, "one sector");\nint g(){return SC_N_COUNTERS;}\n')
    subprocess.run(["g++", "-std=c++17", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(cxx),
                    "-o", str(tmp_path / "t2.o")], check=True)


def fails_loudly_without_a_gpu():
    import torch
    assert not torch.cuda.is_available()
    import singlecarrier_b200 as sc
    assert sc.lib.sc_device_count() == 0
    with pytest.raises(sc.SingleCarrierError) as e:
        sc.ModemBank(8)
    assert "no CUDA device" in str(e.value) and e.value.code == -2
    # stage entry points and the drop-in symbols refuse as well (the latter abort the process)
    assert sc.lib.sc_fir_batch_dev(0, 1, 0, 1, 1, 1, 1, None) == -2
    code = ("import ctypes,singlecarrier_b200 as sc; m=(ctypes.c_float*98)(); x=(ctypes.c_float*16)();"
            "sc.lib.fir(m, False, x, 8)")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode != 0 and "no CUDA device" in r.stderr


def test_fails_loudly_without_a_gpu():
    """The checks above in a child process that sees no device (CUDA_VISIBLE_DEVICES empty), so that they run on
    machines with a GPU as well."""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]; "
            "import test_abi; test_abi.fails_loudly_without_a_gpu()")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]


def test_host_helpers_need_no_gpu():
    """Keystream words (integer LFSR, host side) and bit unpacking."""
    import numpy as np
    import singlecarrier_b200 as sc
    from oracle import pyoracle as po
    o = po.Oracle()
    lfsr = C.c_uint16(0x4A80)
    for n in range(5):
        w = 0
        for i in range(31):
            d = C.c_uint8(0)
            o.lib.sco_scramble2(C.byref(d), C.byref(lfsr))
            w |= (d.value & 1) << (2 * i) | (d.value >> 1) << (2 * i + 1)
        assert sc.keystream_word(n) == w
    # positions beyond one LFSR period (32767 bits = 528.5 calls) are reached by reducing the offset, not by
    # replaying from the seed: check against a straight replay
    lfsr = C.c_uint16(0x4A80)
    want = {}
    for n in range(1200):
        w = 0
        for i in range(31):
            d = C.c_uint8(0)
            o.lib.sco_scramble2(C.byref(d), C.byref(lfsr))
            w |= (d.value & 1) << (2 * i) | (d.value >> 1) << (2 * i + 1)
        want[n] = w
    for n in (5, 527, 528, 529, 1056, 1057, 1199):
        assert sc.keystream_word(n) == want[n], n
    assert sc.keystream_word(32767 * 3 + 11) == want[11]           # 62 * 32767 bits = a whole number of periods
    r = np.zeros(3, sc.RESULT_DTYPE)
    r["bits"] = [0b1011, 0x3FFFFFFFFFFFFFFF, 5]
    r["valid"] = [1, 1, 0]
    rows = sc.unpack_bits(r)
    assert rows[0][:4].tolist() == [1, 1, 0, 1] and rows[1].all() and (rows[2] == 255).all()


def test_new_entry_points_validate_arguments_without_a_gpu():
    """Round-2 entry points: argument errors are reported before any CUDA call; compute refuses without a device."""
    import torch
    import singlecarrier_b200 as sc
    L = sc.lib
    assert L.sc_state_size(None) == 0
    assert L.sc_state_export(None, None, 0) == -1 and L.sc_state_import(None, None, 0) == -1
    assert L.sc_reduce_stats(None, 16, None, None) == -1
    assert L.sc_host_alloc(None, 0, 0, None) == -1 and L.sc_host_free(None) == 0
    out = C.c_double(0)
    assert L.sc_h2d_probe(0, 16, 0, 0, 0.0, 0, C.byref(out)) == -1          # buffer too small
    assert L.sc_ber_stats_dev(0, None, 1, 1, 1, None, 1, None, 0, None, 1, None, None) == -1
    if not torch.cuda.is_available():
        assert L.sc_h2d_probe(0, 1 << 20, 0, 0, 0.0, 0, C.byref(out)) == -2
        p = C.c_void_p()
        assert L.sc_host_alloc(C.byref(p), 4096, 0, None) == -2


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under singlecarrier_b200/ may reference it."""
    bad = []
    for dp, _, fns in os.walk(os.path.join(ROOT, "singlecarrier_b200")):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".c", ".h")):
                txt = open(os.path.join(dp, fn)).read()
                if re.search(r"\boracle\b|sco_|libsc_ref|libsc_oracle", txt):
                    bad.append(fn)
    assert bad == []

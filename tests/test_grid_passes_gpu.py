"""GPU: the persistent and grid-capped kernels past their first pass.

Several kernels loop over their work with a grid capped at the SM count (or at a fixed number of CTAs), so a CTA
handles batch n, n + grid, n + 2 grid, ...  Every test here chooses its shape so that CTAs run more than one pass and
every template instantiation runs, and then compares the kernel with the oracle bit for bit where the operation is
exact, or with float64 under a stated per-output error bound where it is not:

  * the fused tcgen05 front-end (frontend_umma_kernel, SC_FE_SEARCH_TCGEN05): 3 and 4 batches per CTA, both filters;
  * the tcgen05 stage search's proposed correlations (approx) against the proposer's error bound, on the hardware;
  * sc_fir_batch_dev: all 8 instantiations (wide x fast x 128-bit loads), warps striding past the capped grid;
  * sc_fftr_batch_dev / sc_fftri_batch_dev batched, and fft_kernel on both sides of the 48 KB shared-memory switch;
  * sc_track_decide_batch_dev on many CTAs.

Shapes derived from the SM count read it from torch.cuda.get_device_properties(0)."""
import os
import re
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from helpers import compare_results, oracle_results, synth_streams

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_proposer_bound import PRE, preamble_signs, reference_sums, threshold, windows  # noqa: E402

pytestmark = pytest.mark.gpu

F32 = np.float32
U = 2.0 ** -24                                      # unit roundoff of float32
NF = 8                                              # calls per batch in the front-end tests
FE_WIN = 16                                         # stream-frames per batch of frontend_umma_kernel
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


@pytest.fixture(scope="module")
def sms(sc):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def u32(a):
    return np.ascontiguousarray(a).view(np.uint32)


def host_workers():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ================================================================================================================
# A. fused tcgen05 front-end, several batches per CTA
# ================================================================================================================
def pick_slab(n, lo, parts):
    """sc_api.cu pick_slab(): streams per slab."""
    s = max(-(-n // parts), lo)
    return -(-s // 128) * 128


def fe_slabs(n, sms, slab):
    """(first stream, streams, batches, grid) of every slab; the grid is launch_frontend_umma's min(batches, SMs)."""
    out = []
    for s0 in range(0, n, slab):
        ns = min(slab, n - s0)
        nb = -(-ns // FE_WIN)
        out.append((s0, ns, nb, min(nb, sms)))
    return out


def fe_stream(slab, cta, rnd, warp):
    """The stream FIR warp `warp` of CTA `cta` handles in the CTA's batch number `rnd` (None past the slab)."""
    s0, ns, nb, grid = slab
    b = rnd * grid + cta
    return s0 + b * FE_WIN + warp if b < nb and b * FE_WIN + warp < ns else None


def plant_hard_rows(x, rows, rng):
    """Silence, near silence (+-3 LSB), a stream that goes dead mid-way and full-scale noise, in turn."""
    for k, s in enumerate(rows):
        kind = k % 4
        if kind == 0:
            x[s] = 0
        elif kind == 1:
            x[s] = rng.integers(-3, 4, x.shape[1]).astype(np.int16)
        elif kind == 2:
            x[s, x.shape[1] // 2 + 123:] = 0
        else:
            x[s] = rng.integers(-32768, 32768, x.shape[1]).astype(np.int16)


def bank_streams(oracle, ns, seed):
    """150 loop-back streams, then shifted and scaled copies of them: cheap, all different."""
    rng = np.random.default_rng(seed)
    base = synth_streams(oracle, rng, 150, NF)
    x = np.empty((ns, NF * 1880), np.int16)
    for k in range(ns):
        x[k] = np.roll(base[k % 150], 37 * (k // 150)) // (1 + (k // 150) % 3)
    return x, rng


def run_dev(sc, x, mode, wide=False, parts=0, extra=0):
    """rx_frames_dev over NF calls with eq_dbg; extra = samples added to the row stride.  Returns (results, eq, image)."""
    import torch
    from singlecarrier_b200.modem import OPT_FE_SEARCH, OPT_SLAB_PARTS
    ns = x.shape[0]
    bank = sc.ModemBank(ns, wide=wide, debug_eq=True)
    bank.set_option(OPT_FE_SEARCH, mode)
    if parts:
        bank.set_option(OPT_SLAB_PARTS, parts)
    d = torch.zeros((ns, NF * 1880 + extra), dtype=torch.int16, device="cuda")
    d[:, :NF * 1880] = torch.from_numpy(x).cuda()
    res = torch.zeros((ns, NF * 32), dtype=torch.uint8, device="cuda")
    eq = torch.zeros((ns, NF * 10), dtype=torch.float32, device="cuda")
    bank.rx_frames_dev(d, NF, res, eq)
    torch.cuda.synchronize()
    out = (res.cpu().numpy().view(sc.RESULT_DTYPE), eq.cpu().numpy().reshape(ns, NF, 10), bank.state_export())
    bank.close()
    return out


def run_host_split(sc, x, mode, first=3):
    """rx_frames_host in two blocks (first, NF - first): the second block's first call reads the saved history frame."""
    from singlecarrier_b200.modem import OPT_FE_SEARCH
    bank = sc.ModemBank(x.shape[0], debug_eq=True)
    bank.set_option(OPT_FE_SEARCH, mode)
    a, ea = bank.rx_frames_host(np.ascontiguousarray(x[:, :first * 1880]), first)
    b, eb = bank.rx_frames_host(np.ascontiguousarray(x[:, first * 1880:]), NF - first)
    image = bank.state_export()
    bank.close()
    return np.concatenate([a, b], axis=1), np.concatenate([ea, eb], axis=1), image


def same_run(a, b):
    """Every result byte, every eq_dbg bit and the state image after the batch."""
    return a[0].tobytes() == b[0].tobytes() and u32(a[1]).tobytes() == u32(b[1]).tobytes() and np.array_equal(a[2], b[2])


# about 12,000 streams, not a multiple of 16: the device entry point cuts a slab of 8,192 (512 batches, 3 or 4 per CTA
# at 148 SMs) and one of 3,811 whose last batch holds 3 streams
NS_A = 12003


@pytest.fixture(scope="module")
def fe_bank(oracle, sms):
    """The NS_A streams with the hard rows planted where the default device slabs put them in batch 2 or 3 of the first,
    a middle and the last CTA, in different FIR warps; and the streams picked for the oracle."""
    x, rng = bank_streams(oracle, NS_A, 4242)
    slabs = fe_slabs(NS_A, sms, pick_slab(NS_A, 8192, 2))
    assert len(slabs) == 2 and slabs[0][2] >= 3 * sms, slabs           # every CTA of slab 0 runs >= 3 batches
    g = slabs[0][3]
    hard = [fe_stream(slabs[0], c, r, w) for c, r, w in
            ((0, 2, 1), (0, 3, 6), (g // 2, 2, 11), (g - 1, 2, 15), (1, 2, 0), (2, 3, 9), (g - 2, 2, 13), (g // 2, 3, 4))]
    hard = [s for s in hard if s is not None]
    assert len(hard) >= 6
    hard += [fe_stream(slabs[1], 5, 1, 7), NS_A - 1]                  # slab 1: a second batch, and the ragged last one
    plant_hard_rows(x, hard, rng)
    pick = set(hard)
    for c in (0, 1, g // 2, g - 1):                                    # batches 0..3 of four CTAs of slab 0
        for r in range(4):
            pick.update(s for s in (fe_stream(slabs[0], c, r, w) for w in range(FE_WIN)) if s is not None)
    s0, ns, nb, _ = slabs[1]
    pick.update(range(s0 + (nb - 1) * FE_WIN, NS_A))                   # the ragged last batch
    return x, np.array(sorted(pick))


@pytest.mark.parametrize("wide", [False, True], ids=["narrow", "wide"])
def test_fused_frontend_several_batches_per_cta(sc, oracle, fe_bank, wide):
    """SC_FE_SEARCH_TCGEN05 and SC_FE_SEARCH_MMA on the device entry point with the default slabs: every result byte,
    every eq_dbg bit and the state image equal the all-exact front-end's, with 3 or 4 batches per CTA of the persistent
    kernel (the rx_timing prefetch two batches ahead, the mbarrier phases past 0, reused window and B buffers).  With an
    odd row stride the tcgen05 mode falls back to the all-exact kernel for the caller's frames, and the results stay
    the same.  A few hundred streams (batches 0..3 of four CTAs, the ragged last batch, the hard rows) equal the
    oracle."""
    from singlecarrier_b200.modem import FE_SEARCH_DIRECT, FE_SEARCH_MMA, FE_SEARCH_TCGEN05
    x, pick = fe_bank
    ref = run_dev(sc, x, FE_SEARCH_DIRECT, wide)
    assert int(ref[0]["valid"].sum()) > NS_A * 2
    assert same_run(run_dev(sc, x, FE_SEARCH_TCGEN05, wide), ref), "tcgen05 front-end"
    assert same_run(run_dev(sc, x, FE_SEARCH_MMA, wide), ref), "mma front-end"
    assert same_run(run_dev(sc, x, FE_SEARCH_TCGEN05, wide, extra=1), ref), "tcgen05 mode, odd stride"
    obits, ostats = oracle_results(oracle, x[pick], NF, wide=wide)
    assert compare_results(ref[0][pick], ref[1][pick], obits, ostats) == []


def test_fused_frontend_one_cta_four_batches(sc, oracle, sms):
    """SC_OPT_SLAB_PARTS = 1 with 16 (3 SMs) + 1 streams: one slab of 3 SMs + 1 batches, so CTA 0 runs 4 of them and
    its last holds one stream (a hard row)."""
    from singlecarrier_b200.modem import FE_SEARCH_DIRECT, FE_SEARCH_TCGEN05
    ns = FE_WIN * 3 * sms + 1
    x, rng = bank_streams(oracle, ns, 777)
    slab = fe_slabs(ns, sms, pick_slab(ns, 128, 1))
    assert len(slab) == 1 and fe_stream(slab[0], 0, 3, 0) == ns - 1 and fe_stream(slab[0], 1, 3, 0) is None
    hard = [fe_stream(slab[0], 0, 2, 3), fe_stream(slab[0], sms // 2, 2, 8), fe_stream(slab[0], sms - 1, 1, 12), ns - 1]
    plant_hard_rows(x, hard, rng)
    ref = run_dev(sc, x, FE_SEARCH_DIRECT, parts=1)
    assert same_run(run_dev(sc, x, FE_SEARCH_TCGEN05, parts=1), ref)
    pick = np.array(sorted(set(hard) | set(range(FE_WIN * 2 * sms, FE_WIN * 2 * sms + FE_WIN)) | {0, 1, ns - 2}))
    obits, ostats = oracle_results(oracle, x[pick], NF)
    assert compare_results(ref[0][pick], ref[1][pick], obits, ostats) == []


def test_fused_frontend_host_entry_two_blocks(sc, fe_bank):
    """Host entry point, the batch split 3 + 5: the tcgen05 front-end equals the all-exact one (results, eq_dbg, state),
    and both equal one device batch."""
    from singlecarrier_b200.modem import FE_SEARCH_DIRECT, FE_SEARCH_TCGEN05
    x, _ = fe_bank
    ref = run_host_split(sc, x, FE_SEARCH_DIRECT)
    assert same_run(run_host_split(sc, x, FE_SEARCH_TCGEN05), ref)
    whole = run_dev(sc, x, FE_SEARCH_DIRECT)
    assert ref[0].tobytes() == whole[0].tobytes() and u32(ref[1]).tobytes() == u32(whole[1]).tobytes()


# ================================================================================================================
# B. tcgen05 stage search: the proposer's bound on the hardware
# ================================================================================================================
def reference_sums_batch(x, sign):
    """reference_sums() for many windows at once: x float32 [n, 255] -> [n, 128], the same sequential fp32 adds."""
    lags = np.arange(PRE)
    a = np.zeros((x.shape[0], PRE), F32)
    for i in range(PRE):
        a = (a + sign[i] * x[:, lags + i]).astype(F32)
    return a


def search_windows(rng, n, sign):
    """n windows of 255 symbols: the generators of test_proposer_bound in turn, a planted preamble at lag k % 128 in
    every fourth window, and NaN / Inf samples in a few (returned as the third value)."""
    out = np.zeros((n, 2 * PRE - 1), np.complex64)
    gen = iter(())
    planted = 0
    for k in range(n):
        if k % 4 == 3:
            lag = planted % PRE
            planted += 1
            w = rng.normal(0, 1, (2 * PRE - 1, 2))
            w[lag:lag + PRE] += (0.3 + 3 * (planted % 5)) * sign[:, None]
            w *= 10.0 ** rng.integers(-4, 5)
        else:
            try:
                _, w = next(gen)
            except StopIteration:
                gen = windows(rng)
                _, w = next(gen)
        s = w.astype(F32)
        out[k] = s[:, 0] + 1j * s[:, 1]
    bad = np.array([5, 1001, n // 2 + 3, n - 1, n - 7])
    out[bad[0], 50] = np.nan
    out[bad[1], 200] = np.inf
    out[bad[2]] = np.nan + 1j * np.nan
    out[bad[3], 0] = complex(-np.inf, 1.0)
    out[bad[4], 254] = complex(1.0, np.nan)
    return out, planted, bad


def test_tcgen05_search_approx_obeys_the_proposer_bound(sc, oracle, sms):
    """sc_preamble_search_tcgen05_batch_dev with 16 (3 SMs) + 5 windows (at least 3 batches per CTA), row strides 256
    and 260.  max_index / max_value with approx equal those without it and the all-exact kernel's.  Per lag,
    |sqrt(approx) - sqrt(v_ref)| <= sqrt(2) delta + 2^-22 sqrt(max v), with v_ref the reference's float32 sums and also
    with the float64 correlations: each component is within delta = 1.004 2^-13 sum(|d| + |e|) (float64 here), the
    Euclidean norm is 1-Lipschitz and the last term covers the rounding of the squares and their sum.  The reference's
    maximum lag always reaches the candidate threshold.  The worst err / delta (err = |sqrt(approx) - sqrt(v_ref)|) is
    printed and must stay below the 0.6 the kernels' comments claim."""
    import torch
    sign = preamble_signs()
    rng = np.random.default_rng(20261020)
    nw = FE_WIN * 3 * sms + 5
    win, planted, bad = search_windows(rng, nw, sign)
    assert planted >= PRE                                               # every lag has a planted preamble
    approx_seen = None
    for stride in (256, 260):
        buf = (rng.normal(size=(nw, stride)) + 1j * rng.normal(size=(nw, stride))).astype(np.complex64)
        buf[:, :2 * PRE - 1] = win                                      # symbols >= 255 are read (256) or not, never used
        d = dev(buf.view(np.float32))
        out = {}
        for name in ("approx", "plain", "direct"):
            idx = torch.full((nw,), -7, dtype=torch.int32, device="cuda")
            val = torch.full((nw,), -7.0, dtype=torch.float32, device="cuda")
            if name == "direct":
                sc._lib.check(sc.lib.sc_preamble_search_direct_batch_dev(0, nw, d.data_ptr(), stride, idx.data_ptr(),
                                                                         val.data_ptr(), 0))
            else:
                app = torch.full((nw, PRE), -1.0, dtype=torch.float32, device="cuda") if name == "approx" else None
                sc._lib.check(sc.lib.sc_preamble_search_tcgen05_batch_dev(0, nw, d.data_ptr(), stride, idx.data_ptr(),
                                                                          val.data_ptr(),
                                                                          app.data_ptr() if app is not None else None, 0))
            torch.cuda.synchronize()
            out[name] = (idx.cpu().numpy(), val.cpu().numpy())
            if name == "approx":
                approx = app.cpu().numpy()
        for name in ("approx", "plain"):
            assert np.array_equal(out[name][0], out["direct"][0]), (stride, name)
            assert np.array_equal(u32(out[name][1]), u32(out["direct"][1])), (stride, name)
        if approx_seen is None:
            approx_seen = approx
        else:
            assert np.array_equal(u32(approx), u32(approx_seen))          # the layout changes nothing
    gi, gv = out["direct"]
    for k in list(bad) + list(range(0, 24)) + list(range(nw - 24, nw)):  # NaN / Inf windows: the exact fallback
        oi, ov = oracle.search(win[k])
        assert gi[k] == oi and gv[k].view(np.uint32) == F32(ov).view(np.uint32), k

    # ---- the bound, per window and lag
    ok = np.isfinite(win.view(np.float32)).all(axis=1)
    ok[bad] = False
    s = win[ok]
    d = (s.real - s.imag).astype(F32)                                   # qpsk.c:88-96 with pre = v(1 + i)
    e = (s.imag + s.real).astype(F32)
    ref_d, ref_e = reference_sums_batch(d, sign), reference_sums_batch(e, sign)
    for k in range(0, s.shape[0], 997):                                 # the batched form is reference_sums()
        assert np.array_equal(u32(ref_d[k]), u32(reference_sums(d[k], sign)))
        assert np.array_equal(u32(ref_e[k]), u32(reference_sums(e[k], sign)))
    v_ref = ((ref_d * ref_d).astype(F32) + (ref_e * ref_e).astype(F32)).astype(F32)          # cnormf, qpsk.c:75-80
    best = np.argmax(v_ref, axis=1)                                     # first maximum; all zero -> lag 0
    assert np.array_equal(best, gi[ok]) and np.array_equal(u32(v_ref[np.arange(len(best)), best]), u32(gv[ok]))
    app = approx[ok].astype(np.float64)
    assert np.isfinite(app).all() and (app >= 0).all()
    s_abs = np.sum(np.abs(d.astype(np.float64)) + np.abs(e.astype(np.float64)), axis=1)
    delta = s_abs * float.fromhex("0x1.004p-13")
    toep = np.zeros((2 * PRE - 1, PRE))                                 # toep[x, L] = pre[x - L]
    for L in range(PRE):
        toep[L:L + PRE, L] = sign
    ex_d, ex_e = d.astype(np.float64) @ toep, e.astype(np.float64) @ toep
    vmax = np.maximum(app.max(axis=1), v_ref.max(axis=1).astype(np.float64))
    tol = np.sqrt(2.0) * delta[:, None] + 2.0 ** -22 * np.sqrt(vmax)[:, None]
    err = np.abs(np.sqrt(app) - np.sqrt(v_ref.astype(np.float64)))
    err_ex = np.abs(np.sqrt(app) - np.hypot(ex_d, ex_e))
    assert (err <= tol).all(), np.unravel_index(np.argmax(err - tol), err.shape)
    assert (err_ex <= tol).all(), np.unravel_index(np.argmax(err_ex - tol), err.shape)
    aok = approx[ok]
    for k in range(s.shape[0]):                                         # the reference's maximum is a candidate
        delta32 = F32(F32(s_abs[k]) * F32(float.fromhex("0x1.004p-13")))
        assert aok[k, best[k]] >= threshold(aok[k].max(), delta32), (k, best[k])
    pos = delta > 0
    worst = float((err[pos].max(axis=1) / delta[pos]).max())
    print(f"tcgen05 proposer on this GPU: worst |sqrt(approx) - sqrt(v_ref)| / delta = {worst:.4f} "
          f"over {int(pos.sum())} windows x {PRE} lags")
    assert worst < 0.6, worst


# ================================================================================================================
# C. sc_fir_batch_dev, all 8 instantiations, past the grid
# ================================================================================================================
FIR_STREAMS = 4 * 6 * 148 + 37                      # launch_fir_batch caps the grid at 148 x 6 CTAs of 4 warps
FIR_LENGTHS = (1, 48, 49, 319, 320, 321, 1881)
FIR_GAIN = F32(2.2)                                 # fir.h:17
SC_FIR_FAST = 2


def fir_taps(wide):
    text = open(os.path.join(ROOT, "include", "sc_tables.inc")).read()
    name = "SC_TABLE_RRC50" if wide else "SC_TABLE_RRC35"
    body = re.search(name + r" = \{(.*?)\};", text, re.S).group(1)
    taps = np.array([float(t) for t in re.findall(r"-?\d+\.\d+", body)], np.float32)
    assert taps.size == 49
    return taps


def gamma(n):
    return n * U / (1 - n * U)


@pytest.fixture(scope="module")
def fir_inputs():
    """Delay lines and samples of FIR_STREAMS streams with amplitudes spread over 1e-3 .. 1e4."""
    rng = np.random.default_rng(4949)
    ns, n = FIR_STREAMS, max(FIR_LENGTHS)
    amp = 10.0 ** rng.uniform(-3, 4, (ns, 1))
    mem = ((rng.normal(size=(ns, 49)) + 1j * rng.normal(size=(ns, 49))) * amp).astype(np.complex64)
    x = ((rng.normal(size=(ns, n)) + 1j * rng.normal(size=(ns, n))) * amp).astype(np.complex64)
    return mem, x


def fir_layouts(length):
    """(name, row stride, base offset in complex samples): 128-bit loads need an even stride and a 16-byte aligned base."""
    even = length + 7 + (length + 7) % 2
    return (("vec", even, 0), ("scalar", even + 1, 0), ("offset base", even, 1))


def run_fir(sc, mem0, x0, length, mode, stride, offset):
    """One batched call on a padded copy; returns (delay lines, samples [ns, length], padding unchanged?)."""
    import torch
    ns = mem0.shape[0]
    rng = np.random.default_rng(length)
    flat = (rng.normal(size=ns * stride + 2) + 1j * rng.normal(size=ns * stride + 2)).astype(np.complex64)
    rows = flat[offset:offset + ns * stride].reshape(ns, stride)
    rows[:, :length] = x0[:, :length]
    d_x, d_m = dev(flat.view(np.float32)), dev(mem0.view(np.float32))
    sc._lib.check(sc.lib.sc_fir_batch_dev(0, ns, mode, d_m.data_ptr(), d_x.data_ptr() + 8 * offset, stride, length, 0))
    torch.cuda.synchronize()
    got = d_x.cpu().numpy().view(np.complex64)
    got_rows = got[offset:offset + ns * stride].reshape(ns, stride)
    untouched = np.array_equal(u32(np.delete(got.view(np.float32), np.s_[2 * offset:2 * (offset + ns * stride)])),
                               u32(np.delete(flat.view(np.float32), np.s_[2 * offset:2 * (offset + ns * stride)]))) \
        and np.array_equal(u32(got_rows[:, length:]), u32(rows[:, length:]))
    return d_m.cpu().numpy().view(np.complex64), got_rows[:, :length].copy(), untouched


def run_fir_one_by_one(sc, mem0, x0, length, mode):
    """Every stream in a call of its own (one stream: the grid stride never runs)."""
    import torch
    ns = mem0.shape[0]
    stride = fir_layouts(length)[0][1]
    rows = np.zeros((ns, stride), np.complex64)
    rows[:, :length] = x0[:, :length]
    d_x, d_m = dev(rows.view(np.float32)), dev(mem0.view(np.float32))
    for s in range(ns):
        sc._lib.check(sc.lib.sc_fir_batch_dev(0, 1, mode, d_m.data_ptr() + 8 * 49 * s, d_x.data_ptr() + 8 * stride * s,
                                              stride, length, 0))
    torch.cuda.synchronize()
    return d_m.cpu().numpy().view(np.complex64), d_x.cpu().numpy().view(np.complex64)[:, :length].copy()


def oracle_fir(oracle, mem0, x0, length, wide):
    mem, y = mem0.copy(), np.ascontiguousarray(x0[:, :length]).copy()

    def one(s):
        oracle.fir(mem[s], bool(wide), y[s])

    with ThreadPoolExecutor(max_workers=host_workers()) as ex:
        list(ex.map(one, range(mem.shape[0])))
    return mem, y


@pytest.mark.parametrize("wide", [0, 1], ids=["narrow", "wide"])
def test_fir_batch_exact_past_the_grid(sc, oracle, fir_inputs, wide):
    """Exact mode, 128-bit and 64-bit loads: every stream's outputs and delay line equal oracle.fir bit for bit, samples
    beyond `length` are untouched, and one call per stream gives the same bytes."""
    mem0, x0 = fir_inputs
    for length in FIR_LENGTHS:
        want_m, want_y = oracle_fir(oracle, mem0, x0, length, wide)
        for name, stride, offset in fir_layouts(length):
            m, y, untouched = run_fir(sc, mem0, x0, length, wide, stride, offset)
            assert untouched, (length, name)
            bad = np.nonzero((u32(y) != u32(want_y)).any(axis=1) | (u32(m) != u32(want_m)).any(axis=1))[0]
            assert bad.size == 0, (length, name, bad[:10])
        m1, y1 = run_fir_one_by_one(sc, mem0, x0, length, wide)
        assert np.array_equal(u32(y1), u32(want_y)) and np.array_equal(u32(m1), u32(want_m)), length


@pytest.mark.parametrize("wide", [0, 1], ids=["narrow", "wide"])
def test_fir_batch_fast_mode_per_output_bound(sc, fir_inputs, wide):
    """SC_FIR_FAST (one contracted multiply-add per tap, the gain folded into the taps): every output component is
    within gamma_51 g sum_k |x_k| |c_k| of the float64 FIR (49 chained FMAs plus the rounding of tap x FIR_GAIN), a
    bound per output, so a stream of amplitude 1e-3 is held to its own scale.  The delay line holds the raw inputs bit
    for bit, samples beyond `length` are untouched, and the three load layouts and one call per stream give the same
    bytes."""
    mem0, x0 = fir_inputs
    taps = fir_taps(wide).astype(np.float64)
    g = float(FIR_GAIN)
    mode = wide | SC_FIR_FAST
    differs = False
    for length in FIR_LENGTHS:
        ext = np.concatenate([mem0, x0[:, :length]], axis=1).astype(np.complex128)           # ext[49 + j] = x[j]
        y64 = np.zeros((mem0.shape[0], length), np.complex128)
        bre = np.zeros((mem0.shape[0], length))
        bim = np.zeros((mem0.shape[0], length))
        for k in range(49):                                                                  # out[j] = g sum ext[j+1+k] c[k]
            seg = ext[:, 1 + k:1 + k + length]
            y64 += taps[k] * seg
            bre += abs(taps[k]) * np.abs(seg.real)
            bim += abs(taps[k]) * np.abs(seg.imag)
        y64 *= g
        bre *= gamma(51) * g
        bim *= gamma(51) * g
        want_m = ext[:, -49:].astype(np.complex64)                                           # the last 49 raw inputs
        first = None
        for name, stride, offset in fir_layouts(length):
            m, y, untouched = run_fir(sc, mem0, x0, length, mode, stride, offset)
            assert untouched, (length, name)
            assert np.array_equal(u32(m), u32(want_m)), (length, name)
            er, ei = np.abs(y.real - y64.real), np.abs(y.imag - y64.imag)
            assert (er <= bre).all() and (ei <= bim).all(), (length, name, np.argwhere((er > bre) | (ei > bim))[:5])
            if first is None:
                first = y
            assert np.array_equal(u32(y), u32(first)), (length, name)
        m1, y1 = run_fir_one_by_one(sc, mem0, x0, length, mode)
        assert np.array_equal(u32(y1), u32(first)) and np.array_equal(u32(m1), u32(want_m)), length
        _, exact, _ = run_fir(sc, mem0, x0, length, wide, fir_layouts(length)[0][1], 0)      # pinned to the oracle above
        differs |= not np.array_equal(u32(first), u32(exact))
    assert differs                                                                          # really another rounding


# ================================================================================================================
# D. FFT launch configurations past the grid
# ================================================================================================================
def fft_factors(n):
    """sc_api.cu fft_make_plan() (kf_factor, src/fft.c:433-459): the radix of every stage."""
    ps, p = [], 4
    floor_sqrt = np.floor(np.sqrt(F32(n)))
    while True:
        while n % p:
            p = 2 if p == 4 else (3 if p == 2 else p + 2)
            if p > floor_sqrt:
                p = n
        n //= p
        ps.append(p)
        if n <= 1:
            return ps


@pytest.mark.parametrize("nfft,batches", [(6, 1000), (20, 1000), (64, 1000), (250, 1000), (256, 1000), (16384, 100)])
def test_fftr_fftri_batched_past_the_grid(sc, nfft, batches):
    """sc_fftr_batch_dev / sc_fftri_batch_dev with more transforms than CTAs (592, or 64 scratch CTAs at core length
    8,192): every transform equals the same input run alone, bit for bit (the single-transform form is the one pinned
    to the reference's golden vectors).  Without a factor 5 in the core length, both directions are also within
    8 u log2(nfft) sum|input| of numpy's float64 rfft / irfft (a few roundings per radix-2 level of the core transform
    and in the real-FFT pre- / post-processing)."""
    import torch
    rng = np.random.default_rng(nfft)
    h = nfft // 2 + 1
    x = (rng.normal(size=(batches, nfft)) * 10.0 ** rng.uniform(-3, 3, (batches, 1))).astype(np.float32)
    d_x = dev(x)
    spec = torch.zeros((batches, 2 * h), dtype=torch.float32, device="cuda")
    sc._lib.check(sc.lib.sc_fftr_batch_dev(0, batches, nfft, d_x.data_ptr(), spec.data_ptr(), 0))
    back = torch.zeros((batches, nfft), dtype=torch.float32, device="cuda")
    sc._lib.check(sc.lib.sc_fftri_batch_dev(0, batches, nfft, spec.data_ptr(), back.data_ptr(), 0))
    spec1 = torch.zeros_like(spec)
    back1 = torch.zeros_like(back)
    for b in range(batches):
        sc._lib.check(sc.lib.sc_fftr_batch_dev(0, 1, nfft, d_x[b].data_ptr(), spec1[b].data_ptr(), 0))
        sc._lib.check(sc.lib.sc_fftri_batch_dev(0, 1, nfft, spec[b].data_ptr(), back1[b].data_ptr(), 0))
    torch.cuda.synchronize()
    sp, sp1 = spec.cpu().numpy(), spec1.cpu().numpy()
    bk, bk1 = back.cpu().numpy(), back1.cpu().numpy()
    bad = np.nonzero((u32(sp) != u32(sp1)).any(axis=1))[0]
    assert bad.size == 0, ("fftr", bad[:10])
    bad = np.nonzero((u32(bk) != u32(bk1)).any(axis=1))[0]
    assert bad.size == 0, ("fftri", bad[:10])
    if (nfft // 2) % 5 == 0:
        return                                        # the reference's radix-5 butterfly is not a DFT (test_stage_gpu)
    c = 8 * U * np.log2(nfft)
    z = sp.view(np.complex64).astype(np.complex128)
    want = np.fft.rfft(x.astype(np.float64), axis=1)
    lim = c * np.abs(x.astype(np.float64)).sum(axis=1)
    assert (np.abs(z - want).max(axis=1) <= lim).all(), np.max(np.abs(z - want).max(axis=1) / lim)
    want_b = np.fft.irfft(z, n=nfft, axis=1) * nfft
    lim_b = c * 2 * np.abs(z).sum(axis=1)
    assert (np.abs(bk - want_b).max(axis=1) <= lim_b).all(), np.max(np.abs(bk - want_b).max(axis=1) / lim_b)


@pytest.mark.parametrize("n", [3072, 3073, 4093, 4096])
def test_fft_shared_memory_sizes_past_the_grid(sc, n):
    """fft_kernel at 3,072 (48 KB of shared memory, no attribute needed), 3,073 (7 x 439: generic stages), 4,093
    (prime: one generic stage with p = n) and 4,096 (64 KB): 700 transforms, more than the 592 CTAs, forward and
    inverse, out of place and in place, each equal to the same input run alone.  Against the float64 DFT every output
    is within 2 u sum_l (p_l + 3) sum|x| (stage l of radix p_l: a sequential sum of p_l products, the twiddle's own
    rounding and the complex multiply), which for the prime length is the n-term sum of the generic stage."""
    import torch
    batches = 700
    rng = np.random.default_rng(n)
    x = ((rng.normal(size=(batches, n)) + 1j * rng.normal(size=(batches, n)))
         * 10.0 ** rng.uniform(-3, 3, (batches, 1))).astype(np.complex64)
    bound = 2 * U * sum(p + 3 for p in fft_factors(n)) * np.abs(x.astype(np.complex128)).sum(axis=1)
    for inv in (0, 1):
        d_x = dev(x.view(np.float32))
        out = torch.zeros_like(d_x)
        sc._lib.check(sc.lib.sc_fft_batch_dev(0, batches, n, inv, d_x.data_ptr(), out.data_ptr(), 0))
        inplace = d_x.clone()
        sc._lib.check(sc.lib.sc_fft_batch_dev(0, batches, n, inv, inplace.data_ptr(), inplace.data_ptr(), 0))
        alone = torch.zeros_like(d_x)
        for b in range(batches):
            sc._lib.check(sc.lib.sc_fft_batch_dev(0, 1, n, inv, d_x[b].data_ptr(), alone[b].data_ptr(), 0))
        torch.cuda.synchronize()
        y, y_in, y1 = out.cpu().numpy(), inplace.cpu().numpy(), alone.cpu().numpy()
        bad = np.nonzero((u32(y) != u32(y1)).any(axis=1) | (u32(y_in) != u32(y1)).any(axis=1))[0]
        assert bad.size == 0, (inv, bad[:10])
        xx = x.astype(np.complex128)
        want = np.fft.ifft(xx, axis=1) * n if inv else np.fft.fft(xx, axis=1)
        err = np.abs(y.view(np.complex64) - want).max(axis=1)
        assert (err <= bound).all(), (inv, float((err / bound).max()))


# ================================================================================================================
# E. sc_track_decide_batch_dev on many CTAs
# ================================================================================================================
def test_track_decide_batch_many_ctas(sc, oracle):
    """The oracle's own decimated windows (as test_stage_gpu builds them) of 1,037 streams: one launch per call index
    with 1,037 windows (9 CTAs of 128, the last with 13), symbol_stride 300, eq_dbg NULL and non-NULL.  Every field
    equals the oracle's, bit for bit, and rx_timing is updated in place."""
    import torch
    rng = np.random.default_rng(1037)
    ns, nf = 1037, 5
    samples = synth_streams(oracle, rng, ns, nf)
    plant_hard_rows(samples, [100, 500, 900, 1036, 1035, 640, 129, 255], rng)
    per_stream = [None] * ns

    def one(s):
        st = oracle.new_state()
        prev, rec = None, []
        for n in range(nf):
            bits, stats = oracle.rx_frame(st, samples[s, n * 1880:(n + 1) * 1880])
            dec = np.frombuffer(st, np.float32, count=2 * 752, offset=3760 * 8).view(np.complex64)[:290].copy()
            if n >= 2:
                rec.append((n, dec, prev, bits.copy(), stats.copy()))
            prev = int(stats["rx_timing"])
        per_stream[s] = rec

    with ThreadPoolExecutor(max_workers=host_workers()) as ex:
        list(ex.map(one, range(ns)))
    for n in range(2, nf):
        recs = [per_stream[s][n - 2] for s in range(ns)]
        sym = (rng.normal(size=(ns, 300)) + 1j * rng.normal(size=(ns, 300))).astype(np.complex64)
        sym[:, :290] = np.stack([r[1] for r in recs])
        stats = np.array([r[4] for r in recs])
        d_sym = dev(sym.view(np.float32))
        d_mi = dev(stats["max_index"].astype(np.int32))
        d_mv = dev(stats["max_value"].astype(np.float32))
        tin = np.array([r[2] for r in recs], np.int32)
        got = {}
        for with_eq in (False, True):
            d_t = dev(tin)
            d_res = torch.zeros((ns, 32), dtype=torch.uint8, device="cuda")
            d_eq = torch.zeros((ns, 10), dtype=torch.float32, device="cuda") if with_eq else None
            sc._lib.check(sc.lib.sc_track_decide_batch_dev(0, ns, d_sym.data_ptr(), 300, d_mi.data_ptr(), d_mv.data_ptr(),
                                                           d_t.data_ptr(), n, d_res.data_ptr(),
                                                           d_eq.data_ptr() if with_eq else None, 0))
            torch.cuda.synchronize()
            got[with_eq] = (d_res.cpu().numpy().view(sc.RESULT_DTYPE)[:, 0], d_t.cpu().numpy(),
                            d_eq.cpu().numpy() if with_eq else None)
        assert got[False][0].tobytes() == got[True][0].tobytes() and np.array_equal(got[False][1], got[True][1])
        r, t_out, eq = got[True]
        assert np.array_equal(r["valid"].astype(np.int32), stats["valid"]), n
        assert np.array_equal(r["matches"].astype(np.int32), stats["matches"]), n
        assert np.array_equal(r["rx_timing"].astype(np.int32), stats["rx_timing"]), n
        assert np.array_equal(t_out, stats["rx_timing"]), n
        assert np.array_equal(r["max_index"].astype(np.int32), stats["max_index"]), n
        assert np.array_equal(u32(r["max_value"]), u32(stats["max_value"])), n
        assert np.array_equal(u32(r["cost"]), u32(stats["cost"])), n
        assert (r["call_index"] == n).all(), n
        assert np.array_equal(u32(eq), u32(np.ascontiguousarray(stats["eq_coeff"]))), n
        v = stats["valid"].astype(bool)
        assert 0 < v.sum() < ns
        rows = sc.unpack_bits(r)
        assert np.array_equal(rows[v], np.stack([rec[3] for rec in recs])[v]), n

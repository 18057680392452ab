"""CPU: the two parts of packet-mode acquisition's specification (tests/packet_acq_ref.c) that the GPU copies bit for bit
and that only loop-back statistics checked so far, each against a model written from the algorithm:

1. The seeded decision-directed loop (scd_dd_packet_seeded from nu = nu0), which decodes every ACQ record, against a
   float64 model of the loop on the grids and nu0 of real records, under carrier offsets up to 40 Hz.
2. The selection rule of the header comment (stage 1's first maximum, the threshold, the neighbour test outside the
   frame, stage 2's order 0, -1, +1, -2, +2, nu0, freq_hz and the call_index / max_index mapping) as a numpy model on
   the spec's float32 rho and D: it must give exactly the spec's records, also on a stream built to hold an exact tie
   of rho1 between lags of two frames, and on rho with ties and values at the threshold it must accept exactly the
   lags the rule as written accepts.
"""
import functools

import numpy as np
import pytest

import packet_acq_ref as A
from packet_dd_ref import dd_params, loop_streams, po_preamble

FRAME, LAGS, PRE, NDATA = 1880, 376, 128, 248


# ---- 1. the seeded DD loop in float64 ------------------------------------------------------------------------------
def dd_seeded64(S, nu0):
    """The DD loop on the grid S (380 symbols) from p = 1, w = 0, nu = nu0, in complex128: per step i the output
    y = (sum_k conj(w_k) x_k) conj(p) on x = S[i:i+5]; the target d is the preamble symbol (amp, amp) b_i for
    i < 128, else the sign decision of y; e = d - y; w += x conj(e p) mu / (eps + |x|^2); the phase error
    pe = Im(y conj d) / (|y conj d| + peps); nu += beta pe; p *= 1 + j (alpha pe + nu), renormalised.
    -> (y of the 128 training steps, y of the 248 data steps)"""
    mu, alpha, beta, eps, amp, peps = (float(v) for v in dd_params())
    pre = po_preamble()
    S = np.asarray(S, np.complex128)
    w = np.zeros(5, np.complex128)
    p, nu = 1.0 + 0.0j, float(nu0)
    ys = np.zeros(PRE + NDATA, np.complex128)
    for i in range(PRE + NDATA):
        x = S[i:i + 5]
        y = np.sum(np.conj(w) * x) * np.conj(p)
        ys[i] = y
        d = amp * pre[i] * (1 + 1j) if i < PRE else complex(-1.0 if y.real < 0 else 1.0, -1.0 if y.imag < 0 else 1.0)
        q = y * np.conj(d)
        pe = q.imag / (abs(q) + peps)
        w = w + x * np.conj((d - y) * p) * (mu / (eps + np.sum(np.abs(x) ** 2)))
        nu += beta * pe
        p = p * (1 + 1j * (alpha * pe + nu))
        p /= abs(p)
    return ys[:PRE], ys[PRE:]


@pytest.mark.parametrize("sigma", [0.0, 1500.0])
@pytest.mark.parametrize("foff", [0.0, 10.0, -10.0, 20.0, -20.0, 40.0, -40.0])
def test_seeded_loop_agrees_with_the_float64_model(oracle, sigma, foff):
    """Decisions equal where |y| > 1e-3, |z - y| < 1e-2, and matches equal where the training outputs' y.r + y.i are
    clear of 0, on the grid and nu0 of every record the spec finds."""
    rng = np.random.default_rng(int(4000 + sigma + 3 * foff))
    x, _, _ = loop_streams(oracle, rng, 3, 4, sigma=sigma)
    pre = po_preamble()
    n = seeded = 0
    for s in range(x.shape[0]):
        pk, psym, grids = A.acq_run_stream(x[s], foffset=foff)
        for p, z, g in zip(pk, psym, grids):
            yt, y = dd_seeded64(g, float(p["nu0"]))
            big_r, big_i = np.abs(y.real) > 1e-3, np.abs(y.imag) > 1e-3
            assert np.array_equal((y.real < 0)[big_r], (z.real < 0)[big_r]), (s, int(p["grid_sample"]))
            assert np.array_equal((y.imag < 0)[big_i], (z.imag < 0)[big_i]), (s, int(p["grid_sample"]))
            assert np.abs(z - y).max() < 1e-2, (s, int(p["grid_sample"]))
            t = yt.real + yt.imag
            clear = np.abs(t) > 1e-3
            m64 = int(((t * pre) > 0).sum())
            assert abs(int(p["matches"]) - m64) <= int((~clear).sum()), (s, int(p["matches"]), m64)
            if clear.all():
                assert int(p["matches"]) == m64
            n += 1
            seeded += p["nu0"] != 0
    assert n >= 10 and seeded == n           # every record was decoded from a seed, not from nu = 0


# ---- 2. the selection rule in numpy --------------------------------------------------------------------------------
def stage1(rho1, f, tau, W):
    """Stage 1 of frame f on rho1[k + W] (lag k): the lag k* accepted, or None"""
    lo = LAGS * f
    own = rho1[lo + W:lo + LAGS + W]
    ks = lo + int(np.argmax(own))                                      # the first maximum
    best = rho1[ks + W]
    if not best >= tau:
        return None
    for k in range(ks - W, ks + W + 1):
        if lo <= k < lo + LAGS:                                        # only lags outside the frame compete
            continue
        if k < ks and not rho1[k + W] < best:                          # ties go to the earlier lag
            return None
        if k > ks and not rho1[k + W] <= best:
            return None
    return ks


def model_records(x, wide=False, foffset=0.0):
    """The selection rule of the header comment on one stream -> list of (grid_sample, call, max_index, frame,
    metric, nu0, freq_hz) with the float32 values as numpy float32"""
    tau, W, hz_per_rad = A.acq_params()
    nf = x.size // FRAME
    filt = A.acq_filt(x, wide=wide, foffset=foffset)
    rho1 = A.acq_rho_lags(filt, -W, LAGS * nf + 2 * W)                  # lags -W .. 376 nf + W - 1
    out = []
    for f in range(nf - 2):                                            # frame f is decided by call f + 2 < nf
        ks = stage1(rho1, f, tau, W)
        if ks is None:
            continue
        best = None
        for s in (0, -1, 1, -2, 2):
            r, D = A.acq_metric(filt, 5 * ks + s)
            if best is None or r > best[0]:
                best = (r, D, 5 * ks + s)
        r, D, g = best
        nu0 = np.float32(D.imag) / np.float32(D.real) if D.real > 0 else np.float32(0.0)
        call = 2 + g // FRAME                                          # floor division: g may be -1 or -2
        out.append((g, call, (g - (call - 2) * FRAME) // 5, f, np.float32(r), np.float32(nu0),
                    np.float32(np.float32(nu0) * hz_per_rad)))
    return out


def bits(v):
    return int(np.float32(v).view(np.uint32))


def assert_model_is_the_spec(x, wide=False, foffset=0.0):
    pk, _, _ = A.acq_run_stream(x, wide=wide, foffset=foffset)
    got = model_records(x, wide=wide, foffset=foffset)
    want = [(int(p["grid_sample"]), int(p["call"]), int(p["max_index"]), int(p["frame"]), bits(p["metric"]),
             bits(p["nu0"]), bits(p["freq_hz"])) for p in pk]
    assert [(g, c, m, f, bits(r), bits(nu), bits(hz)) for g, c, m, f, r, nu, hz in got] == want
    return len(want)


# the loop-back cases of the GPU acquisition tests (tests/test_packet_passes_gpu.py): (gap, lead_max, frames kept)
CASES = {"gap903": (903, 2000, None), "gap37": (37, 2000, None), "gap0": (0, 2000, None),
         "lead0_60": (903, 61, None), "tail": (0, 1880, 5), "wide": (903, 2000, None), "foffset": (903, 2000, None)}


@pytest.mark.parametrize("case", list(CASES))
def test_model_gives_the_spec_records_on_loop_back(oracle, case):
    gap, lead_max, keep = CASES[case]
    rng = np.random.default_rng(5000 + list(CASES).index(case))
    x, _, starts = loop_streams(oracle, rng, 4, 5, sigma=600.0, gap=gap, lead_max=lead_max)
    if keep is not None:                            # packets start in the last two frames, the last one is cut off
        x = np.ascontiguousarray(x[:, :keep * FRAME])
        assert ((starts >= (keep - 2) * FRAME) & (starts < keep * FRAME)).sum(axis=1).min() >= 2
    n = sum(assert_model_is_the_spec(x[s], wide=case == "wide", foffset=7.5 if case == "foffset" else 0.0)
            for s in range(x.shape[0]))
    assert n >= 4 * (2 if keep else 4)


def test_model_gives_the_spec_records_on_noise_and_degenerate_inputs():
    """Noise at the bench's largest sigma and the degenerate inputs of test_degenerate_inputs_give_no_nan: the spec
    finds nothing on any of them, so this checks that the model, too, rejects every frame there."""
    from singlecarrier_b200.harness import DATA_RMS_LSB
    sigma0 = float(np.sqrt(DATA_RMS_LSB ** 2 * 8000.0 / (2 * 1600.0 * 2.0)))   # the bench's largest: Eb/N0 = 0 dB
    rng = np.random.default_rng(13)
    for _ in range(3):
        x = np.clip(rng.normal(0, sigma0, FRAME * 12), -32767, 32767).round().astype(np.int16)
        assert assert_model_is_the_spec(x) == 0
    n = FRAME * 6
    imp = np.zeros(n, np.int16)
    imp[3000] = 32767
    sat = np.full(n, 32767, np.int16)
    sat[::2] = -32768
    for x in (np.zeros(n, np.int16), np.full(n, 32767, np.int16), sat, imp):
        assert assert_model_is_the_spec(x) == 0


# ---- an exact tie across a frame edge ------------------------------------------------------------------------------
TIE_FRAMES, TIE_K1, TIE_D = 5, 2 * LAGS - 2, 3          # lag 750, the last but one of frame 1, and lag 753 of frame 2


@functools.lru_cache(maxsize=None)
def tie_stream():
    """5 frames in which rho1 of lags TIE_K1 (frame 1) and TIE_K1 + TIE_D (frame 2) are bit-equal and above tau.

    Two packets of the spec's transmitter TIE_D symbols apart, the first on the grid 5 TIE_K1: each lag sees one
    preamble with the other as interference, so their rho1 cross as the second packet's amplitude r grows.  r is
    bisected to the last float32 step below the crossing; then one sample that only the later lag's window sees
    (through outer taps of the matched filter) is moved by a few LSB until the two are equal."""
    po = A.po
    o = po.Oracle()
    rng = np.random.default_rng(1)
    pa, pb = (po.ext_tx_packet(o, o.new_state(), rng.integers(0, 2, 496).astype(np.uint8)).astype(np.float64)
              for _ in range(2))
    k1, k2 = TIE_K1, TIE_K1 + TIE_D
    s1 = 5 * k1 - 48                                               # the two filters' delay

    def make(r):
        x = np.zeros(TIE_FRAMES * FRAME)
        x[s1:s1 + pa.size] += 0.5 * pa
        x[s1 + 5 * TIE_D:s1 + 5 * TIE_D + pb.size] += 0.5 * r * pb
        return np.clip(np.round(x), -32767, 32767).astype(np.int16)

    def gap(x):
        r = A.acq_rho_lags(A.acq_filt(x), k1, TIE_D + 1)
        return float(r[-1]) - float(r[0])

    lo, hi = 1.0, 1.06
    assert gap(make(lo)) < 0 < gap(make(hi))
    for _ in range(40):
        m = (lo + hi) / 2
        lo, hi = (m, hi) if gap(make(m)) < 0 else (lo, m)
    x = make(lo)
    p = 5 * k2 + 5 * (PRE - 1) - 14                                # filt[p .. p + 48] misses lag k1's grid 5 k1 + 5 i
    base = int(x[p])
    for v in sorted(range(-200, 201), key=abs):
        x[p] = base + v
        if gap(x) == 0.0:
            return x
    raise AssertionError("no exact tie")


def test_exact_tie_across_the_frame_edge():
    """Each tied lag is the first maximum of its own frame and the other's neighbour outside it.  Frame 1 keeps its
    lag (a later neighbour may equal it), frame 2 drops its own (an earlier one may not): the spec gives frame 1's
    record only, and so does the model."""
    tau, W, _ = A.acq_params()
    x = tie_stream()
    k1, k2 = TIE_K1, TIE_K1 + TIE_D
    rho1 = A.acq_rho_lags(A.acq_filt(x), -W, LAGS * TIE_FRAMES + 2 * W)
    assert rho1[k1 + W].view(np.uint32) == rho1[k2 + W].view(np.uint32) and rho1[k1 + W] >= tau
    assert LAGS + int(np.argmax(rho1[LAGS + W:2 * LAGS + W])) == k1
    assert 2 * LAGS + int(np.argmax(rho1[2 * LAGS + W:3 * LAGS + W])) == k2
    assert stage1(rho1, 1, tau, W) == k1 and stage1(rho1, 2, tau, W) is None
    assert assert_model_is_the_spec(x) == 1
    pk = A.acq_run_stream(x)[0]
    assert pk["frame"].tolist() == [1] and abs(int(pk["grid_sample"][0]) - 5 * k1) <= 2


def acceptable(rho1, f, tau, W):
    """The lags of frame f that the rule accepts, by its definition: k* is the first maximum of the frame (greater
    than every earlier lag of the frame, not less than any later one), rho1(k*) >= tau, and every lag outside the
    frame within W of k* is below it (before it) or not above it (after it)."""
    lo, hi = LAGS * f, LAGS * (f + 1)
    out = []
    for k in range(lo, hi):
        v = rho1[k + W]
        if not v >= tau:
            continue
        if any(not rho1[j + W] < v for j in range(lo, k)) or any(not rho1[j + W] <= v for j in range(k + 1, hi)):
            continue
        out_lo = [j for j in range(k - W, k) if not lo <= j < hi]
        out_hi = [j for j in range(k + 1, k + W + 1) if not lo <= j < hi]
        if all(rho1[j + W] < v for j in out_lo) and all(rho1[j + W] <= v for j in out_hi):
            out.append(k)
    return out


def test_model_accepts_exactly_what_the_rule_accepts():
    """rho with many exact ties, values at the threshold and peaks at the frame edges: the model's stage 1 accepts a
    lag exactly when the rule does, and no lag that it rejects."""
    tau, W, _ = A.acq_params()
    rng = np.random.default_rng(21)
    levels = np.array([0.0, 0.1, tau, 0.3, 0.6], np.float32)
    nf = 3
    accepted = rejected_ties = 0
    for trial in range(400):
        rho1 = np.zeros(LAGS * nf + 2 * W, np.float32)
        # a few values near each frame edge, drawn from few levels so that ties are common
        for e in range(nf + 1):
            c = LAGS * e + W
            lo, hi = max(0, c - 2 * W), min(rho1.size, c + 2 * W)
            rho1[lo:hi] = rng.choice(levels, hi - lo, p=[0.3, 0.2, 0.15, 0.2, 0.15])
        if trial % 3 == 0:                                             # a peak inside the frame too
            rho1[W + LAGS + int(rng.integers(0, LAGS))] = levels[int(rng.integers(2, 5))]
        for f in range(nf):
            want = acceptable(rho1, f, tau, W)
            assert len(want) <= 1
            got = stage1(rho1, f, tau, W)
            assert ([] if got is None else [got]) == want, (trial, f, got, want)
            accepted += len(want)
            lo = LAGS * f
            ks = lo + int(np.argmax(rho1[lo + W:lo + LAGS + W]))
            out = [j for j in range(ks - W, ks + W + 1) if j != ks and not lo <= j < lo + LAGS]
            if rho1[ks + W] >= tau and any(rho1[j + W] == rho1[ks + W] for j in out):
                rejected_ties += not want
    assert accepted >= 100 and rejected_ties >= 50

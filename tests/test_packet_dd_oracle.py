"""CPU: the specification of packet mode's decision-directed equalizer (SC_FLAG_PACKET_DD, tests/packet_dd_ref.c).

1. The C spec (float32, one rounding per operation) against a float64 model of the same algorithm on the same grids.
2. Bit error rates on loop-back from the spec's packet-mode transmitter, over all 496 bits of the aligned packets.
   Carrier offsets are applied to the grid only (grids64: the receiver's mixer off by the offset, positions found at
   0 Hz), because the reference's detection rarely finds a packet at +-20 Hz.  Measured with these seeds when the
   thresholds were set (BER, aligned packets):
     clean 0 Hz 0.0096 (75), +20 Hz 0.0094 (75), -20 Hz 0.0103 (75); frames 0..6 clean 0 Hz 0.0018
     sigma 1500 LSB +10 Hz 0.0140 (54), -10 Hz 0.0133 (54)
     the reference's equalizer on the same packets, clean 0 Hz: 0.338
   Of the 358 bit errors clean at 0 Hz, 290 are in the last four data symbols, whose pulses the transmitter emits
   only in part (tests/packet_dd_ref.c).
3. Silence, full scale and near silence give finite outputs and defined bits.
"""
import numpy as np
import pytest

from packet_dd_ref import (PACKET_SYMS, aligned, dd_model64, dd_packet, ext_run_stream_dd, grids64, kalman_packet,
                           loop_streams)


@pytest.fixture(scope="module")
def loops(oracle):
    """per sigma: (samples, tx bits, starts, spec runs) of 20 streams x 12 packets"""
    out = {}
    for sigma, seed in ((0.0, 7001), (1500.0, 7002)):
        x, txb, starts = loop_streams(oracle, np.random.default_rng(seed), 20, 12, sigma)
        out[sigma] = (x, txb, starts, [ext_run_stream_dd(x[s]) for s in range(x.shape[0])])
    return out


def errors(loop, foffset, equalizer=None):
    """bit errors [aligned, 496] of the aligned packets with the grids rebuilt at foffset"""
    x, txb, starts, runs = loop
    e = equalizer or (lambda g: dd_packet(g)[0])
    errs = []
    for s, (_, _, pk, _, _) in enumerate(runs):
        a = aligned(pk, starts[s])
        k = np.nonzero(a >= 0)[0]
        for g, kk in zip(grids64(x[s], pk[k], foffset), k):
            errs.append(e(g) != txb[s, a[kk]])
    return np.array(errs)


def test_spec_agrees_with_the_float64_model(loops):
    n = agree = total = 0
    for sigma in loops:
        _, _, _, runs = loops[sigma]
        for _, _, pk, psym, grids in runs:
            for g, z in zip(grids, psym):
                bI, bQ, y = dd_model64(g)
                big_r, big_i = np.abs(y.real) > 1e-3, np.abs(y.imag) > 1e-3
                assert np.array_equal(bI[big_r], (z.real < 0)[big_r])
                assert np.array_equal(bQ[big_i], (z.imag < 0)[big_i])
                assert np.abs(z - y).max() < 1e-2
                agree += int((bI == (z.real < 0)).sum() + (bQ == (z.imag < 0)).sum())
                total += 496
                n += 1
    assert n >= 50 and agree == total


def test_spec_run_keeps_the_packet_list(oracle, loops):
    """the same calls, stats, positions and matches as the reference-equalizer packet mode; grids are the spec's S"""
    from oracle import pyoracle as po
    x, _, _, runs = loops[1500.0]
    for s in range(x.shape[0]):
        bits, stats, pk, psym, grids = runs[s]
        rbits, rstats, rpk = po.ext_run_stream(oracle, x[s], max_packets=x.shape[1] // 1880)
        assert bits.tobytes() == rbits.tobytes() and stats.tobytes() == rstats.tobytes()
        for f in ("call", "max_index", "matches", "timing"):
            assert np.array_equal(pk[f], rpk[f]), f
        for g, p, z in zip(grids, pk, psym):
            b, cost, zz = dd_packet(g)
            assert np.array_equal(b, p["bits"]) and np.float32(cost).view(np.uint32) == p["cost"].view(np.uint32)
            assert np.array_equal(zz.view(np.uint32), z.view(np.uint32))
            assert np.array_equal(kalman_packet(g), rpk["bits"][list(rpk["call"]).index(p["call"])])


@pytest.mark.parametrize("sigma,foffset,limit", [(0.0, 0.0, 0.02), (0.0, 20.0, 0.02), (0.0, -20.0, 0.02),
                                                 (1500.0, 10.0, 0.03), (1500.0, -10.0, 0.03)])
def test_bit_error_rate(loops, sigma, foffset, limit):
    e = errors(loops[sigma], foffset)
    assert len(e) >= 50
    assert e.mean() <= limit, e.mean()


def test_first_seven_frames_and_the_reference_equalizer(loops):
    e = errors(loops[0.0], 0.0)
    assert e[:, :7 * 62].mean() <= 0.01
    r = errors(loops[0.0], 0.0, kalman_packet)
    assert r.mean() >= 0.20


@pytest.mark.parametrize("kind", ["silence", "full_scale", "near_silence"])
def test_degenerate_grids(kind):
    rng = np.random.default_rng(3)
    if kind == "silence":
        g = np.zeros(PACKET_SYMS, np.complex64)
    elif kind == "full_scale":
        g = (np.sign(rng.standard_normal(PACKET_SYMS)) + 1j * np.sign(rng.standard_normal(PACKET_SYMS))) * 1e4
    else:
        g = (rng.standard_normal(PACKET_SYMS) + 1j * rng.standard_normal(PACKET_SYMS)) * 1e-20
    bits, cost, z = dd_packet(np.asarray(g, np.complex64))
    assert np.isfinite(z).all() and np.isfinite(cost)
    assert set(np.unique(bits)) <= {0, 1}
    if kind == "silence":
        assert (z == 0).all() and cost == np.float32(2 * 248)

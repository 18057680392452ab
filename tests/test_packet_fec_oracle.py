"""CPU: the specification of the packet code (tests/packet_fec_ref.c) against its numpy model -- CRC, interleaver,
encoder, LLRs and the Viterbi decoder's maximum-likelihood property -- its behaviour on degenerate LLRs, the payloads
it delivers through the acquisition spec's loop-back, and the entry points' argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_fec_ref as F  # noqa: E402

EPS32 = 2.0 ** -24


def test_crc_check_value():
    assert F.crc16(b"123456789") == 0x29B1 == F.crc16_np(b"123456789")


def test_interleaver_is_a_bijection_and_pads_the_tail():
    p = F.perm()
    assert np.array_equal(p, F.PERM64)
    assert sorted(p.tolist()) == list(range(476))
    rng = np.random.default_rng(1)
    bits = F.encode(rng.integers(0, 256, (500, 27)).astype(np.uint8))
    assert not bits[:, 476:].any()
    assert bits[:, :476].any(axis=0).all()                          # every coded position is used


def test_encoder_equals_the_numpy_model():
    rng = np.random.default_rng(2)
    pay = np.concatenate([rng.integers(0, 256, (10000, 27)), np.zeros((1, 27)), np.full((1, 27), 255)]).astype(np.uint8)
    assert np.array_equal(F.encode(pay), F.encode_np(pay))


def test_keystream_is_the_library_s():
    import singlecarrier_b200 as sc
    assert [int(w) for w in F.keystream()] == [sc.packet_keystream_word(f) for f in range(8)]


def llr64(y):
    """float64 LLRs of blocks complex [n, 248] -> [n, 496], descrambled with the spec's keystream"""
    y = np.asarray(y, np.complex128)
    d = np.where(y.real < 0, -1.0, 1.0) + 1j * np.where(y.imag < 0, -1.0, 1.0)
    v = np.maximum((np.abs(y - d) ** 2).sum(axis=1) / 496.0, 1e-6)[:, None]
    L = np.empty((y.shape[0], 496))
    L[:, 0::2] = 2 * y.imag / v
    L[:, 1::2] = 2 * y.real / v
    ks = F.keystream()
    flip = np.array([(int(ks[k // 62]) >> (k % 62)) & 1 for k in range(496)], bool)
    L[:, flip] = -L[:, flip]
    return L


def test_llrs_match_float64():
    """|L - L64| <= 1e-5 |L64|: S is a sum of 248 non-negative terms over a chain of at most 13 adds, so its float32
    error is ~16 ulps; the divide and the e2 terms add a few more."""
    rng = np.random.default_rng(3)
    for sd in (0.05, 0.3, 1.0, 3.0):
        y = ((1 - 2 * rng.integers(0, 2, (200, 248))) + 1j * (1 - 2 * rng.integers(0, 2, (200, 248)))) * 0.9
        y = (y + sd * (rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape))).astype(np.complex64)
        L, L64 = F.llr(y), llr64(y)
        assert np.all(np.abs(L - L64) <= 1e-5 * np.abs(L64))
        nz = y.view(np.float32).reshape(-1, 248, 2)[:, :, ::-1].reshape(-1, 496) != 0
        assert np.array_equal(np.sign(L)[nz], np.sign(L64)[nz])


def test_llr_hard_decisions_are_the_records_bits(oracle):
    """bit == (L < 0) is the DD slicer's decision, descrambled: the spec's LLR signs give the ACQ spec's record bits"""
    from packet_acq_ref import acq_run_stream
    from packet_dd_ref import loop_streams
    x, _, _ = loop_streams(oracle, np.random.default_rng(4), 2, 3, sigma=1200.0)
    for s in range(2):
        pk, psym, _ = acq_run_stream(x[s])
        assert len(pk)
        L = F.llr(psym)
        nz = L != 0
        assert np.array_equal((L < 0)[nz], pk["bits"].astype(bool)[nz])


def test_noiseless_codewords_decode_exactly():
    rng = np.random.default_rng(5)
    pay = rng.integers(0, 256, (300, 27)).astype(np.uint8)
    for scale in (1.0, 1e-30, 3e5, 1e38):
        L = ((1 - 2.0 * F.encode(pay)) * scale).astype(np.float32)
        L[:, 476:] = 0.0
        d = F.decode(L)
        assert np.array_equal(d["data"], pay) and d["crc_ok"].all() and not d["flipped"].any() and \
            not d["reserved"].any()


def noisy_llrs(rng, n, sd):
    pay = rng.integers(0, 256, (n, 27)).astype(np.uint8)
    bits = F.encode(pay)
    L = ((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2)
    return pay, bits, L.astype(np.float32)


def test_viterbi_is_maximum_likelihood_and_agrees_with_float64():
    """On noisy LLRs the decoded path's float64 correlation is >= the transmitted codeword's; the spec decodes what the
    float64 model decodes except where the two paths' float64 correlations lie within the float32 metrics' rounding
    (476 adds of terms bounded by sum |L'|); the record's fields are those of the decoded path."""
    rng = np.random.default_rng(6)
    differ = 0
    for sd in (0.6, 0.8, 1.0, 1.3):
        pay, bits, L = noisy_llrs(rng, 400, sd)
        d, u, pm = F.decode(L, path=True)
        assert not u[:, 232:].any()
        c = F.code_bits(u)
        bound = 2 * 476 * EPS32 * np.abs(L.astype(np.float64)).sum(axis=1)
        corr = F.correlation64(L, c)
        assert np.all(corr >= F.correlation64(L, bits[:, F.PERM64]) - bound)
        assert np.all(np.abs(corr - pm[:, 0]) <= bound)                 # the survivor into state 0 is the path
        u64, pm64 = F.viterbi64(L)
        same = (u64 == u).all(axis=1)
        assert np.all(same | (np.abs(pm64[:, 0] - corr) <= bound))
        differ += int((~same).sum())
        assert np.array_equal(d["data"], np.packbits(u[:, :216], axis=1))
        crc = np.array([F.crc16_np(row.tobytes()) for row in d["data"]])
        rx = np.packbits(u[:, 216:232], axis=1).astype(np.int64)
        assert np.array_equal(d["crc_ok"], (crc == (rx[:, 0] << 8 | rx[:, 1])).astype(np.uint8))
        assert np.array_equal(d["flipped"], ((L[:, F.PERM64] < 0) != c.astype(bool)).sum(axis=1))
        assert not d["reserved"].any()
    assert differ <= 2


def test_viterbi_ties_and_degenerate_llrs():
    """All-zero LLRs: every comparison ties, so b = 0 at every state and the path is all zeros (CRC of 27 zero bytes is
    not 0: crc_ok = 0).  Integer LLRs (many ties) agree with the float64 model exactly.  NaN, +-Inf and 1e38 decode as
    their sanitised values (0, 0, 2^24)."""
    d, u, _ = F.decode(np.zeros((1, 496), np.float32), path=True)
    assert not u.any() and not d["data"].any() and d["crc_ok"][0] == 0 and d["flipped"][0] == 0
    rng = np.random.default_rng(7)
    L = rng.integers(-2, 3, (300, 496)).astype(np.float32)
    d, u, _ = F.decode(L, path=True)
    u64, _ = F.viterbi64(L)
    assert np.array_equal(u, u64)                                        # small integers: exact in both
    pay, bits, L = noisy_llrs(rng, 200, 0.8)
    bad = L.copy()
    idx = rng.integers(0, 496, (200, 40))
    vals = np.array([np.nan, np.inf, -np.inf, 1e38, -1e38], np.float32)
    bad[np.arange(200)[:, None], idx] = vals[rng.integers(0, 5, idx.shape)]
    clean = np.where(np.isfinite(bad), bad, 0).astype(np.float32)
    clean = np.clip(clean, -2.0 ** 24, 2.0 ** 24).astype(np.float32)
    a, b = F.decode(bad, path=True), F.decode(clean, path=True)
    assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1])
    assert np.isfinite(a[2][:, 0]).all()
    allbad = np.array([[np.nan] * 496, [np.inf] * 496, [1e38] * 496, [-1e38] * 496], np.float32)
    d = F.decode(allbad)
    assert d[:2].tobytes() == F.decode(np.zeros((2, 496), np.float32)).tobytes()


def delivered(oracle, n_streams, n_packets, sigma, foff, seed):
    """loop-back through the ACQ spec: -> (packets sent, records aligned to a packet, of those crc_ok with the payload
    sent, crc_ok with another payload)"""
    from packet_acq_ref import acq_run_stream
    x, pay, starts = F.coded_streams(oracle, np.random.default_rng(seed), n_streams, n_packets, sigma=sigma)
    aligned = good = wrong = 0
    for s in range(n_streams):
        pk, psym, _ = acq_run_stream(x[s], foffset=foff)
        if not len(pk):
            continue
        d = F.decode(F.llr(psym))
        for p, r in zip(pk, d):
            dist = np.abs(starts[s] - (int(p["grid_sample"]) - 48))
            if dist.min() > 10:
                wrong += int(r["crc_ok"])                                # a record of no packet that passes the CRC
                continue
            j = int(dist.argmin())
            aligned += 1
            ok = np.array_equal(r["data"], pay[s, j])
            good += int(r["crc_ok"] and ok)
            wrong += int(r["crc_ok"] and not ok)
    return n_streams * n_packets, aligned, good, wrong


@pytest.mark.parametrize("foff", [0.0, 20.0, -20.0, 40.0, -40.0])
def test_loopback_clean_delivers_every_packet(oracle, foff):
    sent, aligned, good, wrong = delivered(oracle, 6, 4, 0.0, foff, 21)
    assert aligned == good == sent and wrong == 0


def test_loopback_noisy_delivery(oracle):
    """sigma = 1,500 LSB at +-10 Hz, 2 x 12 streams x 4 packets: delivered share measured 1.000 (96 of 96, every
    packet found once, every one with crc_ok and its payload); the threshold sits just below."""
    tot = good = wrong = 0
    for foff, seed in ((10.0, 22), (-10.0, 23)):
        sent, aligned, g, w = delivered(oracle, 12, 4, 1500.0, foff, seed)
        tot, good, wrong = tot + sent, good + g, wrong + w
    print(f"delivered {good} of {tot}")
    assert good / tot >= 0.97 and wrong == 0


def test_no_undetected_error_under_heavy_noise(oracle):
    """sigma = 6,000 LSB (channel Eb/N0 2.6 dB by harness.awgn_sigma), 16 streams x 4 packets, offsets 0 and 15 Hz: the records acquisition
    still finds carry many raw errors; none passes the CRC with a wrong payload."""
    for foff, seed in ((0.0, 24), (15.0, 25)):
        sent, aligned, good, wrong = delivered(oracle, 16, 4, 6000.0, foff, seed)
        print(f"foffset {foff}: {aligned} aligned records, {good} delivered, {wrong} undetected")
        assert wrong == 0


def test_entry_points_reject_bad_arguments_without_a_gpu():
    import singlecarrier_b200 as sc
    L = sc.lib
    ok, mis = C.c_void_p(0x1000), C.c_void_p(0x1004)
    n = C.c_void_p(0x2000)
    assert L.sc_packet_encode_dev(0, None, 1, ok, None) == sc._lib.SC_EINVAL
    assert L.sc_packet_encode_dev(0, ok, 1, None, None) == sc._lib.SC_EINVAL
    assert L.sc_packet_encode_dev(0, ok, -1, ok, None) == sc._lib.SC_EINVAL
    for fn in (L.sc_packet_llr_dev, L.sc_packet_decode_dev):
        assert fn(0, None, 1, n, ok, None) == sc._lib.SC_EINVAL
        assert fn(0, ok, 1, None, ok, None) == sc._lib.SC_EINVAL
        assert fn(0, ok, 1, n, None, None) == sc._lib.SC_EINVAL
        assert fn(0, ok, -1, n, ok, None) == sc._lib.SC_EINVAL
        assert fn(0, mis, 1, n, ok, None) == sc._lib.SC_EINVAL                 # input not 8-byte aligned
    assert L.sc_packet_llr_dev(0, ok, 1, n, mis, None) == sc._lib.SC_EINVAL     # llr not 8-byte aligned
    assert L.sc_packet_decode_dev(0, ok, 1, n, C.c_void_p(0x1002), None) == sc._lib.SC_EINVAL

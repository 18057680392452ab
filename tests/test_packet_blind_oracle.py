"""CPU: blind code detection of the packet code (tests/packet_blind_ref.c, scf_decode_blind) -- one-code masks equal
decode_code, the spec equals the numpy selection model, noiseless codewords decode to their code, the right code is
never lost on noisy LLRs, degenerate and pure-noise LLRs, the loop-back through the acquisition spec with codes that
change packet by packet, and the new entry point's argument checks."""
import ctypes as C
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_blind_ref as B  # noqa: E402
import packet_code_ref as R  # noqa: E402
import packet_fec_ref as F  # noqa: E402

CODES = (0, 1, 2)
MASKS = tuple(range(1, 8))


def random_payloads(rng, n):
    return rng.integers(0, 256, (n, R.PAYLOAD_MAX)).astype(np.uint8)


def decode_all(L):
    """decode_code at the three codes, in parallel chunks (the spec's calls release the GIL)"""
    chunks = np.array_split(np.ascontiguousarray(L, np.float32), max(1, min(8, L.shape[0] // 500)))
    with ThreadPoolExecutor(8) as ex:
        return [np.concatenate(list(ex.map(lambda x: R.decode_code(c, x), chunks))) for c in CODES]


def awgn_llrs(rng, code, bits, ebn0_db):
    """BPSK over AWGN at Eb/N0 per transmitted bit: LLR = 2 y / sigma^2 (sigma^2 = 1 / (2 Eb/N0)), on the N
    transmitted positions"""
    sigma2 = 1.0 / (2.0 * 10.0 ** (ebn0_db / 10.0))
    y = (1 - 2.0 * bits) + np.sqrt(sigma2) * rng.standard_normal(bits.shape)
    L = (2.0 * y / sigma2).astype(np.float32)
    unused = np.ones(496, bool)
    unused[F.PERM64[:R.CODE_CODED[code]]] = False
    L[:, unused] = 0.0
    return L


def hard_llrs(code, bits, scale):
    L = ((1 - 2.0 * bits) * scale).astype(np.float32)
    unused = np.ones(496, bool)
    unused[F.PERM64[:R.CODE_CODED[code]]] = False
    L[:, unused] = 0.0
    return L


def llr_sets(rng):
    """noiseless, noisy, random and adversarial LLRs of every code"""
    sets = []
    for c in CODES:
        bits = R.encode_code(c, random_payloads(rng, 200))
        sets.append(hard_llrs(c, bits, 2.0))
        for db in (0.0, 2.0, 4.0):
            sets.append(awgn_llrs(rng, c, bits, db))
    sets.append(rng.standard_normal((300, 496)).astype(np.float32) * 3)
    sets.append(rng.integers(-2, 3, (300, 496)).astype(np.float32))             # many exact ties
    bad = rng.standard_normal((200, 496)).astype(np.float32)
    k = rng.integers(0, 496, (200, 40))
    bad[np.arange(200)[:, None], k] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e38, -1e38, 2e7], np.float32),
                                                 k.shape)
    sets.append(bad)
    sets.append(np.zeros((4, 496), np.float32))
    return sets


def test_one_code_mask_equals_decode_code():
    rng = np.random.default_rng(200)
    for L in llr_sets(rng):
        for c in CODES:
            assert B.decode_blind(1 << c, L).tobytes() == R.decode_code(c, L).tobytes()


def test_spec_equals_the_numpy_selection_model():
    rng = np.random.default_rng(201)
    for L in llr_sets(rng):
        recs = decode_all(L)
        for mask in MASKS:
            assert B.decode_blind(mask, L).tobytes() == B.select_np(mask, recs).tobytes(), mask


@pytest.mark.parametrize("code", CODES)
def test_noiseless_codewords_decode_to_their_code(code):
    rng = np.random.default_rng(210 + code)
    pay = random_payloads(rng, 100)
    bits = R.encode_code(code, pay)
    nb = R.CODE_BYTES[code]
    for scale in (1.0, 1e-30, 3e5, 1e38):
        L = hard_llrs(code, bits, scale)
        for mask in (m for m in MASKS if (m >> code) & 1):
            d = B.decode_blind(mask, L)
            assert (d["code"] == code).all() and d["crc_ok"].all() and not d["flipped"].any(), (scale, mask)
            assert np.array_equal(d["data"][:, :nb], pay[:, :nb]) and not d["data"][:, nb:].any()


def test_noisy_llrs_the_right_code_is_never_lost():
    """At Eb/N0 0, 2, 4 and 8 dB (BPSK over AWGN, 1,000 payloads per code): no record where the transmitted code's
    decode passes its CRC and blind decoding returns another record; no wrong-code decode passes; flipped / N of the
    right code falls to 0 while the wrong codes' stays above 0.04 -- which is why it can break ties.  A wrong-code
    decode passes its CRC with probability about 2^-16: 24,000 of them give 0.4 expected passes, bounded here at 4."""
    rng = np.random.default_rng(220)
    stats, wrong_total, two_total = {}, 0, 0
    for db in (0.0, 2.0, 4.0, 8.0):
        for c in CODES:
            pay = random_payloads(rng, 1000)
            L = awgn_llrs(rng, c, R.encode_code(c, pay), db)
            recs = decode_all(L)
            d = B.decode_blind(7, L)
            right = recs[c]["crc_ok"] == 1
            assert d.tobytes() == B.select_np(7, recs).tobytes()
            assert (d[right]["code"] == c).all() and (d[right].tobytes() == recs[c][right].tobytes())
            wrong = [o for o in CODES if o != c]
            wrong_pass = sum(int(recs[o]["crc_ok"].sum()) for o in wrong)
            two = int((sum(recs[o]["crc_ok"].astype(int) for o in CODES) >= 2).sum())
            fr = recs[c]["flipped"] / R.CODE_CODED[c]
            fw = min(float((recs[o]["flipped"] / R.CODE_CODED[o]).min()) for o in wrong)
            stats[(db, c)] = (int(right.sum()), wrong_pass, two, float(np.median(fr)), fw)
            wrong_total, two_total = wrong_total + wrong_pass, two_total + two
            if db >= 4.0:
                assert right.mean() >= 0.99 and fw > 0.04 and np.median(fr) < 0.02
            if db >= 8.0:
                assert np.median(fr) == 0.0
    print("(Eb/N0, code): right passes, wrong-code passes, two codes passing, median flipped/N right, "
          "min flipped/N wrong:", stats)
    assert wrong_total <= 4 and two_total <= wrong_total


@pytest.mark.parametrize("mask", MASKS)
def test_zero_llrs_give_the_lowest_code(mask):
    d = B.decode_blind(mask, np.zeros((2, 496), np.float32))
    low = min(c for c in CODES if (mask >> c) & 1)
    assert (d["code"] == low).all() and not d["crc_ok"].any() and not d["flipped"].any() and not d["data"].any()


def test_non_finite_and_huge_llrs():
    """NaN, +-Inf and 1e38 decode as their sanitised values (0, 0, +-2^24) at every candidate, so they neither crash
    the selection nor drive it"""
    rng = np.random.default_rng(230)
    bits = R.encode_code(np.arange(300) % 3, random_payloads(rng, 300))
    L = (((1 - 2.0 * bits) + 0.8 * rng.standard_normal(bits.shape)) * 3.0).astype(np.float32)
    idx = rng.integers(0, 496, (300, 40))
    vals = np.array([np.nan, np.inf, -np.inf, 1e38, -1e38], np.float32)
    L[np.arange(300)[:, None], idx] = vals[rng.integers(0, 5, idx.shape)]
    clean = np.clip(np.where(np.isfinite(L), L, 0), -2.0 ** 24, 2.0 ** 24).astype(np.float32)
    allbad = np.array([[np.nan] * 496, [np.inf] * 496, [-np.inf] * 496, [1e38] * 496, [-1e38] * 496], np.float32)
    for mask in MASKS:
        assert B.decode_blind(mask, L).tobytes() == B.decode_blind(mask, clean).tobytes()
        d = B.decode_blind(mask, allbad)
        low = min(c for c in CODES if (mask >> c) & 1)
        assert (d["code"][:3] == low).all() and not d["crc_ok"][:3].any()
        assert d[3:].tobytes() == B.decode_blind(mask, np.clip(allbad[3:], -2.0 ** 24, 2.0 ** 24)).tobytes()


def test_pure_noise_crc_passes_stay_near_three_times_two_to_the_minus_16():
    """120,000 records of Gaussian LLRs: each of the three candidates passes a garbage CRC with probability about
    2^-16, so blind decoding passes about 3 x 2^-16 of them (5.5 expected); a fixed seed, a bound at 16"""
    rng = np.random.default_rng(240)
    L = (rng.standard_normal((120000, 496)) * 2.0).astype(np.float32)
    recs = decode_all(L)
    per_code = [int(r["crc_ok"].sum()) for r in recs]
    d = B.select_np(7, recs)
    assert d[:3000].tobytes() == B.decode_blind(7, L[:3000]).tobytes()
    passes = int(d["crc_ok"].sum())
    print("pure noise: CRC passes per code", per_code, "blind", passes, "expected", round(3 * 120000 / 65536, 2))
    assert passes == sum(int(x) for x in (sum(r["crc_ok"].astype(int) for r in recs) > 0)) and passes <= 16


@pytest.mark.parametrize("foff", [0.0, 20.0, -20.0])
def test_loopback_per_packet_codes_delivers_every_packet(oracle, foff):
    """3 streams x 3 packets, packet j of stream s at code (s + j) mod 3, through the acquisition spec: every packet
    is delivered at its code by blind decoding, nothing else passes its CRC"""
    from packet_acq_ref import acq_run_stream
    codes = (np.arange(3)[:, None] + np.arange(3)[None, :]) % 3
    x, pay, starts = B.coded_streams_packet_code(oracle, np.random.default_rng(250), codes)
    good = wrong = 0
    for s in range(3):
        pk, psym, _ = acq_run_stream(x[s], foffset=foff)
        d = B.decode_blind(7, F.llr(psym))
        for p, r in zip(pk, d):
            dist = np.abs(starts[s] - (int(p["grid_sample"]) - 48))
            j = int(dist.argmin())
            ok = dist.min() <= 10 and r["code"] == codes[s, j] and np.array_equal(r["data"], pay[s, j])
            good += int(r["crc_ok"] and ok)
            wrong += int(r["crc_ok"] and not ok)
    assert good == 9 and wrong == 0


def test_entry_point_rejects_bad_arguments_without_a_gpu():
    import singlecarrier_b200 as sc
    dec, E = sc.lib.sc_packet_decode_blind_dev, sc._lib.SC_EINVAL
    ok, n = C.c_void_p(0x1000), C.c_void_p(0x2000)
    assert dec(0, None, 1, n, 7, ok, None) == E
    assert dec(0, ok, 1, None, 7, ok, None) == E
    assert dec(0, ok, 1, n, 7, None, None) == E
    assert dec(0, ok, -1, n, 7, ok, None) == E
    for mask in (0, 8, 9, 15, 0x80000001):
        assert dec(0, ok, 1, n, mask, ok, None) == E, mask
    assert dec(0, C.c_void_p(0x1004), 1, n, 7, ok, None) == E             # llr not 8-byte aligned
    assert dec(0, ok, 1, n, 7, C.c_void_p(0x1002), None) == E             # out not 4-byte aligned

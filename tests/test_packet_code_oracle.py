"""CPU: the code rates of the packet code (tests/packet_code_ref.c, scf_encode_code / scf_decode_code) -- sizes,
puncturing maps, layout and free distances; the encoder against its numpy model; code 0 equal to the rate-1/2 spec;
exact and maximum-likelihood decoding, degenerate LLRs, the loop-back through the acquisition spec, and the new entry
points' argument checks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_code_ref as R  # noqa: E402
import packet_fec_ref as F  # noqa: E402

EPS32 = 2.0 ** -24
CODES = (0, 1, 2)


def random_payloads(rng, n):
    """uint8 [n, 41]: B random bytes, then random bytes the code ignores"""
    return rng.integers(0, 256, (n, R.PAYLOAD_MAX)).astype(np.uint8)


def test_sizes():
    import singlecarrier_b200 as sc
    assert [sc.payload_bytes(c) for c in (-1, 0, 1, 2, 3, 255)] == [0, 27, 36, 41, 0, 0]
    assert sc.PAYLOAD_EX_DTYPE == R.PAYLOAD_EX_DTYPE and sc.PAYLOAD_MAX == 41
    assert (sc.CODE_R12, sc.CODE_R23, sc.CODE_R34) == CODES
    for c, (b, t, n) in enumerate(((27, 238, 476), (36, 310, 465), (41, 350, 467))):
        assert R.code_sizes(c) == (b, t, n) and t == 8 * b + 22 and sc.payload_bytes(c) == b
    assert R.code_sizes(3) == (0, 0, 0)


@pytest.mark.parametrize("code", CODES)
def test_puncturing_map_keeps_the_pattern(code):
    m = R.mother_map(code)
    B, T, N = R.code_sizes(code)
    assert m.size == N and np.all(np.diff(m) > 0) and m[-1] < 2 * T
    pat = R.PATTERNS[code]
    kept = {2 * t + i for t in range(T) for i in (0, 1) if pat[t % len(pat)][i]}
    assert set(m.tolist()) == kept
    assert np.array_equal(m, R.mother_map_np(code))


@pytest.mark.parametrize("code", CODES)
def test_layout_zero_outside_the_transmitted_positions(code):
    rng = np.random.default_rng(40 + code)
    bits = R.encode_code(code, random_payloads(rng, 500))
    N = R.code_sizes(code)[2]
    used = np.zeros(496, bool)
    used[F.PERM64[:N]] = True
    assert not bits[:, ~used].any()
    assert bits[:, used].any(axis=0).all()


def test_free_distances():
    assert [R.free_distance(c) for c in CODES] == [10, 6, 5]


@pytest.mark.parametrize("code", CODES)
def test_encoder_equals_the_numpy_model(code):
    rng = np.random.default_rng(50 + code)
    pay = np.concatenate([random_payloads(rng, 10000), np.zeros((1, 41)), np.full((1, 41), 255)]).astype(np.uint8)
    assert np.array_equal(R.encode_code(code, pay), R.encode_code_np(code, pay))
    # the bytes past B do not matter
    other = pay.copy()
    other[:, R.CODE_BYTES[code]:] ^= 0x5A
    assert np.array_equal(R.encode_code(code, other), R.encode_code(code, pay))


def test_invalid_codes_encode_zero_and_decode_to_the_empty_record():
    rng = np.random.default_rng(60)
    pay = random_payloads(rng, 4)
    assert not R.encode_code(np.array([3, 7, 200, 255], np.uint8), pay).any()
    d = R.decode_code(np.array([3, 7, 200, 255], np.uint8), rng.standard_normal((4, 496)).astype(np.float32))
    assert d["code"].tolist() == [3, 7, 200, 255]
    assert not d["data"].any() and not d["crc_ok"].any() and not d["flipped"].any()
    assert not d["reserved0"].any() and not d["reserved1"].any()


def test_code0_equals_the_rate_half_spec():
    rng = np.random.default_rng(61)
    pay = random_payloads(rng, 400)
    assert np.array_equal(R.encode_code(0, pay), F.encode(pay[:, :27]))
    bits = F.encode(pay[:, :27])
    sets = [((1 - 2.0 * bits) * 3.0).astype(np.float32), rng.standard_normal((300, 496)).astype(np.float32)]
    for sd in (0.6, 1.0, 1.5):
        sets.append((((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2)).astype(np.float32))
    sets.append(rng.integers(-2, 3, (300, 496)).astype(np.float32))
    for L in sets:
        a, ua, pa = F.decode(L, path=True)
        b, ub, pb = R.decode_code(0, L, path=True)
        assert np.array_equal(a["data"], b["data"][:, :27]) and not b["data"][:, 27:].any()
        assert np.array_equal(a["crc_ok"], b["crc_ok"]) and np.array_equal(a["flipped"], b["flipped"])
        assert not b["code"].any() and not b["reserved0"].any() and not b["reserved1"].any()
        assert np.array_equal(ua, ub[:, :238]) and np.array_equal(pa.view(np.uint32), pb.view(np.uint32))


def hard_llrs(code, bits, scale=1.0):
    L = ((1 - 2.0 * bits) * scale).astype(np.float32)
    N = R.code_sizes(code)[2]
    unused = np.ones(496, bool)
    unused[F.PERM64[:N]] = False
    L[:, unused] = 0.0
    return L


def check_exact(code, d, pay):
    B = R.CODE_BYTES[code]
    assert np.array_equal(d["data"][:, :B], pay[:, :B]) and not d["data"][:, B:].any()
    assert d["crc_ok"].all() and (d["code"] == code).all()


@pytest.mark.parametrize("code", CODES)
def test_noiseless_codewords_decode_exactly(code):
    rng = np.random.default_rng(70 + code)
    pay = random_payloads(rng, 200)
    bits = R.encode_code(code, pay)
    for scale in (1.0, 1e-30, 3e5, 1e38):
        d = R.decode_code(code, hard_llrs(code, bits, scale))
        check_exact(code, d, pay)
        assert not d["flipped"].any()


@pytest.mark.parametrize("code", (1, 2))
def test_single_and_double_hard_errors_decode_exactly(code):
    """free distance >= 5: every single flipped hard bit, and 2,000 random pairs, are corrected"""
    rng = np.random.default_rng(80 + code)
    N = R.code_sizes(code)[2]
    pos = F.PERM64[:N]
    pay = random_payloads(rng, 1)
    L0 = hard_llrs(code, R.encode_code(code, pay))
    L = np.repeat(L0, N, axis=0)
    L[np.arange(N), pos] *= -1
    d = R.decode_code(code, L)
    check_exact(code, d, np.repeat(pay, N, axis=0))
    assert (d["flipped"] == 1).all()
    pays = random_payloads(rng, 2000)
    L = hard_llrs(code, R.encode_code(code, pays))
    a = rng.integers(0, N, 2000)
    b = (a + rng.integers(1, N, 2000)) % N
    L[np.arange(2000), pos[a]] *= -1
    L[np.arange(2000), pos[b]] *= -1
    d = R.decode_code(code, L)
    check_exact(code, d, pays)
    assert (d["flipped"] == 2).all()


@pytest.mark.parametrize("code", CODES)
def test_viterbi_is_maximum_likelihood_and_agrees_with_float64(code):
    """On noisy LLRs the decoded path's float64 correlation is >= the transmitted codeword's; the spec decodes what a
    float64 Viterbi decodes except within the float32 metrics' rounding of a tie; the record is the decoded path's."""
    rng = np.random.default_rng(90 + code)
    B, T, N = R.code_sizes(code)
    m = R.mother_map(code)
    differ = 0
    for sd in (0.5, 0.7, 0.9, 1.2):
        pay = random_payloads(rng, 300)
        bits = R.encode_code(code, pay)
        L = (((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2)).astype(np.float32)
        d, u, pm = R.decode_code(code, L, path=True)
        u = u[:, :T]
        assert not u[:, 8 * B + 16:].any()
        c = R.mother_bits(u)
        bound = 2 * 2 * T * EPS32 * np.abs(L.astype(np.float64)).sum(axis=1)
        corr = R.correlation64_code(code, L, c)
        sent = R.mother_bits(R.info_bits_code(code, pay))
        assert np.all(corr >= R.correlation64_code(code, L, sent) - bound)
        assert np.all(np.abs(corr - pm[:, 0]) <= bound)
        u64, pm64 = R.viterbi64_code(code, L)
        same = (u64 == u).all(axis=1)
        assert np.all(same | (np.abs(pm64[:, 0] - corr) <= bound))
        differ += int((~same).sum())
        assert np.array_equal(d["data"][:, :B], np.packbits(u[:, :8 * B], axis=1))
        crc = np.array([F.crc16_np(row.tobytes()) for row in d["data"][:, :B]])
        rx = np.packbits(u[:, 8 * B:8 * B + 16], axis=1).astype(np.int64)
        assert np.array_equal(d["crc_ok"], (crc == (rx[:, 0] << 8 | rx[:, 1])).astype(np.uint8))
        Lm = R.mother_llrs64(code, L)
        assert np.array_equal(d["flipped"], ((Lm[:, m] < 0) != c[:, m].astype(bool)).sum(axis=1))
    assert differ <= 2


@pytest.mark.parametrize("code", CODES)
def test_degenerate_llrs(code):
    """All-zero LLRs decode to the all-zero path; NaN, +-Inf and 1e38 decode as their sanitised values (0, 0, 2^24)."""
    B, T, _ = R.code_sizes(code)
    d, u, _ = R.decode_code(code, np.zeros((1, 496), np.float32), path=True)
    assert not u.any() and not d["data"].any() and d["crc_ok"][0] == 0 and d["flipped"][0] == 0
    rng = np.random.default_rng(100 + code)
    bits = R.encode_code(code, random_payloads(rng, 200))
    L = (((1 - 2.0 * bits) + 0.8 * rng.standard_normal(bits.shape)) * 3.0).astype(np.float32)
    idx = rng.integers(0, 496, (200, 40))
    vals = np.array([np.nan, np.inf, -np.inf, 1e38, -1e38], np.float32)
    L[np.arange(200)[:, None], idx] = vals[rng.integers(0, 5, idx.shape)]
    clean = np.clip(np.where(np.isfinite(L), L, 0), -2.0 ** 24, 2.0 ** 24).astype(np.float32)
    a, b = R.decode_code(code, L, path=True), R.decode_code(code, clean, path=True)
    assert a[0].tobytes() == b[0].tobytes() and np.array_equal(a[1], b[1]) and np.isfinite(a[2][:, 0]).all()
    allbad = np.array([[np.nan] * 496, [np.inf] * 496, [1e38] * 496, [-1e38] * 496], np.float32)
    d = R.decode_code(code, allbad)
    assert d[:2].tobytes() == R.decode_code(code, np.zeros((2, 496), np.float32)).tobytes()
    assert np.isfinite(R.decode_code(code, allbad[2:], path=True)[2][:, 0]).all()


@pytest.mark.parametrize("code", CODES)
@pytest.mark.parametrize("foff", [0.0, 20.0, -20.0])
def test_loopback_clean_delivers_every_packet(oracle, code, foff):
    from packet_acq_ref import acq_run_stream
    B = R.CODE_BYTES[code]
    x, pay, starts = R.coded_streams_code(oracle, np.random.default_rng(110 + code), 3, 3, code)
    good = wrong = 0
    for s in range(3):
        pk, psym, _ = acq_run_stream(x[s], foffset=foff)
        d = R.decode_code(code, F.llr(psym))
        for p, r in zip(pk, d):
            dist = np.abs(starts[s] - (int(p["grid_sample"]) - 48))
            j = int(dist.argmin())
            ok = dist.min() <= 10 and np.array_equal(r["data"][:B], pay[s, j, :B])
            good += int(r["crc_ok"] and ok)
            wrong += int(r["crc_ok"] and not ok)
    assert good == 9 and wrong == 0


def test_entry_points_reject_bad_arguments_without_a_gpu():
    import singlecarrier_b200 as sc
    L, E = sc.lib, sc._lib.SC_EINVAL
    ok, mis, n = C.c_void_p(0x1000), C.c_void_p(0x1004), C.c_void_p(0x2000)
    enc = L.sc_packet_encode_ex_dev
    assert enc(0, None, 1, 1, ok, ok, None) == E
    assert enc(0, ok, 1, 1, None, ok, None) == E
    assert enc(0, ok, 1, 1, ok, None, None) == E
    assert enc(0, ok, -1, 1, ok, ok, None) == E
    assert enc(0, ok, 1, 0, ok, ok, None) == E
    dec = L.sc_packet_decode_ex_dev
    assert dec(0, None, ok, 1, n, ok, 1, ok, None) == E
    assert dec(0, ok, None, 1, n, ok, 1, ok, None) == E
    assert dec(0, ok, ok, 1, None, ok, 1, ok, None) == E
    assert dec(0, ok, ok, 1, n, None, 1, ok, None) == E
    assert dec(0, ok, ok, 1, n, ok, 1, None, None) == E
    assert dec(0, ok, ok, -1, n, ok, 1, ok, None) == E
    assert dec(0, ok, ok, 1, n, ok, -1, ok, None) == E
    assert dec(0, mis, ok, 1, n, ok, 1, ok, None) == E                    # llr not 8-byte aligned
    assert dec(0, ok, ok, 1, n, ok, 1, C.c_void_p(0x1002), None) == E     # out not 4-byte aligned

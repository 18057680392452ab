"""CPU: the restatement's soft output (tests/soft_ref.c on the oracle's primitives) -- the equalizer output of every
data step.

The reference keeps that value local (data_eq() returns only crealf(error)), so it cannot be pinned directly.  It is
tied here to outputs that are pinned, by two exact identities:
  sign: a valid call's raw decisions (its bits XOR the keystream word) are (Re < 0, Im < 0) of its symbols;
  cost: an invalid call's cost is the float32 sequential sum of RN(RN(c - Re) * 0.1f), c = Re < 0 ? -1 : 1.
"""
import numpy as np
import pytest

from helpers import synth_streams
from soft_ref import run_stream_soft

N_DATA = 31


def raw_words(sym):
    """Raw (pre-descrambler) decision words of symbols [..., 31]: bit 2i = Im < 0, bit 2i+1 = Re < 0."""
    sh = 2 * np.arange(N_DATA, dtype=np.uint64)
    q = (sym.imag < 0).astype(np.uint64) << sh
    i = (sym.real < 0).astype(np.uint64) << (sh + np.uint64(1))
    return np.bitwise_or.reduce(q | i, axis=-1)


def packed(bits_rows):
    """bit-per-byte rows [..., 62] -> words"""
    return np.bitwise_or.reduce(bits_rows.astype(np.uint64) << np.arange(62, dtype=np.uint64), axis=-1)


def data_cost(sym):
    """float32 sequential sum over the 31 steps of RN(RN(c - Re) * 0.1f), one rounding per operation."""
    re = np.ascontiguousarray(sym.real, np.float32)
    c = np.where(re < 0, np.float32(-1.0), np.float32(1.0)).astype(np.float32)
    e = ((c - re).astype(np.float32) * np.float32(0.1)).astype(np.float32)
    cost = np.zeros(sym.shape[:-1], np.float32)
    for i in range(N_DATA):
        cost = (cost + e[..., i]).astype(np.float32)
    return cost


def check_identities(sym, stats, bits, keystream):
    """Sign identity on valid calls, cost identity on invalid calls.  Returns (n_valid, n_invalid)."""
    v = stats["valid"].astype(bool)
    ks = np.array([keystream(n) for n in range(len(v))], np.uint64)
    assert np.array_equal(raw_words(sym[v]), packed(bits[v]) ^ ks[v])
    assert np.array_equal(data_cost(sym[~v]).view(np.uint32), stats["cost"][~v].view(np.uint32))
    return int(v.sum()), int((~v).sum())


def streams(gold, oracle):
    x = gold("preamble_qpsk_8k.raw")
    out = [("shipped", x[: 14 * 1880], False, 0.0)]
    g = gold("rx_synth.npz")
    out += [(f"synth{s}", g["samples"][s], False, 0.0) for s in range(g["samples"].shape[0])]
    rng = np.random.default_rng(8080)
    loop = synth_streams(oracle, rng, 12, 12)
    out += [(f"loop{s}", loop[s], s % 3 == 1, 7.5 if s % 3 == 2 else 0.0) for s in range(loop.shape[0])]
    return out


def test_soft_run_equals_run_stream_and_identities_hold(gold, oracle):
    import singlecarrier_b200 as sc
    n_valid = n_invalid = 0
    for name, x, wide, foff in streams(gold, oracle):
        bits, stats = oracle.run_stream(x, wide=wide, foffset=foff)
        sbits, sstats, sym = run_stream_soft(x, wide=wide, foffset=foff)
        assert sbits.tobytes() == bits.tobytes(), name
        assert sstats.tobytes() == stats.tobytes(), name
        assert sym.shape == (x.size // 1880, N_DATA) and np.isfinite(sym).all(), name
        a, b = check_identities(sym, stats, bits, sc.keystream_word)
        n_valid += a
        n_invalid += b
    assert n_valid > 50 and n_invalid > 50


def test_silence_gives_signed_zero_symbols(oracle):
    """Exact zeros: every symbol is +-0, the decisions are 0 and the invalid calls' cost is 31 x 0.1f summed."""
    x = np.zeros(6 * 1880, np.int16)
    bits, stats, sym = run_stream_soft(x)
    assert (sym == 0).all()
    assert (raw_words(sym) == 0).all()
    v = stats["valid"].astype(bool)
    assert np.array_equal(data_cost(sym[~v]).view(np.uint32), stats["cost"][~v].view(np.uint32))


@pytest.mark.parametrize("which", ["valid", "invalid"])
def test_identity_checks_detect_a_changed_symbol(oracle, which):
    """The identities are not vacuous: a flipped sign in a valid call, or a changed Re in an invalid one, is caught."""
    import singlecarrier_b200 as sc
    rng = np.random.default_rng(99)
    for x in synth_streams(oracle, rng, 5, 12):
        bits, stats, sym = run_stream_soft(x)
        v = stats["valid"].astype(bool)
        sel = (v if which == "valid" else ~v)[:, None] & (sym.real != 0)
        if sel.any():
            break
    check_identities(sym, stats, bits, sc.keystream_word)
    k, i = np.argwhere(sel)[0]
    bad = sym.copy()
    bad[k, i] = complex(-sym[k, i].real, sym[k, i].imag) if which == "valid" else sym[k, i] + np.float32(0.25)
    with pytest.raises(AssertionError):
        check_identities(bad, stats, bits, sc.keystream_word)

"""CPU: the soft output of packet mode in the restatement (tests/packet_soft_ref.c, scs_ext_run_stream_soft) -- the
equalizer output of the 248 data steps of every packet.

Packet mode has no counterpart in the reference; its specification is oracle/sc_oracle_ext.c.  That file returns only
the packets' bits and cost, so the symbols are tied to them by two exact identities, as for the ordinary calls
(tests/test_soft_oracle.py):
  sign: data frame f's raw decisions (bits[f] XOR the packet keystream word of frame f) are (Im < 0, Re < 0) of
        symbols 31 f .. 31 f + 30;
  cost: the packet's cost is the float32 sequential sum over all 248 steps of RN(RN(c - Re) * 0.1f),
        c = Re < 0 ? -1 : 1 -- for every packet (each of its data steps is a data_eq()).
"""
import numpy as np
import pytest

from packet_soft_ref import ext_run_stream_soft
from test_soft_oracle import packed, raw_words

N_FRAMES, N_DATA = 8, 31


def packet_raw_words(psym):
    """[n, 248] -> raw decision words [n, 8]"""
    return raw_words(np.asarray(psym).reshape(-1, N_FRAMES, N_DATA))


def packet_words(pk_bits):
    """spec bits (bit per byte) [n, 496] -> words [n, 8]"""
    return packed(np.asarray(pk_bits).reshape(-1, N_FRAMES, 62))


def packet_cost(psym):
    """float32 sequential sum over the 248 steps of RN(RN(c - Re) * 0.1f), one rounding per operation"""
    re = np.ascontiguousarray(np.asarray(psym).reshape(-1, N_FRAMES * N_DATA).real, np.float32)
    c = np.where(re < 0, np.float32(-1.0), np.float32(1.0)).astype(np.float32)
    e = ((c - re).astype(np.float32) * np.float32(0.1)).astype(np.float32)
    cost = np.zeros(re.shape[0], np.float32)
    for i in range(N_FRAMES * N_DATA):
        cost = (cost + e[:, i]).astype(np.float32)
    return cost


def check_packet_identities(psym, words, cost, key):
    """words [n, 8] descrambled bits, cost float32 [n], key: the 8 packet keystream words."""
    assert np.array_equal(packet_raw_words(psym), np.asarray(words, np.uint64) ^ np.asarray(key, np.uint64)[None, :])
    assert np.array_equal(packet_cost(psym).view(np.uint32), np.asarray(cost, np.float32).view(np.uint32))


def spec_key():
    """The LFSR seeded with 0x4A80 per packet and advanced 62 steps per data frame (oracle/channel_ref.py)."""
    from oracle import channel_ref
    return np.array(channel_ref.keystream_words(N_FRAMES), np.uint64)


def packet_loop_streams(oracle, rng, n_streams, n_packets, noise_levels=(0.0, 200.0, 1500.0), gap=903):
    """Loop-back streams from the spec's packet-mode transmitter (pyoracle.ext_tx_packet, scrambled): random lead-in,
    gap zeros between packets, additive noise -> int16 [n, n_frames * 1880]."""
    from oracle import pyoracle as po
    total = ((n_packets * (1880 + gap) + 2000 + 2 * 1880) // 1880) * 1880
    out = np.zeros((n_streams, total), np.int16)
    for s in range(n_streams):
        st = oracle.new_state()
        parts = [np.zeros(int(rng.integers(0, 2000)), np.int16)]
        for _ in range(n_packets):
            parts.append(po.ext_tx_packet(oracle, st, rng.integers(0, 2, 496).astype(np.uint8)))
            parts.append(np.zeros(gap, np.int16))
        x = np.concatenate(parts).astype(np.float64)
        x = np.concatenate([x, np.zeros(max(0, total - x.size))])[:total]
        sigma = noise_levels[s % len(noise_levels)]
        if sigma > 0:
            x = x + rng.normal(0, sigma, total)
        out[s] = np.clip(x, -32767, 32767).round().astype(np.int16)
    return out


def streams(gold, oracle):
    from test_soft_gpu import hard_rows
    x = gold("preamble_qpsk_8k.raw")
    out = [("shipped", x[: 14 * 1880], False, 0.0)]
    g = gold("rx_synth.npz")
    out += [(f"synth{s}", g["samples"][s], False, 0.0) for s in range(g["samples"].shape[0])]
    loop = packet_loop_streams(oracle, np.random.default_rng(4242), 6, 4)
    out += [(f"packet{s}", loop[s], s % 3 == 1, 7.5 if s % 3 == 2 else 0.0) for s in range(loop.shape[0])]
    hard = hard_rows(oracle, 12)
    out += [(f"hard{s}", hard[s], False, 0.0) for s in range(hard.shape[0])]
    return out


def test_packet_keystream_word_is_the_per_packet_lfsr():
    import singlecarrier_b200 as sc
    key = spec_key()
    assert [sc.packet_keystream_word(f) for f in range(N_FRAMES)] == [int(w) for w in key]
    assert sc.packet_keystream_word(0) == sc.keystream_word(0)          # the same seed as the call register
    assert sc.packet_keystream_word(-1) == 0 and sc.packet_keystream_word(8) == 0


def test_packet_soft_run_equals_the_spec_and_identities_hold(gold, oracle):
    from oracle import pyoracle as po
    key = spec_key()
    n_packets = 0
    for name, x, wide, foff in streams(gold, oracle):
        bits, stats, pk = po.ext_run_stream(oracle, x, max_packets=x.size // 1880, wide=wide, foffset=foff)
        obits, ostats = oracle.run_stream(x, wide=wide, foffset=foff)
        sbits, sstats, spk, psym = ext_run_stream_soft(x, wide=wide, foffset=foff)
        assert sbits.tobytes() == bits.tobytes() == obits.tobytes(), name
        assert sstats.tobytes() == stats.tobytes() == ostats.tobytes(), name
        assert len(spk) == len(pk) == int(stats["valid"][2:].sum()), name
        for f in ("call", "max_index", "matches", "timing"):
            assert np.array_equal(spk[f], pk[f]), (name, f)
        assert np.array_equal(spk["bits"], pk["bits"]), name
        assert np.array_equal(spk["cost"].view(np.uint32), pk["cost"].view(np.uint32)), name
        assert psym.shape == (len(pk), N_FRAMES * N_DATA) and np.isfinite(psym).all(), name
        check_packet_identities(psym, packet_words(pk["bits"]), pk["cost"], key)
        n_packets += len(pk)
    assert n_packets > 40


@pytest.mark.parametrize("which", ["sign", "cost"])
def test_packet_identity_checks_detect_a_changed_symbol(oracle, which):
    """The identities are not vacuous: a flipped sign, or a changed Re with the same sign, is caught."""
    x = packet_loop_streams(oracle, np.random.default_rng(17), 1, 3)[0]
    _, _, pk, psym = ext_run_stream_soft(x)
    assert len(pk) > 0
    key = spec_key()
    words = packet_words(pk["bits"])
    check_packet_identities(psym, words, pk["cost"], key)
    k, i = np.argwhere(psym.real != 0)[-1]                                # late in the last packet
    bad = psym.copy()
    re = np.float32(psym[k, i].real)
    bad[k, i] = complex(-re if which == "sign" else re * np.float32(1.5), psym[k, i].imag)
    with pytest.raises(AssertionError):
        check_packet_identities(bad, words, pk["cost"], key)

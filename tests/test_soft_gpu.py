"""GPU: soft output (sc_rx_frames_soft_dev / _host) -- the equalizer output of every data step.

Symbols are compared with the restatement's (tests/soft_ref.c) as uint32, like every other float field; results and
the bank's state must be exactly those of the plain entry points, on every schedule.  At sizes where the restatement
is too slow, the sign and cost identities of tests/test_soft_oracle.py tie the symbols to the results."""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from helpers import compare_results, synth_streams
from soft_ref import run_stream_soft

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

NF = 14


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def oracle_soft(oracle, samples, n_frames, wide=False, foffset=0.0):
    """Every stream through soft_ref.run_stream_soft: (bits[ns, nf, 62], stats[ns, nf], symbols complex64 [ns, nf, 31])."""
    from oracle import pyoracle as po
    ns = samples.shape[0]
    bits = np.zeros((ns, n_frames, 62), np.uint8)
    stats = np.zeros((ns, n_frames), po.STATS_DTYPE)
    sym = np.zeros((ns, n_frames, 31), np.complex64)

    def one(s):
        bits[s], stats[s], sym[s] = run_stream_soft(samples[s, : n_frames * 1880], wide=wide, foffset=foffset)

    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        list(ex.map(one, range(ns)))
    return bits, stats, sym


def u32(sym):
    return np.ascontiguousarray(sym).view(np.uint32)


def hard_rows(oracle, n):
    """Loop-back streams plus the hard rows: silence, a stream that goes dead, near silence, full-scale noise."""
    rng = np.random.default_rng(31337 + n)
    x = synth_streams(oracle, rng, n, NF)
    if n > 10:
        x[7] = 0
        x[8, 5000:] = 0
        x[9] = rng.integers(-3, 4, x.shape[1]).astype(np.int16)
        x[10] = rng.integers(-32768, 32768, x.shape[1]).astype(np.int16)
    return x


def identities(sc, res, sym):
    """On every record: raw decisions (bits XOR keystream) are the signs of the symbols; invalid calls' cost is the
    float32 sum of the data_eq() returns computed from Re."""
    from test_soft_oracle import data_cost, raw_words
    calls = np.unique(res["call_index"])
    ks = {int(c): np.uint64(sc.keystream_word(int(c))) for c in calls}
    kw = np.vectorize(lambda c: ks[int(c)], otypes=[np.uint64])(res["call_index"])
    assert np.array_equal(raw_words(sym), res["bits"] ^ kw)
    inv = res["valid"] == 0
    assert np.array_equal(data_cost(sym[inv]).view(np.uint32), res["cost"][inv].view(np.uint32))
    return int(inv.sum())


# ---- against the restatement -----------------------------------------------------------------------------------------

def cases():
    return ["shipped", "synth", "loop1", "loop37", "loop301", "wide", "foffset", "packet_bank"]


@pytest.mark.parametrize("case", cases())
def test_soft_symbols_equal_the_oracle(sc, oracle, gold, case):
    wide, foff, packet = case == "wide", (7.5 if case == "foffset" else 0.0), case == "packet_bank"
    if case == "shipped":
        samples = gold("preamble_qpsk_8k.raw")[: 14 * 1880].reshape(1, -1).copy()
    elif case == "synth":
        samples = np.ascontiguousarray(gold("rx_synth.npz")["samples"])
    elif case.startswith("loop"):
        samples = hard_rows(oracle, int(case[4:]))
    else:
        samples = hard_rows(oracle, 37)
    nf = samples.shape[1] // 1880
    obits, ostats, osym = oracle_soft(oracle, samples, nf, wide=wide, foffset=foff)
    bank = sc.ModemBank(samples.shape[0], wide=wide, foffset_hz=foff, packet=packet)
    res, sym = bank.rx_frames_soft_host(samples, nf)
    bank.close()
    assert compare_results(res, None, obits, ostats) == []
    assert np.array_equal(u32(sym), u32(osym))
    bank = sc.ModemBank(samples.shape[0], wide=wide, foffset_hz=foff, packet=packet)
    plain, _ = bank.rx_frames_host(samples, nf)
    bank.close()
    assert plain.tobytes() == res.tobytes()
    if case == "shipped":
        assert res["valid"][0].tolist() == [1, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0]
    if case == "loop301":
        assert (sym[7] == 0).all()                                   # silence: +-0 throughout
        assert int(res["valid"].sum()) > 301


# ---- schedules --------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bank301(oracle):
    samples = hard_rows(oracle, 301)
    return samples, oracle_soft(oracle, samples, NF)


def test_every_schedule_gives_the_same_bytes(sc, bank301):
    import torch
    from singlecarrier_b200 import modem as md
    samples, (obits, ostats, osym) = bank301
    ns = samples.shape[0]
    b = sc.ModemBank(ns)
    b.set_option(md.OPT_OVERLAP, md.OVERLAP_OFF)
    plain, _ = b.rx_frames_host(samples, NF)
    b.close()
    assert compare_results(plain, None, obits, ostats) == []
    want_sym = u32(osym)
    dev = torch.from_numpy(samples).cuda()
    options = []
    for overlap in (md.OVERLAP_OFF, md.OVERLAP_ON):
        for tracker in (md.TRACKER_THREAD, md.TRACKER_COOP):
            options.append({md.OPT_OVERLAP: overlap, md.OPT_TRACKER: tracker})
    options.append({md.OPT_FE_SEARCH: md.FE_SEARCH_TCGEN05})
    options.append({md.OPT_H2D_MODE: md.H2D_ROWS, md.OPT_SLAB_PARTS: 3})
    for opt in options:
        for splits in ([NF], [1, 2, 3, 1, 7], [2] * 7):
            bank = sc.ModemBank(ns)
            for k, v in opt.items():
                bank.set_option(k, v)
            parts, f0 = [], 0
            for k in splits:
                parts.append(bank.rx_frames_soft_host(np.ascontiguousarray(samples[:, f0 * 1880:(f0 + k) * 1880]), k))
                f0 += k
            bank.close()
            res = np.concatenate([p[0] for p in parts], axis=1)
            sym = np.concatenate([p[1] for p in parts], axis=1)
            assert res.tobytes() == plain.tobytes(), (opt, splits)
            assert np.array_equal(u32(sym), want_sym), (opt, splits)
        # device entry point, one batch and two
        bank = sc.ModemBank(ns)
        for k, v in opt.items():
            bank.set_option(k, v)
        r = torch.zeros((ns, NF * 32), dtype=torch.uint8, device="cuda")
        s = torch.zeros((ns, NF * 62), dtype=torch.float32, device="cuda")
        bank.rx_frames_soft_dev(dev, NF, r, s)
        torch.cuda.synchronize()
        assert r.cpu().numpy().tobytes() == plain.tobytes(), opt
        assert np.array_equal(s.cpu().numpy().view(np.uint32).reshape(want_sym.shape), want_sym), opt
        bank.reset()
        r.zero_()
        s.zero_()
        bank.rx_frames_soft_dev(dev[:, : 6 * 1880], 6, r[:, : 6 * 32], s[:, : 6 * 62])
        bank.rx_frames_soft_dev(dev[:, 6 * 1880:], NF - 6, r[:, 6 * 32:], s[:, 6 * 62:])
        torch.cuda.synchronize()
        bank.close()
        assert r.cpu().numpy().tobytes() == plain.tobytes(), opt
        assert np.array_equal(s.cpu().numpy().view(np.uint32).reshape(want_sym.shape), want_sym), opt


def test_many_slabs(sc, oracle):
    """17,000 streams: several slabs per pipe on the host entry point, serial and overlapped; the first 300 streams
    against the restatement, every record by the identities, and the two schedules byte for byte."""
    from singlecarrier_b200.modem import OPT_OVERLAP, OVERLAP_OFF, OVERLAP_ON
    rng = np.random.default_rng(2468)
    nf = 7
    base = synth_streams(oracle, rng, 150, nf)
    ns = 17000
    samples = np.empty((ns, base.shape[1]), np.int16)
    for k in range(ns):
        samples[k] = np.roll(base[k % 150], 37 * (k // 150)) // (1 + (k // 150) % 3)
    out = {}
    for mode in (OVERLAP_OFF, OVERLAP_ON):
        bank = sc.ModemBank(ns)
        bank.set_option(OPT_OVERLAP, mode)
        a = bank.rx_frames_soft_host(samples[:, : 3 * 1880].copy(), 3)
        b = bank.rx_frames_soft_host(samples[:, 3 * 1880:].copy(), nf - 3)
        bank.close()
        out[mode] = (np.concatenate([a[0], b[0]], axis=1), np.concatenate([a[1], b[1]], axis=1))
    bank = sc.ModemBank(ns)
    plain, _ = bank.rx_frames_host(samples, nf)
    bank.close()
    for mode in (OVERLAP_OFF, OVERLAP_ON):
        assert out[mode][0].tobytes() == plain.tobytes(), mode
        assert np.array_equal(u32(out[mode][1]), u32(out[OVERLAP_OFF][1])), mode
    identities(sc, plain, out[OVERLAP_ON][1])
    _, _, osym = oracle_soft(oracle, samples[:300], nf)
    assert np.array_equal(u32(out[OVERLAP_ON][1][:300]), u32(osym))


# ---- state, alternation, arguments ------------------------------------------------------------------------------------

def test_state_after_soft_equals_plain_and_batches_alternate(sc, bank301):
    import torch
    samples, (_, _, osym) = bank301
    ns = samples.shape[0]
    a = sc.ModemBank(ns)
    plain, _ = a.rx_frames_host(samples, NF)
    img_plain = a.state_export()
    a.close()
    b = sc.ModemBank(ns)
    res, sym = b.rx_frames_soft_host(samples, NF)
    img_soft = b.state_export()
    assert b.call_index == NF
    b.close()
    assert res.tobytes() == plain.tobytes()
    assert img_soft.tobytes() == img_plain.tobytes()
    # soft, plain, soft (device), plain (device) on one handle: the one-shot results, and the state the same batches
    # leave when all of them are plain
    dev = torch.from_numpy(samples).cuda()
    images, outs = [], []
    for soft in (True, False):
        c = sc.ModemBank(ns)
        if soft:
            r1, s1 = c.rx_frames_soft_host(samples[:, : 3 * 1880].copy(), 3)
        else:
            r1, _ = c.rx_frames_host(samples[:, : 3 * 1880].copy(), 3)
        r2, _ = c.rx_frames_host(samples[:, 3 * 1880: 5 * 1880].copy(), 2)
        rd = torch.zeros((ns, 6 * 32), dtype=torch.uint8, device="cuda")
        sd = torch.zeros((ns, 6, 31), dtype=torch.complex64, device="cuda")
        if soft:
            c.rx_frames_soft_dev(dev[:, 5 * 1880: 11 * 1880], 6, rd, sd)
        else:
            c.rx_frames_dev(dev[:, 5 * 1880: 11 * 1880], 6, rd)
        rp = torch.zeros((ns, 3 * 32), dtype=torch.uint8, device="cuda")
        c.rx_frames_dev(dev[:, 11 * 1880:], 3, rp)
        torch.cuda.synchronize()
        if soft:
            sym_dev = sd.cpu().numpy()
        images.append(c.state_export())
        c.close()
        outs.append(np.concatenate([r1, r2, rd.cpu().numpy().view(sc.RESULT_DTYPE),
                                    rp.cpu().numpy().view(sc.RESULT_DTYPE)], axis=1))
    assert outs[0].tobytes() == plain.tobytes() and outs[1].tobytes() == plain.tobytes()
    assert images[0].tobytes() == images[1].tobytes()
    assert np.array_equal(u32(s1), u32(osym[:, :3]))
    assert np.array_equal(u32(sym_dev), u32(osym[:, 5:11]))


def test_result_stride_null_alignment_and_transfer_bytes(sc, bank301):
    import torch
    samples, (_, _, osym) = bank301
    ns, nf, extra = 40, 5, 3
    x = np.ascontiguousarray(samples[:ns, : nf * 1880])
    want = u32(osym[:ns, :nf])
    stride = nf + extra
    # host: records past n_frames keep their NaN / 0xFF sentinels
    bank = sc.ModemBank(ns)
    h0, d0 = bank.transfer_bytes()
    res = np.zeros((ns, stride), sc.RESULT_DTYPE)
    res.view(np.uint8)[:] = 0xFF
    sym = np.full((ns, stride, 31), np.nan + 1j * np.nan, np.complex64)
    sc._lib.check(sc.lib.sc_rx_frames_soft_host(bank._h, x.ctypes.data, x.shape[1], nf, res.ctypes.data, stride,
                                                sym.ctypes.data))
    h1, d1 = bank.transfer_bytes()
    assert d1 - d0 == ns * nf * (32 + 248)
    bank.rx_frames_host(x, nf)                                      # continues the same bank: calls nf .. 2nf-1
    h2, d2 = bank.transfer_bytes()
    assert d2 - d1 == ns * nf * 32 and h2 - h1 == h1 - h0
    bank.close()
    assert np.array_equal(u32(sym[:, :nf]), want)
    assert (res.view(np.uint8).reshape(ns, stride, 32)[:, nf:] == 0xFF).all()
    assert np.isnan(sym[:, nf:].real).all() and np.isnan(sym[:, nf:].imag).all()
    # device, the same with a stride
    bank = sc.ModemBank(ns)
    dev = torch.from_numpy(x).cuda()
    r = torch.full((ns, stride * 32), 0xFF, dtype=torch.uint8, device="cuda")
    s = torch.full((ns, stride * 62), float("nan"), dtype=torch.float32, device="cuda")
    bank.rx_frames_soft_dev(dev, nf, r, s)
    torch.cuda.synchronize()
    sn = s.cpu().numpy().reshape(ns, stride, 62)
    assert np.array_equal(sn[:, :nf].view(np.uint32).reshape(want.shape), want)
    assert np.isnan(sn[:, nf:]).all()
    assert (r.cpu().numpy().reshape(ns, stride, 32)[:, nf:] == 0xFF).all()
    assert r.cpu().numpy().reshape(ns, stride, 32)[:, :nf].tobytes() == res[:, :nf].tobytes()
    # NULL symbols and a misaligned device pointer: SC_EINVAL, nothing queued, the call index unchanged
    k = bank.call_index
    assert sc.lib.sc_rx_frames_soft_dev(bank._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), stride, None, 0) == -1
    assert sc.lib.sc_rx_frames_soft_host(bank._h, x.ctypes.data, nf * 1880, nf, res.ctypes.data, stride, None) == -1
    assert sc.lib.sc_rx_frames_soft_dev(bank._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), stride,
                                        s.data_ptr() + 4, 0) == -1
    assert bank.call_index == k
    bank.close()


# ---- at scale, no restatement -----------------------------------------------------------------------------------------

@pytest.mark.parametrize("ns", [65536, 1024])
def test_at_scale_soft_equals_plain_and_identities_hold(sc, ns):
    """65,536 streams (above SC_OVERLAP_MAX: serial chain, one thread per stream) and 1,024 (overlapped chains,
    cooperative tracker), config-3 style workload."""
    import torch
    from singlecarrier_b200 import harness
    nf = 6
    bank = sc.ModemBank(ns)
    wl = harness.synthesize(bank, nf * 1880, seed=11, config=3)
    r = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    bank.rx_frames_dev(wl.samples, nf, r)
    bank.reset()
    rs = torch.zeros_like(r)
    s = torch.zeros((ns, nf, 31), dtype=torch.complex64, device="cuda")
    bank.rx_frames_soft_dev(wl.samples, nf, rs, s)
    torch.cuda.synchronize()
    bank.close()
    assert torch.equal(r, rs)
    res = rs.cpu().numpy().view(sc.RESULT_DTYPE)
    sym = s.cpu().numpy()
    n_inv = identities(sc, res, sym)
    assert 0 < n_inv < res.size
    soft = sc.soft_bits(res, sym)
    k = np.arange(62, dtype=np.uint64)
    bits = ((res["bits"][..., None] >> k) & np.uint64(1)).astype(bool)
    nz = soft != 0
    assert np.array_equal(bits[nz], (soft < 0)[nz])
    assert nz.any()

"""GPU: packet-mode acquisition (SC_FLAG_PACKET_ACQ) against its specification (tests/packet_acq_ref.c): the record
set keyed by (stream, grid_sample), bit for bit, with the packet symbols; per-call results identical to a DD bank's;
the same records whatever the batching, entry point, slab split or overlap option; the device BER counter from
grid_sample; the flag checks; and sc_reset."""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from packet_acq_ref import acq_run_stream  # noqa: E402
from test_soft_gpu import u32  # noqa: E402

SC_OPT_SLAB_PARTS, SC_OPT_OVERLAP = 1, 6


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def acq_streams(sc, ns, n_packets, seed, gap=903, lead_max=2783):
    """Streams from the library's packet-mode TX and channel: lead-ins of 0 .. lead_max - 1 samples, offsets uniform in
    +-40 Hz, AWGN 0..1500 LSB, a 2-tap echo on every third stream -> (int16 [ns, n], tx bits [ns, n_packets, 8, 62],
    lead-in [ns])"""
    import torch
    bank = sc.ModemBank(ns, packet=True)
    g = torch.Generator(device="cuda").manual_seed(seed)
    lead = torch.randint(0, lead_max, (ns,), generator=g, device="cuda", dtype=torch.int32)
    echo = (torch.arange(ns, device="cuda") % 3 == 0).float()
    ch = {"df_hz": (torch.rand(ns, generator=g, device="cuda") * 80 - 40).float(),
          "phi_rad": (torch.rand(ns, generator=g, device="cuda") * 6.283).float(),
          "sigma_lsb": (torch.arange(ns, device="cuda") % 4).float() * 500.0,
          "echo_amp": echo * 0.3, "echo_theta": (torch.rand(ns, generator=g, device="cuda") * 6.283).float(),
          "echo_delay": torch.randint(1, 6, (ns,), generator=g, device="cuda", dtype=torch.int32)}
    total = ((n_packets * (1880 + gap) + 2783 + 2 * 1880) // 1880) * 1880
    d_in = torch.empty((ns, total), dtype=torch.int16, device="cuda")
    bits = torch.empty((ns, n_packets, 8, 62), dtype=torch.uint8, device="cuda")
    bank.tx_packets_dev(d_in, n_packets, gap_samples=gap, seed=seed, bits_out=bits, lead_in=lead, channel=ch)
    torch.cuda.synchronize()
    bank.close()
    return d_in.cpu().numpy(), bits.cpu().numpy(), lead.cpu().numpy()


def spec_records(samples):
    ns = samples.shape[0]
    outs = [None] * ns

    def one(s):
        outs[s] = acq_run_stream(samples[s])

    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        list(ex.map(one, range(ns)))
    return outs


def keyed(pk, psym=None):
    out = {}
    for k, p in enumerate(pk):
        key = (int(p["stream"]), int(p["grid_sample"]))
        assert key not in out, key
        out[key] = (p, None if psym is None else psym[k])
    return out


def run(sc, samples, nf, soft=True, parts=None, overlap=None, steps=None):
    bank = sc.ModemBank(samples.shape[0], packet=True, dd=True, acq=True)
    if parts is not None:
        bank.set_option(SC_OPT_SLAB_PARTS, parts)
    if overlap is not None:
        bank.set_option(SC_OPT_OVERLAP, overlap)
    res, pks, syms, f = [], [], [], 0
    for step in steps or [nf]:
        k = min(step, nf - f)
        if k <= 0:
            break
        x = np.ascontiguousarray(samples[:, f * 1880:(f + k) * 1880])
        if soft:
            r, _, p, ps, n = bank.rx_packets_soft_host(x, k, call_symbols=True)
            syms.append(ps)
        else:
            r, p, n = bank.rx_packets_host(x, k)
        assert n == len(p)
        res.append(r)
        pks.append(p)
        f += k
    bank.close()
    return np.concatenate(res, axis=1), np.concatenate(pks), (np.concatenate(syms) if soft else None)


@pytest.mark.gpu
def test_acq_records_equal_the_spec(sc):
    ns, npk = 300, 4
    samples, _, _ = acq_streams(sc, ns, npk, 0xAC)
    nf = samples.shape[1] // 1880
    res, pk, psym = run(sc, samples, nf)
    got = keyed(pk, psym)
    want = {}
    for s, (opk, opsym, _) in enumerate(spec_records(samples)):
        for q, qs in zip(opk, opsym):
            want[(s, int(q["grid_sample"]))] = (q, qs)
    assert set(got) == set(want)
    assert len(want) > ns
    rows = sc.unpack_packet_bits(pk)
    row_of = {(int(p["stream"]), int(p["grid_sample"])): k for k, p in enumerate(pk)}
    for key, (q, qs) in want.items():
        p, ps = got[key]
        assert (int(p["call_index"]), int(p["max_index"]), int(p["matches"])) == \
            (int(q["call"]), int(q["max_index"]), int(q["matches"])), key
        for a, b in (("cost", "cost"), ("acq_metric", "metric"), ("acq_freq_hz", "freq_hz")):
            assert np.float32(p[a]).view(np.uint32) == np.float32(q[b]).view(np.uint32), (key, a)
        assert np.array_equal(rows[row_of[key]].reshape(-1), q["bits"]), key
        assert np.array_equal(u32(ps), u32(qs)), key
    # the ordinary calls are those of a DD bank
    bank = sc.ModemBank(ns, packet=True, dd=True)
    dres, dcsym, _, _, _ = bank.rx_packets_soft_host(samples, nf, call_symbols=True)
    bank.close()
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    ares, acsym, _, _, _ = bank.rx_packets_soft_host(samples, nf, call_symbols=True)
    bank.close()
    assert ares.tobytes() == dres.tobytes() == res.tobytes()
    assert np.array_equal(u32(acsym), u32(dcsym))


@pytest.mark.gpu
def test_acq_records_do_not_depend_on_how_the_batch_is_run(sc):
    import torch
    ns, npk = 130, 4
    samples, _, _ = acq_streams(sc, ns, npk, 0xAD)
    nf = samples.shape[1] // 1880
    res, pk, psym = run(sc, samples, nf)
    ref = keyed(pk, psym)

    def same(res2, pk2, psym2):
        assert res2.tobytes() == res.tobytes()
        got = keyed(pk2, psym2)
        assert set(got) == set(ref)
        for key, (p, ps) in got.items():
            assert p.tobytes() == ref[key][0].tobytes(), key
            if ps is not None:
                assert np.array_equal(u32(ps), u32(ref[key][1])), key

    same(*run(sc, samples, nf, steps=[1] * nf))
    same(*run(sc, samples, nf, steps=[2, 1, 3, 1, 100]))
    same(*run(sc, samples, nf, soft=False))
    same(*run(sc, samples, nf, parts=4))
    same(*run(sc, samples, nf, parts=1))
    for ov in (0, 2):
        same(*run(sc, samples, nf, overlap=ov))
    # the device entry points
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    d_in = torch.from_numpy(samples).cuda()
    cap = len(pk) + 8
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_pk = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    d_ps = torch.zeros(cap * 496, dtype=torch.float32, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int64, device="cuda")
    bank.rx_packets_soft_dev(d_in, nf, d_res, d_pk, d_n, d_ps)
    torch.cuda.synchronize()
    n = int(d_n.item())
    same(d_res.cpu().numpy().view(res.dtype).reshape(res.shape), d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE),
         d_ps.cpu().numpy()[:n * 496].view(np.complex64).reshape(n, 248))
    # sc_reset, then the same batch again
    bank.reset()
    d_n.zero_()
    bank.rx_packets_dev(d_in, nf, d_res, d_pk, d_n)
    torch.cuda.synchronize()
    n = int(d_n.item())
    bank.close()
    same(d_res.cpu().numpy().view(res.dtype).reshape(res.shape), d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE),
         None)


@pytest.mark.gpu
def test_acq_ber_counter_aligns_by_grid_sample(sc):
    import torch
    ns, npk = 200, 4
    samples, txb, lead = acq_streams(sc, ns, npk, 0xAE)
    nf = samples.shape[1] // 1880
    res, pk, _ = run(sc, samples, nf, soft=False)
    counters = torch.zeros(32, dtype=torch.int64, device="cuda")
    d_pk = torch.from_numpy(pk.view(np.uint8).copy()).cuda()
    d_n = torch.tensor([len(pk)], dtype=torch.int64, device="cuda")
    d_res = torch.from_numpy(res.view(np.uint8).copy()).cuda()
    d_tx = torch.from_numpy(txb).cuda()
    d_lead = torch.from_numpy(lead).cuda()
    import ctypes as C
    rc = sc.lib.sc_packet_ber_stats_dev(0, C.c_void_p(d_pk.data_ptr()), len(pk), C.c_void_p(d_n.data_ptr()),
                                        C.c_void_p(d_res.data_ptr()), ns, nf, nf, C.c_void_p(d_tx.data_ptr()), npk,
                                        C.c_void_p(d_lead.data_ptr()), 903, None, 1,
                                        C.c_void_p(counters.data_ptr()), None)
    assert rc == 0
    torch.cuda.synchronize()
    c = counters.cpu().numpy()
    # numpy recount
    rows = sc.unpack_packet_bits(pk).reshape(len(pk), 8, 62)
    n_rec = n_al = n_err = 0
    for k, p in enumerate(pk):
        s, n = int(p["stream"]), int(p["call_index"])
        if not (2 <= n < nf):
            continue
        n_rec += 1
        pos = int(p["grid_sample"]) - 48 - int(lead[s])
        j = (pos + 2783 // 2) // 2783
        if 0 <= j < npk and abs(pos - j * 2783) <= 10:
            n_al += 1
            n_err += int((rows[k] != txb[s, j]).sum())
    assert (c[0], c[1], c[2], c[3]) == (n_rec, n_al, 496 * n_al, n_err)
    assert n_al > ns


@pytest.mark.gpu
def test_acq_flag_needs_packet_and_dd(sc):
    import ctypes
    for flags in (0x10, 0x14, 0x18):
        h = ctypes.c_void_p()
        assert sc.lib.sc_create(ctypes.byref(h), 0, 8, flags, 0.0) == -1 and not h.value
    with pytest.raises(sc.SingleCarrierError):
        sc.ModemBank(8, packet=True, acq=True)
    sc.ModemBank(8, packet=True, dd=True, acq=True).close()

"""GPU: soft output of packet mode (sc_rx_packets_soft_dev / _host) -- the equalizer output of the 248 data steps of
every packet record, and optionally of the 31 of every call.

Packet symbols are compared with the restatement's (tests/packet_soft_ref.c, scs_ext_run_stream_soft) as uint32;
records and results must be those of sc_rx_packets_*, per-call symbols those of sc_rx_frames_soft_*.  At sizes where the
restatement is too slow, the sign and cost identities of tests/test_packet_soft_oracle.py tie the symbols to the
records."""
import ctypes
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from packet_soft_ref import ext_run_stream_soft  # noqa: E402
from test_packet_gpu import gpu_packet_streams  # noqa: E402
from test_packet_soft_oracle import check_packet_identities, spec_key  # noqa: E402
from test_soft_gpu import hard_rows, u32  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def by_key(pk):
    return {(int(p["stream"]), int(p["call_index"])): k for k, p in enumerate(pk)}


def check_against_restatement(sc, samples, pk, psym, wide=False, foffset=0.0):
    """pk / psym sorted by (stream, call) == the restatement's packets of every stream, in order."""
    ns = samples.shape[0]
    outs = [None] * ns

    def one(s):
        outs[s] = ext_run_stream_soft(samples[s], wide=wide, foffset=foffset)

    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        list(ex.map(one, range(ns)))
    rows = sc.unpack_packet_bits(pk)
    k = 0
    for s in range(ns):
        _, _, opk, opsym = outs[s]
        for q, qs in zip(opk, opsym):
            p = pk[k]
            assert (p["stream"], p["call_index"], p["max_index"], p["matches"]) == (s, q["call"], q["max_index"],
                                                                                  q["matches"]), (s, q["call"])
            assert np.float32(p["cost"]).view(np.uint32) == np.float32(q["cost"]).view(np.uint32), (s, q["call"])
            assert np.array_equal(rows[k].reshape(-1), q["bits"]), (s, q["call"])
            assert np.array_equal(u32(psym[k]), u32(qs)), (s, q["call"])
            k += 1
    assert k == len(pk)
    return k


def check_identities_and_soft_bits(sc, pk, psym):
    check_packet_identities(psym, pk["bits"], pk["cost"], spec_key())
    soft = sc.packet_soft_bits(pk, psym)
    bits = ((pk["bits"][..., None] >> np.arange(62, dtype=np.uint64)) & np.uint64(1)).astype(bool)
    nz = soft != 0
    assert np.array_equal(bits[nz], (soft < 0)[nz])


# ---- against the restatement and the plain entry points ---------------------------------------------------------------

@pytest.mark.parametrize("case", ["loop1", "loop70", "loop300", "wide", "foffset", "hard"])
def test_packet_symbols_equal_the_restatement(sc, oracle, case):
    wide, foff = case == "wide", (7.5 if case == "foffset" else 0.0)
    if case == "hard":
        samples = hard_rows(oracle, 37)
    else:
        ns, npk, seed = {"loop1": (1, 3, 1), "loop70": (70, 5, 2), "loop300": (300, 4, 3)}.get(case, (70, 4, 5))
        samples, _, _ = gpu_packet_streams(sc, ns, npk, seed)
    ns, nf = samples.shape[0], samples.shape[1] // 1880
    bank = sc.ModemBank(ns, wide=wide, foffset_hz=foff, packet=True)
    res, csym, pk, psym, n = bank.rx_packets_soft_host(samples, nf, call_symbols=True)
    bank.close()
    assert n == len(pk) == len(psym) and psym.shape[1] == 248
    bank = sc.ModemBank(ns, wide=wide, foffset_hz=foff, packet=True)
    res0, pk0, n0 = bank.rx_packets_host(samples, nf)
    bank.close()
    assert res.tobytes() == res0.tobytes()
    assert n == n0 and pk.tobytes() == pk0.tobytes()
    bank = sc.ModemBank(ns, wide=wide, foffset_hz=foff, packet=True)
    res1, sym1 = bank.rx_frames_soft_host(samples, nf)
    bank.close()
    assert res1.tobytes() == res.tobytes()
    assert np.array_equal(u32(csym), u32(sym1))
    assert check_against_restatement(sc, samples, pk, psym, wide=wide, foffset=foff) == n
    check_identities_and_soft_bits(sc, pk, psym)
    if case == "hard":
        silent = pk["stream"] == 7                                      # zeros train perfectly: valid calls
        assert (csym[7] == 0).all() and silent.any() and (psym[silent] == 0).all()    # silence: +-0 throughout
    if ns >= 70:
        assert n > ns


def test_streaming_equals_one_shot(sc):
    """Frames delivered 1, 2, 3, 5 ... at a time (packets whose frames straddle API calls) == one call."""
    ns, npk = 97, 5
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 11)
    nf = samples.shape[1] // 1880
    a = sc.ModemBank(ns, packet=True)
    res, csym, pk, psym, n = a.rx_packets_soft_host(samples, nf, call_symbols=True)
    a.close()
    b = sc.ModemBank(ns, packet=True)
    parts = []
    f = 0
    for step in [1, 2, 1, 3, 1, 1, 5, 2, 100]:
        k = min(step, nf - f)
        if k <= 0:
            break
        parts.append(b.rx_packets_soft_host(np.ascontiguousarray(samples[:, f * 1880:(f + k) * 1880]), k,
                                            call_symbols=True))
        f += k
    b.close()
    assert np.concatenate([p[0] for p in parts], axis=1).tobytes() == res.tobytes()
    assert np.array_equal(u32(np.concatenate([p[1] for p in parts], axis=1)), u32(csym))
    allp = np.concatenate([p[2] for p in parts])
    alls = np.concatenate([p[3] for p in parts])
    order = np.lexsort((allp["call_index"], allp["stream"]))
    assert allp[order].tobytes() == pk.tobytes() and n == len(pk) > ns
    assert np.array_equal(u32(alls[order]), u32(psym))
    straddle = [int(p["call_index"]) for p in pk if int(p["call_index"]) in (1, 3, 4, 7, 8, 9)]
    assert straddle                                                     # first calls of the later batches


def test_slabs_above_the_packet_scratch(sc):
    """70,000 streams: two slabs on the device entry point, each with several packet passes; records as sets against
    sc_rx_packets_dev, and every record checked by the identities and packet_soft_bits."""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = 70000, 6
    bank = sc.ModemBank(ns, packet=True)
    wl = harness.synthesize(bank, nf * 1880, seed=0x5C0DE5, config=4)
    cap = ns * (nf - 2)
    r0 = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    p0 = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    n0 = torch.zeros(1, dtype=torch.int64, device="cuda")
    bank.rx_packets_dev(wl.samples, nf, r0, p0, n0)
    bank.reset()
    r1 = torch.zeros_like(r0)
    p1 = torch.zeros_like(p0)
    n1 = torch.zeros_like(n0)
    ps = torch.zeros((cap, 248), dtype=torch.complex64, device="cuda")
    bank.rx_packets_soft_dev(wl.samples, nf, r1, p1, n1, ps)
    torch.cuda.synchronize()
    bank.close()
    n = int(n0.item())
    assert int(n1.item()) == n and 0 < n <= cap
    assert torch.equal(r0, r1)
    pk0 = p0[: n * 96].cpu().numpy().view(sc.PACKET_DTYPE)
    pk1 = p1[: n * 96].cpu().numpy().view(sc.PACKET_DTYPE)
    psym = ps[:n].cpu().numpy()
    k0, k1 = by_key(pk0), by_key(pk1)
    assert k0.keys() == k1.keys()
    assert all(pk0[k0[key]].tobytes() == pk1[k1[key]].tobytes() for key in k0)
    assert pk1["stream"].max() >= 65536                                 # the second slab has packets
    check_identities_and_soft_bits(sc, pk1, psym)


# ---- the device entry point -------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bank4000(sc):
    ns, npk = 4000, 3
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 21)
    nf = samples.shape[1] // 1880
    host = sc.ModemBank(ns, packet=True)
    res, csym, pk, psym, n = host.rx_packets_soft_host(samples, nf, call_symbols=True)
    host.close()
    return samples, nf, res, csym, pk, psym, n


@pytest.mark.parametrize("start", [0, 5])
def test_device_entry_capacity_and_counter_offset(sc, bank4000, start):
    """capacity too small (start 0) or a counter that starts at 5 with room for all: every packet is counted, the
    kept blocks pair with their records at the counter's offsets, and nothing outside the kept blocks is written."""
    import torch
    samples, nf, res, csym, pk, psym, n = bank4000
    ns = samples.shape[0]
    cap = n // 2 if start == 0 else n + start
    bank = sc.ModemBank(ns, packet=True)
    d_in = torch.from_numpy(samples).cuda()
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_sym = torch.zeros((ns, nf, 31), dtype=torch.complex64, device="cuda")
    d_pk = torch.full((cap * 96,), 0xAB, dtype=torch.uint8, device="cuda")
    d_ps = torch.full((cap * 496 + 1024,), float("nan"), dtype=torch.float32, device="cuda")
    d_n = torch.full((1,), start, dtype=torch.int64, device="cuda")
    bank.rx_packets_soft_dev(d_in, nf, d_res, d_pk, d_n, d_ps, symbols=d_sym)
    torch.cuda.synchronize()
    bank.close()
    assert int(d_n.item()) == start + n
    assert d_res.cpu().numpy().tobytes() == res.tobytes()
    assert np.array_equal(u32(d_sym.cpu().numpy()), u32(csym))
    got = d_pk.cpu().numpy().reshape(cap, 96)
    gps = d_ps.cpu().numpy()
    assert np.isnan(gps[cap * 496:]).all()                              # the sentinel past capacity * 496 floats
    assert (got[:start] == 0xAB).all() and np.isnan(gps[: start * 496]).all()
    kept = min(n, cap - start)
    recs = got[start:start + kept].reshape(-1).view(sc.PACKET_DTYPE)
    blocks = gps[start * 496:(start + kept) * 496].reshape(kept, 248 * 2).view(np.complex64)
    key = by_key(pk)
    for k in range(kept):
        j = key[(int(recs[k]["stream"]), int(recs[k]["call_index"]))]
        assert recs[k].tobytes() == pk[j].tobytes()
        assert np.array_equal(u32(blocks[k]), u32(psym[j]))
    assert (got[start + kept:] == 0xAB).all() and np.isnan(gps[(start + kept) * 496:]).all()


def test_argument_checks(sc):
    import torch
    ns, nf = 64, 3
    x = np.zeros((ns, nf * 1880), np.int16)
    bank = sc.ModemBank(ns, packet=True)
    dev = torch.from_numpy(x).cuda()
    r = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    p = torch.zeros(ns * nf * 96, dtype=torch.uint8, device="cuda")
    ps = torch.zeros(ns * nf * 496 + 2, dtype=torch.float32, device="cuda")
    n = torch.zeros(1, dtype=torch.int64, device="cuda")
    res = np.zeros((ns, nf), sc.RESULT_DTYPE)
    pk = np.zeros(ns * nf, sc.PACKET_DTYPE)
    nh = np.zeros(1, np.uint64)
    k = bank.call_index
    L = sc.lib
    assert L.sc_rx_packets_soft_dev(bank._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), nf, None, p.data_ptr(), ns * nf,
                                    n.data_ptr(), None, 0) == -1
    assert L.sc_rx_packets_soft_dev(bank._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), nf, None, p.data_ptr(), ns * nf,
                                    n.data_ptr(), ps.data_ptr() + 4, 0) == -1
    assert L.sc_rx_packets_soft_host(bank._h, x.ctypes.data, nf * 1880, nf, res.ctypes.data, nf, None, pk.ctypes.data,
                                     ns * nf, nh.ctypes.data_as(ctypes.POINTER(ctypes.c_uint64)), None) == -1
    assert bank.call_index == k
    # symbols = NULL is accepted (silence: the zero windows train perfectly, so there are packets, all of them +-0)
    assert L.sc_rx_packets_soft_dev(bank._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), nf, None, p.data_ptr(), ns * nf,
                                    n.data_ptr(), ps.data_ptr(), 0) == 0
    torch.cuda.synchronize()
    got = int(n.item())
    assert bank.call_index == k + nf and got > 0 and (ps[: got * 496] == 0).all()
    bank.close()
    plain = sc.ModemBank(ns)
    assert L.sc_rx_packets_soft_dev(plain._h, dev.data_ptr(), nf * 1880, nf, r.data_ptr(), nf, None, p.data_ptr(), ns * nf,
                                    n.data_ptr(), ps.data_ptr(), 0) == -1
    with pytest.raises(sc.SingleCarrierError):
        plain.rx_packets_soft_host(x, nf)                               # needs SC_FLAG_PACKET
    assert plain.call_index == 0
    plain.close()


def test_soft_and_plain_packet_batches_alternate(sc):
    """soft host, plain host, soft device, plain device on one handle == the same batches all plain: results, records,
    and the batch after them (which runs on the state they leave; packet banks have no sc_state_export)."""
    import torch
    ns, npk = 150, 5
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 33)
    nf = samples.shape[1] // 1880
    cuts = [0, 3, 5, 7, 9, nf]
    assert nf > 9
    dev = torch.from_numpy(samples).cuda()
    outs = []
    for soft in (True, False):
        c = sc.ModemBank(ns, packet=True)
        rs, pks = [], []
        for b in range(5):
            f0, f1 = cuts[b], cuts[b + 1]
            k = f1 - f0
            if b in (0, 1, 4):
                x = np.ascontiguousarray(samples[:, f0 * 1880:f1 * 1880])
                if soft and b == 0:
                    r, _, p, _, _ = c.rx_packets_soft_host(x, k)
                else:
                    r, p, _ = c.rx_packets_host(x, k)
            else:
                dr = torch.zeros((ns, k * 32), dtype=torch.uint8, device="cuda")
                dp = torch.zeros(ns * k * 96, dtype=torch.uint8, device="cuda")
                dn = torch.zeros(1, dtype=torch.int64, device="cuda")
                if soft and b == 2:
                    ds = torch.zeros((ns * k, 248), dtype=torch.complex64, device="cuda")
                    c.rx_packets_soft_dev(dev[:, f0 * 1880:f1 * 1880], k, dr, dp, dn, ds)
                else:
                    c.rx_packets_dev(dev[:, f0 * 1880:f1 * 1880], k, dr, dp, dn)
                torch.cuda.synchronize()
                r = dr.cpu().numpy().view(sc.RESULT_DTYPE)
                p = dp.cpu().numpy()[: int(dn.item()) * 96].view(sc.PACKET_DTYPE)
            rs.append(r)
            pks.append(p)
        c.close()
        allp = np.concatenate(pks)
        outs.append((np.concatenate(rs, axis=1), allp[np.lexsort((allp["call_index"], allp["stream"]))]))
    assert outs[0][0].tobytes() == outs[1][0].tobytes()
    assert outs[0][1].tobytes() == outs[1][1].tobytes() and len(outs[0][1]) > ns
    one = sc.ModemBank(ns, packet=True)
    res, pk, _ = one.rx_packets_host(samples, nf)
    one.close()
    assert outs[1][0].tobytes() == res.tobytes() and outs[1][1].tobytes() == pk.tobytes()

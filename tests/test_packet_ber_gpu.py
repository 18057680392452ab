"""Bit errors of packet-mode records on the device (sc_packet_ber_stats_dev, ModemBank.packet_ber_stats,
harness.packet_ber_dev) against a plain loop written from the header, one record at a time: hand-made records that
probe every rule of the header, then the records of real SC_FLAG_PACKET batches, across batches, at scale and reduced
over NCCL ranks.  The argument checks need no GPU."""
import ctypes as C

import numpy as np
import pytest

MASK62 = (1 << 62) - 1
OFFSETS = np.array([-11, -10, -1, 0, 1, 10, 11])


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0
    return m


def tx_words(tx_bits):
    """txword(s, j, f) of the header: tx_bits[s][j][f][0..61] & 1 packed, bit i = byte i.  uint64 [ns, n_packets, 8]."""
    return np.packbits(np.asarray(tx_bits) & 1, axis=-1, bitorder="little").view("<u8")[..., 0]


def packet_ber_expected(pk, n_records, res, n_streams, n_frames, tx_bits, lead, gap, group, n_groups):
    """The counters of sc_packet_ber_stats_dev written from include/singlecarrier_b200.h, one record at a time.
    pk: PACKET_DTYPE records (the first n_records count), res: RESULT_DTYPE [n_streams, >= n_frames]."""
    txw = tx_words(tx_bits)
    n_packets, period = txw.shape[1], 1880 + gap
    c = np.zeros((n_groups, 32), np.int64)
    for p in pk[:n_records]:
        s, n = int(p["stream"]), int(p["call_index"])
        if not (0 <= s < n_streams and 2 <= n < n_frames):
            continue
        g = 0 if group is None else int(group[s])
        if not 0 <= g < n_groups:
            continue
        c[g, 0] += 1
        pos = (n - 2) * 1880 + 5 * int(p["max_index"]) + int(res["rx_timing"][s, n - 2]) - 48
        pos -= 0 if lead is None else int(lead[s])
        for j in range(n_packets):
            if abs(pos - j * period) <= 10:
                c[g, 1] += 1
                c[g, 2] += 496
                total = 0
                for f in range(8):
                    e = ((int(p["bits"][f]) ^ int(txw[s, j, f])) & MASK62).bit_count()
                    c[g, 8 + f] += e
                    c[g, 16 + f] += e > 0
                    total += e
                c[g, 3] += total
                c[g, 24 + min(7, total.bit_length())] += 1
    return c


def hand_made(sc, rng, ns, nf, stride, npk, gap, lead, n_rec):
    """Results and records: a third of the records land on packet starts -1..n_packets at offsets -11..+11 (their
    (stream, call) pairs distinct, rx_timing of call n-2 set to aim them), with a chosen number of flipped bits,
    0..496, and bits 62/63 set at random; the rest are anywhere, including streams -1 and ns and calls 0, 1, nf and
    nf + 1.  Half the streams' transmitted bytes carry high bits."""
    period = 1880 + gap
    res = np.zeros((ns, stride), sc.RESULT_DTYPE)
    res["rx_timing"] = rng.integers(-300, 300, (ns, stride))
    tx_bits = rng.integers(0, 2, (ns, npk, 8, 62)).astype(np.uint8)
    tx_bits[::2] |= rng.integers(0, 128, (len(tx_bits[::2]), npk, 8, 62)).astype(np.uint8) << 1
    pk = np.zeros(n_rec, sc.PACKET_DTYPE)
    pk["stream"] = np.where(rng.random(n_rec) < 0.9, rng.integers(0, ns, n_rec), rng.choice([-1, ns], n_rec))
    pk["call_index"] = np.where(rng.random(n_rec) < 0.9, rng.integers(2, nf, n_rec), rng.choice([0, 1, nf, nf + 1], n_rec))
    pk["max_index"] = rng.integers(-20, 128, n_rec)
    pk["matches"] = rng.integers(0, 129, n_rec)
    pk["cost"] = rng.random(n_rec)
    pk["bits"] = rng.integers(0, 2 ** 63, (n_rec, 8), dtype=np.uint64) * np.uint64(2) + \
        rng.integers(0, 2, (n_rec, 8), dtype=np.uint64)
    # aimed records: distinct (stream, call) pairs
    pairs = rng.choice(ns * (nf - 2), min(n_rec // 3, ns * (nf - 2)), replace=False)
    m = pairs.size
    at = rng.choice(n_rec, m, replace=False)
    s, n = pairs // (nf - 2), 2 + pairs % (nf - 2)
    pk["stream"][at], pk["call_index"][at] = s, n
    j = rng.integers(-1, npk + 1, m)
    off = OFFSETS[rng.integers(0, OFFSETS.size, m)]
    pos = j * period + off
    mi = pk["max_index"][at].astype(np.int64)
    t = pos + 48 + (0 if lead is None else lead[s]) - (n - 2) * 1880 - 5 * mi
    assert np.abs(t).max() < 32768
    res["rx_timing"][s, n - 2] = t
    n_flips = np.where(rng.random(m) < 0.6,
                       rng.choice([0, 0, 0, 1, 2, 3, 4, 7, 8, 15, 16, 31, 32, 63, 64, 65, 100, 495, 496], m),
                       rng.integers(0, 497, m))
    flip = (rng.random((m, 496)).argsort(1) < n_flips[:, None]).astype(np.uint8).reshape(m, 8, 62)
    flips = np.packbits(flip, axis=-1, bitorder="little").view("<u8")[..., 0]
    hi = rng.integers(0, 4, (m, 8)).astype(np.uint64) << np.uint64(62)
    jc = np.clip(j, 0, npk - 1)
    pk["bits"][at] = tx_words(tx_bits)[s, jc] ^ flips ^ hi
    return res, pk, tx_bits


@pytest.mark.gpu
@pytest.mark.parametrize("with_lead", [True, False])
def test_packet_ber_counters_on_hand_made_records(sc, with_lead):
    """Offsets -11..+11 around packet starts -1..n_packets, negative positions, every histogram bin, bits 62/63,
    tx_bytes with high bits, out-of-range streams, calls and groups, result_stride > n_frames, NULL and non-NULL
    lead_in and group, counters that already hold values, more records than the grid has threads, *n_found above and
    below capacity, tx_bits / packets bases that are not 16-byte aligned, and more groups than a block keeps in shared
    memory (128: the counters are then added to global memory directly)."""
    import torch
    rng = np.random.default_rng(70 + with_lead)
    ns, nf, stride, npk, gap, n_groups, n_rec = 6000, 9, 11, 4, 903, 3, 320_000
    assert n_rec > 148 * 8 * 256
    lead = rng.integers(0, 3000, ns) if with_lead else None
    res, pk, tx_bits = hand_made(sc, rng, ns, nf, stride, npk, gap, lead, n_rec)
    group = rng.integers(-1, n_groups + 1, ns)
    n_found = n_rec - 5000                                      # the records after it are junk
    pk[n_found:] = pk[rng.choice(n_found, n_rec - n_found)]     # junk that would count
    want = packet_ber_expected(pk, n_found, res, ns, nf, tx_bits, lead, gap, group, n_groups)
    hist = want[:, 24:].sum(0)
    assert (hist > 0).all() and want[:, 1].sum() > 5_000 and (want[:, 0] > want[:, 1]).all()
    assert want[:, 2].tolist() == (496 * want[:, 1]).tolist() and want[:, 4:8].sum() == 0
    assert want[:, 3].tolist() == want[:, 8:16].sum(1).tolist() and want[:, 1].tolist() == want[:, 24:].sum(1).tolist()

    bank = sc.ModemBank(ns)
    d_res = torch.from_numpy(res.view(np.uint8).reshape(ns, stride * 32)).cuda()
    d_pk = torch.from_numpy(pk.view(np.uint8)).cuda()
    d_tx = torch.from_numpy(tx_bits).cuda()
    d_lead = torch.from_numpy(lead.astype(np.int32)).cuda() if with_lead else None
    d_group = torch.from_numpy(group.astype(np.int32)).cuda()
    d_n = torch.tensor([n_found], dtype=torch.int64, device="cuda")

    def run(packets, n, tx, grp, n_grp, prior=None):
        cnt = torch.zeros((n_grp, 32), dtype=torch.int64, device="cuda") if prior is None else \
            torch.from_numpy(prior.copy()).cuda()
        bank.packet_ber_stats(packets, n, d_res, nf, tx, d_lead, gap, cnt, group=grp, n_groups=n_grp)
        torch.cuda.synchronize()
        return cnt.cpu().numpy() - (0 if prior is None else prior)

    prior = rng.integers(0, 2 ** 40, (n_groups, 32))
    assert run(d_pk, d_n, d_tx, d_group, n_groups, prior).tolist() == want.tolist()
    # group NULL: every stream in group 0
    want0 = packet_ber_expected(pk, n_found, res, ns, nf, tx_bits, lead, gap, None, 1)
    assert run(d_pk, d_n, d_tx, None, 1).tolist() == want0.tolist()
    # 300 groups: the global-memory path
    many = rng.integers(-1, 301, ns)
    want_many = packet_ber_expected(pk, n_found, res, ns, nf, tx_bits, lead, gap, many, 300)
    assert run(d_pk, d_n, d_tx, torch.from_numpy(many.astype(np.int32)).cuda(), 300).tolist() == want_many.tolist()
    # tx_bits at an odd address, packets at an address that is 8 but not 16-byte aligned
    raw_tx = torch.empty(d_tx.numel() + 1, dtype=torch.uint8, device="cuda")
    raw_tx[1:] = d_tx.view(-1)
    odd_tx = raw_tx[1:].view(d_tx.shape)
    raw_pk = torch.empty(d_pk.numel() + 8, dtype=torch.uint8, device="cuda")
    raw_pk[8:] = d_pk
    assert odd_tx.data_ptr() % 16 == 1 and raw_pk[8:].data_ptr() % 16 == 8
    assert run(raw_pk[8:], d_n, odd_tx, d_group, n_groups).tolist() == want.tolist()
    # *n_found > capacity: only the first capacity records count
    cap = n_rec - 7000
    big = torch.tensor([10 ** 12], dtype=torch.int64, device="cuda")
    want_cap = packet_ber_expected(pk, cap, res, ns, nf, tx_bits, lead, gap, group, n_groups)
    assert run(d_pk[:cap * 96], big, d_tx, d_group, n_groups).tolist() == want_cap.tolist()
    bank.close()


def run_packets(sc, bank, wl, nf, stream=None, split=None):
    """Cold-started rx_packets_dev over the workload (in two batches at frame `split`) and packet_ber_stats queued
    behind it on the same CUDA stream, with no synchronisation in between.  Returns (results, records, n_found,
    counters [13, 32]) with the streams grouped by Eb/N0."""
    import torch
    ns = bank.n_streams
    cap = ns * nf
    res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device=wl.samples.device)
    pk = torch.zeros(cap * 96, dtype=torch.uint8, device=wl.samples.device)
    n = torch.zeros(1, dtype=torch.int64, device=wl.samples.device)
    cnt = torch.zeros((13, 32), dtype=torch.int64, device=wl.samples.device)
    group = wl.ebn0_db.to(torch.int32)
    torch.cuda.synchronize(wl.samples.device)
    st = torch.cuda.Stream(wl.samples.device) if stream is None else stream
    bank.reset()
    if split is None:
        bank.rx_packets_dev(wl.samples, nf, res, pk, n, stream=st.cuda_stream)
    else:
        bank.rx_packets_dev(wl.samples, split, res, pk, n, stream=st.cuda_stream)
        bank.rx_packets_dev(wl.samples[:, split * 1880:], nf - split, res[:, split * 32:], pk, n, stream=st.cuda_stream)
    bank.packet_ber_stats(pk, n, res, nf, wl.tx_bits, wl.lead, wl.gap, cnt, group=group, n_groups=13,
                          stream=st.cuda_stream)
    st.synchronize()
    n_found = int(n.item())
    assert n_found <= cap
    return res, pk, n_found, cnt.cpu().numpy()


@pytest.fixture(scope="module")
def loopback(sc):
    """300 streams of harness.synthesize(config=4) on a SC_FLAG_PACKET bank, 42 calls."""
    from singlecarrier_b200 import harness
    ns, nf = 300, 42
    bank = sc.ModemBank(ns, packet=True)
    wl = harness.synthesize(bank, nf * 1880, 0xBE5, config=4)
    yield bank, wl, nf
    bank.close()


@pytest.mark.gpu
def test_packet_ber_end_to_end(sc, loopback):
    """rx_packets_dev -> packet_ber_stats on one CUDA stream == the loop over rx_packets_host's records; the errors are
    the payload bits that differ from the transmitted ones, over the aligned records; harness.packet_ber_dev agrees."""
    from singlecarrier_b200 import harness
    bank, wl, nf = loopback
    ns = bank.n_streams
    res, d_pk, n_found, got = run_packets(sc, bank, wl, nf)
    host = sc.ModemBank(ns, packet=True)
    res_h, pk_h, n_h = host.rx_packets_host(wl.samples.cpu().numpy(), nf)
    host.close()
    assert res.cpu().numpy().tobytes() == res_h.tobytes() and n_found == n_h == len(pk_h) > 100
    tx = wl.tx_bits.cpu().numpy()
    lead = wl.lead.cpu().numpy().astype(np.int64)
    group = wl.ebn0_db.cpu().numpy().astype(np.int64)
    want = packet_ber_expected(pk_h, n_h, res_h, ns, nf, tx, lead, wl.gap, group, 13)
    assert got.tolist() == want.tolist()
    # the same errors by plain bit comparison
    s, c = pk_h["stream"].astype(np.int64), pk_h["call_index"].astype(np.int64)
    pos = (c - 2) * 1880 + 5 * pk_h["max_index"].astype(np.int64) + res_h["rx_timing"][s, c - 2] - 48 - lead[s]
    j = np.rint(pos / (1880 + wl.gap)).astype(np.int64)
    ok = (j >= 0) & (j < wl.n_packets) & (np.abs(pos - j * (1880 + wl.gap)) <= 10)
    errors = int((sc.unpack_packet_bits(pk_h[ok]) != tx[s[ok], j[ok]]).sum())
    assert int(ok.sum()) == got[:, 1].sum() > 100 and errors == got[:, 3].sum() > 0
    h = harness.packet_ber_dev(bank, d_pk[:n_found * 96], torch_n(n_found), res, nf, wl, group=wl.ebn0_db, n_groups=13)
    assert h["records"].tolist() == want[:, 0].tolist() and h["errors"].tolist() == want[:, 3].tolist()
    assert h["frame_errors"].tolist() == want[:, 8:16].tolist()
    assert h["frames_in_error"].tolist() == want[:, 16:24].tolist()
    assert h["error_histogram"].tolist() == want[:, 24:].tolist()
    print(f"packet BER, {ns} streams: {got[:, 1].sum()} aligned of {n_found} records, "
          f"BER {got[:, 3].sum() / got[:, 2].sum():.3f}, PER {1 - got[:, 24].sum() / got[:, 1].sum():.3f}")


def torch_n(n):
    import torch
    return torch.tensor([n], dtype=torch.int64, device="cuda")


@pytest.mark.gpu
def test_packet_ber_across_batches(sc, loopback):
    """Records of two successive rx_packets_dev batches (n_found not reset, results written into one array) give the
    counters of one batch."""
    bank, wl, nf = loopback
    _, _, n1, one = run_packets(sc, bank, wl, nf)
    for split in (3, 20):
        _, _, n2, two = run_packets(sc, bank, wl, nf, split=split)
        assert n2 == n1 and two.tolist() == one.tolist(), split


@pytest.mark.gpu
def test_packet_ber_at_scale(sc):
    """70,000 streams, 13 Eb/N0 groups (config 3): the device counters equal the loop."""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = 70_000, 8
    bank = sc.ModemBank(ns, packet=True)
    wl = harness.synthesize(bank, nf * 1880, 0x5CA1E, config=3)
    res, d_pk, n_found, got = run_packets(sc, bank, wl, nf, stream=torch.cuda.current_stream())
    bank.close()
    pk = d_pk[:n_found * 96].cpu().numpy().view(sc.PACKET_DTYPE)
    want = packet_ber_expected(pk, n_found, res.cpu().numpy().view(sc.RESULT_DTYPE), ns, nf, wl.tx_bits.cpu().numpy(),
                               wl.lead.cpu().numpy().astype(np.int64), wl.gap,
                               wl.ebn0_db.cpu().numpy().astype(np.int64), 13)
    assert got.tolist() == want.tolist()
    assert (got[:, 1] > 0).all() and n_found > 1000


@pytest.mark.gpu
def test_packet_ber_reduced_over_nccl(sc, loopback):
    """One rank (a one-device NcclComm) leaves the counters unchanged; with two GPUs, two half-banks on devices 0 and 1
    reduced with sc_reduce_stats equal the whole bank."""
    import torch
    from singlecarrier_b200 import harness
    bank, wl, nf = loopback
    ns = bank.n_streams
    res, pk, n_found, whole = run_packets(sc, bank, wl, nf)
    n = torch_n(n_found)
    plain = harness.packet_ber_dev(bank, pk, n, res, nf, wl, group=wl.ebn0_db, n_groups=13)
    comm = sc.NcclComm.init_all([0])[0]
    one = harness.packet_ber_dev(bank, pk, n, res, nf, wl, group=wl.ebn0_db, n_groups=13, comm=comm)
    comm.close()
    assert all(np.array_equal(one[k], plain[k]) for k in plain) and plain["records"].tolist() == whole[:, 0].tolist()
    if torch.cuda.device_count() < 2:
        return
    parts = []
    for dev, (lo, hi) in enumerate(((0, ns // 2), (ns // 2, ns))):
        torch.cuda.set_device(dev)
        half = sc.ModemBank(hi - lo, device=dev, packet=True)
        sub = harness.Workload(wl.samples[lo:hi].to(f"cuda:{dev}"), wl.tx_bits[lo:hi].to(f"cuda:{dev}"),
                               wl.lead[lo:hi].to(f"cuda:{dev}"), wl.gap, wl.ebn0_db[lo:hi].to(f"cuda:{dev}"),
                               wl.n_packets)
        _, _, _, cnt = run_packets(sc, half, sub, nf)
        half.close()
        parts.append(torch.from_numpy(cnt).to(f"cuda:{dev}"))
    comms = sc.NcclComm.init_all([0, 1])
    nccl = C.CDLL("libnccl.so.2")                     # one process drives both ranks: the calls must be grouped
    nccl.ncclGroupStart()
    for dev, (cm, p) in enumerate(zip(comms, parts)):
        torch.cuda.set_device(dev)
        cm.all_reduce_counters(p)
    nccl.ncclGroupEnd()
    for dev in (0, 1):
        torch.cuda.synchronize(dev)
    assert parts[0].cpu().tolist() == whole.tolist() == parts[1].cpu().tolist()
    for cm in comms:
        cm.close()
    torch.cuda.set_device(0)


def test_packet_ber_stats_rejects_bad_arguments():
    """SC_EINVAL for every NULL or out-of-range argument, before any CUDA call (so also without a GPU); capacity 0,
    n_streams 0 and n_frames < 3 then launch nothing (SC_OK with a device, SC_ECUDA without one)."""
    import singlecarrier_b200 as sc
    P = 4096                                          # a non-NULL address that is never dereferenced
    ok = dict(device=0, packets=P, capacity=4, n_found=P, results=P, n_streams=2, result_stride=5, n_frames=5,
              tx_bits=P, n_packets=1, lead_in=None, gap=903, group=None, n_groups=1, counters=P, stream=None)

    def call(**kw):
        a = dict(ok, **kw)
        return sc.lib.sc_packet_ber_stats_dev(a["device"], a["packets"], a["capacity"], a["n_found"], a["results"],
                                              a["n_streams"], a["result_stride"], a["n_frames"], a["tx_bits"],
                                              a["n_packets"], a["lead_in"], a["gap"], a["group"], a["n_groups"],
                                              a["counters"], a["stream"])

    bad = [("packets", None), ("n_found", None), ("results", None), ("tx_bits", None), ("counters", None),
           ("capacity", -1), ("n_streams", -1), ("n_frames", -1), ("result_stride", 4), ("n_packets", 0),
           ("n_packets", -3), ("gap", -1), ("n_groups", 0), ("n_groups", -1)]
    for k, v in bad:
        assert call(**{k: v}) == -1, k
        assert b"sc_packet_ber_stats_dev" in sc.lib.sc_last_error()
    empty = 0 if sc.lib.sc_device_count() > 0 else -2
    for k, v in (("capacity", 0), ("n_streams", 0), ("n_frames", 2), ("n_frames", 0)):
        assert call(**{k: v, "result_stride": 5}) == empty, k

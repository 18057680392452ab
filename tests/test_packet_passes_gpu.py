"""GPU: packet mode at the schedule of the bench workload, against its specifications.

run_slab (csrc/sc_api.cu) runs the packet pass every pk_chunk = max(1, 65536 / slab streams) calls, so a slab of more
than 32,768 streams, or a batch longer than pk_chunk calls, has several passes per batch, whose first calls read
frames, timings and (on ACQ banks, one call ahead) phasor tables that earlier passes and the table stream left.  The
bench workload (131,072 streams x 42 calls, two slabs of 65,536) has 42.  Here:

- plain, DD and ACQ banks of 9,000 streams x 14 calls with two passes in a slab, through the device soft and hard
  entries and the host soft entry, equal the same bank fed one call per batch, and a subset of streams equals the
  specification (tests/packet_soft_ref.c, packet_dd_ref.c, packet_acq_ref.c);
- an ACQ bank at the bench shape through rx_packets_soft_dev equals 42 one-call batches, and the spec on 2,048 streams;
- ACQ banks equal the spec on a stream with an exact tie of rho1 between the maximum of a frame and a neighbour in
  the next, and with SC_FLAG_WIDE, a bank foffset_hz, back-to-back packets, packets at the start of the stream and
  packets in (and cut off by) the last two frames;
- the ACQ device entry keeps its capacity and counter offset;
- the tracker and front-end search options do not change a DD or ACQ bank's output.
"""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from packet_acq_ref import acq_run_stream  # noqa: E402
from packet_dd_ref import ext_run_stream_dd  # noqa: E402
from packet_soft_ref import ext_run_stream_soft  # noqa: E402
from test_packet_acq_gpu import acq_streams, keyed  # noqa: E402
from test_packet_gpu import gpu_packet_streams  # noqa: E402
from test_soft_gpu import u32  # noqa: E402

FRAME = 1880
SC_OPT_SLAB_PARTS, SC_OPT_FE_SEARCH, SC_OPT_TRACKER = 1, 4, 5
SC_FE_SEARCH_MMA, SC_FE_SEARCH_TCGEN05 = 1, 2
SC_TRACKER_THREAD, SC_TRACKER_COOP, SC_TRACKER_COOP_MAX = 1, 2, 1024

# ---- the schedule of csrc/sc_api.cu, restated ----------------------------------------------------------------------
PK_CAP, N_PIPE, STAGE_BYTES = 65536, 3, 768 << 20


def pick_slab(n, lo, parts):
    """sc_api.cu pick_slab(): streams per slab."""
    s = max(-(-n // parts), lo)
    return -(-s // 128) * 128


def split(n, slab):
    return [(s0, min(slab, n - s0)) for s0 in range(0, n, slab)]


def dev_slabs(n, parts=0):
    """rx_dev_body: the slabs (first stream, streams) of a packet bank's device entry points"""
    return split(n, min(pick_slab(n, 128 if parts else 8192, parts or 2), PK_CAP))


def host_slabs(n, nf, parts=0):
    """rx_host_body for a packet bank and contiguous streams of nf frames: (slabs, frames per block)"""
    if nf * FRAME * 2 * 128 <= STAGE_BYTES and not parts:
        slab = min(STAGE_BYTES // (nf * FRAME * 2) // 128 * 128, pick_slab(n, 128, 2 * N_PIPE), PK_CAP)
        return split(n, slab), nf
    slab = min(pick_slab(n, 128 if parts else 4096, parts or 2 * N_PIPE), PK_CAP)
    return split(n, slab), max(1, min(nf, STAGE_BYTES // (slab * FRAME * 2)))


def passes(ns, nf):
    """run_slab: the packet passes [j_lo, j_hi) of a block of nf calls on a slab of ns streams"""
    chunk = max(1, PK_CAP // ns)
    return [(j, min(j + chunk, nf)) for j in range(0, nf, chunk)]


NS, NF = 9000, 14
BENCH_NS, BENCH_NF = 131072, 42


def test_the_shapes_run_several_passes():
    """What each shape below runs, by the restated schedule."""
    assert dev_slabs(NS, 1) == [(0, NS)] and passes(NS, NF) == [(0, 7), (7, 14)]
    assert dev_slabs(NS) == [(0, 8192), (8192, 808)] and passes(8192, NF) == [(0, 8), (8, 14)]
    assert host_slabs(NS, NF, 1) == ([(0, NS)], NF)
    slabs, fblk = host_slabs(NS, NF)
    assert fblk == NF and len(slabs) >= 2 and all(len(passes(n, NF)) == 1 for _, n in slabs)
    # the bench shape: two slabs, one pass per call
    assert dev_slabs(BENCH_NS) == [(0, 65536), (65536, 65536)]
    assert passes(65536, BENCH_NF) == [(j, j + 1) for j in range(BENCH_NF)]
    # the one-thread tracker runs in a slab of more than SC_TRACKER_COOP_MAX streams, the cooperative one below
    assert 8192 > SC_TRACKER_COOP_MAX and NS > SC_TRACKER_COOP_MAX and 808 <= SC_TRACKER_COOP_MAX


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def flags(flavour):
    return {"dd": flavour != "plain", "acq": flavour == "acq"}


def canon(pk, psym, acq):
    """records (and their symbols) sorted by (stream, grid_sample) on ACQ banks, (stream, call_index) otherwise;
    the keys are unique"""
    second = pk["grid_sample"] if acq else pk["call_index"].astype(np.int64)
    order = np.lexsort((second, pk["stream"]))
    s, k = pk["stream"][order], second[order]
    assert not ((s[1:] == s[:-1]) & (k[1:] == k[:-1])).any(), "duplicate records"
    return pk[order], (None if psym is None else psym[order])


def assert_same(a, b, acq):
    """(results, call symbols or None, records, packet symbols or None) of two runs"""
    assert a[0].tobytes() == b[0].tobytes()
    if a[1] is not None and b[1] is not None:
        assert np.array_equal(u32(a[1]), u32(b[1]))
    pa, sa = canon(a[2], a[3], acq)
    pb, sb = canon(b[2], b[3], acq)
    assert len(pa) == len(pb) and pa.tobytes() == pb.tobytes()
    if sa is not None and sb is not None:
        assert np.array_equal(u32(sa), u32(sb))


def run_host(sc, samples, nf, flavour, steps=None, options=(), soft=True, wide=False, foffset=0.0):
    """host entry points, the batch cut into steps -> (results, call symbols, records, packet symbols)"""
    bank = sc.ModemBank(samples.shape[0], wide=wide, foffset_hz=foffset, packet=True, **flags(flavour))
    for opt, val in options:
        bank.set_option(opt, val)
    res, csym, pks, psyms, f = [], [], [], [], 0
    for k in steps or [nf]:
        x = samples[:, f * FRAME:(f + k) * FRAME]
        if soft:
            r, c, p, ps, n = bank.rx_packets_soft_host(x, k, call_symbols=True)
            csym.append(c)
            psyms.append(ps)
        else:
            r, p, n = bank.rx_packets_host(x, k)
        assert n == len(p)
        res.append(r)
        pks.append(p)
        f += k
    bank.close()
    return (np.concatenate(res, axis=1), np.concatenate(csym, axis=1) if soft else None, np.concatenate(pks),
            np.concatenate(psyms) if soft else None)


def run_dev(sc, samples, nf, flavour, soft=True, options=()):
    """the device entry points, one batch -> (results, call symbols, records, packet symbols)"""
    import torch
    ns = samples.shape[0]
    bank = sc.ModemBank(ns, packet=True, **flags(flavour))
    for opt, val in options:
        bank.set_option(opt, val)
    cap = ns * nf
    d_in = torch.from_numpy(np.ascontiguousarray(samples[:, :nf * FRAME])).cuda()
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_cs = torch.zeros((ns, nf * 62), dtype=torch.float32, device="cuda")
    d_pk = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    d_ps = torch.zeros(cap * 496, dtype=torch.float32, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int64, device="cuda")
    if soft:
        bank.rx_packets_soft_dev(d_in, nf, d_res, d_pk, d_n, d_ps, symbols=d_cs)
    else:
        bank.rx_packets_dev(d_in, nf, d_res, d_pk, d_n)
    torch.cuda.synchronize()
    bank.close()
    n = int(d_n.item())
    assert n <= cap
    res = d_res.cpu().numpy().view(sc.RESULT_DTYPE).reshape(ns, nf)
    pk = d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE)
    if not soft:
        return res, None, pk, None
    return (res, d_cs.cpu().numpy().view(np.complex64).reshape(ns, nf, 31), pk,
            d_ps.cpu().numpy()[:n * 496].view(np.complex64).reshape(n, 248))


def decided_by(pk, acq):
    """the call that decides each record: call_index, or on ACQ banks frame + 2 with frame = floor((g + 2) / 1880)"""
    if acq:
        return (pk["grid_sample"] + 2) // FRAME + 2
    return pk["call_index"].astype(np.int64)


def spec_subset(pk, acq, layouts, nf):
    """The first and last stream of every slab of every layout, and every stream with a record decided by the first or
    second call of a pass after a slab's first (its frames come from the previous pass).  With a packet every 2,783
    samples nearly every stream has such a record, so this is nearly the whole bank; the spec takes about 0.01 s per
    14-frame stream."""
    must, later = set(), set()
    dec = decided_by(pk, acq)
    for slabs in layouts:
        for s0, n in slabs:
            must |= {s0, s0 + n - 1}
            calls = [j for lo, _ in passes(n, nf)[1:] for j in (lo, lo + 1)]
            sel = (pk["stream"] >= s0) & (pk["stream"] < s0 + n) & np.isin(dec, calls)
            later |= set(pk["stream"][sel].tolist())
    assert len(later) >= 1000, "too few records decided by the first calls of a later pass"
    return sorted(must | later)


def spec_of(flavour, x, wide=False, foffset=0.0):
    """the spec's records of one stream as (call, max_index, matches, cost, metric, freq_hz, bits, symbols) rows"""
    if flavour == "acq":
        opk, opsym, _ = acq_run_stream(x, wide=wide, foffset=foffset)
        return [(q["call"], q["max_index"], q["matches"], q["cost"], q["metric"], q["freq_hz"], q["bits"], qs,
                 q["grid_sample"]) for q, qs in zip(opk, opsym)]
    if flavour == "dd":
        _, _, opk, opsym, _ = ext_run_stream_dd(x, wide=wide, foffset=foffset)
    else:
        _, _, opk, opsym = ext_run_stream_soft(x, wide=wide, foffset=foffset)
    return [(q["call"], q["max_index"], q["matches"], q["cost"], None, None, q["bits"], qs, None)
            for q, qs in zip(opk, opsym)]


def bits32(v):
    return int(np.float32(v).view(np.uint32))


def assert_spec(sc, flavour, samples, streams, pk, psym, wide=False, foffset=0.0):
    """the records of `streams` (pk / psym in any order; samples [len(streams), n] their samples) == the spec's"""
    acq = flavour == "acq"
    outs = [None] * len(streams)

    def one(i):
        outs[i] = spec_of(flavour, samples[i], wide=wide, foffset=foffset)

    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        list(ex.map(one, range(len(streams))))
    pk, psym = canon(pk, psym, acq)
    rows = sc.unpack_packet_bits(pk)
    lo = np.searchsorted(pk["stream"], streams, side="left")
    hi = np.searchsorted(pk["stream"], streams, side="right")
    total = 0
    for i, s in enumerate(streams):
        want = outs[i]
        assert hi[i] - lo[i] == len(want), (s, hi[i] - lo[i], len(want))
        for k, (call, mi, m, cost, metric, hz, b, qs, g) in zip(range(lo[i], hi[i]), want):
            p = pk[k]
            key = (s, int(call))
            assert (int(p["call_index"]), int(p["max_index"]), int(p["matches"])) == (int(call), int(mi), int(m)), key
            assert bits32(p["cost"]) == bits32(cost), key
            if acq:
                assert int(p["grid_sample"]) == int(g), key
                assert bits32(p["acq_metric"]) == bits32(metric) and bits32(p["acq_freq_hz"]) == bits32(hz), key
            assert np.array_equal(rows[k].reshape(-1), b), key
            assert np.array_equal(u32(psym[k]), u32(qs)), key
        total += len(want)
    return total


# ---- several passes per batch ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def streams_9k(sc):
    cache = {}

    def get(flavour):
        if flavour not in cache:
            make = acq_streams if flavour == "acq" else gpu_packet_streams
            x = make(sc, NS, 9, {"plain": 0x9A, "dd": 0x9B, "acq": 0x9C}[flavour])[0]
            assert x.shape[1] >= NF * FRAME
            cache[flavour] = np.ascontiguousarray(x[:, :NF * FRAME])
        return cache[flavour]

    return get


@pytest.mark.gpu
@pytest.mark.parametrize("parts", [1, 0], ids=["one_slab", "default_slabs"])
@pytest.mark.parametrize("flavour", ["plain", "dd", "acq"])
def test_several_passes_per_batch(sc, streams_9k, flavour, parts):
    samples = streams_9k(flavour)
    acq = flavour == "acq"
    opts = [(SC_OPT_SLAB_PARTS, parts)] if parts else []
    ref = run_host(sc, samples, NF, flavour, steps=[1] * NF, options=opts)       # one pass per batch
    assert len(ref[2]) > NS
    assert_same(run_dev(sc, samples, NF, flavour, options=opts), ref, acq)
    assert_same(run_dev(sc, samples, NF, flavour, soft=False, options=opts), ref, acq)
    assert_same(run_host(sc, samples, NF, flavour, options=opts), ref, acq)
    layouts = [dev_slabs(NS, parts), host_slabs(NS, NF, parts)[0]]
    assert max(len(passes(n, NF)) for slabs in layouts for _, n in slabs) >= 2
    streams = spec_subset(ref[2], acq, layouts, NF)
    keep = np.isin(ref[2]["stream"], streams)
    n = assert_spec(sc, flavour, samples[streams], streams, ref[2][keep], ref[3][keep])
    assert n > len(streams) // 2


# ---- the bench shape ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bench_shape_acq_bank(sc):
    """131,072 streams x 42 calls of harness.synthesize(config=4) through rx_packets_soft_dev on an ACQ bank: two
    slabs of 65,536 with one packet pass per call.  One batch == 42 one-call batches after sc_reset, byte for byte;
    the records of 2,048 streams from both slabs == the spec."""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = BENCH_NS, BENCH_NF
    cap = ns * 32                                    # packets are 2,783 samples apart: at most 29 per stream here
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    wl = harness.synthesize(bank, nf * FRAME, seed=0xB5, config=4)
    runs = []
    for steps in ([nf], [1] * nf):
        bank.reset()
        res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
        pk = torch.zeros((cap, 96), dtype=torch.uint8, device="cuda")
        ps = torch.zeros((cap, 496), dtype=torch.float32, device="cuda")
        n = torch.zeros(1, dtype=torch.int64, device="cuda")
        f = 0
        for k in steps:
            bank.rx_packets_soft_dev(wl.samples[:, f * FRAME:(f + k) * FRAME], k, res[:, f * 32:(f + k) * 32], pk, n, ps)
            f += k
        torch.cuda.synchronize()
        runs.append((res, pk, ps, int(n.item())))
    bank.close()
    (res1, pk1, ps1, n1), (res2, pk2, ps2, n2) = runs
    runs.clear()
    assert ns < n1 <= cap and n1 == n2
    assert torch.equal(res1, res2)

    def order(pk, n):
        st = pk[:n, 64:68].contiguous().view(torch.int32).view(-1).long()
        g = pk[:n, 88:96].contiguous().view(torch.int64).view(-1)
        return torch.argsort(st * (1 << 20) + g + 16)

    o1, o2 = order(pk1, n1), order(pk2, n2)
    assert torch.equal(pk1[o1], pk2[o2])
    for c in range(0, n1, 1 << 19):
        a, b = o1[c:c + (1 << 19)], o2[c:c + (1 << 19)]
        assert torch.equal(ps1[a].view(torch.int32), ps2[b].view(torch.int32))
    del pk2, ps2, res2, o2                                     # about 8.3 GB, not needed by the spec phase
    torch.cuda.empty_cache()
    # the spec on 2,048 streams of both slabs, the first and last of each among them
    rng = np.random.default_rng(0xB5)
    picks = np.concatenate([[0, 65535, 65536, 131071], rng.choice(np.arange(1, 65535), 1022, replace=False),
                            rng.choice(np.arange(65537, 131071), 1022, replace=False)])
    streams = np.unique(picks).tolist()
    assert len(streams) == 2048
    host_pk = pk1[:n1].cpu().numpy().reshape(-1).view(sc.PACKET_DTYPE)
    sel = np.nonzero(np.isin(host_pk["stream"], streams))[0]
    psym = ps1[torch.from_numpy(sel).cuda()].cpu().numpy().view(np.complex64).reshape(len(sel), 248)
    samples = wl.samples[torch.tensor(streams, device="cuda")].cpu().numpy()
    n = assert_spec(sc, "acq", samples, streams, host_pk[sel], psym)
    assert n > 10 * len(streams)


# ---- an exact tie across a frame edge -------------------------------------------------------------------------------
@pytest.mark.gpu
def test_acq_exact_tie_across_the_frame_edge(sc):
    """tests/test_packet_acq_model.py's tie_stream: rho1 of lag 750 (frame 1) and lag 753 (frame 2) are bit-equal and
    above tau.  The neighbour test keeps frame 1's lag and drops frame 2's, on both entry points, as the spec does."""
    from test_packet_acq_model import TIE_FRAMES, TIE_K1, tie_stream
    ns = 64
    samples = np.ascontiguousarray(np.repeat(tie_stream()[None], ns, axis=0))
    host = run_host(sc, samples, TIE_FRAMES, "acq")
    assert_same(run_dev(sc, samples, TIE_FRAMES, "acq"), host, True)
    assert assert_spec(sc, "acq", samples, list(range(ns)), host[2], host[3]) == ns
    assert (np.abs(host[2]["grid_sample"] - 5 * TIE_K1) <= 2).all()


# ---- acquisition's inputs -------------------------------------------------------------------------------------------
# (gap, lead-ins 0 .. lead_max - 1, frames kept or None, wide, foffset_hz)
ACQ_CASES = {"gap903": (903, 2783, None, False, 0.0), "gap37": (37, 2783, None, False, 0.0),
             "gap0": (0, 2783, None, False, 0.0), "lead0_60": (903, 61, None, False, 0.0),
             "tail": (0, 1880, 6, False, 0.0), "wide": (903, 2783, None, True, 0.0),
             "foffset": (903, 2783, None, False, 7.5)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ACQ_CASES))
def test_acq_inputs_equal_the_spec(sc, case):
    gap, lead_max, keep, wide, foff = ACQ_CASES[case]
    ns, npk = 200, 6
    samples, _, lead = acq_streams(sc, ns, npk, 0xA0 + list(ACQ_CASES).index(case), gap=gap, lead_max=lead_max)
    if keep is not None:
        # gap 0 puts one packet start in every frame: packets start in the last two frames, which are not searched,
        # and the last one is cut off by the stream's end
        samples = np.ascontiguousarray(samples[:, :keep * FRAME])
        starts = lead[:, None] + (FRAME + gap) * np.arange(npk)[None, :]
        assert (((starts >= (keep - 2) * FRAME) & (starts < keep * FRAME)).sum(axis=1) == 2).all()
    nf = samples.shape[1] // FRAME
    res, csym, pk, psym = run_host(sc, samples, nf, "acq", wide=wide, foffset=foff)
    n = assert_spec(sc, "acq", samples, list(range(ns)), pk, psym, wide=wide, foffset=foff)
    assert n >= ns * (2 if keep else 3)
    if case == "gap0":
        assert n >= 0.9 * ns * (nf - 3)              # a packet in (nearly) every searched frame
    if case == "lead0_60":
        assert (pk["grid_sample"] < 48 + 61 + 3).sum() >= ns // 2      # the packets at the start of the stream
    # the ordinary calls are those of a DD bank with the same filter and offset
    dres, dcsym, _, _ = run_host(sc, samples, nf, "dd", wide=wide, foffset=foff)
    assert res.tobytes() == dres.tobytes() and np.array_equal(u32(csym), u32(dcsym))


# ---- the ACQ device entry's capacity and counter ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("start", [0, 5])
def test_acq_device_entry_capacity_and_counter_offset(sc, start):
    import torch
    ns, npk = 1500, 4
    samples, _, _ = acq_streams(sc, ns, npk, 0xA9)
    nf = samples.shape[1] // FRAME
    res, _, pk, psym = run_host(sc, samples, nf, "acq")
    want = keyed(pk, psym)
    n = len(pk)
    assert n > ns
    cap = n // 2 if start == 0 else n + start
    d_in = torch.from_numpy(samples).cuda()
    for soft in (True, False):
        bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
        d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
        d_pk = torch.full((cap * 96,), 0xAB, dtype=torch.uint8, device="cuda")
        d_ps = torch.full((cap * 496,), float("nan"), dtype=torch.float32, device="cuda")
        d_n = torch.full((1,), start, dtype=torch.int64, device="cuda")
        if soft:
            bank.rx_packets_soft_dev(d_in, nf, d_res, d_pk, d_n, d_ps)
        else:
            bank.rx_packets_dev(d_in, nf, d_res, d_pk, d_n)
        torch.cuda.synchronize()
        bank.close()
        assert int(d_n.item()) == start + n                        # every packet counted, kept or not
        assert d_res.cpu().numpy().tobytes() == res.tobytes()
        got = d_pk.cpu().numpy().reshape(cap, 96)
        gps = d_ps.cpu().numpy()
        assert (got[:start] == 0xAB).all()
        kept = min(n, cap - start)
        recs = got[start:start + kept].reshape(-1).view(sc.PACKET_DTYPE)
        blocks = gps[start * 496:(start + kept) * 496].reshape(kept, 496).view(np.complex64)
        seen = set()
        for k in range(kept):
            key = (int(recs[k]["stream"]), int(recs[k]["grid_sample"]))
            assert key in want and key not in seen, key
            seen.add(key)
            assert recs[k].tobytes() == want[key][0].tobytes()
            if soft:
                assert np.array_equal(u32(blocks[k]), u32(want[key][1]))    # the record's block is its own
        assert (got[start + kept:] == 0xAB).all()
        assert np.isnan(gps[:start * 496]).all() and np.isnan(gps[(start + kept) * 496:]).all()
        if not soft:
            assert np.isnan(gps).all()


# ---- schedule options -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("option", [(SC_OPT_TRACKER, SC_TRACKER_THREAD), (SC_OPT_TRACKER, SC_TRACKER_COOP),
                                    (SC_OPT_FE_SEARCH, SC_FE_SEARCH_MMA), (SC_OPT_FE_SEARCH, SC_FE_SEARCH_TCGEN05)],
                         ids=["tracker_thread", "tracker_coop", "fe_search_mma", "fe_search_tcgen05"])
@pytest.mark.parametrize("flavour", ["dd", "acq"])
def test_schedule_options_keep_packet_output(sc, flavour, option):
    """The device entry runs the 1,300 streams as one slab (the one-thread tracker by default), the host entry as
    slabs of 256 (the cooperative one): each option gives both entries' default output."""
    ns, npk = 1300, 5
    make = acq_streams if flavour == "acq" else gpu_packet_streams
    samples = make(sc, ns, npk, 0xC0 + (flavour == "acq"))[0]
    nf = samples.shape[1] // FRAME
    assert dev_slabs(ns) == [(0, ns)] and ns > SC_TRACKER_COOP_MAX
    assert all(n <= SC_TRACKER_COOP_MAX for _, n in host_slabs(ns, nf)[0])
    acq = flavour == "acq"
    ref = run_host(sc, samples, nf, flavour)
    assert len(ref[2]) > ns
    assert_same(run_dev(sc, samples, nf, flavour), ref, acq)
    assert_same(run_dev(sc, samples, nf, flavour, options=[option]), ref, acq)
    assert_same(run_host(sc, samples, nf, flavour, options=[option]), ref, acq)

"""GPU: the packet code's three kernels against their specification (tests/packet_fec_ref.c) -- encoder bytes, LLRs
and decoded records bit for bit, past one grid pass, on real soft output and adversarial input -- the record count
read on the device, the end-to-end loop-back through DD and ACQ banks, and the kernels' SASS."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_fec_ref as F  # noqa: E402
from test_packet_acq_gpu import acq_streams  # noqa: E402
from test_soft_gpu import u32  # noqa: E402


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def gpu_llr(sc, blocks, n_found=None, capacity=None, sentinel=None):
    """blocks float32 [cap, 496] -> (LLRs [cap, 496] as the kernel left them)"""
    import torch
    cap = blocks.shape[0] if capacity is None else capacity
    d_sym = torch.from_numpy(np.ascontiguousarray(blocks, np.float32)).cuda()
    d_llr = torch.full((blocks.shape[0], 496), np.nan if sentinel is None else sentinel, dtype=torch.float32,
                       device="cuda")
    if sentinel is not None:
        d_llr.view(torch.int32).fill_(int(sentinel))
    d_n = torch.tensor([cap if n_found is None else n_found], dtype=torch.int64, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_llr(d_sym[:cap], d_n, d_llr)
    torch.cuda.synchronize()
    bank.close()
    return d_llr.cpu().numpy()


def gpu_decode(sc, llrs, n_found=None, capacity=None):
    import torch
    cap = llrs.shape[0] if capacity is None else capacity
    d_llr = torch.from_numpy(np.ascontiguousarray(llrs, np.float32)).cuda()
    d_out = torch.full((llrs.shape[0] * 32,), 0xA5, dtype=torch.uint8, device="cuda")
    d_n = torch.tensor([cap if n_found is None else n_found], dtype=torch.int64, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_decode(d_llr[:cap], d_n, d_out)
    torch.cuda.synchronize()
    bank.close()
    return d_out.cpu().numpy().view(sc.PAYLOAD_DTYPE)


@pytest.mark.gpu
def test_encode_equals_the_spec(sc):
    """100,003 payloads: more than one pass of the encoder's 296 x 256 threads"""
    import torch
    rng = np.random.default_rng(31)
    pay = rng.integers(0, 256, (100003, 27)).astype(np.uint8)
    pay[0], pay[1] = 0, 255
    bits = torch.full((100003, 8, 62), 7, dtype=torch.uint8, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_encode(torch.from_numpy(pay).cuda(), bits)
    torch.cuda.synchronize()
    # an unaligned output row takes the byte path
    odd = torch.zeros(1 + 5 * 496, dtype=torch.uint8, device="cuda")
    bank.packet_encode(torch.from_numpy(pay[:5]).cuda(), odd[1:])
    torch.cuda.synchronize()
    bank.close()
    want = F.encode(pay)
    assert np.array_equal(bits.cpu().numpy().reshape(-1, 496), want)
    assert np.array_equal(odd.cpu().numpy()[1:].reshape(5, 496), want[:5])


def acq_soft_batch(sc, ns=300, npk=4, seed=0xF1):
    """a real ACQ soft batch: streams with offsets, noise and echo (test_packet_acq_gpu.acq_streams) -> packet
    symbols float32 [n, 496] of the records found"""
    samples, _, _ = acq_streams(sc, ns, npk, seed)
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    _, _, pk, psym, n = bank.rx_packets_soft_host(samples, samples.shape[1] // 1880)
    bank.close()
    assert n == len(pk) > ns
    return psym.view(np.float32).reshape(-1, 496)


@pytest.mark.gpu
def test_llrs_equal_the_spec_on_soft_output_and_adversarial_blocks(sc):
    y = acq_soft_batch(sc)
    assert np.array_equal(u32(gpu_llr(sc, y)), u32(F.llr(y)))
    rng = np.random.default_rng(32)
    specials = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1e30, -1e30, 1e-45, -1e-45, 1e-40, 1.0, -1.0, 3e38],
                        np.float32)
    adv = [np.zeros(496), np.full(496, -0.0), np.full(496, np.nan), np.full(496, np.inf), np.full(496, 1e30),
           np.full(496, 1e-40), rng.choice([-1.0, 1.0], 496), np.tile([1.0, -1.0], 248), np.full(496, 3e38)]
    for _ in range(40):
        b = rng.standard_normal(496) * 10.0 ** rng.uniform(-3, 3)
        k = rng.integers(0, 496, 30)
        b[k] = rng.choice(specials, 30)
        adv.append(b)
    adv = np.array(adv, np.float32)
    assert np.array_equal(u32(gpu_llr(sc, adv)), u32(F.llr(adv)))


@pytest.mark.gpu
def test_blocks_past_the_record_count_are_untouched(sc):
    rng = np.random.default_rng(33)
    y = rng.standard_normal((64, 496)).astype(np.float32)
    want = F.llr(y)
    sentinel = 0x7fc0dead
    for n_found, cap in ((20, 50), (80, 50), (0, 50), (50, 50)):
        got = gpu_llr(sc, y, n_found=n_found, capacity=cap, sentinel=sentinel)
        k = min(n_found, cap)
        assert np.array_equal(u32(got[:k]), u32(want[:k]))
        assert (got[k:].view(np.uint32) == sentinel).all()
        llr = np.where(np.isfinite(want), want, 0).astype(np.float32)
        dec = gpu_decode(sc, llr, n_found=n_found, capacity=cap)
        assert dec[:k].tobytes() == F.decode(llr[:k]).tobytes()
        assert (dec[k:].view(np.uint8) == 0xA5).all()


@pytest.mark.gpu
def test_decode_equals_the_spec(sc):
    rng = np.random.default_rng(34)
    y = acq_soft_batch(sc, ns=200, seed=0xF2)
    sets = [F.llr(y)]
    for sd in (0.4, 0.8, 1.2, 2.0):                                   # noisy codewords
        bits = F.encode(rng.integers(0, 256, (500, 27)).astype(np.uint8))
        sets.append((((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2)).astype(np.float32))
    sets.append(rng.integers(-3, 4, (500, 496)).astype(np.float32))  # ties
    sets.append(np.zeros((3, 496), np.float32))
    bad = rng.standard_normal((200, 496)).astype(np.float32)
    k = rng.integers(0, 496, (200, 30))
    bad[np.arange(200)[:, None], k] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e38, -1e38, 2e7], np.float32),
                                                 k.shape)
    sets.append(bad)
    sets.append(np.full((2, 496), np.nan, np.float32))
    for L in sets:
        assert gpu_decode(sc, L).tobytes() == F.decode(L).tobytes()
    # past one grid pass (148 x 16 blocks x 8 records)
    bits = F.encode(rng.integers(0, 256, (20011, 27)).astype(np.uint8))
    L = (((1 - 2.0 * bits) + 0.9 * rng.standard_normal(bits.shape)) * 2.5).astype(np.float32)
    assert gpu_decode(sc, L).tobytes() == F.decode(L).tobytes()


def fec_run(sc, bank, wl, nf, cap):
    """sc_rx_packets_soft_dev -> sc_packet_llr_dev -> sc_packet_decode_dev on one stream, no host sync between"""
    import torch
    ns = bank.n_streams
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_pk = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    d_ps = torch.zeros((cap, 496), dtype=torch.float32, device="cuda")
    d_llr = torch.zeros((cap, 496), dtype=torch.float32, device="cuda")
    d_out = torch.zeros(cap * 32, dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int64, device="cuda")
    bank.reset()
    bank.rx_packets_soft_dev(wl.samples, nf, d_res, d_pk, d_n, d_ps)
    bank.packet_llr(d_ps, d_n, d_llr)
    bank.packet_decode(d_llr, d_n, d_out)
    torch.cuda.synchronize()
    n = min(int(d_n.item()), cap)
    return d_res, d_pk, n, d_ps.cpu().numpy()[:n], d_llr.cpu().numpy()[:n], d_out.cpu().numpy()[:n * 32]


def record_rows(sc, d_pk, n, d_res, nf, wl, decoded):
    """numpy recount, record by record: (stream, aligned, raw errors over coded bits 0..475, crc_ok, payload equal)
    for every record with call index 2..nf-1; alignment by the rule of sc_packet_ber_stats_dev"""
    ns, n_packets = wl.lead.shape[0], wl.n_packets
    pk = d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE)
    res = d_res.cpu().numpy().view(sc.RESULT_DTYPE).reshape(ns, nf)
    lead, payh = wl.lead.cpu().numpy(), wl.payload.cpu().numpy()
    txb = wl.tx_bits.cpu().numpy().reshape(ns, n_packets, 496)
    rows = sc.unpack_packet_bits(pk).reshape(n, 496)
    out = []
    for k, p in enumerate(pk):
        s, call = int(p["stream"]), int(p["call_index"])
        if not 2 <= call < nf:
            continue
        gs = int(p["grid_sample"])
        pos = (gs if gs else (call - 2) * 1880 + 5 * int(p["max_index"]) + int(res[s, call - 2]["rx_timing"])) \
            - 48 - int(lead[s])
        j = (pos + 2783 // 2) // 2783
        if not (0 <= j < n_packets and abs(pos - j * 2783) <= 10):
            out.append((s, False, 0, False, False))
            continue
        e = int((rows[k][:476] != txb[s, j][:476]).sum())
        out.append((s, True, e, bool(decoded[k]["crc_ok"]), np.array_equal(decoded[k]["data"], payh[s, j])))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("acq", [False, True])
def test_end_to_end_clean_delivers_every_aligned_record(sc, acq):
    """config 2 (clean channel, +-20 Hz): every aligned record that the DD loop decoded with a raw BER below 0.2 is
    delivered, and no record passes the CRC with another payload.  On the ACQ bank that is every aligned record.  On
    the DD bank (grids from the reference's per-call detection, loop started from nu = 0) one of the 162 aligned
    records is a packet on which the DD loop lost lock: raw errors per data frame 5, 10, 17, 27, 32, 31, 32, 21 (175 of
    476), beyond any rate-1/2 code; it is flagged by crc_ok = 0."""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = 256, 14
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=acq)
    n_packets = (nf * 1880 + 2782) // 2783
    g = torch.Generator().manual_seed(35)
    pay = torch.randint(0, 256, (ns, n_packets, 27), generator=g, dtype=torch.uint8).cuda()
    wl = harness.synthesize(bank, nf * 1880, seed=35, config=2, payload=pay)
    d_res, d_pk, n, psym, llr, out = fec_run(sc, bank, wl, nf, ns * nf)
    bank.close()
    dec = out.view(sc.PAYLOAD_DTYPE)
    assert out.tobytes() == F.decode(F.llr(psym)).tobytes()
    c = harness.packet_fec(d_pk, n, out, d_res, nf, wl)
    print({k: int(v.sum()) for k, v in c.items()})
    rows = [r for r in record_rows(sc, d_pk, n, d_res, nf, wl, dec) if r[1]]
    assert len(rows) == c["aligned"][0] > (ns if acq else 100)  # the per-call detection misses most offset packets
    held = [r for r in rows if r[2] <= 0.2 * 476]
    assert all(r[3] and r[4] for r in held)
    assert c["undetected"][0] == 0 and c["correct"][0] == c["crc_ok"][0] == sum(r[3] and r[4] for r in rows)
    assert len(rows) - len(held) <= (0 if acq else 1)


@pytest.mark.gpu
def test_recount_equals_the_spec_decode(sc):
    """config 3 (AWGN 0..12 dB): the device's LLRs and records equal the spec's on the batch's packet symbols, and
    harness.packet_fec counts what a numpy recount of the spec's decode gives"""
    from singlecarrier_b200 import harness
    ns, nf = 260, 14
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    n_packets = (nf * 1880 + 2782) // 2783
    import torch
    g = torch.Generator().manual_seed(36)
    pay = torch.randint(0, 256, (ns, n_packets, 27), generator=g, dtype=torch.uint8).cuda()
    wl = harness.synthesize(bank, nf * 1880, seed=36, config=3, payload=pay)
    group = (torch.arange(ns, device="cuda") % 13).int()
    d_res, d_pk, n, psym, llr, out = fec_run(sc, bank, wl, nf, ns * nf)
    bank.close()
    assert np.array_equal(u32(llr), u32(F.llr(psym)))
    spec = F.decode(llr)
    assert out.tobytes() == spec.tobytes()
    c = harness.packet_fec(d_pk, n, out, d_res, nf, wl, group=group, n_groups=13)
    want = {k: np.zeros(13, np.int64) for k in c}
    for s, al, e, ok, same in record_rows(sc, d_pk, n, d_res, nf, wl, spec):
        gi = s % 13
        want["records"][gi] += 1
        if not al:
            continue
        want["aligned"][gi] += 1
        want["crc_ok"][gi] += ok
        want["correct"][gi] += ok and same
        want["undetected"][gi] += ok and not same
        want["raw_errors"][gi] += e
        want["raw_packet_errors"][gi] += e > 0
    for key in c:
        assert np.array_equal(c[key], want[key]), key
    assert c["aligned"].sum() > ns and c["raw_errors"].sum() > 0


def test_fec_kernels_sass():
    """The Viterbi kernel adds and compares only: no FFMA / FMUL.  The LLR kernel's FFMAs are its 17 IEEE divides'
    (5 each, one FCHK per divide).  None of the three kernels uses local memory."""
    from test_sass_audit import sass
    funcs = sass()
    names = {k: [n for n in funcs if k in n] for k in ("packet_viterbi_kernel", "packet_llr_kernel",
                                                         "packet_encode_kernel")}
    assert all(len(v) == 1 for v in names.values()), names
    op = lambda ins, m: sum(bool(re.match(r"(@!?P\d+\s+)?%s\b" % m, i)) for i in ins)  # noqa: E731
    vit = funcs[names["packet_viterbi_kernel"][0]]
    assert op(vit, "FFMA") == 0 and op(vit, "FMUL") == 0 and op(vit, "FFMA2") == 0
    assert sum("SHFL" in i for i in vit) >= 2 and sum("VOTE" in i for i in vit) >= 2
    llr = funcs[names["packet_llr_kernel"][0]]
    n_chk = sum("FCHK" in i for i in llr)
    assert n_chk == 17 and op(llr, "FFMA") <= 5 * n_chk
    for n in names.values():
        assert not [i for i in funcs[n[0]] if re.search(r"\b(LDL|STL)\b", i)], n

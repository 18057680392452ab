"""GPU: the per-stream code rates of the packet code (sc_packet_encode_ex_dev, sc_packet_decode_ex_dev) against their
specification (tests/packet_code_ref.c, scf_encode_code / scf_decode_code) -- encoder bytes and decoded records bit
for bit past one grid pass, on real soft output and adversarial input, records of streams out of range or with an
invalid code, records past the count untouched, code 0 equal to sc_packet_decode_dev, the end-to-end loop-back through
an ACQ bank with mixed codes, and the new kernels' SASS."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_code_ref as R  # noqa: E402
import packet_fec_ref as F  # noqa: E402
from test_packet_acq_gpu import acq_streams  # noqa: E402


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def records(sc, streams):
    """PACKET_DTYPE records with the given stream indices (the only field the decoder reads)"""
    pk = np.zeros(len(streams), sc.PACKET_DTYPE)
    pk["stream"] = streams
    pk["call_index"] = 7
    return pk


def gpu_decode_ex(sc, llrs, pk, stream_code, n_found=None, capacity=None):
    import torch
    cap = llrs.shape[0] if capacity is None else capacity
    d_llr = torch.from_numpy(np.ascontiguousarray(llrs, np.float32)).cuda()
    d_pk = torch.from_numpy(np.ascontiguousarray(pk).view(np.uint8).copy()).cuda()
    d_code = torch.from_numpy(np.ascontiguousarray(stream_code, np.uint8)).cuda()
    d_out = torch.full((llrs.shape[0] * 48,), 0xA5, dtype=torch.uint8, device="cuda")
    d_n = torch.tensor([cap if n_found is None else n_found], dtype=torch.int64, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_decode_ex(d_llr[:cap], d_pk, d_n, d_code, d_out)
    torch.cuda.synchronize()
    bank.close()
    return d_out.cpu().numpy().view(sc.PAYLOAD_EX_DTYPE)


def spec_decode(pk, stream_code, llrs):
    """the spec's records: a stream out of range reads code 255"""
    s = pk["stream"].astype(np.int64)
    inside = (s >= 0) & (s < len(stream_code))
    codes = np.where(inside, np.asarray(stream_code, np.int64)[np.where(inside, s, 0)], 255).astype(np.uint8)
    return R.decode_code(codes, llrs)


@pytest.mark.gpu
def test_encode_equals_the_spec(sc):
    """100,003 streams x 1 packet with codes 0/1/2 and one invalid code: more than one pass of 296 x 256 threads;
    and 7 streams x 5 packets into an unaligned output (the byte path)"""
    import torch
    rng = np.random.default_rng(131)
    ns = 100003
    pay = rng.integers(0, 256, (ns, 1, 41)).astype(np.uint8)
    pay[0], pay[1] = 0, 255
    code = (np.arange(ns) % 3).astype(np.uint8)
    code[5] = 3
    code[ns - 1] = 255
    bits = torch.full((ns, 1, 8, 62), 7, dtype=torch.uint8, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_encode_ex(torch.from_numpy(pay).cuda(), torch.from_numpy(code).cuda(), bits)
    torch.cuda.synchronize()
    odd = torch.zeros(1 + 35 * 496, dtype=torch.uint8, device="cuda")
    pay2 = rng.integers(0, 256, (7, 5, 41)).astype(np.uint8)
    code2 = np.array([0, 1, 2, 2, 1, 0, 9], np.uint8)
    bank.packet_encode_ex(torch.from_numpy(pay2).cuda(), torch.from_numpy(code2).cuda(), odd[1:])
    torch.cuda.synchronize()
    bank.close()
    want = R.encode_code(code, pay.reshape(ns, 41))
    got = bits.cpu().numpy().reshape(ns, 496)
    assert np.array_equal(got, want)
    assert not got[5].any() and not got[ns - 1].any()
    want2 = R.encode_code(np.repeat(code2, 5), pay2.reshape(35, 41))
    assert np.array_equal(odd.cpu().numpy()[1:].reshape(35, 496), want2)


def acq_soft_batch(sc, ns=300, npk=4, seed=0xC1):
    """a real ACQ soft batch (test_packet_acq_gpu.acq_streams) -> (records PACKET_DTYPE, packet symbols [n, 496])"""
    samples, _, _ = acq_streams(sc, ns, npk, seed)
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    _, _, pk, psym, n = bank.rx_packets_soft_host(samples, samples.shape[1] // 1880)
    bank.close()
    assert n == len(pk) > ns
    return pk, psym.view(np.float32).reshape(-1, 496)


@pytest.mark.gpu
def test_decode_equals_the_spec(sc):
    rng = np.random.default_rng(132)
    # LLRs of a real ACQ soft batch, mixed per-stream codes
    pk, y = acq_soft_batch(sc)
    code = (rng.integers(0, 3, 300)).astype(np.uint8)
    L = F.llr(y)
    got = gpu_decode_ex(sc, L, pk, code)
    assert got.tobytes() == spec_decode(pk, code, L).tobytes()
    # adversarial LLRs at each code: noisy codewords, ties, zeros, non-finite and huge values
    sets = []
    for c in (0, 1, 2):
        bits = R.encode_code(c, rng.integers(0, 256, (300, 41)).astype(np.uint8))
        for sd in (0.5, 1.0, 2.0):
            sets.append((c, (((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2))
                         .astype(np.float32)))
        sets.append((c, rng.integers(-3, 4, (300, 496)).astype(np.float32)))
        sets.append((c, np.zeros((3, 496), np.float32)))
        bad = rng.standard_normal((200, 496)).astype(np.float32)
        k = rng.integers(0, 496, (200, 30))
        bad[np.arange(200)[:, None], k] = rng.choice(
            np.array([np.nan, np.inf, -np.inf, 1e38, -1e38, 2e7], np.float32), k.shape)
        sets.append((c, bad))
        sets.append((c, np.full((2, 496), np.nan, np.float32)))
    for c, L in sets:
        pk = records(sc, np.zeros(L.shape[0], np.int32))
        assert gpu_decode_ex(sc, L, pk, np.array([c], np.uint8)).tobytes() == R.decode_code(c, L).tobytes()
    # 20,011 records, past one grid pass (148 x 16 blocks x 8 records), streams of mixed codes
    n = 20011
    streams = rng.integers(0, 1000, n).astype(np.int32)
    code = (np.arange(1000) % 3).astype(np.uint8)
    bits = R.encode_code(code[streams], rng.integers(0, 256, (n, 41)).astype(np.uint8))
    L = (((1 - 2.0 * bits) + 0.9 * rng.standard_normal(bits.shape)) * 2.5).astype(np.float32)
    pk = records(sc, streams)
    assert gpu_decode_ex(sc, L, pk, code).tobytes() == spec_decode(pk, code, L).tobytes()


@pytest.mark.gpu
def test_records_not_decoded(sc):
    """a stream outside 0..n_streams-1 (code 255) or a code that is not 0..2: data 0, crc_ok 0, flipped 0, the code
    as read"""
    rng = np.random.default_rng(133)
    code = np.array([0, 1, 2, 3, 77, 255], np.uint8)
    streams = np.array([0, 1, 2, 3, 4, 5, 6, -1, 1 << 30, -(1 << 31), 2], np.int32)
    L = rng.standard_normal((streams.size, 496)).astype(np.float32) * 4
    pk = records(sc, streams)
    got = gpu_decode_ex(sc, L, pk, code)
    assert got.tobytes() == spec_decode(pk, code, L).tobytes()
    assert got["code"].tolist() == [0, 1, 2, 3, 77, 255, 255, 255, 255, 255, 2]
    assert not got["data"][3:10].any() and not got["crc_ok"][3:10].any() and not got["flipped"][3:10].any()
    assert not got["reserved0"].any() and not got["reserved1"].any()
    # n_streams = 0: every record is out of range
    import torch
    d_llr = torch.from_numpy(L[:3]).cuda()
    d_pk = torch.from_numpy(pk[:3].view(np.uint8).copy()).cuda()
    d_code = torch.zeros(1, dtype=torch.uint8, device="cuda")
    d_out = torch.full((3 * 48,), 0xA5, dtype=torch.uint8, device="cuda")
    d_n = torch.tensor([3], dtype=torch.int64, device="cuda")
    assert sc.lib.sc_packet_decode_ex_dev(0, d_llr.data_ptr(), d_pk.data_ptr(), 3, d_n.data_ptr(), d_code.data_ptr(), 0,
                                          d_out.data_ptr(), None) == 0
    torch.cuda.synchronize()
    got = d_out.cpu().numpy().view(sc.PAYLOAD_EX_DTYPE)
    assert (got["code"] == 255).all() and not got["data"].any() and not got["crc_ok"].any()


@pytest.mark.gpu
def test_records_past_the_count_are_untouched(sc):
    rng = np.random.default_rng(134)
    L = (rng.standard_normal((64, 496)) * 3).astype(np.float32)
    code = np.array([0, 1, 2], np.uint8)
    pk = records(sc, np.arange(64, dtype=np.int32) % 3)
    want = spec_decode(pk, code, L)
    for n_found, cap in ((20, 50), (80, 50), (0, 50), (50, 50)):
        got = gpu_decode_ex(sc, L, pk, code, n_found=n_found, capacity=cap)
        k = min(n_found, cap)
        assert got[:k].tobytes() == want[:k].tobytes()
        assert (got[k:].view(np.uint8) == 0xA5).all()


@pytest.mark.gpu
def test_code0_agrees_with_the_rate_half_decoder(sc):
    import torch
    pk, y = acq_soft_batch(sc, ns=200, seed=0xC2)
    # the soft batch's LLRs (its streams carry random bits: no CRC passes), then noisy codewords (most pass)
    rng = np.random.default_rng(136)
    bits = F.encode(rng.integers(0, 256, (500, 27)).astype(np.uint8))
    noisy = (((1 - 2.0 * bits) + 0.8 * rng.standard_normal(bits.shape)) * 3.0).astype(np.float32)
    L = np.concatenate([F.llr(y), noisy])
    pk = np.concatenate([pk, records(sc, np.zeros(500, np.int32))])
    ex = gpu_decode_ex(sc, L, pk, np.zeros(200, np.uint8))
    d_llr = torch.from_numpy(L).cuda()
    d_out = torch.zeros(L.shape[0] * 32, dtype=torch.uint8, device="cuda")
    d_n = torch.tensor([L.shape[0]], dtype=torch.int64, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_decode(d_llr, d_n, d_out)
    torch.cuda.synchronize()
    bank.close()
    old = d_out.cpu().numpy().view(sc.PAYLOAD_DTYPE)
    assert np.array_equal(ex["data"][:, :27], old["data"]) and not ex["data"][:, 27:].any()
    assert np.array_equal(ex["crc_ok"], old["crc_ok"]) and np.array_equal(ex["flipped"], old["flipped"])
    assert ex["crc_ok"][-500:].sum() > 400


@pytest.mark.gpu
def test_end_to_end_mixed_codes_on_an_acq_bank(sc):
    """config 2 (clean channel, +-20 Hz), ACQ bank, code s mod 3: the device records equal the spec's decode of the
    batch's packet symbols; every aligned record without a raw error over its code's transmitted bits is delivered;
    no record passes its CRC with another payload"""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = 255, 14
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    n_packets = (nf * 1880 + 2782) // 2783
    g = torch.Generator().manual_seed(135)
    pay = torch.randint(0, 256, (ns, n_packets, 41), generator=g, dtype=torch.uint8).cuda()
    code = (torch.arange(ns) % 3).to(torch.uint8).cuda()
    wl = harness.synthesize(bank, nf * 1880, seed=135, config=2, payload=pay, stream_code=code)
    cap = ns * nf
    d_res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
    d_pk = torch.zeros(cap * 96, dtype=torch.uint8, device="cuda")
    d_ps = torch.zeros((cap, 496), dtype=torch.float32, device="cuda")
    d_llr = torch.zeros((cap, 496), dtype=torch.float32, device="cuda")
    d_out = torch.zeros(cap * 48, dtype=torch.uint8, device="cuda")
    d_n = torch.zeros(1, dtype=torch.int64, device="cuda")
    bank.reset()
    bank.rx_packets_soft_dev(wl.samples, nf, d_res, d_pk, d_n, d_ps)
    bank.packet_llr(d_ps, d_n, d_llr)
    bank.packet_decode_ex(d_llr, d_pk, d_n, code, d_out)
    torch.cuda.synchronize()
    bank.close()
    n = min(int(d_n.item()), cap)
    pk = d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE)
    out = d_out.cpu().numpy()[:n * 48].view(sc.PAYLOAD_EX_DTYPE)
    codes = code.cpu().numpy()
    assert out.tobytes() == spec_decode(pk, codes, F.llr(d_ps.cpu().numpy()[:n])).tobytes()
    # record by record: aligned by grid_sample (every ACQ record has one), raw errors over the transmitted positions
    lead, payh = wl.lead.cpu().numpy(), pay.cpu().numpy()
    txb = wl.tx_bits.cpu().numpy().reshape(ns, n_packets, 496)
    rows = sc.unpack_packet_bits(pk).reshape(n, 496)
    sent = np.zeros(3, np.int64)
    for c in range(3):
        sent[c] = (codes == c).sum() * n_packets
    delivered, aligned, clean = np.zeros(3, np.int64), np.zeros(3, np.int64), 0
    for k, p in enumerate(pk):
        s, call = int(p["stream"]), int(p["call_index"])
        if not 2 <= call < nf:
            continue
        c = int(codes[s])
        B, _, N = R.code_sizes(c)
        pos = int(p["grid_sample"]) - 48 - int(lead[s])
        j = (pos + 2783 // 2) // 2783
        same = 0 <= j < n_packets and np.array_equal(out[k]["data"][:B], payh[s, j, :B])
        assert not (out[k]["crc_ok"] and not same)                      # no undetected error
        if not (0 <= j < n_packets and abs(pos - j * 2783) <= 10):
            continue
        aligned[c] += 1
        delivered[c] += int(out[k]["crc_ok"] and same)
        raw = int((rows[k][F.PERM64[:N]] != txb[s, j][F.PERM64[:N]]).sum())
        if raw == 0:
            clean += 1
            assert out[k]["crc_ok"] and same
    c = harness.packet_fec(d_pk, n, d_out, d_res, nf, wl, group=code, n_groups=3)
    assert np.array_equal(c["correct"], delivered) and np.array_equal(c["aligned"], aligned)
    assert c["undetected"].sum() == 0
    assert np.array_equal(c["payload_bytes"], delivered * np.array(R.CODE_BYTES))
    print("delivered share per code:", {k: f"{delivered[k]}/{sent[k]} = {delivered[k] / sent[k]:.3f}" for k in range(3)},
          "aligned:", aligned.tolist(), "without raw errors:", clean)
    assert clean > ns and (aligned == delivered).all()


def test_code_kernels_sass():
    """The new decoder adds and compares only (no FFMA / FMUL / FFMA2) and has its shuffles and ballots; neither new
    kernel uses local memory; the three existing FEC kernel names still match exactly one function each."""
    from test_sass_audit import sass
    funcs = sass()
    names = {k: [n for n in funcs if k in n] for k in ("packet_viterbi_kernel", "packet_llr_kernel",
                                                         "packet_encode_kernel", "packet_code_viterbi_kernel",
                                                         "packet_code_encode_kernel")}
    assert all(len(v) == 1 for v in names.values()), names
    op = lambda ins, m: sum(bool(re.match(r"(@!?P\d+\s+)?%s\b" % m, i)) for i in ins)  # noqa: E731
    vit = funcs[names["packet_code_viterbi_kernel"][0]]
    assert op(vit, "FFMA") == 0 and op(vit, "FMUL") == 0 and op(vit, "FFMA2") == 0
    assert sum("SHFL" in i for i in vit) >= 2 and sum("VOTE" in i for i in vit) >= 2
    for k in ("packet_code_viterbi_kernel", "packet_code_encode_kernel"):
        assert not [i for i in funcs[names[k][0]] if re.search(r"\b(LDL|STL)\b", i)], k

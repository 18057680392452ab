"""GPU: blind code detection of the packet code (sc_packet_decode_blind_dev) against its specification
(tests/packet_blind_ref.c, scf_decode_blind) -- records byte for byte for every mask on a real ACQ soft batch with
per-packet codes, on adversarial LLRs and past one grid pass; records past the count untouched; one-code masks equal
to sc_packet_decode_ex_dev; the end-to-end loop-back with codes that change packet by packet; the per-packet layout
of sc_packet_encode_ex_dev; and the kernel's SASS."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import packet_blind_ref as B  # noqa: E402
import packet_code_ref as R  # noqa: E402
import packet_fec_ref as F  # noqa: E402

MASKS = tuple(range(1, 8))


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def gpu_blind(sc, llrs, mask, n_found=None, capacity=None):
    import torch
    cap = llrs.shape[0] if capacity is None else capacity
    d_llr = torch.from_numpy(np.ascontiguousarray(llrs, np.float32)).cuda()
    d_out = torch.full((llrs.shape[0] * 48,), 0xA5, dtype=torch.uint8, device="cuda")
    d_n = torch.tensor([cap if n_found is None else n_found], dtype=torch.int64, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_decode_blind(d_llr[:cap], d_n, d_out, code_mask=mask)
    torch.cuda.synchronize()
    bank.close()
    return d_out.cpu().numpy().view(sc.PAYLOAD_EX_DTYPE)


def per_packet_batch(sc, ns, nf, seed, config, blind=True):
    """an ACQ bank over harness.synthesize(..., packet_code=(s + j) mod 3) -> (workload, codes, records, n, d_pk,
    d_res, d_llr, d_n, d_out) with the device batch, its LLRs and (blind) sc_packet_decode_blind_dev's records, mask 7"""
    import torch
    from singlecarrier_b200 import harness
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    n_packets = (nf * 1880 + 2782) // 2783
    g = torch.Generator().manual_seed(seed)
    pay = torch.randint(0, 256, (ns, n_packets, 41), generator=g, dtype=torch.uint8).cuda()
    codes = ((torch.arange(ns)[:, None] + torch.arange(n_packets)[None, :]) % 3).to(torch.uint8).cuda()
    wl = harness.synthesize(bank, nf * 1880, seed=seed, config=config, payload=pay, packet_code=codes)
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
    if blind:
        bank.packet_decode_blind(d_llr, d_n, d_out)
    torch.cuda.synchronize()
    bank.close()
    n = min(int(d_n.item()), cap)
    return wl, codes, n, d_pk, d_res, d_llr, d_n, d_out


@pytest.mark.gpu
def test_decode_blind_equals_the_spec(sc):
    rng = np.random.default_rng(300)
    # a real ACQ soft batch whose packets carry per-packet codes, at Eb/N0 0..12 dB: every mask
    _, _, n, _, _, d_llr, _, _ = per_packet_batch(sc, 130, 10, 301, config=4, blind=False)
    L = d_llr.cpu().numpy()[:n]
    assert n > 130
    for mask in MASKS:
        want = B.decode_blind(mask, L)
        assert gpu_blind(sc, L, mask).tobytes() == want.tobytes(), mask
        if mask == 7:
            assert want["crc_ok"].sum() > n // 4 and len(set(want["code"][want["crc_ok"] == 1].tolist())) == 3
    # adversarial LLRs: noisy codewords, ties, zeros, non-finite and huge values
    sets = []
    for c in (0, 1, 2):
        bits = R.encode_code(c, rng.integers(0, 256, (200, 41)).astype(np.uint8))
        for sd in (0.5, 1.0, 2.0):
            sets.append((((1 - 2.0 * bits) + sd * rng.standard_normal(bits.shape)) * (2 / sd ** 2)).astype(np.float32))
    sets.append(rng.integers(-3, 4, (300, 496)).astype(np.float32))
    sets.append(np.zeros((3, 496), np.float32))
    bad = rng.standard_normal((200, 496)).astype(np.float32)
    k = rng.integers(0, 496, (200, 30))
    bad[np.arange(200)[:, None], k] = rng.choice(np.array([np.nan, np.inf, -np.inf, 1e38, -1e38, 2e7], np.float32),
                                                 k.shape)
    sets.append(bad)
    sets.append(np.array([[np.nan] * 496, [np.inf] * 496, [1e38] * 496, [-1e38] * 496], np.float32))
    L = np.concatenate(sets)
    for mask in MASKS:
        assert gpu_blind(sc, L, mask).tobytes() == B.decode_blind(mask, L).tobytes(), mask
    # 20,011 records, past one grid pass (148 x 16 blocks x 8 records), codes mixed record by record
    n = 20011
    code = (np.arange(n) % 3).astype(np.uint8)
    bits = R.encode_code(code, rng.integers(0, 256, (n, 41)).astype(np.uint8))
    L = (((1 - 2.0 * bits) + 0.9 * rng.standard_normal(bits.shape)) * 2.5).astype(np.float32)
    got = gpu_blind(sc, L, 7)
    assert got.tobytes() == B.decode_blind(7, L).tobytes()
    assert (got["code"][got["crc_ok"] == 1] == code[got["crc_ok"] == 1]).all()


@pytest.mark.gpu
def test_records_past_the_count_are_untouched(sc):
    rng = np.random.default_rng(302)
    L = (rng.standard_normal((64, 496)) * 3).astype(np.float32)
    want = B.decode_blind(5, L)
    for n_found, cap in ((20, 50), (80, 50), (0, 50), (50, 50)):
        got = gpu_blind(sc, L, 5, n_found=n_found, capacity=cap)
        k = min(n_found, cap)
        assert got[:k].tobytes() == want[:k].tobytes()
        assert (got[k:].view(np.uint8) == 0xA5).all()


@pytest.mark.gpu
def test_one_code_masks_equal_decode_ex(sc):
    """mask 1 << c against sc_packet_decode_ex_dev with every stream at code c, on the same records"""
    import torch
    _, _, n, d_pk, _, d_llr, d_n, _ = per_packet_batch(sc, 100, 10, 303, config=4, blind=False)
    bank = sc.ModemBank(1)
    for c in (0, 1, 2):
        ex = torch.full((n * 48,), 0x5A, dtype=torch.uint8, device="cuda")
        bl = torch.full((n * 48,), 0xA5, dtype=torch.uint8, device="cuda")
        bank.packet_decode_ex(d_llr[:n], d_pk, d_n, torch.full((100,), c, dtype=torch.uint8, device="cuda"), ex)
        bank.packet_decode_blind(d_llr[:n], d_n, bl, code_mask=1 << c)
        torch.cuda.synchronize()
        assert torch.equal(ex, bl), c
    bank.close()


@pytest.mark.gpu
def test_end_to_end_per_packet_codes_on_an_acq_bank(sc):
    """config 2 (clean channel, +-20 Hz), ACQ bank, packet j of stream s at code (s + j) mod 3: the device records
    equal the spec's; every aligned record whose transmitted bits arrived without a raw error is delivered at its code;
    no record passes its CRC at another code or with another payload"""
    from singlecarrier_b200 import harness
    ns, nf = 255, 14
    wl, codes, n, d_pk, d_res, d_llr, _, d_out = per_packet_batch(sc, ns, nf, 304, config=2)
    pk = d_pk.cpu().numpy()[:n * 96].view(sc.PACKET_DTYPE)
    out = d_out.cpu().numpy()[:n * 48].view(sc.PAYLOAD_EX_DTYPE)
    assert out.tobytes() == B.decode_blind(7, d_llr.cpu().numpy()[:n]).tobytes()
    codes = codes.cpu().numpy()
    lead, payh = wl.lead.cpu().numpy(), wl.payload.cpu().numpy()
    txb = wl.tx_bits.cpu().numpy().reshape(ns, wl.n_packets, 496)
    rows = sc.unpack_packet_bits(pk).reshape(n, 496)
    delivered, aligned, clean = np.zeros(3, np.int64), np.zeros(3, np.int64), 0
    for k, p in enumerate(pk):
        s, call = int(p["stream"]), int(p["call_index"])
        if not 2 <= call < nf:
            continue
        pos = int(p["grid_sample"]) - 48 - int(lead[s])
        j = (pos + 2783 // 2) // 2783
        inside = 0 <= j < wl.n_packets
        c = int(codes[s, j]) if inside else -1
        nb = R.CODE_BYTES[c] if inside else 0
        same = inside and out[k]["code"] == c and np.array_equal(out[k]["data"][:nb], payh[s, j, :nb])
        assert not (out[k]["crc_ok"] and not same)                      # no undetected error, no wrong code
        if not (inside and abs(pos - j * 2783) <= 10):
            continue
        aligned[c] += 1
        delivered[c] += int(out[k]["crc_ok"] and same)
        N = R.CODE_CODED[c]
        if not (rows[k][F.PERM64[:N]] != txb[s, j][F.PERM64[:N]]).any():
            clean += 1
            assert out[k]["crc_ok"] and same
    f = harness.packet_fec(d_pk, n, d_out, d_res, nf, wl)
    assert f["wrong_code"].sum() == 0 and f["undetected"].sum() == 0
    assert f["correct"].sum() == delivered.sum() and f["aligned"].sum() == aligned.sum()
    assert f["payload_bytes"].sum() == (delivered * np.array(R.CODE_BYTES)).sum()
    print("delivered per code:", delivered.tolist(), "aligned:", aligned.tolist(), "without raw errors:", clean)
    assert clean > ns and (aligned == delivered).all() and (delivered > 0).all()


@pytest.mark.gpu
def test_encoder_per_packet_layout_equals_the_spec(sc):
    """payloads [n_streams * n_packets][1][41] with one code per packet, n_packets = 1: the bits land in the
    [n_streams][n_packets][8][62] layout, packet j of stream s encoded at its code"""
    import torch
    rng = np.random.default_rng(305)
    ns, npk = 37, 5
    pay = rng.integers(0, 256, (ns, npk, 41)).astype(np.uint8)
    codes = rng.integers(0, 3, (ns, npk)).astype(np.uint8)
    bits = torch.full((ns, npk, 8, 62), 7, dtype=torch.uint8, device="cuda")
    bank = sc.ModemBank(1)
    bank.packet_encode_ex(torch.from_numpy(pay.reshape(ns * npk, 1, 41)).cuda(),
                          torch.from_numpy(codes.reshape(-1)).cuda(), bits)
    torch.cuda.synchronize()
    bank.close()
    want = R.encode_code(codes.reshape(-1), pay.reshape(-1, 41)).reshape(ns, npk, 496)
    assert np.array_equal(bits.cpu().numpy().reshape(ns, npk, 496), want)


def test_blind_kernel_sass():
    """The blind decoder adds and compares only (no FFMA / FMUL / FFMA2), has its shuffles and ballots and no local
    memory; the existing FEC kernel names still match exactly one function each."""
    from test_sass_audit import sass
    funcs = sass()
    names = {k: [n for n in funcs if k in n] for k in ("packet_viterbi_kernel", "packet_llr_kernel",
                                                         "packet_encode_kernel", "packet_code_viterbi_kernel",
                                                         "packet_code_encode_kernel", "packet_blind_decode_kernel")}
    assert all(len(v) == 1 for v in names.values()), names
    op = lambda ins, m: sum(bool(re.match(r"(@!?P\d+\s+)?%s\b" % m, i)) for i in ins)  # noqa: E731
    ins = funcs[names["packet_blind_decode_kernel"][0]]
    assert op(ins, "FFMA") == 0 and op(ins, "FMUL") == 0 and op(ins, "FFMA2") == 0
    assert sum("SHFL" in i for i in ins) >= 2 and sum("VOTE" in i for i in ins) >= 2
    assert not [i for i in ins if re.search(r"\b(LDL|STL)\b", i)]

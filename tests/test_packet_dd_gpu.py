"""GPU: packet mode with the decision-directed equalizer (SC_FLAG_PACKET_DD) against its specification
(tests/packet_dd_ref.c, scd_ext_run_stream_dd): records, cost and packet symbols compared as uint32; per-call results
identical to a plain packet bank's; and the bit error rate through the library's own transmitter and channel.
The SASS check at the end needs only cuobjdump."""
import os
import re
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from packet_dd_ref import ext_run_stream_dd  # noqa: E402
from test_packet_gpu import gpu_packet_streams  # noqa: E402
from test_soft_gpu import hard_rows, u32  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sc():
    import singlecarrier_b200 as m
    assert m.lib.sc_device_count() > 0, "no CUDA device"
    return m


def by_key(pk):
    return {(int(p["stream"]), int(p["call_index"])): k for k, p in enumerate(pk)}


def check_against_spec(sc, samples, pk, psym, wide=False, foffset=0.0):
    """pk / psym sorted by (stream, call) == the spec's packets of every stream, in order (psym None: records only)."""
    ns = samples.shape[0]
    outs = [None] * ns

    def one(s):
        outs[s] = ext_run_stream_dd(samples[s], wide=wide, foffset=foffset)

    with ThreadPoolExecutor(max_workers=max(1, min(32, os.cpu_count() or 1))) as ex:
        list(ex.map(one, range(ns)))
    rows = sc.unpack_packet_bits(pk)
    k = 0
    for s in range(ns):
        _, _, opk, opsym, _ = outs[s]
        for q, qs in zip(opk, opsym):
            p = pk[k]
            assert (p["stream"], p["call_index"], p["max_index"], p["matches"]) == (s, q["call"], q["max_index"],
                                                                                  q["matches"]), (s, q["call"])
            assert np.float32(p["cost"]).view(np.uint32) == np.float32(q["cost"]).view(np.uint32), (s, q["call"])
            assert np.array_equal(rows[k].reshape(-1), q["bits"]), (s, q["call"])
            if psym is not None:
                assert np.array_equal(u32(psym[k]), u32(qs)), (s, q["call"])
            k += 1
    assert k == len(pk)
    return k


def host_forms(sc, samples, nf, dd, wide=False, foff=0.0):
    bank = sc.ModemBank(samples.shape[0], wide=wide, foffset_hz=foff, packet=True, dd=dd)
    res, csym, pk, psym, n = bank.rx_packets_soft_host(samples, nf, call_symbols=True)
    bank.close()
    bank = sc.ModemBank(samples.shape[0], wide=wide, foffset_hz=foff, packet=True, dd=dd)
    res0, pk0, n0 = bank.rx_packets_host(samples, nf)
    bank.close()
    assert res.tobytes() == res0.tobytes() and n == n0 == len(pk) and pk.tobytes() == pk0.tobytes()
    return res, csym, pk, psym


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["loop1", "loop70", "loop300", "wide", "foffset", "hard"])
def test_dd_packets_equal_the_spec(sc, oracle, case):
    wide, foff = case == "wide", (7.5 if case == "foffset" else 0.0)
    if case == "hard":
        samples = hard_rows(oracle, 37)
    else:
        ns, npk, seed = {"loop1": (1, 3, 1), "loop70": (70, 5, 2), "loop300": (300, 4, 3)}.get(case, (70, 4, 5))
        samples, _, _ = gpu_packet_streams(sc, ns, npk, seed)
    ns, nf = samples.shape[0], samples.shape[1] // 1880
    res, csym, pk, psym = host_forms(sc, samples, nf, True, wide, foff)
    # the ordinary calls and the record list are those of a plain packet bank
    pres, pcsym, ppk, _ = host_forms(sc, samples, nf, False, wide, foff)
    assert res.tobytes() == pres.tobytes() and np.array_equal(u32(csym), u32(pcsym))
    for f in ("stream", "call_index", "max_index", "matches"):
        assert np.array_equal(ppk[f], pk[f]), f
    assert check_against_spec(sc, samples, pk, psym, wide=wide, foffset=foff) == len(pk)
    assert np.isfinite(psym).all()
    # the sign identity of packet soft output holds for y
    raw = sc.unpack_packet_bits(pk).reshape(len(pk), 248, 2) ^ \
        np.array([(np.uint64(sc.packet_keystream_word(f)) >> np.arange(62, dtype=np.uint64)) & np.uint64(1)
                  for f in range(8)], np.uint8).reshape(248, 2)[None]
    assert np.array_equal(raw[..., 0], (psym.imag < 0).astype(np.uint8))
    assert np.array_equal(raw[..., 1], (psym.real < 0).astype(np.uint8))
    if ns >= 70:
        assert len(pk) > ns


@pytest.mark.gpu
def test_dd_streaming_equals_one_shot(sc):
    ns, npk = 97, 5
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 11)
    nf = samples.shape[1] // 1880
    a = sc.ModemBank(ns, packet=True, dd=True)
    res, csym, pk, psym, n = a.rx_packets_soft_host(samples, nf, call_symbols=True)
    a.close()
    b = sc.ModemBank(ns, packet=True, dd=True)
    parts, f = [], 0
    for step in [1, 2, 1, 3, 1, 1, 5, 2, 100]:
        k = min(step, nf - f)
        if k <= 0:
            break
        parts.append(b.rx_packets_soft_host(np.ascontiguousarray(samples[:, f * 1880:(f + k) * 1880]), k))
        f += k
    b.close()
    assert np.concatenate([p[0] for p in parts], axis=1).tobytes() == res.tobytes()
    allp = np.concatenate([p[2] for p in parts])
    alls = np.concatenate([p[3] for p in parts])
    order = np.lexsort((allp["call_index"], allp["stream"]))
    assert allp[order].tobytes() == pk.tobytes() and n == len(pk) > ns
    assert np.array_equal(u32(alls[order]), u32(psym))


@pytest.mark.gpu
@pytest.mark.parametrize("start", [0, 5])
def test_dd_device_entry_capacity_and_counter_offset(sc, start):
    import torch
    ns, npk = 4000, 3
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 21)
    nf = samples.shape[1] // 1880
    res, csym, pk, psym = host_forms(sc, samples, nf, True)
    n = len(pk)
    cap = n // 2 if start == 0 else n + start
    d_in = torch.from_numpy(samples).cuda()
    for soft in (True, False):
        bank = sc.ModemBank(ns, packet=True, dd=True)
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
        assert int(d_n.item()) == start + n
        assert d_res.cpu().numpy().tobytes() == res.tobytes()
        got = d_pk.cpu().numpy().reshape(cap, 96)
        gps = d_ps.cpu().numpy()
        assert (got[:start] == 0xAB).all()
        kept = min(n, cap - start)
        recs = got[start:start + kept].reshape(-1).view(sc.PACKET_DTYPE)
        blocks = gps[start * 496:(start + kept) * 496].reshape(kept, 496).view(np.complex64)
        key = by_key(pk)
        for k in range(kept):
            j = key[(int(recs[k]["stream"]), int(recs[k]["call_index"]))]
            assert recs[k].tobytes() == pk[j].tobytes()
            if soft:
                assert np.array_equal(u32(blocks[k]), u32(psym[j]))
        assert (got[start + kept:] == 0xAB).all()
        assert np.isnan(gps).all() if not soft else np.isnan(gps[(start + kept) * 496:]).all()


@pytest.mark.gpu
def test_dd_flag_alone_is_refused(sc):
    with pytest.raises(sc.SingleCarrierError):
        sc.ModemBank(8, dd=True)
    import ctypes
    h = ctypes.c_void_p()
    assert sc.lib.sc_create(ctypes.byref(h), 0, 8, 0x8, 0.0) == -1 and not h.value


@pytest.mark.gpu
def test_dd_and_plain_packet_banks_alternate(sc):
    """A DD bank and a plain packet bank fed the same batches in turn, in one process: each equals its own one-shot
    run, and the per-call results of the two are identical."""
    ns, npk = 150, 5
    samples, _, _ = gpu_packet_streams(sc, ns, npk, 33)
    nf = samples.shape[1] // 1880
    cuts = [0, 3, 5, 9, nf]
    banks = {dd: sc.ModemBank(ns, packet=True, dd=dd) for dd in (True, False)}
    got = {dd: ([], []) for dd in (True, False)}
    for b in range(4):
        x = np.ascontiguousarray(samples[:, cuts[b] * 1880:cuts[b + 1] * 1880])
        for dd in ((True, False) if b % 2 == 0 else (False, True)):
            r, p, _ = banks[dd].rx_packets_host(x, cuts[b + 1] - cuts[b])
            got[dd][0].append(r)
            got[dd][1].append(p)
    for bank in banks.values():
        bank.close()
    one = {}
    for dd in (True, False):
        bank = sc.ModemBank(ns, packet=True, dd=dd)
        one[dd] = bank.rx_packets_host(samples, nf)
        bank.close()
        allp = np.concatenate(got[dd][1])
        assert np.concatenate(got[dd][0], axis=1).tobytes() == one[dd][0].tobytes()
        assert allp[np.lexsort((allp["call_index"], allp["stream"]))].tobytes() == one[dd][1].tobytes()
    assert one[True][0].tobytes() == one[False][0].tobytes()
    assert not np.array_equal(one[True][1]["bits"], one[False][1]["bits"])


@pytest.mark.gpu
def test_dd_bit_error_rate_at_scale(sc):
    """65,536 streams through sc_tx_channel_dev with a carrier offset only (uniform in +-20 Hz, random phase and
    lead-in): the packets the receiver finds decode with BER < 2 % where the reference's equalizer is above 30 %."""
    import torch
    from singlecarrier_b200 import harness
    ns, nf = 65536, 12
    out = {}
    for dd in (False, True):
        bank = sc.ModemBank(ns, packet=True, dd=dd)
        wl = harness.synthesize(bank, nf * 1880, seed=0xDD, config=2)
        res = torch.zeros((ns, nf * 32), dtype=torch.uint8, device="cuda")
        pk = torch.zeros(ns * nf * 96, dtype=torch.uint8, device="cuda")
        n = torch.zeros(1, dtype=torch.int64, device="cuda")
        bank.rx_packets_dev(wl.samples, nf, res, pk, n)
        out[dd] = harness.packet_ber_dev(bank, pk, n, res, nf, wl)
        bank.close()
    for dd in (False, True):
        assert out[dd]["aligned"][0] > 1000
    assert np.array_equal(out[True]["records"], out[False]["records"])
    ber = {dd: out[dd]["errors"][0] / out[dd]["bits"][0] for dd in (False, True)}
    assert ber[True] < 0.02 and ber[False] > 0.30, ber


def test_dd_kernels_in_the_library_without_spills():
    """Both instantiations of packet_track_dd_kernel are compiled for sm_100a, and they touch local memory no more than
    the reference-equalizer kernel does (its only local arrays: the keystream words and the record being built)."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump not available")
    lib = os.path.join(ROOT, "singlecarrier_b200", "libsinglecarrier_b200.so")
    out = subprocess.run([exe, "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs, cur, arch = {}, None, None
    for ln in out.splitlines():
        m = re.search(r"arch = (sm_\w+)", ln)
        if m:
            arch = m.group(1)
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            funcs[cur] = (arch, [])
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", ln):
            funcs[cur][1].append(ln.split("*/", 1)[1].split("/*")[0].strip())

    def local(ins):
        return sum(bool(re.search(r"\b(LDL|STL)\b", i)) for i in ins)

    for soft in (0, 1):
        dd = [v for k, v in funcs.items() if f"packet_track_dd_kernelILb{soft}E" in k]
        ref = [v for k, v in funcs.items() if f"packet_track_kernelILb{soft}E" in k]
        assert len(dd) == 1 and len(ref) == 1
        assert dd[0][0] == "sm_100a"
        assert local(dd[0][1]) <= local(ref[0][1]), (local(dd[0][1]), local(ref[0][1]))

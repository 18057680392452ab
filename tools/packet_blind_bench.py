"""Blind code detection of the packet code (sc_packet_decode_blind_dev) against a genie that knows each packet's code:
delivered payloads, wrong codes and false deliveries per Eb/N0 group, and kernel times.

Workload: the bench's, 131,072 streams x 42 calls (harness.synthesize(config=4): +-20 Hz offset, random phase and
lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index; the same channel in every case), every packet
carrying a random payload at its own code (harness.synthesize(packet_code=...)).  A SC_FLAG_PACKET | SC_FLAG_PACKET_DD |
SC_FLAG_PACKET_ACQ bank runs one cold-started sc_rx_packets_soft_dev batch, then sc_packet_llr_dev, on one CUDA stream.
  random  each packet's code drawn uniformly from 0..2 with a fixed seed
  group   the code of each Eb/N0 group that profiles/r07_packet_code.md chose (the most payload per packet)
  blind   sc_packet_decode_blind_dev, mask 7
  genie   the blind kernel at each one-code mask (1, 2, 4); per record the decode at the code of its packet j (the
          aligned packet, or the nearest one for a record that is not aligned), taken on the host
harness.packet_fec recounts both on the host.
  kernels CUDA events, after a warm-up, on the random case's records: blind at mask 7 and at each one-code mask,
          alternated with sc_packet_decode_ex_dev at each code; with --compare-lib, sc_packet_decode_ex_dev of another
          build of the library as well (its records checked byte for byte against this build's)
The card's name, power limit and max SM clock are read before and after.
usage: python tools/packet_blind_bench.py [--out FILE.json] [--md FILE.md] [--reps R] [--streams N] [--compare-lib SO]"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import singlecarrier_b200 as sc  # noqa: E402
from singlecarrier_b200 import harness  # noqa: E402
from packet_code_bench import gpu_info, timed_alternating  # noqa: E402

NF, FRAME, N_GROUPS = 42, 1880, 13
GROUP_CODE = [0, 0, 0, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2]     # profiles/r07_packet_code.json, "mixed" / "group_code"


def rates(c, extra, transmitted):
    """harness.packet_fec counters and this tool's extra counters (summed) -> the profile's rates"""
    r = lambda x: round(float(x), 6)  # noqa: E731
    al = int(c["aligned"])
    return {"transmitted": int(transmitted), "aligned": al, "per": r(1 - c["correct"] / max(al, 1)),
            "delivered": int(c["correct"]), "goodput": r(c["payload_bytes"] / max(transmitted, 1)),
            "payload_bytes": int(c["payload_bytes"]), "wrong_code": int(c["wrong_code"]),
            "undetected": int(c["undetected"]), "not_aligned": int(c["records"] - c["aligned"]),
            **{k: int(v) for k, v in extra.items()}}


def markdown(out):
    w, k = out["workload"], out["kernels"]
    L = ["# Blind code detection of the packet code: blind against genie, and kernel times", "",
         f"`python tools/packet_blind_bench.py` on one {out['gpu']['device']} ({out['gpu']['nvidia_smi']}: name, power "
         f"limit, max SM clock; after the run: {out['gpu_after']['nvidia_smi']}).  Raw output: "
         "`profiles/r08_packet_blind.json`.", "",
         f"Workload: the bench's, {w['streams']:,} streams x {w['calls']} calls (`harness.synthesize(config=4, "
         "payload=random, packet_code=...)`: +-20 Hz offset uniform per stream, random phase and lead-in, AWGN at Eb/N0 "
         f"0..12 dB striped over 13 groups; the same channel in both cases), {w['packets_per_stream']} packets per "
         "stream, each at its own code.  Bank `SC_FLAG_PACKET | SC_FLAG_PACKET_DD | SC_FLAG_PACKET_ACQ`: "
         "`sc_rx_packets_soft_dev` -> `sc_packet_llr_dev` -> `sc_packet_decode_blind_dev` (mask 7) on one CUDA stream.",
         "",
         "- **random**: each packet's code drawn uniformly from 1/2, 2/3, 3/4 with a fixed seed.",
         "- **group**: each Eb/N0 group at the code r07 chose for it (" +
         ", ".join(f"{g} dB: {['1/2', '2/3', '3/4'][c]}" for g, c in enumerate(GROUP_CODE)) + ").",
         "- **genie**: the blind kernel at each one-code mask; each record takes the decode at its packet's code.", "",
         "PER: aligned records (+-10 samples) not delivered (CRC passes, code and payload those sent).  goodput: payload "
         "bytes delivered per transmitted packet.  wrong code: aligned records whose CRC passes at another code (also "
         "in undetected).  undet.: aligned records whose CRC passes with another payload or code.  false: CRC passes "
         "among records not aligned to a packet.  two: aligned records that pass their CRC at two or more codes.", ""]
    for case in ("random", "group"):
        o = out[case]
        L += [f"## {case}", "",
              "| Eb/N0 dB | aligned | PER blind | PER genie | goodput blind | goodput genie | wrong code | undet. blind "
              "| undet. genie | not aligned | false blind | false genie | two |", "|---" * 13 + "|"]
        rows = [(str(g), o["blind"]["per_ebn0"][g], o["genie"]["per_ebn0"][g]) for g in range(N_GROUPS)]
        rows.append(("all", o["blind"]["all"], o["genie"]["all"]))
        for name, b, g in rows:
            L.append(f"| {name} | {b['aligned']:,} | {b['per']:.5f} | {g['per']:.5f} | {b['goodput']:.3f} | "
                     f"{g['goodput']:.3f} | {b['wrong_code']} | {b['undetected']} | {g['undetected']} | "
                     f"{b['not_aligned']:,} | {b['false']} | {g['false']} | {b['two_pass']} |")
        L += ["", f"Payload bytes delivered: {o['blind']['all']['payload_bytes']:,} blind, "
              f"{o['genie']['all']['payload_bytes']:,} genie; largest PER difference over the groups "
              f"{o['max_per_diff']:.6f}.", ""]
    L += ["## Kernel time", "",
          f"CUDA events around each launch, {out['reps']} rounds after a warm-up, the steps alternated in each round, on "
          f"the random case's {k['records']:,} records (their LLRs, {k['records'] * 496 * 4 / 1e9:.2f} GB: beyond L2).  "
          "decode_ex: every stream set to the code.", "",
          "| step | median ms | min | max | ms per 10^6 records |", "|---|---|---|---|---|"]
    for name, v in k["steps"].items():
        L.append(f"| {name} | {v['median']:.3f} | {v['min']:.3f} | {v['max']:.3f} | {v['ms_per_million']:.3f} |")
    if "compare_lib_records_equal" in k:
        L += ["", f"Records of `sc_packet_decode_ex_dev` of the compared build equal this build's at every code: "
              f"{k['compare_lib_records_equal']}."]
    L.append("")
    return "\n".join(L) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--md", help="also write the tables as markdown here")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0xFEC)
    ap.add_argument("--compare-lib", help="another build of libsinglecarrier_b200.so whose sc_packet_decode_ex_dev is "
                                          "timed and checked on the same records")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_blind_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps}
    ns, dev = a.streams, torch.device("cuda", 0)
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    cap = ns * (NF - 2)                         # every call n >= 2 can give a record
    res = torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev)
    pk = torch.empty(cap * 96, dtype=torch.uint8, device=dev)
    psym = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    llr = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    dec = torch.empty(cap * 48, dtype=torch.uint8, device=dev)
    one = [torch.empty(cap * 48, dtype=torch.uint8, device=dev) for _ in range(3)]
    n_found = torch.zeros(1, dtype=torch.int64, device=dev)
    g = torch.Generator(device=dev)
    n_packets = (NF * FRAME + harness.PERIOD - 1) // harness.PERIOD
    group = (torch.arange(ns, device=dev) % N_GROUPS).to(torch.int32)
    per_group = [int((group == k).sum().item()) * n_packets for k in range(N_GROUPS)]

    def run(packet_code):
        g.manual_seed(a.seed)
        pay = torch.randint(0, 256, (ns, n_packets, sc.PAYLOAD_MAX), generator=g, device=dev, dtype=torch.uint8)
        wl = harness.synthesize(bank, NF * FRAME, seed=a.seed, config=4, payload=pay, packet_code=packet_code)
        assert torch.equal(wl.ebn0_db.to(torch.int32), group), "Eb/N0 groups are striped by stream index"
        bank.reset()
        n_found.zero_()
        bank.rx_packets_soft_dev(wl.samples, NF, res, pk, n_found, psym)
        bank.packet_llr(psym, n_found, llr)
        bank.packet_decode_blind(llr, n_found, dec, code_mask=7)
        for c in range(3):
            bank.packet_decode_blind(llr, n_found, one[c], code_mask=1 << c)
        torch.cuda.synchronize()
        n = int(n_found.item())
        assert n <= cap, "capacity"
        recs = [x[:n * 48].cpu().numpy().view(sc.PAYLOAD_EX_DTYPE) for x in one]
        s, j, ok, al = harness.packet_alignment(pk, n, res, NF, wl)
        sent = packet_code.cpu().numpy().astype(np.int64)[s, j]
        genie = recs[0].copy()
        for c in (1, 2):
            genie[sent == c] = recs[c][sent == c]
        blind = dec[:n * 48].cpu().numpy().view(sc.PAYLOAD_EX_DTYPE)
        two = (sum(r["crc_ok"].astype(np.int64) for r in recs) >= 2) & al
        grp = group.cpu().numpy()[s]
        out_case = {"records_found": n}
        for name, d in (("blind", blind), ("genie", genie)):
            c = harness.packet_fec(pk, n, d, res, NF, wl, group=group, n_groups=N_GROUPS)
            false = ok & ~al & (d["crc_ok"] != 0)
            extra = {"false": np.bincount(grp[false], minlength=N_GROUPS),
                     "two_pass": np.bincount(grp[two], minlength=N_GROUPS)}
            out_case[name] = {"all": rates({k: v.sum() for k, v in c.items()}, {k: v.sum() for k, v in extra.items()},
                                           sum(per_group)),
                              "per_ebn0": [dict(ebn0_db=k, **rates({q: v[k] for q, v in c.items()},
                                                                  {q: v[k] for q, v in extra.items()}, per_group[k]))
                                           for k in range(N_GROUPS)]}
        out_case["max_per_diff"] = max(abs(out_case["blind"]["per_ebn0"][k]["per"] - out_case["genie"]["per_ebn0"][k]["per"])
                                       for k in range(N_GROUPS))
        return out_case

    out["workload"] = {"streams": ns, "calls": NF, "config": 4, "packets_per_stream": n_packets}
    out["group"] = run(torch.tensor(GROUP_CODE, dtype=torch.uint8, device=dev)[group.long()][:, None]
                       .expand(ns, n_packets).contiguous())
    print("group:", out["group"]["blind"]["all"], out["group"]["genie"]["all"], flush=True)
    gc = torch.Generator(device=dev)
    gc.manual_seed(a.seed + 1)
    out["random"] = run(torch.randint(0, 3, (ns, n_packets), generator=gc, device=dev, dtype=torch.uint8))
    print("random:", out["random"]["blind"]["all"], out["random"]["genie"]["all"], flush=True)

    # kernel times on the records of the last batch (the random case's), whose LLRs are those now in llr
    n = int(n_found.item())
    codes = {c: torch.full((ns,), c, dtype=torch.uint8, device=dev) for c in range(3)}
    steps = {"blind mask 7 (packet_blind_decode_kernel)": lambda: bank.packet_decode_blind(llr, n_found, dec, 7)}
    for c in range(3):
        steps[f"decode_ex code {c} (packet_code_viterbi_kernel)"] = (
            lambda c=c: bank.packet_decode_ex(llr, pk, n_found, codes[c], one[c]))
    for c in range(3):
        steps[f"blind mask {1 << c}"] = lambda c=c: bank.packet_decode_blind(llr, n_found, dec, 1 << c)
    if a.compare_lib:
        other = C.CDLL(os.path.abspath(a.compare_lib))
        fn = other.sc_packet_decode_ex_dev
        fn.restype = C.c_int
        fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                       C.c_void_p]
        ref = torch.empty(cap * 48, dtype=torch.uint8, device=dev)

        def other_decode(c):
            assert fn(0, llr.data_ptr(), pk.data_ptr(), cap, n_found.data_ptr(), codes[c].data_ptr(), ns, ref.data_ptr(),
                      None) == 0

        equal = {}
        for c in range(3):
            bank.packet_decode_ex(llr, pk, n_found, codes[c], one[c])
            other_decode(c)
            torch.cuda.synchronize()
            equal[c] = bool(torch.equal(one[c][:n * 48], ref[:n * 48]))
        for c in range(3):
            steps[f"decode_ex code {c}, compared build"] = lambda c=c: other_decode(c)
    for f in steps.values():
        f()
    torch.cuda.synchronize()
    out["kernels"] = {"records": n, "steps": timed_alternating(steps, a.reps, {k: n for k in steps})}
    if a.compare_lib:
        out["kernels"]["compare_lib_records_equal"] = equal
    bank.close()
    out["gpu_after"] = gpu_info()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
    if a.md:
        with open(a.md, "w") as f:
            f.write(markdown(out))


if __name__ == "__main__":
    main()

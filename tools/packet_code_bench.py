"""Code rates of the packet code (sc_packet_encode_ex_dev, sc_packet_decode_ex_dev): delivered payloads per Eb/N0 group
and code, and kernel times per code.

Workload: the bench's, 131,072 streams x 42 calls (harness.synthesize(config=4): +-20 Hz offset, random phase and
lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index; the same channel in every run), every packet
carrying a random payload at its stream's code.  A SC_FLAG_PACKET | SC_FLAG_PACKET_DD | SC_FLAG_PACKET_ACQ bank runs
one cold-started sc_rx_packets_soft_dev batch, then sc_packet_llr_dev and sc_packet_decode_ex_dev on the same CUDA
stream; harness.packet_fec recounts the records on the host.
  uniform  every stream on code 0, then on 1, then on 2
  mixed    the code of each Eb/N0 group is the one with the most payload bytes delivered per transmitted packet in
           the uniform runs
  kernels  CUDA events, after a warm-up, on the mixed batch's records: sc_packet_decode_ex_dev and
           sc_packet_encode_ex_dev per code, and code 0 through packet_code_viterbi_kernel next to
           packet_viterbi_kernel (sc_packet_decode_dev), the two alternated in the same run
The card's name, power limit and max SM clock are read before and after.
usage: python tools/packet_code_bench.py [--out FILE.json] [--md FILE.md] [--reps R] [--streams N]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import singlecarrier_b200 as sc  # noqa: E402
from singlecarrier_b200 import harness  # noqa: E402

NF, FRAME, N_GROUPS = 42, 1880, 13
CODES = (sc.CODE_R12, sc.CODE_R23, sc.CODE_R34)
RATE = {0: "1/2", 1: "2/3", 2: "3/4"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def summary(ts, per):
    m = statistics.median(ts)
    return {"median": round(m, 4), "min": round(min(ts), 4), "max": round(max(ts), 4),
            "ms_per_million": round(m / (per / 1e6), 4), "all": [round(x, 4) for x in ts]}


def timed_alternating(fns, reps, per):
    """each step of fns once per round, reps rounds -> {name: summary}"""
    ts = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            ts[k].append(event_ms(f))
    return {k: summary(v, per[k]) for k, v in ts.items()}


def rates(c, transmitted):
    """harness.packet_fec counters (summed) -> the profile's rates"""
    r = lambda x: round(float(x), 5)  # noqa: E731
    al = int(c["aligned"])
    return {"transmitted": transmitted, "aligned": al, "per_decoded": r(1 - c["correct"] / max(al, 1)),
            "delivered": int(c["correct"]), "delivered_share": r(c["correct"] / max(transmitted, 1)),
            "undetected": int(c["undetected"]), "payload_bytes": int(c["payload_bytes"]),
            "goodput": r(c["payload_bytes"] / max(transmitted, 1))}


def markdown(out):
    w, k = out["workload"], out["kernels"]
    L = ["# Code rates of the packet code: delivered payloads and kernel times", "",
         f"`python tools/packet_code_bench.py` on one {out['gpu']['device']} ({out['gpu']['nvidia_smi']}: name, power "
         f"limit, max SM clock; after the run: {out['gpu_after']['nvidia_smi']}).  Raw output: "
         "`profiles/r07_packet_code.json`.", "",
         f"Workload: the bench's, {w['streams']:,} streams x {w['calls']} calls (`harness.synthesize(config=4, "
         "payload=random, stream_code=...)`: +-20 Hz offset uniform per stream, random phase and lead-in, AWGN at Eb/N0 "
         f"0..12 dB striped over 13 groups; the same channel in every run), {w['packets_per_stream']} packets per "
         "stream.  Bank `SC_FLAG_PACKET | SC_FLAG_PACKET_DD | SC_FLAG_PACKET_ACQ`: `sc_rx_packets_soft_dev` -> "
         "`sc_packet_llr_dev` -> `sc_packet_decode_ex_dev` on one CUDA stream.", "",
         "PER: aligned records (+-10 samples) not delivered.  delivered: payloads delivered (CRC passes and payload "
         "equals the one sent) over packets transmitted (including the two per stream cut by the stream's end).  "
         "goodput: payload bytes delivered per transmitted packet.  undetected: aligned records whose CRC passes with "
         "another payload.", "",
         "## Per Eb/N0 group and code", "",
         "| Eb/N0 dB | " + " | ".join(f"PER {RATE[c]} | delivered {RATE[c]} | goodput {RATE[c]} | undet. {RATE[c]}"
                                      for c in CODES) + " | mixed: code | mixed goodput |",
         "|---" * (2 + 4 * len(CODES) + 1) + "|"]
    for gi in range(N_GROUPS):
        cells = []
        for c in CODES:
            r = out["uniform"][str(c)]["per_ebn0"][gi]
            cells += [f"{r['per_decoded']:.4f}", f"{r['delivered_share']:.4f}", f"{r['goodput']:.2f}",
                      str(r["undetected"])]
        m = out["mixed"]["per_ebn0"][gi]
        L.append(f"| {gi} | " + " | ".join(cells) + f" | {RATE[out['mixed']['group_code'][gi]]} | {m['goodput']:.2f} |")
    cells = []
    for c in CODES:
        r = out["uniform"][str(c)]["all"]
        cells += [f"{r['per_decoded']:.4f}", f"{r['delivered_share']:.4f}", f"{r['goodput']:.2f}", str(r["undetected"])]
    L.append("| all | " + " | ".join(cells) + f" | mixed | {out['mixed']['all']['goodput']:.2f} |")
    L += ["", f"Mixed run: {out['mixed']['all']['payload_bytes']:,} payload bytes delivered against "
          + ", ".join(f"{out['uniform'][str(c)]['all']['payload_bytes']:,} at rate {RATE[c]}" for c in CODES)
          + f"; {out['mixed']['all']['undetected']} undetected errors.", "",
          "## Kernel time", "",
          f"CUDA events around each launch, {out['reps']} rounds after a warm-up, the steps of a table alternated in each "
          f"round.  Decoders on the mixed batch's {k['records']:,} records (its LLRs, "
          f"{k['records'] * 496 * 4 / 1e9:.2f} GB: beyond L2), every stream set to the code; encoder on "
          f"{k['payloads']:,} payloads.", "",
          "| step | median ms | min | max | ms per 10^6 records |", "|---|---|---|---|---|"]
    for name, v in k["steps"].items():
        L.append(f"| {name} | {v['median']:.3f} | {v['min']:.3f} | {v['max']:.3f} | {v['ms_per_million']:.3f} |")
    L.append("")
    return "\n".join(L) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--md", help="also write the tables as markdown here")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0xFEC)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_code_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps}
    ns, dev = a.streams, torch.device("cuda", 0)
    bank = sc.ModemBank(ns, packet=True, dd=True, acq=True)
    cap = ns * (NF - 2)                         # every call n >= 2 can give a record
    res = torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev)
    pk = torch.empty(cap * 96, dtype=torch.uint8, device=dev)
    psym = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    llr = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    dec = torch.empty(cap * 48, dtype=torch.uint8, device=dev)
    dec_old = torch.empty(cap * 32, dtype=torch.uint8, device=dev)
    n_found = torch.zeros(1, dtype=torch.int64, device=dev)
    g = torch.Generator(device=dev)
    n_packets = (NF * FRAME + harness.PERIOD - 1) // harness.PERIOD
    group = None

    def run(stream_code):
        nonlocal group
        g.manual_seed(a.seed)
        pay = torch.randint(0, 256, (ns, n_packets, sc.PAYLOAD_MAX), generator=g, device=dev, dtype=torch.uint8)
        wl = harness.synthesize(bank, NF * FRAME, seed=a.seed, config=4, payload=pay, stream_code=stream_code)
        group = wl.ebn0_db.to(torch.int32)
        bank.reset()
        n_found.zero_()
        bank.rx_packets_soft_dev(wl.samples, NF, res, pk, n_found, psym)
        bank.packet_llr(psym, n_found, llr)
        bank.packet_decode_ex(llr, pk, n_found, stream_code, dec)
        torch.cuda.synchronize()
        n = int(n_found.item())
        assert n <= cap, "capacity"
        c = harness.packet_fec(pk, n, dec, res, NF, wl, group=group, n_groups=N_GROUPS)
        per_group = [int((group == k).sum().item()) * n_packets for k in range(N_GROUPS)]
        return {"records_found": n, "all": rates({k: v.sum() for k, v in c.items()}, sum(per_group)),
                "per_ebn0": [dict(ebn0_db=k, **rates({q: v[k] for q, v in c.items()}, per_group[k]))
                             for k in range(N_GROUPS)]}

    out["workload"] = {"streams": ns, "calls": NF, "config": 4, "packets_per_stream": n_packets}
    out["uniform"] = {}
    for c in CODES:
        out["uniform"][str(c)] = run(torch.full((ns,), c, dtype=torch.uint8, device=dev))
        print(f"code {c}: {out['uniform'][str(c)]['all']}", flush=True)
    best = [max(CODES, key=lambda c: out["uniform"][str(c)]["per_ebn0"][gi]["payload_bytes"]) for gi in range(N_GROUPS)]
    mixed = run(torch.tensor(best, dtype=torch.uint8, device=dev)[(torch.arange(ns, device=dev) % N_GROUPS)])
    assert torch.equal(group.cpu(), (torch.arange(ns) % N_GROUPS).int()), "Eb/N0 groups are striped by stream index"
    out["mixed"] = dict(group_code=best, **mixed)
    print(f"mixed {best}: {mixed['all']}", flush=True)

    # kernel times on the records of the last batch (the mixed run's), whose LLRs are those now in llr
    n = int(n_found.item())
    codes = {c: torch.full((ns,), c, dtype=torch.uint8, device=dev) for c in CODES}
    pay = torch.randint(0, 256, (ns, n_packets, sc.PAYLOAD_MAX), generator=g, device=dev, dtype=torch.uint8)
    bits = torch.empty((ns, n_packets, 8, 62), dtype=torch.uint8, device=dev)
    steps = {"decode_ex code 0 (packet_code_viterbi_kernel)": lambda: bank.packet_decode_ex(llr, pk, n_found, codes[0],
                                                                                              dec),
             "decode code 0 (packet_viterbi_kernel)": lambda: bank.packet_decode(llr, n_found, dec_old)}
    for c in (1, 2):
        steps[f"decode_ex code {c}"] = (lambda c=c: bank.packet_decode_ex(llr, pk, n_found, codes[c], dec))
    for c in CODES:
        steps[f"encode_ex code {c}"] = (lambda c=c: bank.packet_encode_ex(pay, codes[c], bits))
    pay27 = pay[:, :, :27].contiguous()
    steps["encode code 0 (packet_encode_kernel)"] = lambda: bank.packet_encode(pay27, bits)
    for f in steps.values():
        f()
    torch.cuda.synchronize()
    per = {k: (ns * n_packets if "encode" in k else n) for k in steps}
    timed = timed_alternating({k: f for k, f in steps.items() if "decode" in k}, a.reps, per)
    timed.update(timed_alternating({k: f for k, f in steps.items() if "encode" in k}, a.reps, per))
    out["kernels"] = {"records": n, "payloads": ns * n_packets, "steps": timed}
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

"""The coded payload of packet-mode packets (sc_packet_encode_dev, sc_packet_llr_dev, sc_packet_decode_dev): kernel
times and delivered payloads.

Workload: the bench's, 131,072 streams x 42 calls (harness.synthesize(config=4, payload=random): +-20 Hz offset,
random phase and lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index), every packet carrying a
random 27-byte payload through the packet code.  Each of a SC_FLAG_PACKET | SC_FLAG_PACKET_DD bank ("dd") and one with
SC_FLAG_PACKET_ACQ as well ("acq") runs one cold-started sc_rx_packets_soft_dev batch, then sc_packet_llr_dev and
sc_packet_decode_dev on the same CUDA stream; harness.packet_fec recounts the records on the host.
  kernels  CUDA events around each kernel, repeated: the LLR and Viterbi kernels on the acq batch's records, the
           encoder on the workload's payloads; the acq soft batch itself for comparison
  curve    per Eb/N0 group and bank: aligned share, raw coded-bit BER, PER without and with the code, delivered
           payloads over transmitted packets, undetected errors
  offsets  the acq bank on clean channels with a carrier offset only, 0, +-10 and +-20 Hz
The card's name, power limit and max SM clock are read before and after.
usage: python tools/packet_fec_bench.py [--out FILE.json] [--md FILE.md] [--reps R] [--streams N]"""
import argparse
import json
import math
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
HBM_TBS = 7.7                                   # HGX B200 data sheet, one GPU
PAYLOAD_DB = 10 * math.log10(496 / 216)         # Eb/N0 per payload bit = per channel bit + 3.61 dB


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return {"median": round(statistics.median(ts), 4), "min": round(min(ts), 4), "max": round(max(ts), 4),
            "all": [round(x, 4) for x in ts]}


def rates(c, transmitted):
    """harness.packet_fec counters (summed) -> the profile's rates"""
    r = lambda x: round(float(x), 5)  # noqa: E731
    al = int(c["aligned"])
    return {"transmitted": transmitted, "records": int(c["records"]), "aligned": al,
            "aligned_share": r(al / max(transmitted, 1)), "raw_ber": r(c["raw_errors"] / max(476 * al, 1)),
            "per_uncoded": r(c["raw_packet_errors"] / max(al, 1)), "per_decoded": r(1 - c["correct"] / max(al, 1)),
            "delivered": int(c["correct"]), "delivered_share": r(c["correct"] / max(transmitted, 1)),
            "crc_ok": int(c["crc_ok"]), "undetected": int(c["undetected"])}


def markdown(out):
    t, w, k = out["acq_batch_ms"], out["workload"], out["kernels"]
    L = ["# Coded payload of packet-mode packets: kernel times and delivered payloads", "",
         f"`python tools/packet_fec_bench.py` on one {out['gpu']['device']} ({out['gpu']['nvidia_smi']}: name, power "
         f"limit, max SM clock; after the run: {out['gpu_after']['nvidia_smi']}).  Raw output: "
         "`profiles/r06_packet_fec.json`.", "",
         f"Workload: the bench's, {w['streams']:,} streams x {w['calls']} calls (`harness.synthesize(config=4, "
         "payload=random)`: +-20 Hz offset uniform per stream, random phase and lead-in, AWGN at Eb/N0 0..12 dB striped "
         f"over 13 groups), {w['packets_per_stream']} packets per stream, each carrying a random 27-byte payload through "
         "the packet code.  Banks `SC_FLAG_PACKET | SC_FLAG_PACKET_DD` (\"dd\") and the same with `SC_FLAG_PACKET_ACQ` "
         "(\"acq\"): `sc_rx_packets_soft_dev` -> `sc_packet_llr_dev` -> `sc_packet_decode_dev` on one CUDA stream.", "",
         "## Kernel time", "",
         f"CUDA events around each launch, {out['reps']} launches after a warm-up; the LLR and Viterbi kernels on the acq "
         f"batch's {k['records']:,} records (packet symbols and LLRs {k['llr_bytes'] / 1e9:.2f} GB: far beyond L2), the "
         f"encoder on the workload's {k['payloads']:,} payloads.  One acq `sc_rx_packets_soft_dev` batch: median "
         f"{t['median']:.1f} ms (min {t['min']:.1f}, max {t['max']:.1f}).", "",
         "| kernel | median ms | min | max | ms per 10^6 records | share of the acq batch |", "|---|---|---|---|---|---|"]
    for name in ("llr", "decode", "encode"):
        v = k[name]
        L.append(f"| {name} | {v['median']:.3f} | {v['min']:.3f} | {v['max']:.3f} | {v['ms_per_million']:.3f} | "
                 f"{v['median'] / t['median']:.4f} |")
    L += ["", f"LLR kernel: {k['llr_bytes'] / 1e9:.2f} GB moved (2 x 1,984 B per record) in {k['llr']['median']:.3f} ms "
          f"= {k['llr_tbs']:.2f} TB/s, {k['llr_hbm_share']:.3f} of {HBM_TBS} TB/s (data sheet; bytes over time, "
          "the bound is the memory).", "",
          "## Rates per Eb/N0 group", "",
          "Eb/N0 per channel bit is the harness's; per payload bit it is +3.61 dB (10 log10(496/216)).  aligned share: "
          "records aligned (+-10 samples) over packets transmitted (including the two per stream cut by the stream's "
          "end).  raw BER: hard-decision errors over coded bits 0..475 of aligned records.  PER uncoded: aligned "
          "records with any such error.  PER decoded: aligned records not delivered (CRC passes and payload equals "
          "the one sent).  delivered: payloads delivered over packets transmitted.  undetected: aligned records whose "
          "CRC passes with another payload.", ""]
    for bank in ("dd", "acq"):
        L += [f"### {bank}", "", "| Eb/N0 dB (channel) | (payload) | aligned share | raw BER | PER uncoded | PER decoded "
              "| delivered | undetected |", "|---|---|---|---|---|---|---|---|"]
        for row in out["curve"][bank]["per_ebn0"] + [out["curve"][bank]["all"] | {"ebn0_db": "all"}]:
            e = row["ebn0_db"]
            ep = f"{e + PAYLOAD_DB:.2f}" if e != "all" else "all"
            L.append(f"| {e} | {ep} | {row['aligned_share']:.4f} | {row['raw_ber']:.4f} | {row['per_uncoded']:.4f} | "
                     f"{row['per_decoded']:.4f} | {row['delivered_share']:.4f} | {row['undetected']} |")
        L.append("")
    L += ["## Clean channel, carrier offset only (acq bank; random phase and lead-in, the same offset on every stream)",
          "", "| offset Hz | aligned share | raw BER | PER uncoded | PER decoded | delivered | undetected |",
          "|---|---|---|---|---|---|---|"]
    for df, row in out["offsets_hz"].items():
        L.append(f"| {float(df):+.0f} | {row['aligned_share']:.4f} | {row['raw_ber']:.4f} | {row['per_uncoded']:.4f} | "
                 f"{row['per_decoded']:.4f} | {row['delivered_share']:.4f} | {row['undetected']} |")
    return "\n".join(L) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--md", help="also write the tables as markdown here")
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0xFEC)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_fec_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps}
    ns, dev = a.streams, torch.device("cuda", 0)
    banks = {"dd": sc.ModemBank(ns, packet=True, dd=True), "acq": sc.ModemBank(ns, packet=True, dd=True, acq=True)}
    cap = ns * (NF - 2)                         # every call n >= 2 can give a record
    res = torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev)
    pk = torch.empty(cap * 96, dtype=torch.uint8, device=dev)
    psym = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    llr = torch.empty((cap, 496), dtype=torch.float32, device=dev)
    dec = torch.empty(cap * 32, dtype=torch.uint8, device=dev)
    n_found = torch.zeros(1, dtype=torch.int64, device=dev)

    def batch(name, samples):
        banks[name].reset()
        n_found.zero_()
        banks[name].rx_packets_soft_dev(samples, NF, res, pk, n_found, psym)

    def run(name, wl, group, n_groups):
        batch(name, wl.samples)
        banks[name].packet_llr(psym, n_found, llr)
        banks[name].packet_decode(llr, n_found, dec)
        torch.cuda.synchronize()
        n = int(n_found.item())
        assert n <= cap, "capacity"
        return n, harness.packet_fec(pk, n, dec, res, NF, wl, group=group, n_groups=n_groups)

    g = torch.Generator(device=dev)
    g.manual_seed(a.seed)
    n_packets = (NF * FRAME + harness.PERIOD - 1) // harness.PERIOD
    pay = torch.randint(0, 256, (ns, n_packets, 27), generator=g, device=dev, dtype=torch.uint8)
    wl = harness.synthesize(banks["dd"], NF * FRAME, seed=a.seed, config=4, payload=pay)
    group = wl.ebn0_db.to(torch.int32)
    out["workload"] = {"streams": ns, "calls": NF, "config": 4, "packets_per_stream": wl.n_packets}

    curve = {}
    for name in ("dd", "acq"):                  # acq last: its records stay in the buffers for the kernel timing
        n, c = run(name, wl, group, N_GROUPS)
        per_group = [int((group == k).sum().item()) * wl.n_packets for k in range(N_GROUPS)]
        curve[name] = {"records_found": n, "all": rates({k: v.sum() for k, v in c.items()}, sum(per_group)),
                       "per_ebn0": [dict(ebn0_db=k, **rates({q: v[k] for q, v in c.items()}, per_group[k]))
                                    for k in range(N_GROUPS)]}
    out["curve"] = curve

    # kernel times on the acq batch's records
    n = int(n_found.item())
    enc_bits = torch.empty((ns, n_packets, 8, 62), dtype=torch.uint8, device=dev)
    steps = {"llr": lambda: banks["acq"].packet_llr(psym, n_found, llr),
             "decode": lambda: banks["acq"].packet_decode(llr, n_found, dec),
             "encode": lambda: banks["acq"].packet_encode(pay, enc_bits)}
    for f in steps.values():
        f()
    torch.cuda.synchronize()
    kern = {"records": n, "payloads": ns * n_packets, "llr_bytes": n * 2 * 496 * 4}
    for name, f in steps.items():
        v = timed(f, a.reps)
        v["ms_per_million"] = round(v["median"] / ((ns * n_packets if name == "encode" else n) / 1e6), 4)
        kern[name] = v
    kern["llr_tbs"] = round(kern["llr_bytes"] / (kern["llr"]["median"] * 1e-3) / 1e12, 4)
    kern["llr_hbm_share"] = round(kern["llr_tbs"] / HBM_TBS, 4)
    assert torch.equal(enc_bits, wl.tx_bits), "encoder output changed between calls"
    out["kernels"] = kern
    out["acq_batch_ms"] = timed(lambda: batch("acq", wl.samples), max(3, a.reps // 3))
    del wl

    offsets = {}
    for df in (0.0, 10.0, -10.0, 20.0, -20.0):
        g.manual_seed(a.seed + int(df) + 100)
        lead = torch.randint(0, harness.PERIOD, (ns,), generator=g, device=dev, dtype=torch.int32)
        ch = {"df_hz": torch.full((ns,), df, device=dev),
              "phi_rad": (torch.rand(ns, generator=g, device=dev) * (2 * math.pi)).float()}
        opay = torch.randint(0, 256, (ns, n_packets, 27), generator=g, device=dev, dtype=torch.uint8)
        samples = torch.empty((ns, NF * FRAME), dtype=torch.int16, device=dev)
        bits = torch.empty((ns, n_packets, 8, 62), dtype=torch.uint8, device=dev)
        banks["acq"].packet_encode(opay, bits)
        banks["acq"].tx_packets_dev(samples, n_packets, gap_samples=harness.PERIOD - FRAME, bits=bits, lead_in=lead,
                                    channel=ch)
        torch.cuda.synchronize()
        owl = harness.Workload(samples, bits, lead, harness.PERIOD - FRAME, None, n_packets, ch, opay)
        _, c = run("acq", owl, None, 1)
        offsets[str(df)] = rates({k: v.sum() for k, v in c.items()}, ns * n_packets)
        del samples, bits, opay
    out["offsets_hz"] = offsets
    for b in banks.values():
        b.close()
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

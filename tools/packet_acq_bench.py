"""Packet mode with and without acquisition (SC_FLAG_PACKET_ACQ), both decoded by the decision-directed equalizer:
time, packets found and bit error rate.

Workload: the bench's, 131,072 streams x 42 calls (harness.synthesize(config=4): +-20 Hz offset, random phase and
lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index), input resident in HBM.
  timing   one cold-started sc_rx_packets_dev batch on a SC_FLAG_PACKET | SC_FLAG_PACKET_DD bank ("dd", records from
           the reference's per-call detection) and on one with SC_FLAG_PACKET_ACQ as well ("acq"), alternating, CUDA
           events; median, min and max
  curve    sc_packet_ber_stats_dev per Eb/N0 group for both: records, aligned records and their share of the packets
           transmitted, BER per data frame, BER, packet error rate
  offsets  the same counters on clean channels with a carrier offset only, 0, +-10 and +-20 Hz
           (random phase and lead-in)
The card's name, power limit and max SM clock are read before and after.
usage: python tools/packet_acq_bench.py [--out FILE.json] [--md FILE.md] [--reps R] [--warmup W] [--streams N]"""
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

NF, FRAME, PK_BYTES, N_GROUPS = 42, 1880, 96, 13
NAMES = {False: "dd", True: "acq"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(c, transmitted):
    """per-group counters (harness.packet_counters) -> BER, BER per data frame, PER, aligned"""
    r4 = lambda x: round(float(x), 4)  # noqa: E731
    al = int(c["aligned"].sum())
    return {"records": int(c["records"].sum()), "aligned": al, "transmitted": transmitted,
            "aligned_of_transmitted": r4(al / max(transmitted, 1)), "ber": r4(c["errors"].sum() / max(c["bits"].sum(), 1)),
            "ber_per_frame": [r4(c["frame_errors"][:, f].sum() / max(62 * al, 1)) for f in range(8)],
            "per": r4((al - c["error_histogram"][:, 0].sum()) / max(al, 1))}


def markdown(out):
    t, w = out["timing_ms"], out["workload"]
    L = ["# Packet-mode acquisition (`SC_FLAG_PACKET_ACQ`): packets found, bit error rate, time", "",
         f"`python tools/packet_acq_bench.py` on one {out['gpu']['device']} ({out['gpu']['nvidia_smi']}: name, power "
         f"limit, max SM clock; after the run: {out['gpu_after']['nvidia_smi']}).  Raw output: "
         "`profiles/r05_packet_acq.json`.", "",
         f"Workload: the bench's, {w['streams']:,} streams x {w['calls']} calls (`harness.synthesize(config=4)`: +-20 Hz "
         "offset uniform per stream, random phase and lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups), "
         f"{w['packets_per_stream']} packets synthesised per stream (the last two are cut by the stream's end).  Banks "
         "`SC_FLAG_PACKET | SC_FLAG_PACKET_DD` (\"dd\", records from the reference's per-call detection) and the same "
         f"with `SC_FLAG_PACKET_ACQ` (\"acq\").  Per-call results byte-identical: {out['results_identical']}.", "",
         "## Time", "", "One cold-started `sc_rx_packets_dev` batch, CUDA events, banks alternating.", "",
         "| bank | median ms | min | max |", "|---|---|---|---|"]
    for k in ("dd", "acq"):
        L.append(f"| {k} | {t[k]['median']:.2f} | {t[k]['min']:.2f} | {t[k]['max']:.2f} |")
    L += ["", f"acq / dd: {out['acq_over_dd']:.3f}.", "", "## Aligned packets and bit error rate per Eb/N0", "",
          "aligned / transmitted: the share of the packets synthesised that a record lines up with (+-10 samples).", "",
          "| Eb/N0 dB | transmitted | dd aligned | dd share | acq aligned | acq share | dd BER | acq BER | dd PER | acq PER |",
          "|---|---|---|---|---|---|---|---|---|---|"]
    rows = zip(out["curve"]["dd"]["per_ebn0"], out["curve"]["acq"]["per_ebn0"])
    for d, q in list(rows) + [(out["curve"]["dd"]["all"] | {"ebn0_db": "all"}, out["curve"]["acq"]["all"] | {"ebn0_db": "all"})]:
        L.append(f"| {d['ebn0_db']} | {d['transmitted']:,} | {d['aligned']:,} | {d['aligned_of_transmitted']:.4f} | "
                 f"{q['aligned']:,} | {q['aligned_of_transmitted']:.4f} | {d['ber']:.4f} | {q['ber']:.4f} | {d['per']:.4f} | "
                 f"{q['per']:.4f} |")
    L += ["", "acq BER per data frame, all groups: " + ", ".join(f"{x:.4f}" for x in out["curve"]["acq"]["all"]["ber_per_frame"]),
          "", "## Carrier offset only (clean channel, random phase and lead-in, the same offset on every stream)", "",
          "| offset Hz | dd records | dd aligned | acq records | acq aligned | acq share | dd BER | acq BER | acq PER |",
          "|---|---|---|---|---|---|---|---|---|"]
    for df, v in out["offsets_hz"].items():
        d, q = v["dd"], v["acq"]
        dber = f"{d['ber']:.4f}" if d["aligned"] else "—"
        L.append(f"| {float(df):+.0f} | {d['records']:,} | {d['aligned']:,} | {q['records']:,} | {q['aligned']:,} | "
                 f"{q['aligned_of_transmitted']:.4f} | {dber} | {q['ber']:.4f} | {q['per']:.4f} |")
    return "\n".join(L) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--md", help="also write the tables as markdown here")
    ap.add_argument("--kernels", action="store_true", help="only: per-kernel CUDA time of one acq batch (torch.profiler)")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0xACB)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_acq_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps, "warmup": a.warmup}
    ns, dev = a.streams, torch.device("cuda", 0)
    banks = {acq: sc.ModemBank(ns, packet=True, dd=True, acq=acq) for acq in (False, True)}
    cap = ns * (NF - 2)                     # every call n >= 2 can be valid (silence is, F6)
    res = {dd: torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev) for dd in banks}
    pk = {dd: torch.empty(cap * PK_BYTES, dtype=torch.uint8, device=dev) for dd in banks}
    n_found = {dd: torch.zeros(1, dtype=torch.int64, device=dev) for dd in banks}

    def batch(dd, samples):
        banks[dd].reset()
        n_found[dd].zero_()
        banks[dd].rx_packets_dev(samples, NF, res[dd], pk[dd], n_found[dd])

    def counters(dd, wl, group, n_groups):
        assert int(n_found[dd].item()) <= cap, "capacity"
        return harness.packet_ber_dev(banks[dd], pk[dd], n_found[dd], res[dd], NF, wl, group=group, n_groups=n_groups)

    wl = harness.synthesize(banks[False], NF * FRAME, seed=a.seed, config=4)
    group = wl.ebn0_db.to(torch.int32)
    if a.kernels:
        batch(True, wl.samples)
        torch.cuda.synchronize()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batch(True, wl.samples)
            torch.cuda.synchronize()
        ev = prof.key_averages()
        tot = {e.key: (e.count, e.device_time_total / 1e3) for e in ev if e.device_time_total > 0}
        print(json.dumps({"gpu": gpu_info(), "kernels_ms": {k: {"launches": c, "ms": round(t, 3)}
                                                              for k, (c, t) in sorted(tot.items(), key=lambda x: -x[1][1])}},
                         indent=1))
        return
    for _ in range(a.warmup):
        for dd in banks:
            batch(dd, wl.samples)
    torch.cuda.synchronize()
    times = {NAMES[dd]: [] for dd in banks}
    for r in range(a.reps):
        for dd in ((False, True) if r % 2 == 0 else (True, False)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            batch(dd, wl.samples)
            e1.record()
            torch.cuda.synchronize()
            times[NAMES[dd]].append(e0.elapsed_time(e1))
    out["workload"] = {"streams": ns, "calls": NF, "config": 4, "packets_per_stream": wl.n_packets,
                       "note": "transmitted counts every packet synthesised, including those cut by the stream's end"}
    out["timing_ms"] = {k: {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4),
                            "all": [round(x, 4) for x in v]} for k, v in times.items()}
    out["acq_over_dd"] = round(statistics.median(times["acq"]) / statistics.median(times["dd"]), 4)

    # the last timed batches' records: the curve per Eb/N0 group
    curve = {}
    for dd in banks:
        batch(dd, wl.samples)
        c = counters(dd, wl, group, N_GROUPS)
        per_group = [int((group == g).sum().item()) * wl.n_packets for g in range(N_GROUPS)]
        curve[NAMES[dd]] = {"all": summary(c, sum(per_group)), "per_ebn0": [
            dict(ebn0_db=g, **summary({k: v[g:g + 1] for k, v in c.items()}, per_group[g])) for g in range(N_GROUPS)]}
    out["curve"] = curve
    same = bool(torch.equal(res[False], res[True]))
    out["results_identical"] = same
    del wl

    offsets = {}
    for df in (0.0, 10.0, -10.0, 20.0, -20.0):
        g = torch.Generator(device=dev)
        g.manual_seed(a.seed + int(df) + 100)
        period = harness.PERIOD
        n_packets = (NF * FRAME + period - 1) // period
        lead = torch.randint(0, period, (ns,), generator=g, device=dev, dtype=torch.int32)
        ch = {"df_hz": torch.full((ns,), df, device=dev),
              "phi_rad": (torch.rand(ns, generator=g, device=dev) * (2 * math.pi)).float()}
        samples = torch.empty((ns, NF * FRAME), dtype=torch.int16, device=dev)
        bits = torch.empty((ns, n_packets, 8, 62), dtype=torch.uint8, device=dev)
        banks[False].tx_packets_dev(samples, n_packets, gap_samples=period - FRAME, seed=a.seed + 7, bits_out=bits,
                                    lead_in=lead, channel=ch)
        torch.cuda.synchronize()
        owl = harness.Workload(samples, bits, lead, period - FRAME, None, n_packets, ch)
        offsets[str(df)] = {}
        for dd in banks:
            batch(dd, samples)
            offsets[str(df)][NAMES[dd]] = summary(counters(dd, owl, None, 1), ns * n_packets)
        del samples, bits
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
    assert same, "per-call results differ between the two banks"


if __name__ == "__main__":
    main()

"""Packet mode with and without the decision-directed equalizer (SC_FLAG_PACKET_DD): time and bit error rate.

Workload: the bench's, 131,072 streams x 42 calls (harness.synthesize(config=4): +-20 Hz offset, random phase and
lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index), input resident in HBM.
  timing   one cold-started sc_rx_packets_dev batch on a SC_FLAG_PACKET bank ("kalman", the reference's equalizer) and
           on a SC_FLAG_PACKET | SC_FLAG_PACKET_DD bank ("dd"), alternating, CUDA events; median, min and max
  curve    sc_packet_ber_stats_dev per Eb/N0 group for both equalizers: BER per data frame, BER, packet error rate
  offsets  the same per-equalizer counters on clean channels with a carrier offset only, 0, +-10 and +-20 Hz
           (random phase and lead-in)
The card's name, power limit and max SM clock are read before and after.
usage: python tools/packet_dd_bench.py [--out FILE] [--reps R] [--warmup W] [--streams N]"""
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
NAMES = {False: "kalman", True: "dd"}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(c):
    """per-group counters (harness.packet_counters) -> BER, BER per data frame, PER, aligned"""
    r4 = lambda x: round(float(x), 4)  # noqa: E731
    al = int(c["aligned"].sum())
    return {"records": int(c["records"].sum()), "aligned": al, "ber": r4(c["errors"].sum() / max(c["bits"].sum(), 1)),
            "ber_per_frame": [r4(c["frame_errors"][:, f].sum() / max(62 * al, 1)) for f in range(8)],
            "per": r4((al - c["error_histogram"][:, 0].sum()) / max(al, 1))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0xDDB)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_dd_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps, "warmup": a.warmup}
    ns, dev = a.streams, torch.device("cuda", 0)
    banks = {dd: sc.ModemBank(ns, packet=True, dd=dd) for dd in (False, True)}
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
    out["workload"] = {"streams": ns, "calls": NF, "config": 4}
    out["timing_ms"] = {k: {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4),
                            "all": [round(x, 4) for x in v]} for k, v in times.items()}
    out["dd_over_kalman"] = round(statistics.median(times["dd"]) / statistics.median(times["kalman"]), 4)

    # the last timed batches' records: the curve per Eb/N0 group
    curve = {}
    for dd in banks:
        batch(dd, wl.samples)
        c = counters(dd, wl, group, N_GROUPS)
        curve[NAMES[dd]] = {"all": summary(c), "per_ebn0": [
            dict(ebn0_db=g, **summary({k: v[g:g + 1] for k, v in c.items()})) for g in range(N_GROUPS)]}
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
            offsets[str(df)][NAMES[dd]] = summary(counters(dd, owl, None, 1))
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
    assert same, "per-call results differ between the two banks"


if __name__ == "__main__":
    main()

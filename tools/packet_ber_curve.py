"""Packet-mode bit error rate against Eb/N0 from the device counter (sc_packet_ber_stats_dev), and its cost.

Workload: 65,536 streams x 42 calls (harness.synthesize(config=3) on a SC_FLAG_PACKET bank: +-20 Hz offset, random
phase and lead-in, AWGN at Eb/N0 0..12 dB striped over 13 groups by stream index), input resident in HBM.  One
sc_rx_packets_dev batch, then the counters of its records per Eb/N0 group: BER per data frame, the share of aligned
packets with an error in each frame, the histogram of bit errors per packet, the packet error rate.  The counters are
checked against a host recount of the same records (numpy, vectorised) in the same run.

Timing, CUDA events after warm-up, medians over the repetitions:
  batch        one cold-started sc_rx_packets_dev batch
  counter_l2   sc_packet_ber_stats_dev, `launches` back-to-back launches per repetition (its inputs stay in L2)
  counter_hbm  one launch per repetition after a 512 MB buffer has been overwritten (its inputs come from HBM)
The counter is timed with the 13 groups (each block sums in shared memory), with the same 13 groups among 129
(above 128 groups the atomics go to global memory directly) and with one group.
--dd decodes the packets with the decision-directed equalizer (SC_FLAG_PACKET_DD) instead of the reference's.
usage: python tools/packet_ber_curve.py [--out FILE] [--reps R] [--warmup W] [--launches L] [--streams N] [--dd]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import singlecarrier_b200 as sc  # noqa: E402
from singlecarrier_b200 import harness  # noqa: E402

NF, FRAME, PK_BYTES, N_GROUPS = 42, 1880, 96, 13


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def host_recount(pk, res, wl, group):
    """The counters from the records on the host: alignment as in the header, errors by comparing unpacked bits."""
    lead = wl.lead.cpu().numpy().astype(np.int64)
    tx = wl.tx_bits.cpu().numpy() & 1
    period = FRAME + wl.gap
    s, n = pk["stream"].astype(np.int64), pk["call_index"].astype(np.int64)
    keep = (s >= 0) & (s < res.shape[0]) & (n >= 2) & (n < NF)
    s, n, pk = s[keep], n[keep], pk[keep]
    pos = (n - 2) * FRAME + 5 * pk["max_index"].astype(np.int64) + res["rx_timing"][s, n - 2].astype(np.int64) - 48 \
        - lead[s]
    j = np.floor_divide(pos + period // 2, period)
    ok = (j >= 0) & (j < wl.n_packets) & (np.abs(pos - j * period) <= 10)
    err = (sc.unpack_packet_bits(pk[ok]) != tx[s[ok], j[ok]]).sum(-1)        # [aligned, 8]
    tot = err.sum(-1)
    b = np.where(tot == 0, 0, np.minimum(7, np.floor(np.log2(np.maximum(tot, 1))).astype(np.int64) + 1))
    c = np.zeros((N_GROUPS, 32), np.int64)
    g, ga = group[s], group[s[ok]]
    np.add.at(c[:, 0], g, 1)
    np.add.at(c[:, 1], ga, 1)
    c[:, 2] = 496 * c[:, 1]
    np.add.at(c[:, 3], ga, tot)
    for f in range(8):
        np.add.at(c[:, 8 + f], ga, err[:, f])
        np.add.at(c[:, 16 + f], ga, (err[:, f] > 0).astype(np.int64))
    np.add.at(c, (ga, 24 + b), 1)
    return c


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--streams", type=int, default=65536)
    ap.add_argument("--seed", type=int, default=0xBE4C)
    ap.add_argument("--dd", action="store_true", help="decode with the decision-directed equalizer (SC_FLAG_PACKET_DD)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_ber_curve needs a CUDA device"
    out = {"gpu": gpu_info(), "reps": a.reps, "warmup": a.warmup, "launches": a.launches, "dd": a.dd}
    ns, dev = a.streams, torch.device("cuda", 0)
    bank = sc.ModemBank(ns, packet=True, dd=a.dd)
    wl = harness.synthesize(bank, NF * FRAME, seed=a.seed, config=3)
    cap = ns * 8
    res = torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev)
    pk = torch.empty(cap * PK_BYTES, dtype=torch.uint8, device=dev)
    n_found = torch.zeros(1, dtype=torch.int64, device=dev)
    group = wl.ebn0_db.to(torch.int32)
    scratch = torch.zeros((129, 32), dtype=torch.int64, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def batch():
        bank.reset()
        n_found.zero_()
        bank.rx_packets_dev(wl.samples, NF, res, pk, n_found)

    def counter(grp, n_grp):
        bank.packet_ber_stats(pk, n_found, res, NF, wl.tx_bits, wl.lead, wl.gap, scratch[:n_grp], group=grp,
                              n_groups=n_grp)

    def timed(fn, k=1, before=None):
        if before:
            before()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    variants = {"13_groups": lambda: counter(group, N_GROUPS), "13_of_129_groups": lambda: counter(group, 129),
                "1_group": lambda: counter(None, 1)}
    for _ in range(a.warmup):
        batch()
        for v in variants.values():
            v()
    torch.cuda.synchronize()
    times = {"batch": []}
    for name in variants:
        times[f"counter_l2_{name}"], times[f"counter_hbm_{name}"] = [], []
    for _ in range(a.reps):
        times["batch"].append(timed(batch))
        for name, v in variants.items():
            times[f"counter_l2_{name}"].append(timed(v, a.launches))
            times[f"counter_hbm_{name}"].append(timed(v, before=lambda: flush.fill_(1)))

    # the counters of the last batch's records, on one CUDA stream straight behind it, and the host recount
    batch()
    cnt = torch.zeros((N_GROUPS, 32), dtype=torch.int64, device=dev)
    bank.packet_ber_stats(pk, n_found, res, NF, wl.tx_bits, wl.lead, wl.gap, cnt, group=group, n_groups=N_GROUPS)
    torch.cuda.synchronize()
    c = cnt.cpu().numpy()
    n = int(n_found.item())
    assert n <= cap, "capacity"
    recs = pk[: n * PK_BYTES].cpu().numpy().view(sc.PACKET_DTYPE)
    host = host_recount(recs, res.cpu().numpy().view(sc.RESULT_DTYPE), wl, wl.ebn0_db.cpu().numpy().astype(np.int64))
    bank.close()

    med = {k: statistics.median(v) for k, v in times.items()}
    out["workload"] = {"streams": ns, "calls": NF, "config": 3, "records": n, "aligned": int(c[:, 1].sum()),
                       "records_counted": int(c[:, 0].sum())}
    out["timing_ms"] = {k: {"median": round(med[k], 5), "all": [round(x, 5) for x in v]} for k, v in times.items()}
    out["counter_over_batch"] = round(med["counter_hbm_13_groups"] / med["batch"], 6)
    out["device_equals_host_recount"] = bool(np.array_equal(c, host))
    r4 = lambda x: round(float(x), 4)  # noqa: E731
    curve = []
    for g in range(N_GROUPS):
        al = int(c[g, 1])
        curve.append({"ebn0_db": g, "records": int(c[g, 0]), "aligned": al,
                      "ber": r4(c[g, 3] / max(c[g, 2], 1)),
                      "ber_per_frame": [r4(c[g, 8 + f] / max(62 * al, 1)) for f in range(8)],
                      "frames_in_error": [r4(c[g, 16 + f] / max(al, 1)) for f in range(8)],
                      "error_histogram": c[g, 24:].tolist(),
                      "per": r4((al - c[g, 24]) / max(al, 1))})
    out["curve"] = curve
    tot = c.sum(0)
    out["all"] = {"aligned": int(tot[1]), "ber": r4(tot[3] / max(tot[2], 1)),
                  "ber_per_frame": [r4(tot[8 + f] / max(62 * tot[1], 1)) for f in range(8)],
                  "error_histogram": tot[24:].tolist(), "per": r4((tot[1] - tot[24]) / max(tot[1], 1))}
    out["gpu_after"] = gpu_info()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

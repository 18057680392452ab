"""Cost of the packet soft output, and the constellation of the packet symbols.

Workload: 131,072 streams x 42 calls (10 s at 8 kHz), harness.synthesize(config=4) on a SC_FLAG_PACKET bank, input
resident in HBM.  After a warm-up of each, every repetition times `steps` batches of
  plain   sc_rx_packets_dev
  soft    sc_rx_packets_soft_dev, packet symbols only
  soft+   sc_rx_packets_soft_dev with the per-call symbols as well
with CUDA events, in that order.  Results and packet records (as sets keyed by stream and call) are checked identical
between the three.  For each data frame 1..8 of the packets that sit on a transmitted packet it reports the RMS error
vector of the packet symbols against the transmitted QPSK point (+-1 +-1j, the slicer's reference; transmitted dibit =
payload XOR packet keystream) and the bit error rate.  Prints one JSON object.
usage: python tools/packet_soft_bench.py [--out FILE] [--steps K] [--reps R] [--warmup W] [--streams N]"""
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

SPP, FRAME, NF, PK_BYTES, PK_SYM_BYTES, CALL_SYM_BYTES = 80000, 1880, 42, 96, 248 * 8, 31 * 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def sorted_records(pk_bytes, n):
    pk = pk_bytes[: n * PK_BYTES].cpu().numpy().view(sc.PACKET_DTYPE)
    order = np.lexsort((pk["call_index"], pk["stream"]))
    return pk, order


def constellation(res, pk, psym, wl):
    """Per data frame of the packets aligned to a transmitted packet: RMS |sym - transmitted point| and BER."""
    lead = wl.lead.cpu().numpy().astype(np.int64)
    tx = wl.tx_bits.cpu().numpy()                                      # payload bits [ns, n_packets, 8, 62]
    period = FRAME + wl.gap
    s_, c_ = pk["stream"].astype(np.int64), pk["call_index"].astype(np.int64)
    t_prev = res["rx_timing"][s_, c_ - 2].astype(np.int64)            # rx_timing at entry of call n-1
    pos = (c_ - 2) * FRAME + 5 * pk["max_index"].astype(np.int64) + t_prev - 48 - lead[s_]
    j = np.rint(pos / period).astype(np.int64)
    ok = (j >= 0) & (j < tx.shape[1]) & (np.abs(pos - j * period) <= 10)
    key = np.array([sc.packet_keystream_word(f) for f in range(8)], np.uint64)
    kbits = ((key[:, None] >> np.arange(62, dtype=np.uint64)) & np.uint64(1)).astype(np.uint8)   # [8, 62]
    sent = tx[s_[ok], j[ok]] ^ kbits[None]                             # transmitted (scrambled) dibits [m, 8, 62]
    point = ((1.0 - 2.0 * sent[..., 1::2]) + 1j * (1.0 - 2.0 * sent[..., 0::2])).astype(np.complex64)   # [m, 8, 31]
    sym = psym[ok].reshape(-1, 8, 31)
    ev = np.abs(sym.astype(np.complex128) - point)
    rms = np.sqrt((ev ** 2).mean(axis=(0, 2)))
    bits = sc.unpack_packet_bits(pk[ok])
    ber = (bits != tx[s_[ok], j[ok]]).mean(axis=(0, 2))
    mag = np.abs(sym).astype(np.float64)
    r4 = lambda a: [round(float(x), 4) for x in a]                     # noqa: E731
    return {"aligned_packets": int(ok.sum()), "packets": int(len(pk)),
            "rms_error_vector_per_frame": r4(rms),
            "median_error_vector_per_frame": r4(np.median(ev.transpose(1, 0, 2).reshape(8, -1), axis=1)),
            "mean_abs_symbol_per_frame": r4(mag.mean(axis=(0, 2))),
            "median_abs_symbol_per_frame": r4(np.median(mag.transpose(1, 0, 2).reshape(8, -1), axis=1)),
            "p90_abs_symbol_per_frame": r4(np.percentile(mag.transpose(1, 0, 2).reshape(8, -1), 90, axis=1)),
            "ber_per_frame": r4(ber)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--seed", type=int, default=0x5C0DE5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "packet_soft_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "steps": a.steps, "reps": a.reps, "warmup": a.warmup}
    ns = a.streams
    dev = torch.device("cuda", 0)
    bank = sc.ModemBank(ns, packet=True)
    wl = harness.synthesize(bank, SPP, seed=a.seed, config=4)
    cap = ns * 8
    res = {k: torch.empty((ns, NF * 32), dtype=torch.uint8, device=dev) for k in ("plain", "soft", "soft+")}
    pks = {k: torch.empty(cap * PK_BYTES, dtype=torch.uint8, device=dev) for k in res}
    cnt = {k: torch.zeros(1, dtype=torch.int64, device=dev) for k in res}
    psym = torch.empty((cap, 248), dtype=torch.complex64, device=dev)
    csym = torch.empty((ns, NF, 31), dtype=torch.complex64, device=dev)

    def run(kind):
        bank.reset()
        cnt[kind].zero_()
        if kind == "plain":
            bank.rx_packets_dev(wl.samples, NF, res[kind], pks[kind], cnt[kind])
        else:
            bank.rx_packets_soft_dev(wl.samples, NF, res[kind], pks[kind], cnt[kind], psym,
                                     symbols=csym if kind == "soft+" else None)

    kinds = ("plain", "soft", "soft+")
    for _ in range(a.warmup):
        for k in kinds:
            run(k)
    torch.cuda.synchronize()
    times = {k: [] for k in kinds}
    for _ in range(a.reps):
        for k in kinds:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                run(k)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / a.steps)
    n = {k: int(cnt[k].item()) for k in kinds}
    assert n["plain"] <= cap, "capacity"
    recs = {k: sorted_records(pks[k], n[k]) for k in kinds}
    same_results = all(torch.equal(res["plain"], res[k]) for k in kinds)
    p0, o0 = recs["plain"]
    same_records = all(n[k] == n["plain"] and recs[k][0][recs[k][1]].tobytes() == p0[o0].tobytes() for k in kinds)
    med = {k: statistics.median(v) for k, v in times.items()}
    sym_steps = ns * NF * 376
    out["workload"] = {"streams": ns, "calls": NF, "config": 4, "packets": n["plain"],
                       "packets_per_call": round(n["plain"] / (ns * NF), 4)}
    out["timing"] = {k: {"ms_median": round(med[k], 3), "ms_all": [round(x, 3) for x in times[k]],
                         "gsym_s": round(sym_steps / (med[k] * 1e-3) / 1e9, 3),
                         "over_plain": round(med[k] / med["plain"], 4)} for k in kinds}
    out["extra_bytes"] = {"soft_packet_symbols_gb": round(n["plain"] * PK_SYM_BYTES / 1e9, 4),
                          "soft+_call_symbols_gb": round(ns * NF * CALL_SYM_BYTES / 1e9, 4)}
    out["results_identical"] = bool(same_results)
    out["records_identical"] = bool(same_records)
    pk, _ = recs["soft+"]                                              # psym holds the last soft+ batch's blocks
    out["constellation"] = constellation(res["plain"].cpu().numpy().view(sc.RESULT_DTYPE), pk,
                                         psym[: n["soft+"]].cpu().numpy(), wl)
    bank.close()
    out["gpu_after"] = gpu_info()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

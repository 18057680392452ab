"""Cost of the soft output: sc_rx_frames_dev against sc_rx_frames_soft_dev (and the _host pair), alternating in one
process on the same input, after a warm-up of both.

  large   bench.py's workload: 131,072 streams x 42 calls, input resident in HBM (serial call chain, one thread per
          stream -- the bank is above SC_OVERLAP_MAX)
  small   1,024 streams x 42 calls, input resident in HBM (overlapped chains, cooperative tracker)
  host    the host entry points end to end from pinned memory (copies in, kernels, results and symbols out)

Each repetition times `steps` batches of the plain entry point, then `steps` of the soft one, with CUDA events (host:
a wall clock around work that ends in a synchronise).  The soft output adds 248 B per stream-frame (31 complex
floats) to the 3,760 B of samples read and the 32 B result written.  Results are checked byte-identical between
the two entry points.  Prints one JSON object.
usage: python tools/soft_bench.py [--out FILE] [--steps K] [--reps R] [--host-streams N]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import singlecarrier_b200 as sc  # noqa: E402
from bench import synth_input  # noqa: E402

FRAME, SYM_PER_FRAME, SOFT_BYTES, IN_BYTES, RES_BYTES = 1880, 376, 248, 3760, 32
SPP = 80000                      # samples per stream, as bench.py: 10 s at 8 kHz = 42 calls


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def summary(ns, nf, plain_ms, soft_ms):
    p, s = statistics.median(plain_ms), statistics.median(soft_ms)
    gsym = lambda ms: ns * nf * SYM_PER_FRAME / (ms * 1e-3) / 1e9       # noqa: E731
    return {"streams": ns, "calls": nf, "plain_ms_median": round(p, 4), "soft_ms_median": round(s, 4),
            "plain_ms_all": [round(x, 4) for x in plain_ms], "soft_ms_all": [round(x, 4) for x in soft_ms],
            "plain_gsym_s": round(gsym(p), 4), "soft_gsym_s": round(gsym(s), 4), "soft_over_plain_time": round(s / p, 4),
            "extra_bytes_per_stream_frame": SOFT_BYTES, "plain_bytes_per_stream_frame": IN_BYTES + RES_BYTES,
            "extra_bytes_fraction": round(SOFT_BYTES / (IN_BYTES + RES_BYTES), 4)}


def run_dev(ns, nf, seed, steps, reps, warmup):
    dev = torch.device("cuda", 0)
    bank = sc.ModemBank(ns)
    d_in = synth_input(sc, torch, bank, ns, SPP, seed, 0)
    res_p = torch.empty((ns, nf * 32), dtype=torch.uint8, device=dev)
    res_s = torch.empty_like(res_p)
    sym = torch.empty((ns, nf * 62), dtype=torch.float32, device=dev)

    def plain():
        bank.reset()
        bank.rx_frames_dev(d_in, nf, res_p)

    def soft():
        bank.reset()
        bank.rx_frames_soft_dev(d_in, nf, res_s, sym)

    for _ in range(warmup):
        plain()
        soft()
    torch.cuda.synchronize()
    times = {plain: [], soft: []}
    for _ in range(reps):
        for fn in (plain, soft):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[fn].append(e0.elapsed_time(e1) / steps)
    same = bool(torch.equal(res_p, res_s))
    bank.close()
    out = summary(ns, nf, times[plain], times[soft])
    out["results_identical"] = same
    return out


def run_host(ns, nf, seed, steps, reps, warmup):
    bank = sc.ModemBank(ns)
    d_in = synth_input(sc, torch, bank, ns, SPP, seed, 0)
    buf = sc.PinnedBuffer(ns * SPP * 2 + ns * nf * (32 + 32 + SOFT_BYTES))
    x = buf.array(np.int16, (ns, SPP))
    x[:] = d_in.cpu().numpy()
    del d_in
    off = ns * SPP * 2
    res_p = buf.array(sc.RESULT_DTYPE, (ns, nf), off)
    res_s = buf.array(sc.RESULT_DTYPE, (ns, nf), off + ns * nf * 32)
    sym = buf.array(np.complex64, (ns, nf, 31), off + ns * nf * 64)

    def plain():
        bank.reset()
        sc._lib.check(sc.lib.sc_rx_frames_host(bank._h, x.ctypes.data, SPP, nf, res_p.ctypes.data, nf, None))

    def soft():
        bank.reset()
        sc._lib.check(sc.lib.sc_rx_frames_soft_host(bank._h, x.ctypes.data, SPP, nf, res_s.ctypes.data, nf,
                                                    sym.ctypes.data))

    for _ in range(warmup):
        plain()
        soft()
    times = {plain: [], soft: []}
    for _ in range(reps):
        for fn in (plain, soft):
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()                                   # returns after everything has landed
            times[fn].append((time.perf_counter() - t0) * 1e3 / steps)
    same = res_p.tobytes() == res_s.tobytes()
    bank.close()
    out = summary(ns, nf, times[plain], times[soft])
    out["results_identical"] = same
    buf.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON here")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--streams", type=int, default=131072)
    ap.add_argument("--small-streams", type=int, default=1024)
    ap.add_argument("--host-streams", type=int, default=16384)
    ap.add_argument("--seed", type=int, default=0x5C0DE5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "soft_bench needs a CUDA device"
    out = {"gpu": gpu_info(), "steps": a.steps, "reps": a.reps, "warmup": a.warmup}
    nf = SPP // FRAME
    out["large"] = run_dev(a.streams, nf, a.seed, a.steps, a.reps, a.warmup)
    out["small"] = run_dev(a.small_streams, nf, a.seed + 1, 4 * a.steps, a.reps, a.warmup)
    out["host"] = run_host(a.host_streams, nf, a.seed + 2, max(1, a.steps // 2), a.reps, a.warmup)
    out["gpu_after"] = gpu_info()
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()

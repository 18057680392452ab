#!/usr/bin/env python
"""bench.py -- demodulated Msym/s of the batched RX chain on B200 (BASELINE.json metric).

A "step" is one cold-start pass of the RX hot path (N lock-step copies of the reference's
``while(1){fread; qpsk_rx_frame()}`` loop, /root/reference/src/qpsk.c:436-458) over one batch of
synthetic streams.  Workload at every N: BASELINE.json configs[3]'s per-GPU shard -- 131,072
streams per GPU (1M streams on 8 GPUs), 10 s = 80,000 samples = 42 calls each, weak scaling.
Input is synthesised on the device by the library's own TX + channel kernels (reference packet
structure, random frequency/phase offset, AWGN at Eb/N0 0..12 dB), 21 GB per GPU, so every step
streams far more than the 126 MB L2.

  value     whole-job Msym/s with the int16 samples already resident in HBM (CUDA events, max over ranks)
  e2e       the same metric through the host-buffer entry point (sc_rx_frames_host): pinned host samples
            -> H2D -> kernels -> D2H results, all inside the timed region
  roofline  the dominant kernel's algorithmic bytes / its average launch duration, measured live with
            CUDA events on the launching stream (single slab, so launches do not overlap)
  cpu_baseline  the reference's own C objects (oracle/_ref) -- or the oracle port when absent -- timed on
            this box's host cores on a bounded sample of the same input (rank 0, N=1 only)

``--impl reference`` times only that CPU implementation (all host threads) and prints the same line
with "impl": "reference".

``--dump-outputs DIR`` writes what the last timed step computed (rank 0's results for a seeded sample of
its streams, and the lock/bit counters) as float32 / float64 .npy files, so that two builds run with the
same arguments can be compared output for output (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME = 1880
SYM_PER_FRAME = 376
METRIC = "demodulated_msym_per_s"
UNIT = "Msym/s"

# algorithmic bytes / FP32 operations per stream-frame (DESIGN.md section 5)
FE_BYTES = 1494 * 2 + 198 * 8 + 8          # int16 samples the 290 decimated outputs depend on + tracker window + (idx,val)
TK_BYTES = 198 * 8 + 12 + 32 + 4           # tracker window + (idx,val,timing) + result record + timing
CHAIN_BYTES = 1880 * 2 + 32                # int16 frame in + result record out
FE_OPS = 2 * 1494 + 290 * 198 + 2 * 255 + 128 * 128 * 2 + 128 * 3
TK_OPS = 128 * 398 + 31 * 397


def ncu_traffic():
    """DRAM traffic per stream-frame of the two RX kernels, parsed from the newest committed
    profiles/rNN_ncu_raw.csv (written by tools/profile_summary.py from one `ncu --set full` capture; the
    first line carries the git hash the capture was taken at).  {kernel: (bytes per stream-frame, source)}."""
    import csv
    import glob
    out = {}
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_raw.csv")))
    if not files:
        return out
    path = files[-1]
    rows = list(csv.reader(open(path)))
    git = rows[0][1] if rows and len(rows[0]) > 1 else "?"
    per = {}
    for r in rows[2:]:
        if len(r) < 6 or r[3] not in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            continue
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r[4], 1.0)
        grid = int(r[1].strip("()").split(",")[0])
        k = per.setdefault(r[0], {"grid": grid, "bytes": 0.0})
        k["bytes"] += float(r[5]) * scale
    for name, k in per.items():
        # frontend_kernel: 4 streams per CTA; track_kernel: 128 streams per CTA
        streams = k["grid"] * (4 if "frontend" in name else 128)
        key = "frontend_kernel" if "frontend" in name else "track_kernel" if "track_kernel" in name else name
        out[key] = (k["bytes"] / streams, f"{os.path.relpath(path, ROOT)} (ncu --set full, dram__bytes_read.sum + "
                    f"dram__bytes_write.sum of a {streams}-stream launch, captured at git {git}), scaled to this launch's streams")
    return out


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("sm_max_mhz", 1965.0)), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML from a background thread,
    every 5 ms; falls back to `nvidia-smi -lms` when NVML is unavailable)."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = False
        self._thread = None
        self._proc = None
        self._path = None

    def _run(self, pynvml, h):
        while not self._stop:
            try:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self._thread = threading.Thread(target=self._run, args=(pynvml, h), daemon=True)
            self._thread.start()
            return
        except Exception:
            self._thread = None
        try:
            fd, self._path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                           "--format=csv,noheader,nounits", "-lms", "100"],
                                          stdout=open(self._path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self._proc = None

    def mark(self):
        """Call at the start of the timed region: earlier samples (warm-up) are dropped."""
        self.samples = []

    def stop(self) -> dict:
        if self._thread is not None:
            self._stop = True
            self._thread.join(timeout=2)
            sm = self.samples
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_min_mhz": float(min(sm)) if sm else None,
                    "sm_max_mhz": self.max_mhz, "samples": len(sm), "reasons": sorted(self.reasons), "source": "nvml, 5 ms"}
        if self._proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no clock source available"]}
        self._proc.terminate()
        try:
            self._proc.wait(timeout=5)
        except Exception:
            self._proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self._path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self._path)
        busy = sorted(sm)[len(sm) // 2:] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100 (incl. warm-up)"}


def synth_input(sc, torch, bank, streams, samples_per_stream, seed, rank):
    """Device-side synthesis of the step's input: reference packet structure + channel."""
    dev = torch.device("cuda", bank.device)
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 7919 * rank)
    period = FRAME + 903
    n_packets = (samples_per_stream + period - 1) // period + 1
    lead = torch.randint(0, period, (streams,), generator=g, device=dev, dtype=torch.int32)
    df = (torch.rand(streams, generator=g, device=dev) * 40.0 - 20.0).float()
    phi = (torch.rand(streams, generator=g, device=dev) * (2 * np.pi)).float()
    ebn0_db = (torch.arange(streams, device=dev) % 13).float()            # 0..12 dB
    # real AWGN: sigma^2 = P_sig * Fs / (2 * Rs * Es/N0), Es/N0 = 2 Eb/N0 (SURVEY 8d); P_sig of the data section
    p_sig = 0.5 * (16384.0 * 0.48) ** 2 * 2.0
    esn0 = 2.0 * 10.0 ** (ebn0_db / 10.0)
    sigma = torch.sqrt(torch.tensor(p_sig, device=dev) * 8000.0 / (2.0 * 1600.0 * esn0)).float()
    out = torch.empty((streams, samples_per_stream), dtype=torch.int16, device=dev)
    bank.tx_packets_dev(out, n_packets, gap_samples=903, seed=seed + rank, lead_in=lead,
                        channel={"df_hz": df, "phi_rad": phi, "sigma_lsb": sigma})
    torch.cuda.synchronize(dev)
    return out


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation on this box's host cores.  Nothing of the
    product is loaded: the input is synthesised on the CPU by the workers themselves (oracle TX + numpy channel,
    the same packet structure / offsets / AWGN ladder as the device generator), then every reference build that
    can run here is timed -- the parity-flag build all parity claims are pinned to, and the -O3 AVX2/AVX-512
    builds.  The line's value is the FASTEST of them, so the speed-up quoted against it is the conservative one."""
    if rank != 0:
        return
    from oracle import cpu_bench
    from oracle import pyoracle as po
    po.build()
    n_frames = args.seconds * 8000 // FRAME
    streams = args.ref_streams
    source = f"synth:{args.seed}:{streams}"
    builds = cpu_bench.available_builds() if po.have_ref() else []
    if not builds:
        builds = ["port"]
    runs = {}
    for bname in builds:
        r = cpu_bench.run(source, n_frames, None, args.warmup + args.steps, bname)
        walls = r["wall_s"][args.warmup:]
        total_sym = r["streams"] * n_frames * SYM_PER_FRAME * len(walls)
        runs[bname] = {"value": total_sym / sum(walls) / 1e6, "ms_per_step": 1e3 * sum(walls) / len(walls), "cores": r["cores"],
                       "kind": r["kind"], "flags": r["flags"], "valid_frames": r["valid_frames"], "streams": r["streams"]}
    best = max(runs, key=lambda k: runs[k]["value"])
    rb = runs[best]
    value = rb["value"]
    sample_desc = (f"{rb['streams']} streams x {n_frames} calls per step of the same workload, synthesised on the CPU "
                   f"(oracle TX + numpy channel); {rb['cores']} processes, one per core; build '{best}' ({rb['flags']}) is the "
                   f"fastest of {sorted(runs)} and is the one quoted")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": rb["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, streams_override=rb["streams"]),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": rb["cores"], "kind": rb["kind"], "sample": sample_desc,
                         "build": best, "flags": rb["flags"]},
        "cpu_builds": {k: {"value": v["value"], "flags": v["flags"], "ms_per_step": v["ms_per_step"]} for k, v in runs.items()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_RESULT_BUDGET = 48 << 20             # bytes of sampled per-call results; the whole dump stays under 64 MB
DUMP_MAX_STREAMS = 16384


def dump_outputs(out_dir, d_res, counters, n_frames, seed):
    """The timed step's outputs as .npy: for a fixed sample of streams (chosen by --seed; every stream when the
    bank is small enough) each field of the sc_frame_result records the step returned, plus the 16 lock/bit
    counters.  Integer fields are stored as float32 (all exact); the 62 packed bits as two float64 halves
    (bits 0-31 and 32-61) so that they stay exact; the counters as float64."""
    import singlecarrier_b200 as sc
    import torch
    streams = d_res.shape[0]
    per_stream = n_frames * (7 * 4 + 2 * 8)
    k = max(1, min(streams, DUMP_MAX_STREAMS, DUMP_RESULT_BUDGET // per_stream))
    idx = np.sort(np.random.default_rng(seed).choice(streams, k, replace=False))
    rows = d_res[torch.from_numpy(idx).to(d_res.device)].cpu().numpy()
    res = np.ascontiguousarray(rows).view(sc.RESULT_DTYPE).reshape(k, n_frames)
    os.makedirs(out_dir, exist_ok=True)
    out = {"results_stream_index": idx.astype(np.float64)}
    for name in ("valid", "max_index", "matches", "rx_timing", "call_index", "max_value", "cost"):
        out["results_" + name] = res[name].astype(np.float32)
    bits = res["bits"].astype(np.uint64)
    out["results_bits_lo32"] = (bits & np.uint64(0xFFFFFFFF)).astype(np.float64)
    out["results_bits_hi32"] = (bits >> np.uint64(32)).astype(np.float64)
    out["lock_stats"] = counters.cpu().numpy().astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(args, streams_override=None):
    return {
        "workload": "BASELINE.json configs[3] per-GPU shard: 131072 streams/GPU x 10 s (1M streams on 8 GPUs), "
                    "reference packets (640 preamble + 8x155 data + 903 dead air), df~U(-20,20) Hz, random phase, "
                    "AWGN Eb/N0 0..12 dB",
        "streams_per_gpu": streams_override if streams_override is not None else args.streams,
        "seconds_per_stream": args.seconds, "calls_per_stream": args.seconds * 8000 // FRAME,
        "samples_per_stream": args.seconds * 8000, "l2": "input per step (>= 2.6 GB at defaults) >> 126 MB L2; no flush needed",
        "filter": "alpha=0.35 (firwide=false)", "parallelism": "streams sharded by rank, no hot-path collective",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=131072, help="streams per GPU")
    ap.add_argument("--seconds", type=int, default=10, help="seconds of 8 kHz audio per stream")
    ap.add_argument("--seed", type=int, default=0x5C0DE5)
    ap.add_argument("--ref-streams", type=int, default=4096, help="streams per step of the CPU reference arm")
    ap.add_argument("--cpu-streams", type=int, default=4096, help="streams of the cpu_baseline sample")
    ap.add_argument("--slab-parts", type=int, default=0, help="override the library's slab split (0 = default)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.slab_parts > 0:
        os.environ["SC_SLAB_PARTS"] = str(args.slab_parts)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import singlecarrier_b200 as sc
    from singlecarrier_b200.modem import OPT_PROFILE, OPT_SLAB_PARTS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; singlecarrier_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    streams, spp = args.streams, args.seconds * 8000
    n_frames = spp // FRAME
    bank = sc.ModemBank(streams, device=local_rank)
    d_in = synth_input(sc, torch, bank, streams, spp, args.seed, rank)
    d_res = torch.empty((streams, n_frames * 32), dtype=torch.uint8, device=dev)
    counters = torch.zeros(16, dtype=torch.int64, device=dev)
    stream_handle = torch.cuda.current_stream(dev).cuda_stream
    # the path's only collective lives in the C ABI (sc_reduce_stats -> ncclAllReduce); torch.distributed only
    # carries the NCCL unique id to the other ranks and provides the barrier / max-over-ranks of the timing
    comm = None
    if world > 1:
        ids = [sc.NcclComm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        comm = sc.NcclComm.init_rank(world, rank, ids[0], local_rank)

    def step():
        bank.reset()
        bank.rx_frames_dev(d_in, n_frames, d_res, stream=stream_handle)
        counters.zero_()
        bank.lock_stats(d_res, n_frames, counters, stream=stream_handle)
        if comm is not None:
            comm.all_reduce_counters(counters, stream=stream_handle)   # the only collective: lock / bit statistics

    sampler = ClockSampler(local_rank)          # started before the warm-up (same workload) so that
    sampler.start()                             # nvidia-smi is already sampling when the timed steps run
    for _ in range(args.warmup):
        step()
    barrier()
    sampler.mark()
    launches0 = sc.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    launches = sc.launch_count() - launches0
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    sym_per_step = world * streams * n_frames * SYM_PER_FRAME
    value = sym_per_step * args.steps / (ms_total * 1e-3) / 1e6
    stats = counters.cpu().numpy().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_res, counters, n_frames, args.seed)      # before the passes below reuse d_res

    # ---- roofline: per-kernel durations with events on the launching stream, one slab ----------------
    hbm_peak, sm_max, peak_src = peaks()
    bank.set_option(OPT_SLAB_PARTS, 1)
    bank.set_option(OPT_PROFILE, 1)
    bank.reset()
    bank.rx_frames_dev(d_in, n_frames, d_res, stream=stream_handle)
    prof = bank.profile_read()
    # the same pass with the front-end's search proposed on tcgen05 (SC_FE_SEARCH_TCGEN05, opt-in; sc_frontend_umma.cu):
    # per-launch time of that kernel, and that every result byte is the same
    from singlecarrier_b200.modem import FE_SEARCH_DIRECT, FE_SEARCH_TCGEN05, OPT_FE_SEARCH
    res_default = d_res.clone()
    bank.set_option(OPT_FE_SEARCH, FE_SEARCH_TCGEN05)
    bank.reset()
    bank.rx_frames_dev(d_in, min(n_frames, 3), d_res, stream=stream_handle)    # one-time set-up (attributes, the master table)
    bank.profile_read()
    bank.reset()
    bank.rx_frames_dev(d_in, n_frames, d_res, stream=stream_handle)
    prof_tc = bank.profile_read()
    fe_tc_ms = prof_tc["frontend_ms"] / max(prof_tc["frontend_launches"], 1)
    fe_tc_same = bool(torch.equal(res_default, d_res))
    del res_default
    bank.set_option(OPT_FE_SEARCH, FE_SEARCH_DIRECT)
    bank.set_option(OPT_PROFILE, 0)
    bank.set_option(OPT_SLAB_PARTS, args.slab_parts)
    fe_ms = prof["frontend_ms"] / max(prof["frontend_launches"], 1)
    tk_ms = prof["track_ms"] / max(prof["track_launches"], 1)
    clk = (clocks.get("sm_mhz") or sm_max) * 1e6
    fp32_peak = 148 * 128 * clk

    def roof(name, ms_launch, bytes_sf, ops_sf, traffic_sf):
        gbs = streams * bytes_sf / (ms_launch * 1e-3) / 1e9
        ops = streams * ops_sf / (ms_launch * 1e-3)
        return {"kernel": name, "bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                "traffic": streams * traffic_sf[0] if traffic_sf else None,
                "traffic_source": traffic_sf[1] if traffic_sf else "no committed profiles/rNN_ncu_raw.csv",
                "algorithmic_bytes_per_launch": streams * bytes_sf,
                "ms_per_launch": ms_launch, "bytes_per_stream_frame": bytes_sf,
                "fp32_issue": {"achieved_tops": ops / 1e12, "peak_tops": fp32_peak / 1e12, "frac": ops / fp32_peak,
                               "ops_per_stream_frame": ops_sf, "note": "exact-order FP32 (no FMA): the true bound, SURVEY F8"}}

    traffic = ncu_traffic()
    fe = roof("frontend_kernel", fe_ms, FE_BYTES, FE_OPS, traffic.get("frontend_kernel"))
    tk = roof("track_kernel", tk_ms, TK_BYTES, TK_OPS, traffic.get("track_kernel"))
    dom, other = (tk, fe) if tk_ms >= fe_ms else (fe, tk)
    roofline = dict(dom)
    roofline["peak_source"] = peak_src
    roofline["timing"] = ("CUDA events around every launch, on the launching stream, in one extra single-slab pass over the "
                          "same input right after the timed steps (the timed steps run two slabs on two streams, whose "
                          "launches overlap and cannot be timed individually)")
    roofline["other_kernel"] = other
    roofline["frontend_tcgen05"] = {
        "kernel": "frontend_umma_kernel", "ms_per_launch": fe_tc_ms, "identical_results": fe_tc_same,
        "note": "opt-in mode SC_OPT_FE_SEARCH = SC_FE_SEARCH_TCGEN05 (persistent, 16 FIR warps + 4 search warps per SM, "
                "proposer on tcgen05.mma, exact verification); not used by the timed steps"}
    chain_gbs = streams * n_frames * CHAIN_BYTES * args.steps / (ms_total * 1e-3) / 1e9
    roofline["chain"] = {"bytes_per_symbol": CHAIN_BYTES / SYM_PER_FRAME, "achieved_gbs": chain_gbs,
                         "frac_of_hbm": chain_gbs / hbm_peak,
                         "ops_per_symbol": (FE_OPS + TK_OPS) / SYM_PER_FRAME,
                         "fp32_issue_frac": (value / world) * 1e6 * (FE_OPS + TK_OPS) / SYM_PER_FRAME / fp32_peak}

    # ---- BASELINE.json configs[1]: a 1,024-stream bank, where a call is latency- and not throughput-bound ----------
    small = None
    if rank == 0 and world == 1:
        small = run_small_bank(args, sc, torch, dev, n_frames)

    # ---- e2e: host buffers through sc_rx_frames_host ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, sc, torch, dist, bank, d_in, streams, n_frames, world, rank, dev, barrier)

    # ---- CPU baseline on a bounded sample (rank 0, N=1) --------------------------------------------
    cpu = None
    cpu_fast = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu, cpu_fast = run_cpu_baseline(args, d_in, n_frames)

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args),
            "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_fast": cpu_fast, "e2e": e2e, "small_bank": small,
            "gpu_launches": int(launches), "clocks": clocks,
            "collective": ("sc_reduce_stats (ncclAllReduce of 16 uint64 through the C ABI), once per step" if comm is not None
                           else "none at N=1"),
            "wall_ms_per_step": 1e3 * wall / args.steps,
            "realtime_factor": value * 1e6 / (world * streams * 1600.0),
            "lock_stats": {"calls": stats[0], "valid": stats[1], "sum_matches": stats[2], "bit_popcount": stats[5],
                           "bit_checksum": stats[6]},
        }
        print(json.dumps(line), flush=True)
    bank.close()
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def run_small_bank(args, sc, torch, dev, n_frames, streams=1024):
    """The same chain on a bank far too small to fill the GPU (BASELINE.json configs[1]), input resident in HBM: the
    library's default for this size (the even and the odd calls as two overlapped chains, lane-cooperative training
    kernel) beside the serial call-by-call chain the large bank uses.  Same results either way (tests)."""
    from singlecarrier_b200.modem import OPT_OVERLAP, OPT_TRACKER, OVERLAP_OFF, TRACKER_THREAD
    out = {"streams": streams, "unit": UNIT, "calls_per_step": n_frames, "steps": args.steps,
           "workload": "BASELINE.json configs[1]: 1,024 loop-back streams, random offset/phase, one bank on one GPU"}
    res = torch.empty((streams, n_frames * 32), dtype=torch.uint8, device=dev)
    for name, serial in (("value", False), ("serial_chain_value", True)):
        bank = sc.ModemBank(streams, device=dev.index)
        if serial:
            bank.set_option(OPT_OVERLAP, OVERLAP_OFF)
            bank.set_option(OPT_TRACKER, TRACKER_THREAD)
        d_in = synth_input(sc, torch, bank, streams, args.seconds * 8000, args.seed + 1, 0)
        for _ in range(args.warmup):
            bank.reset()
            bank.rx_frames_dev(d_in, n_frames, res)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            bank.reset()
            bank.rx_frames_dev(d_in, n_frames, res)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / args.steps
        out[name] = streams * n_frames * SYM_PER_FRAME / (ms * 1e-3) / 1e6
        out["us_per_call" if not serial else "serial_chain_us_per_call"] = 1e3 * ms / n_frames
        bank.close()
    return out


def run_e2e(args, sc, torch, dist, bank, d_in, streams, n_frames, world, rank, dev, barrier):
    """Host-buffer path: pinned int16 samples in, results out, copies inside the timed region.  Before it, every
    rank measures plain pinned-host -> device copies AT THE SAME TIME (sc_h2d_probe): that is the platform's
    PCIe / host-memory ceiling at this N, against which the end-to-end number is reported."""
    import psutil
    from singlecarrier_b200.modem import H2D_COLUMNS, H2D_COLUMNS_3D, H2D_FULL, OPT_H2D_MODE
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))

    def rank_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def rank_min(x):
        return -rank_max(-x)

    # ---- the ceiling: contiguous copies and the 3,248-byte-row pattern, all ranks concurrently ----------
    probe_bytes = 512 << 20
    barrier()
    contig = sc.h2d_probe(bank.device, probe_bytes, min_seconds=1.0)
    barrier()
    strided = sc.h2d_probe(bank.device, probe_bytes, row_bytes=1624 * 2, src_pitch_bytes=FRAME * 2 * n_frames, min_seconds=1.0)
    barrier()
    d2h = sc.h2d_probe(bank.device, 64 << 20, min_seconds=0.3, d2h=True)
    contig_min, strided_min = rank_min(contig), rank_min(strided)
    # Msym/s one GPU could reach if the host->device copy were the only cost, per copy pattern
    ceil_full = contig_min * 1e9 / (FRAME * 2 / SYM_PER_FRAME) / 1e6
    ceil_cols = strided_min * 1e9 / (1624 * 2 / SYM_PER_FRAME) / 1e6

    budget = psutil.virtual_memory().available * 0.6 / max(local_world, 1)
    e_streams = streams
    while e_streams * n_frames * FRAME * 2 > budget and e_streams > 1024:
        e_streams //= 2
    e_streams = int(rank_min(e_streams))                        # same size on every rank
    in_bytes = e_streams * n_frames * FRAME * 2
    pin_in = sc.PinnedBuffer(in_bytes, device=bank.device)       # page-locked on the GPU's NUMA node
    pin_res = sc.PinnedBuffer(e_streams * n_frames * 32, device=bank.device)
    x = pin_in.array(np.int16, (e_streams, n_frames * FRAME))
    r = pin_res.array(sc.RESULT_DTYPE, (e_streams, n_frames))
    torch.from_numpy(x).copy_(d_in[:e_streams, : n_frames * FRAME])
    ebank = bank if e_streams == streams else sc.ModemBank(e_streams, device=bank.device)

    def step():
        ebank.reset()
        ebank.rx_frames_host(x, n_frames, results=r)

    def timed(k):
        barrier()
        t0 = time.perf_counter()
        for _ in range(k):
            step()
        torch.cuda.synchronize(dev)
        return rank_max(time.perf_counter() - t0) / k

    # ---- pick the copy pattern by measurement (identical results in every mode) ------------------------------
    names = {H2D_COLUMNS: "columns (2-D copy per frame, 86 % of the bytes)", H2D_COLUMNS_3D: "columns (one 3-D copy per block)",
             H2D_FULL: "full frames (plain 1-D copies)"}
    trial = {}
    for mode in (H2D_COLUMNS, H2D_COLUMNS_3D, H2D_FULL):
        ebank.set_option(OPT_H2D_MODE, mode)
        step()
        trial[mode] = timed(2)
    best = min(trial, key=lambda m: trial[m])
    ebank.set_option(OPT_H2D_MODE, best)
    steps = args.steps
    h0, o0 = ebank.transfer_bytes()
    dt = timed(steps)
    h1, o1 = ebank.transfer_bytes()
    h2d, d2h_b = (h1 - h0) // steps, (o1 - o0) // steps
    val = world * e_streams * n_frames * SYM_PER_FRAME / dt / 1e6
    valid = int(r["valid"].sum())
    ebank.set_option(OPT_H2D_MODE, H2D_COLUMNS)
    if ebank is not bank:
        ebank.close()
    pcie = h2d / dt / 1e9
    pattern_peak = contig_min if best == H2D_FULL else strided_min
    ceiling = (ceil_full if best == H2D_FULL else ceil_cols)
    out = {"value": val, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h_b), "steps": steps,
           "streams_per_gpu": e_streams, "ms_per_step": 1e3 * dt,
           "api": "sc_rx_frames_host (pinned host int16 in, sc_frame_result out)",
           "timer": "host wall clock around the blocking call, max over ranks", "valid_calls_last_step": valid,
           "host_input_bytes_per_step": int(in_bytes), "pcie_gbs": pcie,
           "h2d_peak_gbs": contig_min,
           "h2d_probe": {"what": "sc_h2d_probe: plain cudaMemcpyAsync / cudaMemcpy2DAsync from pinned host memory, all ranks "
                                 "at the same time, >= 1 s each, CUDA events; min over ranks, per GPU",
                         "contiguous_gbs": contig_min, "rows_3248B_gbs": strided_min, "d2h_contiguous_gbs": rank_min(d2h),
                         "contiguous_gbs_max_rank": rank_max(contig), "rows_3248B_gbs_max_rank": rank_max(strided),
                         "ceiling_msym_per_gpu": {"full_frames": ceil_full, "columns": ceil_cols}},
           "h2d_mode": names[best], "h2d_mode_trials_ms": {names[m]: 1e3 * t for m, t in trial.items()},
           "frac_of_h2d_probe": pcie / pattern_peak if pattern_peak else None,
           "frac_of_h2d_ceiling": val / (world * max(ceil_full, ceil_cols)) if max(ceil_full, ceil_cols) else None,
           "pinned_numa_node": pin_in.numa_node}
    pin_in.close()
    pin_res.close()
    return out


def run_cpu_baseline(args, d_in, n_frames):
    """Rank 0, N=1: the reference's objects on a bounded sample of this run's own input -- the parity-flag build
    (cpu_baseline) and the fastest of the -O3 builds that can run on this CPU (cpu_baseline_fast)."""
    from oracle import cpu_bench
    ns = min(args.cpu_streams, d_in.shape[0])
    path = os.path.join(tempfile.gettempdir(), f"sc_cpu_sample_{os.getpid()}.npy")
    np.save(path, d_in[:ns, : n_frames * FRAME].cpu().numpy())

    def one(build):
        out = subprocess.run([sys.executable, "-m", "oracle.cpu_bench", path, str(n_frames), "0", "1"] + ([build] if build else []),
                             cwd=ROOT, capture_output=True, text=True, timeout=600)
        r = json.loads(out.stdout.strip().splitlines()[-1])
        return {"value": r["msym_per_s"][0], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "build": r["build"],
                "flags": r["flags"],
                "sample": f"first {r['streams']} streams x {n_frames} calls of rank 0's input "
                          f"({r['streams'] * n_frames} qpsk_rx_frame calls, {r['wall_s'][0]:.2f} s wall, one process per core)",
                "per_core": r["msym_per_s"][0] / r["cores"]}

    base, fast = None, None
    try:
        base = one(None)
        for b in cpu_bench.available_builds():
            if b == "parity":
                continue
            f = one(b)
            if fast is None or f["value"] > fast["value"]:
                fast = f
    except Exception as e:
        if base is None:
            base = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": f"failed: {e}"}
    finally:
        if os.path.exists(path):
            os.unlink(path)
    return base, fast


if __name__ == "__main__":
    main()

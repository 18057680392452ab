"""The numbers behind SC_FLAG_PACKET_ACQ's threshold tau (DESIGN.md section 8b), from the C specification on the CPU
(tests/packet_acq_ref.c): the stage-1 frame maximum of rho1 for
  loop-back streams   (tests/packet_dd_ref.loop_streams: 4 packets, gap 903, offsets -20 / 0 / +20 Hz), split into
                      frames whose accepted candidate lies within 4 samples of a packet start ("packet") and the others
  noise only          at the bench's largest sigma (Eb/N0 = 0 dB), 40 frames per stream
  dead air            all-zero samples
Accepted means: the first maximum passes the neighbour test (the threshold is what is being chosen).
usage: python tools/packet_acq_roc.py [--streams N] [--noise-streams M]"""
import argparse
import math
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import packet_acq_ref as A  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from packet_dd_ref import loop_streams  # noqa: E402
from singlecarrier_b200.harness import DATA_RMS_LSB  # noqa: E402


def sigma_of(ebn0_db):
    """harness.awgn_sigma in float64"""
    return math.sqrt(DATA_RMS_LSB ** 2 * 8000.0 / (2 * 1600.0 * 2.0 * 10 ** (ebn0_db / 10)))


def stage1(x, W, foff=0.0):
    """(k*, rho1(k*), passes the neighbour test) of every frame the spec searches"""
    filt = A.acq_filt(x, foffset=foff)
    nf = x.size // 1880
    r = A.acq_rho_lags(filt, -W, 376 * nf + 2 * W)                  # r[W + k] = rho1(k)
    out = []
    for f in range(nf - 2):
        seg = r[W + 376 * f: W + 376 * f + 376]
        kb = int(np.argmax(seg))
        best, k = seg[kb], 376 * f + kb
        ok = all(not (k - d < 376 * f and r[W + k - d] >= best) and not (k + d >= 376 * f + 376 and r[W + k + d] > best)
                 for d in range(1, W + 1))
        out.append((k, float(best), ok))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=60)
    ap.add_argument("--noise-streams", type=int, default=400)
    a = ap.parse_args()
    oracle = po.Oracle()
    tau, W, _ = A.acq_params()
    print(f"spec: tau {tau}, W {W}")

    def loop_job(args):
        sg, seed, foff = args
        x, _, st = loop_streams(oracle, np.random.default_rng(seed), 1, 4, sigma=sg)
        pk, other = [], []
        for k, b, ok in stage1(x[0], W, foff):
            if ok:
                (pk if np.abs(5 * k - (st[0] + 48)).min() <= 4 else other).append(b)
        return pk, other

    with ThreadPoolExecutor(max(1, min(32, os.cpu_count() or 1))) as ex:
        for name, sg in [("clean", 0.0), ("sigma 1500", 1500.0)] + [(f"{eb} dB", sigma_of(eb)) for eb in (0, 3, 6, 12)]:
            res = list(ex.map(loop_job, [(sg, 100 + i, 20.0 * (i % 3 - 1)) for i in range(a.streams)]))
            p = np.concatenate([np.array(r[0]) for r in res])
            o = np.concatenate([np.array(r[1]) for r in res])
            print(f"{name:>10}: packets found {p.size} of {4 * a.streams}, rho1 1/10/50 % quantiles "
                  f"{np.round(np.quantile(p, [0.01, 0.1, 0.5]), 3).tolist()}, found with rho1 >= tau {(p >= tau).sum()}; "
                  f"other accepted candidates: max {o.max() if o.size else 0:.3f}")

        def noise_job(seed):
            rng = np.random.default_rng(seed)
            x = np.clip(rng.normal(0, sigma_of(0), 1880 * 40), -32767, 32767).round().astype(np.int16)
            return [b for _, b, ok in stage1(x, W) if ok]

        n = np.concatenate([np.array(v) for v in ex.map(noise_job, range(1000, 1000 + a.noise_streams))])
    print(f"noise at Eb/N0 0 dB ({sigma_of(0):.0f} LSB): {n.size} accepted frame maxima, 99 / 99.9 % quantiles "
          f"{np.round(np.quantile(n, [0.99, 0.999]), 4).tolist()}, max {n.max():.4f}, above tau {(n >= tau).sum()}")
    z = stage1(np.zeros(1880 * 20, np.int16), W)
    print(f"dead air: largest rho1 {max(b for _, b, _ in z):.3f}")


if __name__ == "__main__":
    main()

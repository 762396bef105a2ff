"""S4b: one blocking kdeb200_sample_batch / kdeb200_resample_batch call of 256 problems against a loop of 256 single
sample / resample calls.  python tools/bench_sample_batch.py <outdir> [reps] writes <outdir>/r05_sample_batch.json.

Workloads, as a belief-propagation round produces them (256 densities of N = 100..200 points, d = 2 and 3 alternating):
  (a) sample_batch, Np = N                       against [sample(p, N, seed=s)]
  (b) resample_batch, Np = N                     against [resample(p, N, seed=s)]
  (c) sample_batch, Np = N except every 16th problem Np = 5000 (above SB_MAX = 2048: the single call's route inside the
      batch), against the loop of single calls
Per workload: median, min and max wall time of the batch call and of the loop over `reps` alternating repetitions
after one warm-up of each (host clock around whole calls; every call ends in a device synchronise; the cumulative-weight
tables are built in the warm-up), and the batch call's kernel time (kdeb200_last_kernel_ms).  The batch outputs must
equal the loop's bit for bit on the timed inputs; a run that fails the check stops without writing a record.  The
card's name and power limit are read in the same run and recorded with the numbers."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import kde_b200 as K
from tests.util import mixture, silverman

B = 256


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers still stand, without their label
        return "unknown (%s)" % e


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def same_samples(a, b):
    return len(a) == len(b) and all(np.array_equal(bits(x[0]), bits(y[0])) and np.array_equal(x[1], y[1])
                                    for x, y in zip(a, b))


def same_densities(a, b):
    return len(a) == len(b) and all(np.array_equal(bits(x.bandwidth), bits(y.bandwidth)) and
                                    np.array_equal(bits(x.means), bits(y.means)) for x, y in zip(a, b))


def timed(fn, reps, loop_fn):
    fn()
    loop_fn()
    tb, tl, km = [], [], []
    out = ref = None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        tb.append((time.perf_counter() - t0) * 1e3)
        km.append(K.last_kernel_ms()[0])
        t0 = time.perf_counter()
        ref = loop_fn()
        tl.append((time.perf_counter() - t0) * 1e3)
    return out, ref, {"batch_ms": float(np.median(tb)), "loop_ms": float(np.median(tl)),
                      "speedup": float(np.median(tl) / np.median(tb)), "kernel_ms": float(np.median(km)),
                      "batch_ms_min": float(np.min(tb)), "batch_ms_max": float(np.max(tb)),
                      "loop_ms_min": float(np.min(tl)), "loop_ms_max": float(np.max(tl))}


def main():
    outdir = sys.argv[1]
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 9
    os.makedirs(outdir, exist_ok=True)
    K.init(0)  # no device: this fails, there is no fallback
    label = gpu_label()
    rng = np.random.default_rng(12)
    dens = []
    for b in range(B):
        pts = mixture(rng, 2 + b % 2, int(rng.integers(100, 201)))
        dens.append(K.kde(pts, silverman(pts)))
    Np = [K.Npts(p) for p in dens]
    Np_mix = [5000 if b % 16 == 0 else n for b, n in enumerate(Np)]
    seeds = [int(x) for x in rng.integers(0, 2 ** 63, size=B)]
    res = {"gpu": label, "reps": reps, "B": B, "shapes": {
        "sample": "256 densities, N 100..200, d = 2 / 3 alternating, Np = N",
        "resample": "the same densities, resample with Np = N",
        "sample_mix": "the same densities, Np = N except every 16th problem Np = 5000 (> SB_MAX = 2048)"}}

    out, ref, r = timed(lambda: K.sample_batch(dens, Np, seeds=seeds), reps,
                        lambda: [K.sample(p, n, seed=s) for p, n, s in zip(dens, Np, seeds)])
    if not same_samples(out, ref):
        raise SystemExit("sample: batch outputs differ from the single calls: no record written")
    res["sample"] = r
    print("sample", r, flush=True)

    out, ref, r = timed(lambda: K.resample_batch(dens, Np, seeds=seeds), reps,
                        lambda: [K.resample(p, n, seed=s) for p, n, s in zip(dens, Np, seeds)])
    if not same_densities(out, ref):
        raise SystemExit("resample: batch densities differ from the single calls: no record written")
    res["resample"] = r
    print("resample", r, flush=True)

    out, ref, r = timed(lambda: K.sample_batch(dens, Np_mix, seeds=seeds), reps,
                        lambda: [K.sample(p, n, seed=s) for p, n, s in zip(dens, Np_mix, seeds)])
    if not same_samples(out, ref):
        raise SystemExit("sample_mix: batch outputs differ from the single calls: no record written")
    res["sample_mix"] = r
    print("sample_mix", r, flush=True)

    res["gpu_after"] = gpu_label()
    with open(os.path.join(outdir, "r05_sample_batch.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""K2b: one blocking kdeb200_eval_batch call of B problems against a loop of B single evaluateDualTree calls, and
kde_batch (kdeb200_kde_lcv_batch) against a loop of kde(points).  python tools/bench_eval_batch.py <outdir> [reps]
writes <outdir>/r03_eval_batch.json.

Shapes, as a belief-propagation round produces them: B in {1, 16, 256, 1024} densities of N = 100..200 points, d = 1..3
(cycled), each evaluated at its own M = 100..200 query points; the same B with lvFlag (each density at its own points,
leave-one-out); kde_batch of B sets of 100 points, d = 2.  Per B: median wall time of the batch call and of the loop
over `reps` alternating repetitions after one warm-up of each (host clock around whole calls; every call ends in a
device synchronise), and the batch call's kernel time (kdeb200_last_kernel_ms).  The batch outputs must equal the
loop's bit for bit; a run that fails the check stops without writing a record.  The card's name and power limit are
recorded with the numbers."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import kde_b200 as K
from tests.util import mixture, silverman

BATCH = [1, 16, 256, 1024]


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers still stand, without their label
        return "unknown (%s)" % e


def same(a, b):
    return len(a) == len(b) and all(np.array_equal(np.ascontiguousarray(x).view(np.int64),
                                                   np.ascontiguousarray(y).view(np.int64)) for x, y in zip(a, b))


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
                      "batch_ms_min": float(np.min(tb)), "loop_ms_min": float(np.min(tl))}


def main():
    outdir = sys.argv[1]
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    os.makedirs(outdir, exist_ok=True)
    K.init(0)
    rng = np.random.default_rng(11)
    nmax = max(BATCH)
    dens, queries = [], []
    for b in range(nmax):
        d = 1 + b % 3
        pts = mixture(rng, d, int(rng.integers(100, 201)))
        dens.append(K.kde(pts, silverman(pts)))
        queries.append(mixture(rng, d, int(rng.integers(100, 201))))
    sets = [mixture(rng, 2, 100) for _ in range(nmax)]
    res = {"gpu": gpu_label(), "reps": reps, "shapes": {
        "eval": "N 100..200, d 1..3 cycled, M 100..200 per density", "eval_loo": "the same densities, lvFlag",
        "kde": "sets of 100 points, d = 2"}, "eval": {}, "eval_loo": {}, "kde": {}}
    for B in BATCH:
        ds, qs = dens[:B], queries[:B]
        out, ref, r = timed(lambda: K.evaluateDualTree_batch(ds, qs), reps,
                            lambda: [K.evaluateDualTree(b, q) for b, q in zip(ds, qs)])
        if not same(out, ref):
            raise SystemExit("eval B=%d: batch outputs differ from the single calls: no record written" % B)
        res["eval"][str(B)] = r
        print("eval", B, r, flush=True)
        out, ref, r = timed(lambda: K.evaluateDualTree_batch(ds, ds, [True] * B), reps,
                            lambda: [K.evaluateDualTree(b, b, True) for b in ds])
        if not same(out, ref):
            raise SystemExit("eval_loo B=%d: batch outputs differ from the single calls: no record written" % B)
        res["eval_loo"][str(B)] = r
        print("eval_loo", B, r, flush=True)
        ss = sets[:B]
        out, ref, r = timed(lambda: K.kde_batch(ss), reps, lambda: [K.kde(p) for p in ss])
        if not same([K.getBW(p)[:, 0] for p in out], [K.getBW(p)[:, 0] for p in ref]):
            raise SystemExit("kde B=%d: batch bandwidths differ from kde(points): no record written" % B)
        res["kde"][str(B)] = r
        print("kde", B, r, flush=True)
    with open(os.path.join(outdir, "r03_eval_batch.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

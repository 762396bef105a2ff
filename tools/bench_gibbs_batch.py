"""K1b: one blocking kdeb200_gibbs_batch call of B problems against a loop of B single prodAppxMSGibbsS calls with the
same seeds, and kdeb200_product_kde_batch against a loop of prod.  python tools/bench_gibbs_batch.py <outdir> [reps]
writes <outdir>/r03_gibbs_batch.json.

Shapes: C1 (2 densities x 100 components, 2-D, Np 100, Niter 5: the README product) and testProds (6 x 100, 3-D,
Np 100, Niter 5), each problem with its own trees.  Per B: median wall time of the batch call and of the loop (host
clock around calls that end in a device synchronise), the batch call's split (host checks + schedule assembly +
packing, the one host-to-device copy, kernels = kdeb200_last_kernel_ms, the copies back), and an output check against
the loop, which takes the default single-call route (K1w at these sizes): labels identical, points within 1e-10; a
run that fails the check stops without writing a record.  The first call of each B (not timed) also builds the draw
templates, which the library keeps per tree, of the trees no smaller B used; "first_plan_ms" is that call's host time.  The card's name and power
limit are recorded with the numbers."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import kde_b200 as K
from tests.util import mixture, silverman

SHAPES = {"C1": (2, 2, 100, 100), "testProds": (3, 6, 100, 100)}  # d, densities, components, Np
BATCH = [1, 16, 64, 256, 1024]
PROD_BATCH = [16, 256]
T = 5


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers still stand, without their label
        return "unknown (%s)" % e


def close(a, b):
    scale = np.maximum(np.abs(b), 1e-3 * np.max(np.abs(b)) + 1e-300)
    return float(np.max(np.abs(a - b) / scale))


def main():
    outdir = sys.argv[1]
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    os.makedirs(outdir, exist_ok=True)
    K.init(0)
    res = {"gpu": gpu_label(), "reps": reps, "Niter": T, "shapes": {}}
    for name, (d, M, N, Np) in SHAPES.items():
        rng = np.random.default_rng(7)
        pool = []
        for b in range(max(BATCH)):
            ts = []
            for j in range(M):
                p = mixture(rng, d, N, 0.25 * j)
                ts.append(K.kde(p, silverman(p)))
            pool.append(ts)
        shape = {"d": d, "densities": M, "components": N, "Np": Np, "gibbs": {}, "prod": {}}
        for B in BATCH:
            lists, seeds = pool[:B], list(range(1, B + 1))
            K.prodAppxMSGibbsS_batch(lists, [Np] * B, Niter=T, seeds=seeds)  # warm-up: modules, pools, staging, templates
            first_plan = K.gibbs_batch_split()[0]
            loop = [K.prodAppxMSGibbsS(None, ts, None, None, Niter=T, Np=Np, seed=s) for ts, s in zip(lists, seeds)]
            tb, tl, split = [], [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                out = K.prodAppxMSGibbsS_batch(lists, [Np] * B, Niter=T, seeds=seeds)
                tb.append((time.perf_counter() - t0) * 1e3)
                split.append(K.gibbs_batch_split() + (K.last_kernel_ms()[0],))
                t0 = time.perf_counter()
                loop = [K.prodAppxMSGibbsS(None, ts, None, None, Niter=T, Np=Np, seed=s) for ts, s in zip(lists, seeds)]
                tl.append((time.perf_counter() - t0) * 1e3)
            sp = np.median(np.array(split), axis=0)
            labels_ok = all(np.array_equal(o[1], l[1]) for o, l in zip(out, loop))
            err = max(close(o[0], l[0]) for o, l in zip(out, loop))
            if not labels_ok or not err <= 1e-10:
                raise SystemExit("%s B=%d: batch outputs differ from the single calls (labels identical: %s, max point "
                                 "relative error %.3g): no record written" % (name, B, labels_ok, err))
            shape["gibbs"][str(B)] = {
                "batch_ms": float(np.median(tb)), "loop_ms": float(np.median(tl)),
                "speedup": float(np.median(tl) / np.median(tb)),
                "plan_ms": float(sp[0]), "first_plan_ms": first_plan, "h2d_ms": float(sp[1]), "kernel_ms": float(sp[3]), "d2h_ms": float(sp[2]),
                "labels_identical": bool(labels_ok), "max_point_relerr": err}
            print(name, B, shape["gibbs"][str(B)], flush=True)
        for B in PROD_BATCH:
            lists, seeds = pool[:B], list(range(1, B + 1))
            K.prod_batch(lists, seeds=seeds)
            tb, tl = [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                out = K.prod_batch(lists, seeds=seeds)
                tb.append((time.perf_counter() - t0) * 1e3)
                kms = K.last_kernel_ms()[0]
                t0 = time.perf_counter()
                loop = [K.prod(ts, seed=s) for ts, s in zip(lists, seeds)]
                tl.append((time.perf_counter() - t0) * 1e3)
            err = max(close(K.getPoints(o), K.getPoints(l)) for o, l in zip(out, loop))
            bw_err = max(close(K.getBW(o)[:, 0], K.getBW(l)[:, 0]) for o, l in zip(out, loop))
            if not err <= 1e-10:
                raise SystemExit("%s prod B=%d: product points differ from the prod loop (max relative error %.3g): no "
                                 "record written" % (name, B, err))
            shape["prod"][str(B)] = {"batch_ms": float(np.median(tb)), "loop_ms": float(np.median(tl)),
                                     "speedup": float(np.median(tl) / np.median(tb)), "kernel_ms": kms,
                                     "max_point_relerr": err, "max_bw_relerr": bw_err}
            print(name, "prod", B, shape["prod"][str(B)], flush=True)
        res["shapes"][name] = shape
    with open(os.path.join(outdir, "r03_gibbs_batch.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

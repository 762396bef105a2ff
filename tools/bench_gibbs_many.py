"""K1m: single Gibbs products of more than 16 densities against today's 16-density route.
python tools/bench_gibbs_many.py <outdir> [reps] [--variant <libkdeb200_*.so>] writes <outdir>/r07_gibbs_many.json.

Shapes (Niter 5, Philox): "C1" -- 2-D densities of 100 components, Np 100 (the README product, grown in M); and
"throughput" -- 3-D densities of 1024 components, Np 100 000.  M = 16 runs the existing routes (K1w at C1, K1x at
throughput); M = 17, 24, 32, 64 run K1m.  Per (shape, M): median wall time of the call (host clock around a blocking
kdeb200_gibbs), median kernel time (kdeb200_last_kernel_ms, device events), and kernel time per evaluated node (kernel
time / (Np x kernel evaluations per sample from kdeb200_gibbs_sizes)).  Each K1m shape is first checked against the
oracle under injected streams on a 64-sample prefix (labels identical, points within 1e-10); a failure stops the run
without writing a record.  --variant also times the throughput shape with another build of the library (an occupancy
sweep: tools' build_variant with GB_MINBLOCKS), in a subprocess.  The card's name and power limit are recorded with the
numbers, read in the same run."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

SHAPES = {"C1": (2, 100, 100), "throughput": (3, 1024, 100_000)}  # d, components, Np
MS = [16, 17, 24, 32, 64]
T = 5


def gpu_label():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # the numbers still stand, without their label
        return "unknown (%s)" % e


def trees_for(K, d, N, M, seed=7):
    from tests.util import mixture, silverman
    rng = np.random.default_rng(seed)
    pts = [mixture(rng, d, N, 0.05 * j) for j in range(M)]
    return [K.kde(p, silverman(p)) for p in pts], pts, [silverman(p) for p in pts]


def check(K, trees, pts, bws):
    from oracle import oracle as O
    ot = [O.OKDE.kde_bw(p, b) for p, b in zip(pts, bws)]
    rng = np.random.default_rng(1)
    nU, nN = O.prod_sizes(ot, 64, T)
    U, G = rng.random(nU), rng.standard_normal(nN)
    ep, ei = O.gibbs(ot, 64, T, U, G, nthreads=O.max_threads())
    gp, gi = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=64, randU=U, randN=G)
    scale = np.maximum(np.abs(ep), 1e-3 * np.max(np.abs(ep)) + 1e-300)
    if not np.array_equal(gi, ei) or float(np.max(np.abs(gp - ep) / scale)) >= 1e-10:
        raise SystemExit("K1m differs from the oracle at M=%d" % len(trees))


def time_shape(K, d, N, Np, M, reps, verify):
    trees, pts, bws = trees_for(K, d, N, M)
    if verify and M > 16:
        check(K, trees, pts, bws)
    L, _, _, evals = K.gibbs_sizes(trees, T)
    K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=3)  # warm-up: schedule, module load
    wall, kern = [], []
    for r in range(reps):
        t0 = time.perf_counter()
        K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=100 + r)
        wall.append(1e3 * (time.perf_counter() - t0))
        kern.append(K.last_kernel_ms()[0])
    km = float(np.median(kern))
    return {"M": M, "route": "K1m" if M > 16 else "existing", "levels": L, "evals_per_sample": int(evals),
            "call_ms": float(np.median(wall)), "kernel_ms": km, "ns_per_node": 1e6 * km / (Np * evals),
            "call_ms_all": wall, "kernel_ms_all": kern}


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    variant = sys.argv[sys.argv.index("--variant") + 1] if "--variant" in sys.argv else None
    if variant in args:
        args.remove(variant)
    if "--child" in sys.argv:  # one throughput sweep with the library named by KDEB200_SO, JSON on stdout
        import kde_b200 as K
        K.init(0)
        d, N, Np = SHAPES["throughput"]
        print(json.dumps([time_shape(K, d, N, Np, M, int(args[0]), False) for M in MS if M > 16]))
        return
    outdir = args[0]
    reps = int(args[1]) if len(args) > 1 else 5
    os.makedirs(outdir, exist_ok=True)
    import kde_b200 as K
    K.init(0)
    res = {"gpu": gpu_label(), "reps": reps, "Niter": T, "shapes": {}}
    for name, (d, N, Np) in SHAPES.items():
        res["shapes"][name] = {"d": d, "components": N, "Np": Np,
                               "runs": [time_shape(K, d, N, Np, M, reps, True) for M in MS]}
        for r in res["shapes"][name]["runs"]:
            print(name, "M=%d" % r["M"], "call %.3f ms  kernel %.3f ms  %.4g ns/node" % (
                r["call_ms"], r["kernel_ms"], r["ns_per_node"]), flush=True)
    if variant:
        env = dict(os.environ, KDEB200_SO=os.path.abspath(variant))
        out = subprocess.run([sys.executable, os.path.abspath(__file__), str(reps), "--child"], env=env,
                             capture_output=True, text=True, check=True).stdout
        res["variant"] = {"so": os.path.basename(variant), "throughput": json.loads(out.strip().splitlines()[-1])}
        for r in res["variant"]["throughput"]:
            print("variant", "M=%d" % r["M"], "kernel %.3f ms" % r["kernel_ms"], flush=True)
    res["gpu_after"] = gpu_label()
    with open(os.path.join(outdir, "r07_gibbs_many.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

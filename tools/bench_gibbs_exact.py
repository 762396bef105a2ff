"""K1x (certified FP32 decisions, FP64 results) against K1 (all FP64), alternating in one process:
python tools/bench_gibbs_exact.py [Np] [dims] [reps] -> one JSON object.  dims is a comma list (default 3 = the C4 shape:
8 densities x 4096 components, Niter 5).  Kernel times are the library's own CUDA-event times.  `redone_*` are the
lane-draws / warp-draws K1x redid in FP64 per leaf-level draw; `identical` compares points and labels bit for bit.
Also reports the card's name and power limit: the times belong to them."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import kde_b200 as K
from tests.util import mixture, silverman

Np = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
dims = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "3").split(",")]
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
os.environ["KDEB200_GIBBS_WARP_MAX"] = "0"
K.init(0)
K.set_gibbs_precision(K.F64)
out = {"samples": Np, "reps": reps}
try:
    out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                capture_output=True, text=True, timeout=60).stdout.strip()
except Exception as e:  # the numbers still stand, without their label
    out["gpu"] = "unknown (%s)" % e


def run(route, trees):
    os.environ["KDEB200_GIBBS_EXACT"] = route
    res = K.prodAppxMSGibbsS(None, trees, None, None, Niter=5, Np=Np, seed=1)
    return res, K.last_kernel_ms()[0]


for d in dims:
    rng = np.random.default_rng(2)
    trees = []
    for j in range(8):
        p = mixture(rng, d, 4096, 0.25 * j)
        trees.append(K.kde(p, silverman(p)))
    r = {"k1_ms": [], "k1x_ms": []}
    run("1", trees)  # schedule, records and scratch are built on the first call
    K.gibbs_exact_redone()
    for _ in range(reps):
        ref, ms = run("0", trees)
        r["k1_ms"].append(ms)
        new, ms = run("1", trees)
        r["k1x_ms"].append(ms)
    lanes, warps = K.gibbs_exact_redone()
    L, pu, pn, ev = K.gibbs_sizes(trees, 5)
    leaf_levels = sum(1 for l in range(1, L + 1) if min(2 ** l, 4096) == 4096)
    leaf_draws = reps * Np * 8 * 6 * leaf_levels
    r["redone_lane_frac"] = lanes / leaf_draws
    r["redone_warp_frac"] = warps / (leaf_draws / 32)
    r["identical"] = bool(all(np.array_equal(a, b) for a, b in zip(ref, new)))
    r["k1_samples_per_s"] = Np / min(r["k1_ms"]) * 1e3
    r["k1x_samples_per_s"] = Np / min(r["k1x_ms"]) * 1e3
    r["speedup"] = min(r["k1_ms"]) / min(r["k1x_ms"])
    out["d%d" % d] = r
os.environ.pop("KDEB200_GIBBS_EXACT", None)
print(json.dumps(out, indent=1))

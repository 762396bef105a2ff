"""K1x (certified FP32 decisions, FP64 results) against K1 (all FP64), alternating in one process:
python tools/bench_gibbs_exact.py [Np] [dims] [reps] -> one JSON object.  dims is a comma list (default 3 = the C4 shape:
8 densities x 4096 components, Niter 5).  Kernel times are the library's own CUDA-event times.  `redone_*` are the
lane-draws / warp-draws K1x redid in FP64 per leaf-level draw, `redone_b_*` the same per sampleIndices! draw of an
internal level, `redone_int_*` per sampleIndex draw of an internal level; `tier3_lanes` / `tier3_warps` count the
redone lane-draws / warp-draws (all classes, per call) that the warp-parallel FP64 sums could not decide either, which
were summed serially in node order; `identical` compares points and labels bit for bit.
Also reports the card's name and power limit: the times belong to them."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import kde_b200 as K
from tests.util import mixture, silverman

Np = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
dims = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "3").split(",")]
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
T = 5
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
    res = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=1)
    return res, K.last_kernel_ms()[0]


for d in dims:
    rng = np.random.default_rng(2)
    trees = []
    for j in range(8):
        p = mixture(rng, d, 4096, 0.25 * j)
        trees.append(K.kde(p, silverman(p)))
    r = {"k1_ms": [], "k1x_ms": []}
    run("1", trees)  # schedule, records and scratch are built on the first call
    counters = {"": K.gibbs_exact_redone, "_b": K.gibbs_exact_redone_b, "_int": K.gibbs_exact_redone_internal}
    for f in list(counters.values()) + [K.gibbs_exact_tier3]:
        f()
    for _ in range(reps):
        ref, ms = run("0", trees)
        r["k1_ms"].append(ms)
        new, ms = run("1", trees)
        r["k1x_ms"].append(ms)
    # every draw is certified: per level and density one sampleIndices! draw and T sampleIndex draws; a level of
    # min(2^l, N) = N nodes is a leaf level (variant A for all T + 1), every other level is internal (B once, C T times)
    L = K.gibbs_sizes(trees, T)[0]
    leaf = sum(1 for l in range(1, L + 1) if 2 ** l >= 4096)
    draws = {"": reps * Np * 8 * (T + 1) * leaf, "_b": reps * Np * 8 * (L - leaf), "_int": reps * Np * 8 * T * (L - leaf)}
    for cls, f in counters.items():
        lanes, warps = f()
        r["redone%s_lane_frac" % cls] = lanes / max(draws[cls], 1)
        r["redone%s_warp_frac" % cls] = warps / max(draws[cls] / 32, 1)
    r["tier3_lanes"], r["tier3_warps"] = [v / reps for v in K.gibbs_exact_tier3()]
    r["identical"] = bool(all(np.array_equal(a, b) for a, b in zip(ref, new)))
    r["k1_samples_per_s"] = Np / min(r["k1_ms"]) * 1e3
    r["k1x_samples_per_s"] = Np / min(r["k1x_ms"]) * 1e3
    r["speedup"] = min(r["k1_ms"]) / min(r["k1x_ms"])
    out["d%d" % d] = r
os.environ.pop("KDEB200_GIBBS_EXACT", None)
print(json.dumps(out, indent=1))

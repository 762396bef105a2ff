"""What the undecided draws of K1x cost at the C4 shape (8 densities x 4096 components, 3-D, Niter 5):
python tools/gibbs_exact_redo_share.py [Np] [inflates] [reps] -> one JSON object.

KDEB200_GIBBS_EXACT_INFLATE only widens the FP32 bound, so the labels stay K1's at every value >= 1 while more draws
are left undecided.  For each inflate (comma list, default 1,2,4,8) the K1x kernel time (library CUDA events, min of
`reps`) and the undecided lane-draws / warp-draws per class are recorded; the least-squares slope of time against the
undecided warp-draws of all classes is the cost of one, and slope x warp-draws at inflate 1 over the time at inflate 1
is the share of K1x's time the undecided draws take.  Where the library counts them, `tier3_*` are the draws that
needed the serial FP64 sweep.  Also reports the card's name, power limit and SM clock: the times belong to them."""
import json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import kde_b200 as K
from tests.util import mixture, silverman

Np = int(sys.argv[1]) if len(sys.argv) > 1 else 1000000
inflates = [float(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "1,2,4,8").split(",")]
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
T = 5
os.environ["KDEB200_GIBBS_WARP_MAX"] = "0"
os.environ["KDEB200_GIBBS_EXACT"] = "1"
K.init(0)
K.set_gibbs_precision(K.F64)
out = {"samples": Np, "reps": reps}
try:
    out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                capture_output=True, text=True, timeout=60).stdout.strip()
except Exception as e:  # the numbers still stand, without their label
    out["gpu"] = "unknown (%s)" % e

rng = np.random.default_rng(2)
trees = []
for j in range(8):
    p = mixture(rng, 3, 4096, 0.25 * j)
    trees.append(K.kde(p, silverman(p)))
counters = {"": K.gibbs_exact_redone, "_b": K.gibbs_exact_redone_b, "_int": K.gibbs_exact_redone_internal}
tier3 = getattr(K, "gibbs_exact_tier3", None)


def run():
    res = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=1)
    return res, K.last_kernel_ms()[0]


run()  # schedule, records and scratch are built on the first call
ref = None
rows = []
for inf in inflates:
    os.environ["KDEB200_GIBBS_EXACT_INFLATE"] = repr(inf)
    for f in counters.values():
        f()
    if tier3:
        tier3()
    ms = []
    for _ in range(reps):
        res, t = run()
        ms.append(t)
        if ref is None:
            ref = res
        elif not all(np.array_equal(a, b) for a, b in zip(ref, res)):
            raise SystemExit("inflate %g changed the result" % inf)
    row = {"inflate": inf, "k1x_ms": ms, "k1x_ms_min": min(ms)}
    for cls, f in counters.items():
        lanes, warps = f()
        row["redone%s_lanes" % cls] = lanes / reps
        row["redone%s_warps" % cls] = warps / reps
    if tier3:
        row["tier3_lanes"], row["tier3_warps"] = [v / reps for v in tier3()]
    row["redone_warps_all"] = sum(row["redone%s_warps" % c] for c in counters)
    rows.append(row)
os.environ.pop("KDEB200_GIBBS_EXACT_INFLATE", None)
out["rows"] = rows
if len(rows) > 1:
    x = np.array([r["redone_warps_all"] for r in rows])
    y = np.array([r["k1x_ms_min"] for r in rows])
    slope, icpt = np.polyfit(x, y, 1)
    out["ms_per_redone_warp_draw"] = slope
    out["ms_without_redo_extrapolated"] = icpt
    out["redo_share_at_first_inflate"] = slope * x[0] / y[0]
print(json.dumps(out, indent=1))

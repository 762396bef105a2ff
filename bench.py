#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 hot path (contract: see the task statement).

Main workload (BASELINE.json configs[3], the one `metric` is quoted on; it fits one GPU):
    C4: prodAppxMSGibbsS of 8 densities x 4096 components, 3-D, Niter=5, 1,000,000 product samples
    per GPU per step, free-running Philox streams, synthetic Gaussian-mixture data (SURVEY.md 8d).
A "step" is one such call.  `value` = product samples/s with the trees resident in HBM
(kdeb200_gibbs_device on torch's current stream, CUDA events, L2 flushed between steps);
`e2e` = the same through the host API (prodAppxMSGibbsS mirror -> kdeb200_gibbs): tree
flatten + H2D and the D2H of points and labels inside the timed region.

N > 1 (torchrun, one rank per GPU): chains are addressed by global sample index, so results do not
depend on N.  Two curves are measured in the same run:
  weak   (the headline line, "scaling": "weak"): every rank draws its own 1M-sample slice of an N x 1M-sample run
  strong ("strong" sub-record; BASELINE.json configs[3] "1M samples at 1/2/4/8 GPUs"): 1M samples in total,
         1M / N per rank
both with the NCCL all-gather of points + labels inside the timed step, and after the timed loops every rank
recomputes a 4096-sample slice that a FOREIGN rank produced and compares it bit for bit with what the all-gather
delivered ("gather_checked").

`secondary` carries the other BASELINE configurations measured in the same run, each with its own roofline
(algorithmic and issued) and cpu_baseline: C5 (1M x 1M brute-force evaluation, FP64 and FP32) and C3 (kde! LOOCV of
100k x 4-D points: one nLOO_LL launch and the whole bandwidth search); at N > 1 their sharded forms.

Issued-instruction and DRAM-traffic figures come from profiles/ncu_issued.json (tools/ncu_issued.py: ncu counters
keyed by a hash of the kernel sources); if the sources changed since the capture they are reported as stale (null),
never silently reused.

`--impl reference` times the CPU arm: the literal C restatement of the reference (oracle/, kind "port"; the
reference itself is Julia and there is no julia binary on the box) with all host threads over independent
chains, on a bounded sample of the same workload.
"""
import argparse
import ctypes as C
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20261017
NDENS, NCOMP, DIM, NITER = 8, 4096, 3, 5
SAMPLES_PER_GPU = 1_000_000
GATHER_CHECK = 4096
# algorithmic FP64-pipe slots per sample for this shape (SURVEY.md 8d): 393216 leaf-level
# evaluations x 22 + 196512 internal-level evaluations x 47
ALG_SLOTS_PER_SAMPLE = 393216 * 22 + 196512 * 47
ALG_SLOTS_EVAL = {1: 17, 3: 21}  # 2d + 1 + 14 (SURVEY.md 8d, C3 / C5)
DUMP_LIMIT = 64 << 20  # bytes written by --dump-outputs, .npy headers included


def synth_points(j):
    """Density j: K=4 isotropic Gaussians (sigma 0.6) on corners of {+-2}^3, shifted 0.25*j along dim 1."""
    rng = np.random.default_rng(SEED + j)
    corners = np.array([[-2, -2, -2], [-2, -2, 2], [-2, 2, -2], [-2, 2, 2]], dtype=np.float64)
    comp = rng.integers(0, 4, size=NCOMP)
    pts = corners[comp].T + 0.6 * rng.standard_normal((DIM, NCOMP))
    pts[0, :] += 0.25 * j
    return pts


def mixture(rng, d, N, sigma=0.6):
    """K=4 isotropic Gaussians on the first 4 corners of {+-2}^d (the C3 / C5 inputs; same law as tests/util.py)."""
    corners = np.array([[(-2.0 if (c >> (d - 1 - k)) & 1 == 0 else 2.0) for k in range(d)] for c in range(min(4, 2 ** d))])
    comp = rng.integers(0, len(corners), size=N)
    return corners[comp].T + sigma * rng.standard_normal((d, N))


def silverman(pts):
    d, N = pts.shape
    return pts.std(axis=1, ddof=1) * (4.0 / ((d + 2.0) * N)) ** (1.0 / (d + 4.0))


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """--dump-outputs: writes every float32 / float64 array of `arrays` (name -> array, one row per sample) as
    out_dir/<name>.npy, so that two builds can be compared output for output.  If the rows do not fit in `limit`
    bytes, the same fixed, seeded sample of rows is taken from every array and its row indices go to rows.npy."""
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise ValueError("--dump-outputs writes float32 / float64 only: %s is %s" % (name, a.dtype))
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.itemsize * (a.size // max(n, 1)) for a in arrays.values())
    header = 128  # .npy header of a 1- or 2-D array
    if n * row_bytes + len(arrays) * header > limit:
        k = (limit - (len(arrays) + 1) * header) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(SEED).choice(n, size=k, replace=False))
        arrays = dict({name: a[rows] for name, a in arrays.items()}, rows=rows.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def _build_module():
    spec = importlib.util.spec_from_file_location("kdeb200_build", os.path.join(ROOT, "kerneldensityestimate.jl_b200", "build.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def issued_record(label, err=sys.stderr):
    """Entry `label` of profiles/ncu_issued.json if it was captured on the current kernel sources, else None."""
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "ncu_issued.json")))[label]
    except Exception as e:  # noqa: BLE001
        print("[bench] no ncu record for %s (%s): issued/traffic figures are null" % (label, e), file=err)
        return None
    cur = _build_module().kernel_source_hash(rec["kind"])
    if cur != rec["source_hash"]:
        print("[bench] STALE ncu record for %s: kernel sources %s != profiled %s -- re-run tools/ncu_issued.py; "
              "issued/traffic figures are null" % (label, cur, rec["source_hash"]), file=err)
        return None
    return rec


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def run_reference(args, rank, world):
    """CPU arm: oracle port, all host threads, bounded sample of the same workload."""
    if rank != 0:
        return
    from oracle import oracle as O
    trees = [O.OKDE.kde_bw(synth_points(j), silverman(synth_points(j))) for j in range(NDENS)]
    cores = host_cores()  # torchrun exports OMP_NUM_THREADS=1: ask the OS instead
    n = args.ref_samples if args.ref_samples > 0 else 16 * cores
    nU, nN = O.prod_sizes(trees, n, NITER)
    rng = np.random.default_rng(SEED)
    U, G = rng.random(nU), rng.standard_normal(nN)
    for _ in range(args.warmup if args.warmup < 1 else 1):
        O.gibbs(trees, min(n, cores), NITER, U, G, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pts, ind = O.gibbs(trees, n, NITER, U, G, nthreads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"points": pts.T, "indices": ind.T.astype(np.float32)})
    val = n / dt
    sample = "%d of %d samples per step (C4 shape, injected numpy streams), %d OpenMP threads over chains" % (
        n, SAMPLES_PER_GPU, cores)
    print(json.dumps({
        "impl": "reference", "metric": "product samples/sec (Gibbs, Niter=5)", "value": val, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(world),
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(world=1):
    return {"workload": "C4: prodAppxMSGibbsS, 8 densities x 4096 components, 3-D, Niter=5, 1M samples per GPU per step",
            "ndens": NDENS, "components": NCOMP, "dims": DIM, "niter": NITER, "samples_per_gpu": SAMPLES_PER_GPU,
            "rng": "Philox4x32-10 (seed %d), free-running" % SEED,
            "bandwidth": "Silverman", "l2": "flushed between timed steps (256 MiB write); trees (5.3 MB) are L2-resident by design",
            "multi_gpu": "weak (headline): rank r draws samples [r*1M,(r+1)*1M) of one N*1M-sample run; strong (sub-record "
                         "'strong', BASELINE configs[3]): 1M samples in total, 1M/N per rank; both with the NCCL all-gather of "
                         "points+labels in the timed step and a bit-exact check of a foreign rank's gathered slice afterwards",
            "secondary": "C5 (1M x 1M evaluation) and C3 (kde! LOOCV, 100k x 4-D) measured in the same run: key 'secondary'"}


# ------------------------------------------------------------------------------------------ secondary workloads ----
def eval_roofline(label, d, evals, k_ms, dfma, kernel):
    alg = ALG_SLOTS_EVAL[d]
    rec = issued_record(label)
    r = {"bound": "fp64_fma_pipe", "kernel": kernel, "kernel_ms": k_ms, "algorithmic_fp64_slots_per_eval": alg,
         "achieved": evals * alg * 2 / (k_ms * 1e-3) / 1e12, "peak": dfma * 2 / 1e12, "unit": "TFLOP/s",
         "frac": evals * alg / (k_ms * 1e-3) / dfma, "issued_fp64_instr_per_eval": None, "issued_frac": None,
         "traffic": None, "peak_source": "DFMA microbenchmark (kdeb200_pipe_peak) in this run"}
    if rec:
        r["issued_fp64_instr_per_eval"] = rec["fp64_lane_instr_per_unit"]
        r["issued_frac"] = rec["fp64_lane_instr_per_unit"] * evals / (k_ms * 1e-3) / dfma
        r["traffic_bytes_per_eval_ncu"] = rec["dram_bytes_per_unit"]
        r["issued_source"] = "profiles/ncu_issued.json[%s] (source hash %s)" % (label, rec["source_hash"])
    return r


def secondary_single(K, dfma, mufu, args):
    """C5 and C3 on one GPU (N = 1): kernel time via the library's own CUDA-event bracket (kdeb200_last_kernel_ms),
    end-to-end wall through the host API, CPU port on a bounded sample."""
    from oracle import oracle as O
    out = {}
    cores = host_cores()
    # ---- C5: brute-force evaluation of a 1M-component 3-D KDE at 1M query points
    N = M = args.c5_n
    rng = np.random.default_rng(SEED)
    pts, pos = mixture(rng, 3, N), mixture(rng, 3, M)
    bw = silverman(pts)
    t0 = time.perf_counter(); p = K.kde(pts, bw); t_build = time.perf_counter() - t0
    K.evaluateDualTree(p, pos[:, :4096])  # H2D of the tree, module warm-up
    evals = float(N) * M
    rec = {"workload": "C5: brute-force evaluation, %d components x %d queries, 3-D, Silverman bandwidth" % (N, M),
           "evals": evals, "tree_build_host_s": t_build}
    for prec, name in ((K.F64, "f64"), (K.F32, "f32")):
        t0 = time.perf_counter(); v = K.evaluateDualTree(p, pos, precision=prec); wall = time.perf_counter() - t0
        ms, nl = K.last_kernel_ms()
        e = {"value": evals / (ms * 1e-3), "unit": "evals/s", "kernel_ms": ms, "launches": nl,
             "e2e": {"value": evals / wall, "unit": "evals/s", "wall_s": wall, "h2d_bytes": 8 * 3 * M, "d2h_bytes": 8 * M,
                     "api": "kde_b200.evaluateDualTree -> kdeb200_eval (host buffers)"}}
        if prec == K.F64:
            e["roofline"] = eval_roofline("eval_c5", 3, evals, ms, dfma, "eval_kernel<3,2,false>")
            ref = v
        else:
            e["roofline"] = {"bound": "mufu_ex2", "achieved": evals / (ms * 1e-3) / 1e12, "peak": mufu / 1e12,
                             "unit": "T ex2/s (1 per eval)", "frac": evals / (ms * 1e-3) / mufu, "kernel": "eval_f32_kernel<3,false>"}
            e["max_rel_err_vs_f64"] = float(np.max(np.abs(v - ref) / ref))
        rec[name] = e
    # the error-bounded tile-pruned route (csrc/eval_pruned.cu; the reference's dual-tree evaluation re-thought for the
    # GPU): same arithmetic on the pairs it keeps, so the pipe roofline applies to the EVALUATED pairs; the nominal
    # N x M rate is what a caller sees
    K.evaluateDualTree(p, pos[:, :8192], precision=K.F64_BOUNDED)
    t0 = time.perf_counter(); vb = K.evaluateDualTree(p, pos, precision=K.F64_BOUNDED); wall = time.perf_counter() - t0
    ms, nl = K.last_kernel_ms()
    kept, redo = K.pruned_stats()
    rec["f64_bounded"] = {
        "value": evals / (ms * 1e-3), "unit": "evals/s (nominal N x M)", "kernel_ms": ms, "launches": nl,
        "kept_pair_fraction": kept, "rows_recomputed_exactly": redo, "evaluated_pairs_per_s": evals * kept / (ms * 1e-3),
        "max_rel_err_vs_brute_force": float(np.max(np.abs(vb - ref) / ref)), "guaranteed_rel_err": 1e-13,
        "e2e": {"value": evals / wall, "unit": "evals/s (nominal)", "wall_s": wall, "h2d_bytes": 8 * 3 * M, "d2h_bytes": 8 * M,
                "api": "kde_b200.evaluateDualTree(precision=F64_BOUNDED) -> kdeb200_eval (host buffers)"},
        "roofline": {"bound": "fp64_fma_pipe", "note": "on the evaluated pairs (kept fraction of block x tile pairs); includes "
                     "the Morton sort, box and mask passes in kernel_ms",
                     "frac": evals * kept * ALG_SLOTS_EVAL[3] / (ms * 1e-3) / dfma},
        "speedup_vs_brute_force": rec["f64"]["kernel_ms"] / ms}
    K.evaluateDualTree(p, pos[:, :8192], precision=K.F32_BOUNDED)
    t0 = time.perf_counter(); vf = K.evaluateDualTree(p, pos, precision=K.F32_BOUNDED); wall = time.perf_counter() - t0
    ms, nl = K.last_kernel_ms()
    kept32, redo32 = K.pruned_stats()
    rec["f32_bounded"] = {"value": evals / (ms * 1e-3), "unit": "evals/s (nominal N x M)", "kernel_ms": ms, "launches": nl,
                          "kept_pair_fraction": kept32, "rows_recomputed_in_fp64": redo32,
                          "max_rel_err_vs_f64": float(np.max(np.abs(vf - ref) / ref)),
                          "e2e": {"value": evals / wall, "unit": "evals/s (nominal)", "wall_s": wall},
                          "roofline": {"bound": "mufu_ex2", "frac": evals * kept32 / (ms * 1e-3) / mufu,
                                       "note": "on the evaluated pairs; kernel_ms includes sort / box / mask passes"},
                          "speedup_vs_fp32_brute_force": rec["f32"]["kernel_ms"] / ms}
    o = O.OKDE.kde_bw(pts, bw)
    mq = 128 * cores
    t0 = time.perf_counter(); ov = o.evaluate(pos[:, :mq], nthreads=cores); tn = time.perf_counter() - t0
    rec["cpu_baseline"] = {"value": float(N) * mq / tn, "unit": "evals/s", "cores": cores, "kind": "port",
                           "sample": "%d of %d queries against all %d components in %.1f s (oracle, OpenMP over queries)" % (mq, M, N, tn)}
    rec["parity_max_rel_err_vs_oracle"] = float(np.max(np.abs(ref[:mq] - ov) / ov))
    rec["f64_bounded"]["parity_max_rel_err_vs_oracle"] = float(np.max(np.abs(vb[:mq] - ov) / ov))
    out["c5"] = rec
    p._invalidate()
    # ---- C3: kde! LOOCV bandwidth selection on 100k synthetic 4-D mixture points
    N = args.c3_n
    pts = mixture(np.random.default_rng(3), 4, N)
    p1 = K.marginal(K.kde(pts, [1.0]), [1])
    evals = float(N) * N

    def one_nloo(mode):
        K.set_pruning(mode)
        K.entropy(p1)
        t0 = time.perf_counter(); H = K.entropy(p1); wall = time.perf_counter() - t0
        ms, nl = K.last_kernel_ms()
        return H, wall, ms, nl
    H0, one0, ms0, nl0 = one_nloo(0)   # reference-order brute force: every ordered pair (eval_kernel<1,6,true>)
    H, one, ms, nl = one_nloo(1)       # default: each unordered pair once + tile pruning (loo_sym_kernel<1,8>)
    kept, redo = K.pruned_stats()
    rsym = issued_record("loo_sym_c3")
    sym_roof = {"bound": "fp64_fma_pipe", "kernel": "loo_sym_kernel<1,8>", "kernel_ms": ms,
                # per UNORDERED pair: 2d+1 (distance) + 14 (exp) + 2 (credit both rows) = 19 slots at d = 1
                "algorithmic_fp64_slots_per_unordered_pair": 19, "unordered_pairs_evaluated": evals * kept,
                "frac": evals * kept * 19 / (ms * 1e-3) / dfma, "peak": dfma * 2 / 1e12, "unit": "TFLOP/s",
                "achieved": evals * kept * 19 * 2 / (ms * 1e-3) / 1e12,
                "note": "kept = fraction of (row block x tile) pairs evaluated: ~0.5 is the triangle, less is pruning; kernel_ms "
                        "includes the box / mask / order / finalize / exact-pass launches",
                "issued_fp64_instr_per_nominal_eval": None, "issued_frac": None}
    if rsym:
        sym_roof["issued_fp64_instr_per_nominal_eval"] = rsym["fp64_lane_instr_per_unit"]
        sym_roof["issued_source"] = "profiles/ncu_issued.json[loo_sym_c3] (source hash %s)" % rsym["source_hash"]
    K.kde(pts[:, :3000])
    t0 = time.perf_counter(); pk = K.kde(pts); total = time.perf_counter() - t0
    K.set_pruning(0)
    t0 = time.perf_counter(); pk0 = K.kde(pts); total_brute = time.perf_counter() - t0
    K.set_pruning(1)
    rec = {"workload": "C3: kde!(points) LOOCV bandwidth selection, %d points, 4-D" % N,
           "one_nLOO_LL": {"value": evals / (ms * 1e-3), "unit": "evals/s (nominal N x N)", "kernel_ms": ms, "wall_ms": one * 1e3,
                           "launches": nl, "H": H, "kept_pair_fraction": kept, "rows_recomputed_exactly": redo,
                           "rel_diff_vs_reference_order_sum": abs(H - H0) / abs(H0), "roofline": sym_roof,
                           "speedup_vs_brute_force": ms0 / ms},
           "one_nLOO_LL_brute_force": {"value": evals / (ms0 * 1e-3), "unit": "evals/s", "kernel_ms": ms0, "wall_ms": one0 * 1e3,
                                       "launches": nl0, "H": H0,
                                       "roofline": eval_roofline("eval_c3", 1, evals, ms0, dfma, "eval_kernel<1,6,true>")},
           "full_kde": {"value": total, "unit": "s", "higher_is_better": False, "bandwidth": K.getBW(pk)[:, 0].tolist(),
                        "brute_force_only_s": total_brute, "bandwidth_brute_force_only": K.getBW(pk0)[:, 0].tolist(),
                        "note": "default policy: the LOO likelihood is summed each-pair-once (symmetric kernel) and tile-pruned, "
                                "within 1e-13 relative of the reference-order sum; kdeb200_set_pruning(0) = brute force only",
                        "api": "kde_b200.kde(points) -> kdeb200_kde_lcv (host points in, d bandwidths out)",
                        "h2d_bytes": 8 * 2 * N * 4, "d2h_bytes": 8 * 4}}
    o1 = O.OKDE.kde_bw(K.getPoints(p1), K.getBW(p1)[:, 0], K.getWeights(p1))
    mq = 256 * cores
    t0 = time.perf_counter(); rows = o1.loo_rows(0, mq, nthreads=cores); tn = time.perf_counter() - t0
    rec["cpu_baseline"] = {"value": float(N) * mq / tn, "unit": "evals/s", "cores": cores, "kind": "port",
                           "sample": "%d of %d LOO rows of one nLOO_LL in %.2f s (oracle evalDirect rows, OpenMP)" % (mq, N, tn),
                           "extrapolated_one_nLOO_LL_s": tn * N / mq}
    out["c3"] = rec
    return out


def secondary_sharded(K, kd, torch, dist, rank, world, dev, args):
    """C5 with the queries block-partitioned (all-gather of the densities) and C3 with the rows of every nLOO_LL step
    block-partitioned (all-reduce per step) -- strong scaling, timed as max over ranks."""
    from kde_b200 import _lib
    L = _lib.lib()
    out = {}
    n = args.c5_n
    rng = np.random.default_rng(SEED)
    pts, pos = mixture(rng, 3, n), mixture(rng, 3, n)
    p = K.kde(pts, silverman(pts))
    a, b = kd.shard_range(n, rank, world)
    d_pos = torch.from_numpy(np.ascontiguousarray(pos[:, a:b].T)).to(dev)
    d_out = torch.empty(b - a, dtype=torch.float64, device=dev)
    g_out = torch.empty(n, dtype=torch.float64, device=dev)

    def step():
        _lib.check(L.kdeb200_eval_device(p._dev(), d_pos.data_ptr(), b - a, 0, K.F64, d_out.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream))
        if n % world == 0:
            dist.all_gather_into_tensor(g_out, d_out)
        else:
            g_out.copy_(kd.all_gather_blocks(d_out, n))
    step()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); step(); step(); e1.record()
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 2], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # content check: the first 1024 densities of the NEXT rank's block, recomputed here
    fa, _ = kd.shard_range(n, (rank + 1) % world, world)
    chk = K.evaluateDualTree(p, pos[:, fa:fa + 1024])
    got = g_out[fa:fa + 1024].cpu().numpy()  # rows are independent; the component-split count differs with the block size
    rel = np.abs(chk - got) / np.maximum(np.abs(chk), 1e-300)
    worst = float(np.max(rel)) if np.all(np.isfinite(rel)) else float("inf")
    ok = torch.tensor([int(worst < 1e-12)], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    wt = torch.tensor([worst], dtype=torch.float64, device=dev)
    dist.all_reduce(wt, op=dist.ReduceOp.MAX)
    out["c5"] = {"workload": "C5: %d components x %d queries, 3-D, f64, queries sharded over %d GPUs + NCCL all-gather" % (n, n, world),
                 "value": float(n) * n / (float(t.item()) * 1e-3), "unit": "evals/s", "ms_per_call": float(t.item()),
                 "scaling": "strong", "gather_checked": bool(ok.item()), "gather_max_rel_diff": float(wt.item())}
    p._invalidate()
    n3 = args.c3_n
    pts = mixture(np.random.default_rng(3), 4, n3)
    kd.kde_sharded(pts[:, :3000])
    dist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter(); pk = kd.kde_sharded(pts); torch.cuda.synchronize(); dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out["c3"] = {"workload": "C3: kde!(points) LOOCV, %d points, 4-D, rows of every nLOO_LL step sharded over %d GPUs" % (n3, world),
                 "full_kde": {"value": float(t.item()), "unit": "s", "higher_is_better": False, "bandwidth": K.getBW(pk)[:, 0].tolist()},
                 "scaling": "strong", "route": "one process per GPU (torch.distributed): row shards + one vector all-reduce per step"}
    # The library's own multi-GPU route (kdeb200_init_multi: ONE process drives all GPUs through the C-ABI, symmetric LOO
    # kernel sharing the triangle of pairs, peer copies) cannot be timed from inside a torchrun job -- the other ranks'
    # NCCL barrier kernels would occupy the GPUs it drives -- so it is measured by tools/bench_multi_inproc.py and
    # examples/product_multi_c.c (profiles/r02_inproc_n{2,4,8}.json, r02_product_multi_c_n{2,4,8}.json).
    out["in_process_route"] = "see profiles/r02_inproc_n%d.json and profiles/r02_product_multi_c_n%d.json" % (world, world)
    return out


# ------------------------------------------------------------------------------------------------------ main ----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--samples", type=int, default=SAMPLES_PER_GPU, help="samples per GPU per step (default = the named config)")
    ap.add_argument("--ref-samples", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the C5 / C3 secondary records")
    ap.add_argument("--c5-n", type=int, default=1_000_000)
    ap.add_argument("--c3-n", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the points and labels of the last timed step to "
                    "DIR/points.npy (float64) and DIR/indices.npy (float32), one row per sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3  # timing rule: W >= 3
    # stdout carries exactly ONE JSON line: NCCL writes its banner / logs to stdout by default (seen at 4 and 8
    # GPUs even at WARN level), so send them to stderr whatever level the caller asked for
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"

    import torch
    import torch.distributed as dist
    import kde_b200 as K
    from kde_b200 import _lib, api as _api, dist as _dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    K.init(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = _lib.lib()
    n_per = args.samples
    Np_total = n_per * world
    s0, s1 = rank * n_per, (rank + 1) * n_per

    pts = [synth_points(j) for j in range(NDENS)]
    trees = [K.kde(p, silverman(p)) for p in pts]
    handles = _api._handles(trees)
    nlev, perU, perN, evals = K.gibbs_sizes(trees, NITER)
    tree_bytes = 0
    for t in trees:
        b = C.c_int64(0)
        L.kdeb200_tree_info(t._dev(gibbs=True), None, None, None, C.byref(b))
        tree_bytes += b.value

    dev = torch.device("cuda", local)
    d_pts = torch.empty((n_per, DIM), dtype=torch.float64, device=dev)
    d_idx = torch.empty((n_per, NDENS), dtype=torch.int64, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    g_pts = g_idx = None
    if world > 1:
        g_pts = torch.empty((Np_total, DIM), dtype=torch.float64, device=dev)
        g_idx = torch.empty((Np_total, NDENS), dtype=torch.int64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, warmup, sample_clocks=False):
        """W untimed + K timed steps, CUDA events on the launching stream, L2 flush between steps (outside the bracket),
        barrier + synchronize on both sides, MAX over ranks."""
        for _ in range(warmup):
            step_fn()
        barrier()
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            time.sleep(0.3)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        tw0 = time.time()
        for a, b in evs:
            flush.fill_(1)
            a.record()
            step_fn()
            b.record()
        barrier()
        tw1 = time.time()
        tot = float(sum(a.elapsed_time(b) for a, b in evs))
        if world > 1:
            tt = torch.tensor([tot], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            tot = float(tt.item())
        return tot, (sampler.stop(tw0, tw1) if sampler else None)

    def gather_check(total, gp, gi):
        """Recompute GATHER_CHECK samples from the block of rank+1 locally and compare with the gathered rows, bit for bit."""
        fa, fb = _dist.shard_range(total, (rank + 1) % world, world)
        n = min(GATHER_CHECK, fb - fa)
        cp = torch.empty((n, DIM), dtype=torch.float64, device=dev)
        ci = torch.empty((n, NDENS), dtype=torch.int64, device=dev)
        _lib.check(L.kdeb200_gibbs_device(handles, NDENS, total, NITER, 1, None, None, 0, None, 0, SEED, fa, fa + n,
                                          cp.data_ptr(), ci.data_ptr(), None, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        ok = torch.tensor([int(torch.equal(cp, gp[fa:fa + n]) and torch.equal(ci, gi[fa:fa + n]))], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        return bool(ok.item())

    # ---- headline: weak scaling (1M samples per GPU per step) -------------------------------------------------
    def step():  # the sharded product: this rank's block + NCCL all-gather (kde_b200.dist)
        _dist.prod_sharded_device(handles, NDENS, DIM, Np_total, NITER, SEED, d_pts, d_idx, g_pts, g_idx)

    total_ms, clocks = timed(step, args.steps, args.warmup, sample_clocks=True)
    value = Np_total * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:  # the legs below overwrite d_pts / d_idx
        out_pts, out_idx = (g_pts, g_idx) if world > 1 else (d_pts, d_idx)
        dump_outputs(args.dump_outputs, {"points": out_pts.cpu().numpy(),
                                         "indices": out_idx.to(torch.float32).cpu().numpy()})
    gather_ok = gather_check(Np_total, g_pts, g_idx) if world > 1 else None

    # ---- strong scaling: BASELINE configs[3], 1M samples in total ---------------------------------------------
    strong = None
    if world > 1:
        tot_s = SAMPLES_PER_GPU - SAMPLES_PER_GPU % world
        a, b = _dist.shard_range(tot_s, rank, world)
        sp, si = d_pts[: b - a], d_idx[: b - a]
        gsp, gsi = g_pts[:tot_s], g_idx[:tot_s]

        def step_strong():
            _dist.prod_sharded_device(handles, NDENS, DIM, tot_s, NITER, SEED, sp, si, gsp, gsi)
        ms_s, _ = timed(step_strong, args.steps, args.warmup)
        strong = {"value": tot_s * args.steps / (ms_s * 1e-3), "unit": "samples/s", "ms_per_step": ms_s / args.steps,
                  "samples_total": tot_s, "samples_per_gpu": b - a, "steps": args.steps, "warmup": args.warmup,
                  "scaling": "strong", "gather_checked": gather_check(tot_s, gsp, gsi),
                  "note": "efficiency = value / (n_gpus x the 1-GPU headline value of the same run series)"}

    # kernel-only duration for the roofline: same launch, no collective, events on the launch stream
    kms = []
    for _ in range(max(2, min(args.steps, 3))):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        st = torch.cuda.current_stream().cuda_stream
        _lib.check(L.kdeb200_gibbs_device(handles, NDENS, Np_total, NITER, 1, None, None, 0, None, 0, SEED, s0, s1,
                                          d_pts.data_ptr(), d_idx.data_ptr(), None, st))
        b.record()
        torch.cuda.synchronize()
        kms.append(a.elapsed_time(b))
    k_ms = float(np.mean(kms))

    # e2e through the host API with host buffers (tree flatten + H2D, D2H of points and labels).  At N > 1 this is the
    # "consumer is host memory" variant of SURVEY.md 8e: every rank copies its own shard straight to the host, no gather.
    e2e_n = n_per
    e2e_t = []
    for i in range(1 + max(1, min(args.steps, 2))):
        for t in trees:
            t._invalidate()
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p_host, i_host = K.prodAppxMSGibbsS(None, trees, None, None, Niter=NITER, Np=Np_total, seed=SEED, s0=s0,
                                            s1=s0 + e2e_n)
        float(p_host[0, 0])
        dt = time.perf_counter() - t0
        if i > 0:
            e2e_t.append(dt)
    e2e_dt = float(np.mean(e2e_t))
    if world > 1:
        tt = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_dt = float(tt.item())
    e2e_val = e2e_n * world / e2e_dt
    handles = _api._handles(trees)  # the e2e leg rebuilt the device trees

    # ---- K1f: the same call with the label probabilities in packed FP32 (statistical mode (b) only; NOT the headline:
    # labels are not bit-exact against the reference).  MUFU-pipe roofline: 1 ex2 per leaf-level / sampleIndices! node,
    # rsqrt + ex2 per internal sampleIndex node (SURVEY.md 8d "FP32 variant").
    c4_f32 = None
    if not args.no_secondary and world == 1 and rank == 0:
        nchk = min(65536, n_per)
        st = torch.cuda.current_stream().cuda_stream
        K.set_gibbs_precision(K.F32)
        try:
            fms = []
            for i in range(4):
                flush.fill_(1)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                _lib.check(L.kdeb200_gibbs_device(handles, NDENS, Np_total, NITER, 1, None, None, 0, None, 0, SEED, s0, s1,
                                                  d_pts.data_ptr(), d_idx.data_ptr(), None, st))
                b.record()
                torch.cuda.synchronize()
                if i > 0:
                    fms.append(a.elapsed_time(b))
            p32, i32 = d_pts[:nchk].clone(), d_idx[:nchk].clone()
            slow = K.gibbs_f32_slow_draws()
        finally:
            K.set_gibbs_precision(K.F64)
        _lib.check(L.kdeb200_gibbs_device(handles, NDENS, Np_total, NITER, 1, None, None, 0, None, 0, SEED, s0, s0 + nchk,
                                          d_pts.data_ptr(), d_idx.data_ptr(), None, st))
        torch.cuda.synchronize()
        same = (d_idx[:nchk] == i32).all(dim=1)
        f_ms = float(np.mean(fms))
        mufu0, _ = K.pipe_peak(2, 200000)
        leaf = NDENS * 2 * NCOMP * (1 + NITER)
        internal = evals - leaf
        mufu_per_sample = leaf + internal * (NITER * 2 + 1) / (1.0 + NITER)
        c4_f32 = {"workload": "C4 with kdeb200_set_gibbs_precision(KDEB200_F32): same trees, seed and sample range as the headline",
                  "value": n_per / (f_ms * 1e-3), "unit": "samples/s", "kernel_ms": f_ms, "dtype": "f32 label probabilities, f64 chain state and points",
                  "parity": "statistical (mode b): fraction of samples whose 8 labels equal the FP64 kernel's under the same Philox streams",
                  "same_labels_as_f64": float(same.float().mean().item()), "samples_compared": nchk,
                  "max_point_diff_where_labels_agree": float((d_pts[:nchk][same] - p32[same]).abs().max().item()) if bool(same.any()) else None,
                  "draws_redone_in_fp64": slow, "speedup_vs_f64_kernel": k_ms / f_ms,
                  "roofline": {"bound": "mufu (ex2 / rsqrt)", "mufu_lane_ops_per_sample": mufu_per_sample,
                               "achieved": mufu_per_sample * n_per / (f_ms * 1e-3) / 1e12, "peak": mufu0 / 1e12, "unit": "T MUFU/s",
                               "frac": mufu_per_sample * n_per / (f_ms * 1e-3) / mufu0, "kernel": "gibbs_f32_kernel<3,8>",
                               "peak_source": "MUFU.EX2 microbenchmark (kdeb200_pipe_peak) in this run",
                               "note": "ncu (profiles/r02_gibbs_f32_ncu.txt): issue slots 61 %, XU pipe ~58 %, LSU data pipe ~75 % busy -- "
                                       "no single pipe saturated; see DESIGN.md K1f"}}

    secondary = None
    if not args.no_secondary:
        if world > 1:
            secondary = secondary_sharded(K, _dist, torch, dist, rank, world, dev, args)
        elif rank == 0:
            dfma0, _ = K.pipe_peak(0, 200000)
            mufu0, _ = K.pipe_peak(2, 200000)
            secondary = secondary_single(K, dfma0, mufu0, args)
            secondary["c4_f32"] = c4_f32

    if rank == 0:
        # roofline denominators measured live (SURVEY.md 8d): dependency-free DFMA stream
        dfma, _ = K.pipe_peak(0, 200000)
        ach = ALG_SLOTS_PER_SAMPLE * n_per / (k_ms * 1e-3)  # algorithmic FP64-pipe slots / s
        peaks_file = {}
        try:
            peaks_file = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        alg_bytes = tree_bytes + n_per * (DIM * 8 + NDENS * 8)
        rec = issued_record("gibbs_c4")
        roof = {"bound": "fp64_fma_pipe", "achieved": ach * 2 / 1e12, "peak": dfma * 2 / 1e12, "unit": "TFLOP/s",
                "frac": ach / dfma, "kernel": "gibbs_kernel<3,false>", "kernel_ms": k_ms,
                # DRAM bytes of ONE launch (ncu dram__bytes_read + write, scaled per sample to this launch's samples)
                "traffic": None, "traffic_ratio": None, "algorithmic_bytes": alg_bytes,
                # honest "issued" view next to the algorithmic one (SURVEY.md 8d asks for both): the kernel issues fewer
                # FP64 instructions per sample than the model's 17.9e6 slots (exp costs 7 instead of 14), so frac can exceed 1
                "issued_fp64_instr_per_sample": None, "issued_frac": None,
                "algorithmic_fp64_slots_per_sample": ALG_SLOTS_PER_SAMPLE, "kernel_evals_per_sample": evals,
                "peak_source": "DFMA microbenchmark (kdeb200_pipe_peak) measured in this run; nominal 64/clk/SM x 148 x 1.965 GHz = 37.2 TFLOP/s",
                "hbm_view": {"algorithmic_bytes": alg_bytes, "achieved_GBs": alg_bytes / (k_ms * 1e-3) / 1e9,
                             "peak_GBs": peaks_file.get("hbm_gbs"),
                             "frac": (alg_bytes / (k_ms * 1e-3) / 1e9 / peaks_file["hbm_gbs"]) if peaks_file.get("hbm_gbs") else None},
                "note": "path is FP64-FMA-pipe bound, not HBM/tensor (SURVEY.md 8d): the HBM view is ~1e-5 of the measured copy bandwidth"}
        if rec:
            roof["issued_fp64_instr_per_sample"] = rec["fp64_lane_instr_per_unit"]
            roof["issued_other_instr_per_sample"] = rec["other_lane_instr_per_unit"]
            roof["issued_frac"] = rec["fp64_lane_instr_per_unit"] * n_per / (k_ms * 1e-3) / dfma
            roof["traffic"] = rec["dram_bytes_per_unit"] * n_per
            roof["traffic_ratio"] = roof["traffic"] / alg_bytes
            roof["traffic_source"] = ("profiles/ncu_issued.json[gibbs_c4]: dram__bytes_read+write of a %d-sample launch "
                                      "(source hash %s), scaled per sample" % (int(rec["units_per_launch"]), rec["source_hash"]))
            roof["fp64_pipe_active_pct_ncu"] = rec["fp64_pipe_active_pct"]
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            from oracle import oracle as O
            otrees = [O.OKDE.kde_bw(p, silverman(p)) for p in pts]
            cores = host_cores()
            rng = np.random.default_rng(SEED)
            n0 = 2 * cores
            nU, nN = O.prod_sizes(otrees, n0, NITER)
            U, G = rng.random(nU), rng.standard_normal(nN)
            t0 = time.perf_counter()
            O.gibbs(otrees, n0, NITER, U, G, nthreads=cores)
            pilot = time.perf_counter() - t0
            n = int(max(n0, min(65536, n0 * args.cpu_seconds / max(pilot, 1e-3))))
            n = (n // cores) * cores
            nU, nN = O.prod_sizes(otrees, n, NITER)
            U, G = rng.random(nU), rng.standard_normal(nN)
            t0 = time.perf_counter()
            O.gibbs(otrees, n, NITER, U, G, nthreads=cores)
            dt = time.perf_counter() - t0
            t0 = time.perf_counter()
            O.gibbs(otrees, 16, NITER, U, G, nthreads=1)
            one = 16 / (time.perf_counter() - t0)
            cpu = {"value": n / dt, "unit": "samples/s", "cores": cores, "kind": "port", "one_thread_value": one,
                   "sample": "%d of %d samples of the same workload in %.1f s (literal C restatement of the reference, OpenMP over chains; the reference itself is single-threaded Julia, not installed)" % (n, n_per, dt)}
        out = {
            "metric": "product samples/sec (Gibbs, Niter=5)", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(world), "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "samples/s", "h2d_bytes_per_step": tree_bytes,
                    "d2h_bytes_per_step": e2e_n * (DIM * 8 + NDENS * 8), "ms_per_step": e2e_dt * 1e3,
                    "api": "kde_b200.prodAppxMSGibbsS -> kdeb200_tree_create x8 + kdeb200_gibbs (host buffers; at N > 1 every "
                           "rank copies its own shard to the host: the no-gather variant of SURVEY.md 8e)"},
            "gpu_launches": args.steps, "roofline": roof, "cpu_baseline": cpu,
            "kernel_evals_per_s": evals * value, "strong": strong, "gather_checked": gather_ok, "secondary": secondary,
        }
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

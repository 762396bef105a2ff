"""The issued-instruction / DRAM-traffic figures that bench.py quotes come from profiles/ncu_issued.json, keyed by the
profiled kernels' compiled code and launch sources (build.kernel_source_hash, tools/ncu_issued.py).  A kernel change
without a new capture must fail loudly here, not let the bench line carry stale numbers (VERDICT r1: a hard-coded count had gone stale silently)."""
import json
import os

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ncu_issued_records_match_the_current_kernel_sources():
    recs = json.load(open(os.path.join(ROOT, "profiles", "ncu_issued.json")))
    kb = bench._build_module()
    assert {"gibbs_c4", "eval_c5", "eval_c3", "loo_sym_c3", "eval_pruned_c5"} <= set(recs)
    stale = {k: (e["source_hash"], kb.kernel_source_hash(e["kind"])) for k, e in recs.items()
             if e["source_hash"] != kb.kernel_source_hash(e["kind"])}
    assert not stale, "re-run tools/r02_evidence.sh (ncu captures) and copy gpurun_out/ncu_issued.json to profiles/: %r" % stale
    for k, e in recs.items():
        assert e["fp64_warp_instr"] > 0 and e["duration_ns"] > 0 and e["units_per_launch"] > 0, k
        assert bench.issued_record(k, err=open(os.devnull, "w")) is not None

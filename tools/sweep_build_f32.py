"""Tuning variants of the FP32 Gibbs kernel (d = 3 only): python tools/sweep_build_f32.py tag:DEF1,DEF2 ...
-> kerneldensityestimate.jl_b200/libkdeb200_<tag>.so, selected at run time with KDEB200_SO=<path>."""
import importlib.util, os, sys
from concurrent.futures import ThreadPoolExecutor
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("b", os.path.join(ROOT, "kerneldensityestimate.jl_b200", "build.py"))
b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
b.build()
jobs = []
for a in sys.argv[1:]:
    tag, defs = a.split(":")
    jobs.append((tag, ["GF_ONLY_D3"] + [d for d in defs.split(",") if d]))
with ThreadPoolExecutor(max_workers=6) as ex:
    for r in ex.map(lambda j: b.build_variant(*j), jobs):
        print("built", r)

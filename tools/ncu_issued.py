"""Machine-readable issued-instruction / DRAM-traffic summary of the hot kernels, keyed by build.kernel_source_hash
(the profiled kernels' SASS and resource usage as compiled, plus their launch sources).

Run ON THE GPU BOX right after the metric captures, so that the hashes describe the sources that were profiled:

  M=smsp__inst_executed_pipe_fp64.sum,smsp__inst_executed.sum,dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active
  ncu --metrics $M --clock-control none --csv --log-file gpurun_out/issued_gibbs.csv -k regex:gibbs_kernel python tools/prof_gibbs.py 75776 1
  ncu --metrics $M --clock-control none --csv --log-file gpurun_out/issued_eval.csv  -k regex:eval_kernel  python tools/prof_eval.py 200000
  python tools/ncu_issued.py gpurun_out/ncu_issued.json \\
      gibbs_c4:gibbs:gpurun_out/issued_gibbs.csv:gibbs_kernel<3:75776:sample \\
      eval_c5:eval:gpurun_out/issued_eval.csv:eval_kernel<3:4e10:eval  eval_c3:eval:gpurun_out/issued_eval.csv:eval_kernel<1:4e10:eval

then copy gpurun_out/ncu_issued.json to profiles/ncu_issued.json (tracked).  bench.py reads it and quotes the issued
numbers only while build.kernel_source_hash(kind) still equals the recorded hash.
spec = label:kind:csv:kernel-name-substring:units-per-launch:unit   (the LAST matching launch of the csv is used)"""
import csv
import importlib.util
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec_ = importlib.util.spec_from_file_location("kb", os.path.join(ROOT, "kerneldensityestimate.jl_b200", "build.py"))
kb = importlib.util.module_from_spec(spec_)
spec_.loader.exec_module(kb)


def parse(path, needle):
    rows = [r for r in csv.reader(open(path)) if len(r) >= 15 and r[0].isdigit()]
    launches = {}
    for r in rows:
        if needle in r[4]:
            launches.setdefault(int(r[0]), {"kernel": r[4], "grid": r[8], "block": r[7]})[r[12]] = (r[13], float(r[14].replace(",", "")))
    if not launches:
        raise SystemExit("no launch of %r in %s" % (needle, path))
    return launches[max(launches)]


def to_bytes(unit, v):
    return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)


def to_ns(unit, v):
    return v * {"ns": 1, "us": 1e3, "ms": 1e6, "s": 1e9}.get(unit, 1)


out_path, specs = sys.argv[1], sys.argv[2:]
out = {}
for s in specs:
    label, kind, path, needle, units, unit = s.split(":")
    m = parse(path, needle)
    units = float(units)
    e = {"kernel": m["kernel"], "grid": m["grid"], "block": m["block"], "kind": kind,
         "source_hash": kb.kernel_source_hash(kind), "units_per_launch": units, "unit": unit,
         "fp64_warp_instr": m["smsp__inst_executed_pipe_fp64.sum"][1],
         "warp_instr": m["smsp__inst_executed.sum"][1],
         "dram_read_bytes": to_bytes(*m["dram__bytes_read.sum"]), "dram_write_bytes": to_bytes(*m["dram__bytes_write.sum"]),
         "duration_ns": to_ns(*m["gpu__time_duration.sum"]),
         "fp64_pipe_active_pct": m["sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active"][1], "csv": os.path.basename(path)}
    if "smsp__inst_executed_pipe_xu.sum" in m:  # MUFU / conversions (the FP32 Gibbs kernel's bound)
        e["xu_warp_instr"] = m["smsp__inst_executed_pipe_xu.sum"][1]
        e["xu_lane_instr_per_unit"] = e["xu_warp_instr"] * 32 / units
    e["fp64_lane_instr_per_unit"] = e["fp64_warp_instr"] * 32 / units
    e["other_lane_instr_per_unit"] = (e["warp_instr"] - e["fp64_warp_instr"]) * 32 / units
    e["dram_bytes_per_unit"] = (e["dram_read_bytes"] + e["dram_write_bytes"]) / units
    out[label] = e
json.dump(out, open(out_path, "w"), indent=1)
print(json.dumps(out, indent=1))

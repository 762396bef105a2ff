"""Builds libkdeb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import os
import re
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libkdeb200.so")
SOURCES = ["context.cu", "tree.cu", "eval.cu", "eval_pruned.cu", "eval_f32.cu", "extras.cu", "lcv.cu", "gibbs.cu", "gibbs_f32.cu", "gibbs_exact.cu", "gibbs_batch.cu", "gibbs_many.cu", "eval_batch.cu", "sample_batch.cu", "peaks.cu", "capi.cu"] + [
    "gibbs_d%d.cu" % d for d in range(1, 9)] + ["gibbs_f32_d%d.cu" % d for d in range(1, 9)] + [
    "gibbs_exact_d%d.cu" % d for d in range(1, 9)] + ["gibbs_batch_d%d.cu" % d for d in range(1, 9)] + [
    "gibbs_many_d%d.cu" % d for d in range(1, 9)]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-ccbin", "/usr/bin/g++", "-Xptxas", "-v"]


# What each Nsight Compute record in profiles/ncu_issued.json (tools/ncu_issued.py) describes, per kind: the object of
# the library build that holds the profiled kernels, their mangled names, and the launch sources -- the host code that
# decides the profiled launch's shape (grid, schedule, chunk and tile sizes).  The key hashes the kernels' SASS and
# resource usage as compiled, plus the launch sources' text, so edits that change neither (comments, other kernels,
# other host code) leave the records valid.  bench.py refuses to quote a record whose key no longer matches.
KERNEL_KEYS = {
    "gibbs": ("gibbs_d3", ["_ZN7kdeb20012gibbs_kernelILi3ELb0ELi8EEEvNS_11GibbsParamsE"],
              ["gibbs_plan.cuh", "gibbs_kernel.cuh"]),
    "gibbs_f32": ("gibbs_f32_d3", ["_ZN7kdeb20016gibbs_f32_kernelILi3ELi8EEEvNS_11GibbsParamsE"],
                  ["gibbs_plan.cuh", "gibbs_f32_kernel.cuh"]),
    "eval": ("eval", ["_ZN7kdeb20011eval_kernelILi3ELi2ELb0EEEvNS_10EvalParamsE",
                      "_ZN7kdeb20011eval_kernelILi1ELi6ELb1EEEvNS_10EvalParamsE"], ["eval.cu"]),
    "eval_pruned": ("eval_pruned", ["_ZN7kdeb20018eval_pruned_kernelILi3ELb0EEEvNS_12PrunedParamsE",
                                    "_ZN7kdeb20014loo_sym_kernelILi1ELi8EEEvNS_9SymParamsE"], ["eval_pruned.cu"]),
}


def _cuobjdump(*args):
    exe = os.path.join(os.path.dirname(NVCC), "cuobjdump")
    if not os.path.exists(exe):
        raise RuntimeError("kernel_source_hash needs cuobjdump next to nvcc (%s)" % exe)
    return subprocess.run([exe] + list(args), check=True, capture_output=True, text=True).stdout


def kernel_source_hash(kind):
    import hashlib
    obj, funcs, launch_sources = KERNEL_KEYS[kind]
    build()
    o = os.path.join(HERE, "build", obj + ".o")
    usage = _cuobjdump("-res-usage", o).splitlines()
    h = hashlib.sha256()
    for fn in funcs:
        sass = _cuobjdump("-sass", "-fun", fn, o)
        at = sass.find("Function : " + fn)  # the header before it names the source file's path
        use = [usage[i + 1] for i, line in enumerate(usage[:-1]) if line.strip() == "Function %s:" % fn]
        if at < 0 or len(use) != 1:
            raise RuntimeError("kernel_source_hash(%r): %s not found in %s" % (kind, fn, o))
        h.update(fn.encode() + b"\0" + sass[at:].encode() + b"\0" + use[0].strip().encode() + b"\0")
    for f in launch_sources:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def _stale():
    if not os.path.exists(OUT):
        return True
    if not all(os.path.exists(os.path.join(HERE, "build", s.replace(".cu", ".o"))) for s in SOURCES):
        return True  # kernel_source_hash and build_variant read the objects
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "kdeb200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_variant(tag, defines):
    """Experimental builds (tuning sweeps): libkdeb200_<tag>.so with extra -D flags, selected at run time with
    KDEB200_SO=<path>.  Every Gibbs source is rebuilt with the flags: the host code plans each route's chunks and tiles
    with the same constants (GB_TILE_N, GB_MAXCK_N, unroll depths) its kernel is compiled with.  With GB_ONLY_D3 or
    GF_ONLY_D3 the host code launches d = 3 only, and the other instantiations are left out."""
    out = os.path.join(HERE, "libkdeb200_%s.so" % tag)
    bdir = os.path.join(HERE, "build", tag)
    os.makedirs(bdir, exist_ok=True)
    only_d3 = any("ONLY_D3" in d for d in defines)
    procs, objs = [], []
    build()
    for s in SOURCES:
        if not s.startswith("gibbs"):  # everything else comes from the main build
            objs.append(os.path.join(HERE, "build", s.replace(".cu", ".o")))
            continue
        inst = re.search(r"_d(\d)\.cu$", s)  # one instantiation per dimension
        if only_d3 and inst and inst.group(1) != "3":
            continue
        o = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [NVCC] + FLAGS + ["-D%s" % d for d in defines] + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        o, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(o)
            raise RuntimeError("nvcc failed on %s (%s)" % (s, tag))
        lines = o.splitlines()
        for i, line in enumerate(lines):
            if "Function properties" in line and "gibbs_kernelILi3ELb0" in line:
                print(tag, " ".join(x.strip() for x in lines[i + 1:i + 3]))
    subprocess.check_call([NVCC, "-shared", "-o", out] + objs + ["-ccbin", "/usr/bin/g++"])
    return out


def build(force=False, verbose=False):
    if not force and not _stale():
        return OUT
    objs = []
    bdir = os.path.join(HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    procs = []
    for s in SOURCES:
        o = os.path.join(bdir, s.replace(".cu", ".o"))
        objs.append(o)
        src = os.path.join(CSRC, s)
        if not force and os.path.exists(o) and all(
                os.path.getmtime(o) > os.path.getmtime(os.path.join(CSRC, f)) for f in os.listdir(CSRC)
                if f.endswith((".cuh", ".h")) or f == s) and os.path.getmtime(o) > os.path.getmtime(
                    os.path.join(HERE, "..", "include", "kdeb200.h")):
            continue
        cmd = [NVCC] + FLAGS + ["-c", src, "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for s, p in procs:
        out, _ = p.communicate()
        log.append("== %s ==\n%s" % (s, out))
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError("nvcc failed on %s" % s)
    with open(os.path.join(bdir, "ptxas.log"), "a" if not force else "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    subprocess.check_call([NVCC, "-shared", "-o", OUT] + objs + ["-ccbin", "/usr/bin/g++"])
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))

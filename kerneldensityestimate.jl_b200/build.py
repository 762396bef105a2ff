"""Builds libkdeb200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libkdeb200.so")
SOURCES = ["context.cu", "tree.cu", "eval.cu", "eval_pruned.cu", "eval_f32.cu", "extras.cu", "lcv.cu", "gibbs.cu", "gibbs_f32.cu", "gibbs_exact.cu", "peaks.cu", "capi.cu"] + [
    "gibbs_d%d.cu" % d for d in range(1, 9)] + ["gibbs_f32_d%d.cu" % d for d in range(1, 9)] + [
    "gibbs_exact_d%d.cu" % d for d in range(1, 9)]
GIBBS_TUNED = ["gibbs.cu", "gibbs_d3.cu"]  # what the tuning variants rebuild (GB_ONLY_D3)
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-ccbin", "/usr/bin/g++", "-Xptxas", "-v"]


# the sources that determine each hot kernel's instruction stream (tools/ncu_issued.py keys its ncu counters by this
# hash; bench.py refuses to quote issued-instruction numbers measured on other sources)
# (device code and the host code that shapes a launch; tree.cuh -- the host-side handle struct -- is deliberately not in)
KERNEL_SOURCES = {
    "gibbs": ["gibbs_kernel.cuh", "gibbs.cu", "common.cuh"],
    "eval": ["eval.cu", "eval_shared.cuh", "common.cuh"],
    "eval_pruned": ["eval_pruned.cu", "eval_shared.cuh", "common.cuh"],
    "eval_f32": ["eval_f32.cu", "common.cuh"],
    "lcv": ["lcv.cu", "eval_shared.cuh", "common.cuh"],
    "gibbs_f32": ["gibbs_f32_kernel.cuh", "gibbs_f32.cu", "gibbs_kernel.cuh", "common.cuh"],
    "gibbs_exact": ["gibbs_exact_kernel.cuh", "gibbs_exact.cu", "gibbs_f32_kernel.cuh", "gibbs_kernel.cuh", "common.cuh"],
}


def kernel_source_hash(kind):
    import hashlib
    h = hashlib.sha256()
    for f in KERNEL_SOURCES[kind]:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()[:16]


def _stale():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "kdeb200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_variant(tag, defines, tuned=None):
    """Experimental builds (tuning sweeps): libkdeb200_<tag>.so with extra -D flags on the sources in `tuned`
    (default: the Gibbs kernel); selected at run time with KDEB200_SO=<path>."""
    global GIBBS_TUNED
    saved = GIBBS_TUNED
    if tuned is not None:
        GIBBS_TUNED = list(tuned)
    try:
        return _build_variant(tag, defines)
    finally:
        GIBBS_TUNED = saved


def _build_variant(tag, defines):
    out = os.path.join(HERE, "libkdeb200_%s.so" % tag)
    bdir = os.path.join(HERE, "build", tag)
    os.makedirs(bdir, exist_ok=True)
    procs, objs = [], []
    build()
    for s in SOURCES:
        if s not in GIBBS_TUNED:  # everything else comes from the main build
            if not (s.startswith("gibbs_d") and any("GB_ONLY_D3" in d for d in defines)) and not (
                    s.startswith("gibbs_f32_d") and s != "gibbs_f32_d3.cu" and any("GF_ONLY_D3" in d for d in defines)):
                objs.append(os.path.join(HERE, "build", s.replace(".cu", ".o")))
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

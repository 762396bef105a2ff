"""Builds tools/micro/mufu_err.cu in a temporary directory and prints its JSON line: the largest relative error of
ex2.approx.ftz.f32 over every float in [-126, 0] and of rsqrt.approx.ftz.f32 over every positive normal float, plus the
card it ran on.  K1x's error bound (csrc/gibbs_exact.cu, GX_EX2_ERR = 2^-21)
uses more than three times the measured ex2 figure."""
import json, os, subprocess, sys, tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
with tempfile.TemporaryDirectory() as tmp:
    exe = os.path.join(tmp, "mufu_err")
    subprocess.check_call([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-gencode", "arch=compute_100a,code=sm_100a",
                           "-O3", "-o", exe, os.path.join(HERE, "micro", "mufu_err.cu")])
    out = json.loads(subprocess.check_output([exe], text=True))
out["gpu"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True).stdout.strip()
print(json.dumps(out))

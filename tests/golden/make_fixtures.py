"""Regenerates tests/golden/reference_fixtures.json from the reference's own test data.

Run with a checkout of KernelDensityEstimate.jl (the tests only read the JSON it writes):
    python tests/golden/make_fixtures.py <path to KernelDensityEstimate.jl>

The reference's fixtures (test/testdata/*Result.txt) are MATLAB print-outs of complete
BallTreeDensity structs with 0-based indices; test/runtests.jl:8-18 parses them and
:42-83 compares them (indices after a +1 shift).  The inline inputs of
UnitTest1D01 / UnitTest2D01 / UnitTest2Dvar01 (test/runtests.jl:90-153) are recorded next to
them, together with the tolerance each reference test uses.
"""
import json
import os
import sys

REF = os.path.join(sys.argv[1], "test", "testdata")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_fixtures.json")


def parse_result(path):
    d = {}
    with open(path) as f:
        for line in f:
            line = line.strip()
            if not line or "=" not in line:
                continue
            name, rhs = line.split("=", 1)
            body = rhs.split("[", 1)[1].split("]", 1)[0]
            d[name.strip()] = [float(x) for x in body.split(",") if x.strip()]
    return d


def read_numbers(path):
    with open(path) as f:
        return [[float(x) for x in line.split()] for line in f if line.strip()]


cases = {
    # name: (input points as d x N rows, bandwidth std-devs or None for LOOCV, fixture, tol, enabled, cite)
    "UnitTest1D01": dict(points=[[.1, .45, .55, 3.8]], ks=[0.08], fixture="test1DResult.txt", tol=1e-5,
                         enabled=True, cite="test/runtests.jl:90-101"),
    "UnitTest2D01": dict(points=[[0.5172, 0.7169, 0.4049], [0.0312, 1.0094, 2.0204]], ks=[0.1],
                         fixture="test2DResult.txt", tol=1e-5, enabled=True, cite="test/runtests.jl:118-129"),
    "UnitTest2Dvar01": dict(points=[[0.5172, 7.169, 4.049], [0.0312, 10.0094, -2.0204]], ks=[0.1, 1.0],
                            fixture="test2DvarResult.txt", tol=1e-4, enabled=True, cite="test/runtests.jl:143-153"),
    "UnitTest1Dlcv01": dict(points_file="test1Dlcv100.txt", ks=None, fixture="test1Dlcv100Result.txt", tol=1e-4,
                            enabled=True, cite="test/runtests.jl:104-116"),
    # disabled in the reference (test/runtests.jl:236,238): MATLAB-era single-bandwidth semantics.
    "UnitTest2Dlcv01": dict(points_file="test2Dlcv100.txt", ks=None, fixture="test2Dlcv100Result.txt", tol=1e-4,
                            enabled=False, cite="test/runtests.jl:131-141"),
    "UnitTest2Dvarlcv01": dict(points_file="test2Dvarlcv100.txt", ks=None, fixture="test2Dvarlcv100Result.txt",
                               tol=2e-3, enabled=False, cite="test/runtests.jl:155-165"),
}

out = {}
for name, c in cases.items():
    if "points_file" in c:
        rows = read_numbers(os.path.join(REF, c["points_file"]))  # N rows x d columns (readdlm(...)')
        d = len(rows[0])
        pts = [[r[k] for r in rows] for k in range(d)]
    else:
        pts = c["points"]
    out[name] = dict(points=pts, ks=c["ks"], tol=c["tol"], enabled=c["enabled"], cite=c["cite"],
                     source=c["fixture"], expected=parse_result(os.path.join(REF, c["fixture"])))

with open(OUT, "w") as f:
    json.dump(out, f)
print("wrote", OUT, os.path.getsize(OUT), "bytes")

"""-m gpu: in-process multi-GPU behind the C-ABI (kdeb200_init_multi, SURVEY.md 8b S0 / 8e).

One host process, several device contexts: the host-buffer entry points shard samples / query points / leaf rows over
the set and every device copies its shard straight into the caller's buffers.  Results must not depend on the number of
GPUs.  On a single-GPU box the set is made of several contexts on device 0 (kdeb200_init_multi_devices with a repeated
device), which exercises the same replication, threading and scatter code; with >= 2 GPUs the real devices are used."""
import os
import subprocess

import numpy as np
import pytest

import kde_b200 as K
from kde_b200 import _lib
from oracle.oracle import OKDE
from tests.util import mixture, relerr, silverman

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_count():
    import ctypes as C
    n = C.c_int(0)
    _lib.check(_lib.lib().kdeb200_device_count(C.byref(n)))
    return n.value


@pytest.fixture(params=["oversubscribed-3", "all-devices"])
def multi(request):
    K.init(0)
    if request.param == "all-devices":
        if device_count() < 2:
            pytest.skip("one visible GPU: the real multi-device set needs >= 2")
        n = K.init_multi(0)
    else:
        n = K.init_multi(devices=[0, 0, 0])
    assert n == K.multi_count() and n >= 2
    yield n
    assert K.init_multi(1) == 1


def test_gibbs_sharded_in_process_equals_one_gpu(multi):
    rng = np.random.default_rng(7)
    trees = [K.kde(mixture(rng, 3, 500, 0.25 * j), [0.3, 0.35, 0.4]) for j in range(4)]
    Np, T = 20_000 + 37, 3                      # ragged blocks
    pm, im, rm = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=11, recordLabels=True)
    L, perU, perN, _ = K.gibbs_sizes(trees, T)
    U, G = K.philox_streams(11, Np, perU, perN)
    pj, ij = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, randU=U, randN=G)   # injected streams, sharded
    assert np.array_equal(pm, pj) and np.array_equal(im, ij)
    sub, subi = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=11, s0=5000, s1=15_001)
    assert np.array_equal(sub, pm[:, 5000:15_001]) and np.array_equal(subi, im[:, 5000:15_001])
    K.init_multi(1)
    p1, i1, r1 = K.prodAppxMSGibbsS(None, trees, None, None, Niter=T, Np=Np, seed=11, recordLabels=True)
    assert np.array_equal(pm, p1) and np.array_equal(im, i1) and np.array_equal(rm, r1)


def test_eval_loo_entropy_and_lcv_sharded_in_process(multi):
    rng = np.random.default_rng(8)
    N, M = 30_000, 50_001
    pts, pos = mixture(rng, 3, N), mixture(rng, 3, M)
    w = rng.random(N) + 0.1
    p = K.kde(pts, silverman(pts), w)
    em, lm, Hm = K.evaluateDualTree(p, pos), K.evaluateDualTree(p, p), K.entropy(p)
    fm = K.evaluateDualTree(p, pos, precision=K.F32)
    x4 = mixture(rng, 2, 40_000)
    bwm = K.lcv_bandwidths(x4)
    K.init_multi(1)
    e1, l1, H1 = K.evaluateDualTree(p, pos), K.evaluateDualTree(p, p), K.entropy(p)
    # rows are independent; only the number of component splits per launch (and so the order of a few partial sums)
    # depends on the block size
    assert relerr(em, e1) < 1e-13 and relerr(lm, l1) < 1e-13 and abs(Hm - H1) <= 1e-13 * abs(H1)
    assert relerr(fm, e1) < 1e-5
    o = OKDE.kde_bw(pts, silverman(pts), w)
    assert relerr(em[:300], o.evaluate(pos[:, :300], nthreads=8)) < 1e-12
    perm = p.bt.permutation[N:] - 1
    assert relerr(lm[perm[:200]], o.loo_rows(0, 200, nthreads=8)) < 1e-12   # host-side scatter of the leaf-ordered rows
    bw1 = K.lcv_bandwidths(x4)
    assert relerr(bwm, bw1) < 1e-9


def test_small_calls_stay_on_one_device_and_errors_propagate(multi):
    rng = np.random.default_rng(9)
    trees = [K.kde(rng.normal(size=(2, 50)) + j, [0.5, 0.5]) for j in range(2)]
    a = K.prodAppxMSGibbsS(None, trees, None, None, Niter=2, Np=100, seed=3)
    K.init_multi(1)
    b = K.prodAppxMSGibbsS(None, trees, None, None, Niter=2, Np=100, seed=3)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    K.init_multi(devices=[0, 0])
    with pytest.raises(K.KDEError):
        K.init_multi(devices=[0, 99])
    with pytest.raises(K.KDEError):          # too-short injected streams are refused before any device work
        K.prodAppxMSGibbsS(None, trees, None, None, Niter=2, Np=10_000, randU=np.zeros(10), randN=np.zeros(10))


def test_c_example_drives_all_gpus_from_one_process(tmp_path):
    """examples/product_multi_c.c: one plain-C process, kdeb200_init_multi, C4-shaped product; the multi-GPU result
    equals the 1-GPU result bit for bit (the example's exit code)."""
    so_dir = os.path.dirname(_lib.SO_PATH)
    exe = tmp_path / "product_multi_c"
    subprocess.check_call(["/usr/bin/gcc", "-std=c99", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "product_multi_c.c"), "-o", str(exe), "-L", so_dir, "-lkdeb200",
                           "-lm", "-Wl,-rpath," + so_dir])
    r = subprocess.run([str(exe), "0", "20000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert '"identical_to_one_gpu": true' in r.stdout

"""GPU parity of the drop-in entry points against the compiled reference CPU path: same synthetic
MS in, solved Jones within 1e-5 relative (north_star tolerance), residuals alike."""
import numpy as np
import pytest

from util import small_problem, relerr, known
from sagecal_b200 import synth
from util import Bound

pytestmark = pytest.mark.gpu

JONES_TOL = 1e-5


def run_both(api, ref, b, fn="sagefit_visibilities", **kw):
    pr = b.pr
    out = []
    for lib in (ref, api):
        x = pr.x.copy()
        pp = pr.pp0.copy()
        r = getattr(lib, fn)(pr.u, pr.v, pr.w, x, pr.N, pr.Nbase, pr.tilesz, b.fresh_barr(), b.sky,
                             pr.coh, pp, **kw)
        out.append((r, x, pp))
    return out


SAGE_CASES = [
    ("C1-lm", dict(N=8, M=2, tilesz=10, seed=20260922), dict(solver_mode=1, max_iter=5)),
    ("lm-qr", dict(N=8, M=2, tilesz=10, seed=5), dict(solver_mode=1, max_iter=4, linsolv=1)),
    ("lm-svd", dict(N=8, M=2, tilesz=10, seed=6), dict(solver_mode=1, max_iter=3, linsolv=2,
                                                      max_lbfgs=0)),
    ("lm-multi", dict(N=13, M=5, tilesz=8, seed=31, kmean=2.0), dict(solver_mode=1, max_iter=3)),
    ("lm-hybrid", dict(N=12, M=4, tilesz=10, seed=32, nchunk=[1, 2, 1, 5]),
     dict(solver_mode=1, max_iter=3)),
    ("oslm", dict(N=10, M=3, tilesz=20, seed=33, kmean=1.0), dict(solver_mode=0, max_iter=4)),
    ("rlm", dict(N=8, M=2, tilesz=10, seed=34, outliers=0.02), dict(solver_mode=2, max_iter=3)),
    ("osrlm", dict(N=8, M=2, tilesz=20, seed=35, outliers=0.02), dict(solver_mode=3, max_iter=3)),
    # tile counts per chunk are multiples of the OS subset count: the reference's OS-LM pairs J rows
    # and residual rows of different tiles otherwise (clmfit.c:1313-1356, DESIGN.md "flagged quirks")
    ("rlm-multi", dict(N=13, M=4, tilesz=20, seed=37, kmean=1.0, outliers=0.02, nchunk=[1, 2, 1, 4]),
     dict(solver_mode=2, max_iter=2)),
    ("lm-nolbfgs", dict(N=35, M=3, tilesz=6, seed=34), dict(solver_mode=1, max_iter=2,
                                                           max_lbfgs=0)),
]


@pytest.mark.parametrize("name,prob,args", SAGE_CASES, ids=[c[0] for c in SAGE_CASES])
def test_sagefit_matches_reference(api, ref, name, prob, args):
    b = small_problem(**prob)
    kw = dict(max_emiter=3, max_lbfgs=10, lbfgs_m=7, randomize=0)
    kw.update(args)
    (rr, xr, ppr), (rg, xg, ppg) = run_both(api, ref, b, **kw)
    assert rr[0] == rg[0]
    assert abs(rr[1] - rg[1]) < 1e-9                    # mean nu
    assert abs(rr[2] - rg[2]) <= 1e-10 * rr[2]          # res_0
    assert relerr(ppg, ppr) < JONES_TOL, (name, relerr(ppg, ppr))
    assert relerr(xg, xr) < 1e-5 * max(1.0, np.max(np.abs(b.pr.x)) / np.max(np.abs(xr)))
    assert abs(rr[3] - rg[3]) <= 1e-5 * rr[3]           # res_1


@pytest.mark.parametrize("mode,nu", [(1, 2.0), (2, 4.0)], ids=["gauss", "robust"])
def test_bfgsfit_matches_reference(api, ref, mode, nu):
    b = small_problem(N=9, M=3, tilesz=8, seed=41, kmean=1.0, outliers=0.02 if mode == 2 else 0.0)
    (rr, xr, ppr), (rg, xg, ppg) = run_both(api, ref, b, fn="bfgsfit_visibilities", max_lbfgs=8,
                                            lbfgs_m=5, solver_mode=mode, mean_nu=nu)
    assert rr[0] == rg[0]
    assert abs(rr[1] - rg[1]) <= 1e-10 * rr[1]
    assert relerr(ppg, ppr) < JONES_TOL, relerr(ppg, ppr)
    assert abs(rr[2] - rg[2]) <= 1e-5 * rr[2]


def test_index_helpers_bit_exact(api, ref):
    for N, T in ((8, 10), (5, 3), (33, 2)):
        Nbase = N * (N - 1) // 2
        from sagecal_b200.dirac_api import barr_to_numpy
        a = barr_to_numpy(ref.generate_baselines(Nbase, T, N), Nbase * T)
        g = barr_to_numpy(api.generate_baselines(Nbase, T, N), Nbase * T)
        assert np.array_equal(a[0], g[0]) and np.array_equal(a[1], g[1])
    rng = np.random.default_rng(0)
    n = 100
    flag = (rng.uniform(0, 1, n) < 0.3).astype(np.float64) * rng.integers(1, 3, n)
    xs = rng.normal(0, 1, 8 * n)
    res = []
    for lib in (ref, api):
        barr = lib.generate_baselines(n, 1, 15)
        x = xs.copy()
        lib.preset_flags_and_data(flag.copy(), barr, x)
        res.append((barr_to_numpy(barr, n)[2], x))
    k = known(res[0][1])
    assert np.array_equal(res[0][0], res[1][0])
    assert np.array_equal(res[0][1][k], res[1][1][k])


@pytest.mark.parametrize("switch", ["DIRAC_B200_CUSOLVER", "DIRAC_B200_NO_TMA", "DIRAC_B200_CP_UNSPLIT"])
def test_alternate_paths_agree(api, switch):
    """The library fallbacks (cuSOLVER instead of the cluster Cholesky, register-staged instead of
    TMA-fed kernels, unsplit gradient pass) solve the same problem to the same Jones: they differ in
    summation order only."""
    import json
    import os
    import subprocess
    import sys
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fallback_check.py")

    def run(env_extra):
        env = dict(os.environ)
        for k in ("DIRAC_B200_CUSOLVER", "DIRAC_B200_NO_TMA", "DIRAC_B200_CP_UNSPLIT"):
            env.pop(k, None)
        env.update(env_extra)
        out = subprocess.run([sys.executable, script], env=env, capture_output=True, text=True,
                             timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        return json.loads(out.stdout.strip().splitlines()[-1])

    base = run({})
    alt = run({switch: "1"})
    assert relerr(np.array(alt["pp"]), np.array(base["pp"])) < 1e-7
    assert abs(alt["r"][3] - base["r"][3]) <= 1e-7 * base["r"][3]


EDGE_CASES = [
    # a third of the rows flagged, 2 % under the uv cut
    ("heavy-flags", dict(N=10, M=2, tilesz=10, seed=51, flag_frac=0.3, uvcut_frac=0.02),
     dict(solver_mode=1, max_iter=3)),
    # a single timeslot
    ("one-slot", dict(N=9, M=2, tilesz=1, seed=52, uvcut_frac=0.0), dict(solver_mode=1, max_iter=3)),
    # 8N = 512: the largest system the cluster Cholesky takes
    ("n512", dict(N=64, M=1, tilesz=2, seed=53), dict(solver_mode=1, max_iter=2, max_emiter=1,
                                                     max_lbfgs=2)),
    # 8N = 520: one station more, the damped solves fall back to cuSOLVER
    ("n520", dict(N=65, M=1, tilesz=2, seed=54), dict(solver_mode=1, max_iter=2, max_emiter=1,
                                                     max_lbfgs=2)),
    # 8N not a multiple of the 32-wide blocks, several clusters
    ("n264", dict(N=33, M=3, tilesz=4, seed=55, kmean=1.0), dict(solver_mode=1, max_iter=2)),
]


@pytest.mark.parametrize("name,prob,args", EDGE_CASES, ids=[c[0] for c in EDGE_CASES])
def test_sagefit_edge_cases(api, ref, name, prob, args):
    b = small_problem(**prob)
    kw = dict(max_emiter=3, max_lbfgs=6, lbfgs_m=5, randomize=0)
    kw.update(args)
    (rr, xr, ppr), (rg, xg, ppg) = run_both(api, ref, b, **kw)
    assert rr[0] == rg[0]
    assert abs(rr[2] - rg[2]) <= 1e-10 * rr[2]          # res_0
    assert relerr(ppg, ppr) < JONES_TOL, (name, relerr(ppg, ppr))
    assert abs(rr[3] - rg[3]) <= 1e-5 * rr[3]           # res_1


def test_sagefit_at_the_solution_stops_like_the_reference(api, ref):
    """Noise-free data and the true Jones as the starting point: the residual is at rounding level,
    every LM run stops on its entry tests (clmfit.c:300-340, applied after the fact by the deferred
    path of lm_core) and the Jones come back unchanged in both libraries."""
    b = small_problem(N=8, M=3, tilesz=6, seed=61, noise_rel=0.0, flag_frac=0.0, uvcut_frac=0.0)
    pr = b.pr
    out = []
    for lib in (ref, api):
        x = pr.x.copy()
        pp = pr.jones_true.copy()
        r = lib.sagefit_visibilities(pr.u, pr.v, pr.w, x, pr.N, pr.Nbase, pr.tilesz, b.fresh_barr(),
                                     b.sky, pr.coh, pp, max_emiter=2, max_iter=3, max_lbfgs=0,
                                     lbfgs_m=5, solver_mode=1, randomize=0)
        out.append((r, pp))
    (rr, ppr), (rg, ppg) = out
    assert np.max(np.abs(ppr - pr.jones_true)) < 1e-9
    assert np.max(np.abs(ppg - pr.jones_true)) < 1e-9
    assert rg[2] < 1e-12 and rr[2] < 1e-12


RANDOMIZE_CASES = [
    # the reference driver runs with randomize = 1 (data.cpp:78): every other SAGE sweep shares the
    # iteration budget out by the clusters' last cost reductions (lmfit.c:880-887,996-998) and the
    # ordered-subsets solvers walk a random permutation of their subsets drawn with rand()
    # (lmfit.c:1085-1099, clmfit.c:1376-1379).  Both libraries live on the process's libc: seeding it
    # before each call gives them the same draws.
    ("lm-rand", dict(N=10, M=4, tilesz=10, seed=101, kmean=1.0), dict(solver_mode=1, max_iter=3)),
    ("oslm-rand", dict(N=10, M=3, tilesz=20, seed=102, kmean=1.0), dict(solver_mode=0, max_iter=4)),
    ("osrlm-rand", dict(N=8, M=2, tilesz=20, seed=103, outliers=0.02), dict(solver_mode=3, max_iter=3)),
    ("rtr-rand", dict(N=10, M=3, tilesz=10, seed=104), dict(solver_mode=4, max_iter=3)),
]


@pytest.mark.parametrize("name,prob,args", RANDOMIZE_CASES, ids=[c[0] for c in RANDOMIZE_CASES])
def test_sagefit_randomize_matches_reference(api, ref, name, prob, args):
    import ctypes
    libc = ctypes.CDLL(None)
    b = small_problem(**prob)
    pr = b.pr
    kw = dict(max_emiter=4, max_lbfgs=4, lbfgs_m=5, randomize=1)
    kw.update(args)
    out = []
    for lib in (ref, api):
        libc.srand(12345)
        x, pp = pr.x.copy(), pr.pp0.copy()
        r = lib.sagefit_visibilities(pr.u, pr.v, pr.w, x, pr.N, pr.Nbase, pr.tilesz, b.fresh_barr(),
                                     b.sky, pr.coh, pp, **kw)
        out.append((r, pp))
    (rr, ppr), (rg, ppg) = out
    assert rr[0] == rg[0]
    assert relerr(ppg, ppr) < JONES_TOL, (name, relerr(ppg, ppr))
    assert abs(rr[3] - rg[3]) <= 1e-5 * rr[3]

"""CPU: pins the restated oracle (oracle/dirac_oracle.c) against the compiled reference
(oracle/_ref, built from /root/reference by oracle/Makefile).  Runs without a GPU."""
import numpy as np
import pytest

import orcdirac
from util import small_problem, perturbed_jones, relerr
from sagecal_b200.dirac_api import barr_to_numpy

CASES = [
    dict(N=8, M=2, tilesz=10, seed=11),
    dict(N=7, M=3, tilesz=6, seed=12, kmean=2.0),
    dict(N=9, M=3, tilesz=10, seed=15, nchunk=[3, 1, 4]),
    dict(N=10, M=4, tilesz=10, seed=14, nchunk=[1, 2, 1, 5]),
]


@pytest.fixture(params=range(len(CASES)), ids=lambda i: "case%d" % i)
def bound(request):
    return small_problem(**CASES[request.param])


@pytest.fixture(scope="module", autouse=True)
def _need_oracle():
    if not orcdirac.available():
        pytest.skip("oracle/liboracle.so not built")


def test_index_helpers_bit_exact(ref):
    L = orcdirac.Oracle(small_problem().pr).L
    for N, T in ((8, 10), (5, 3), (33, 2)):
        Nbase = N * (N - 1) // 2
        a = barr_to_numpy(ref.generate_baselines(Nbase, T, N), Nbase * T)
        s1 = np.zeros(Nbase * T, dtype=np.int32)
        s2 = np.zeros(Nbase * T, dtype=np.int32)
        L.orc_generate_baselines(Nbase, T, N, s1.ctypes.data_as(orcdirac.ip),
                                 s2.ctypes.data_as(orcdirac.ip))
        assert np.array_equal(a[0], s1) and np.array_equal(a[1], s2)


def test_predict_cost_grad(ref, bound):
    pr = bound.pr
    orc = orcdirac.Oracle(pr)
    pp = perturbed_jones(pr)
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, robust_nu=3.0)
    assert relerr(orc.predict_full(pp), ref.predict_full(pp, md, bound.n)) < 1e-14
    for k in range(pr.M):
        mdk = ref.me_data(pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, clus=k)
        assert relerr(orc.predict_cluster(k, pp), ref.predict_cluster(pp, mdk, bound.n)) < 1e-14
    for robust in (False, True):
        cw = ref.cost(pp, pr.x, md, robust=robust)
        assert abs(orc.cost(pp, pr.x, robust, 3.0) - cw) <= 1e-12 * abs(cw)
        assert relerr(orc.grad(pp, pr.x, robust, 3.0), ref.grad(pp, pr.x, md, robust=robust)) < 1e-12


def test_normal_equations(ref, bound):
    pr = bound.pr
    orc = orcdirac.Oracle(pr)
    pp = perturbed_jones(pr, seed=7)
    off = 0
    for k in range(pr.M):
        for ck in range(pr.nchunk[k]):
            t0, nt = orc.chunk_tiles(k, ck)
            pblk = pp[off:off + 8 * pr.N].copy()
            off += 8 * pr.N
            if nt <= 0:
                continue
            md = ref.me_data(pr.N, pr.Nbase, nt, bound.barr, bound.sky, pr.coh, clus=k, tileoff=t0)
            nn = 8 * nt * pr.Nbase
            xs = pr.x[8 * t0 * pr.Nbase: 8 * (t0 + nt) * pr.Nbase]
            ee, JTe_ref, JTJ_ref = ref.normal_eq(pblk, xs, md)
            c, JTJ, JTe = orc.normal_eq(k, t0, nt, pblk, xs)
            assert abs(c - ee) <= 1e-12 * ee
            assert relerr(JTe, JTe_ref) < 1e-12
            assert relerr(JTJ, JTJ_ref) < 1e-12
            rng = np.random.default_rng(3)
            wt = rng.uniform(0.3, 1.2, nn)
            c, JTJ, JTe = orc.normal_eq(k, t0, nt, pblk, xs, wt)
            _, JTe_ref, JTJ_ref = ref.normal_eq(pblk, xs, md, wt)
            assert relerr(JTJ, JTJ_ref) < 1e-12
            assert relerr(JTe, JTe_ref) < 1e-12


@pytest.mark.parametrize("os_", [False, True], ids=["lm", "oslm"])
@pytest.mark.parametrize("linsolv", [0, 1], ids=["chol", "qr"])
def test_lm_chunk(ref, os_, linsolv):
    b = small_problem(N=8, M=2, tilesz=20, seed=51)
    pr = b.pr
    orc = orcdirac.Oracle(pr)
    k = 1
    pblk = pr.pp0[8 * pr.N * k: 8 * pr.N * (k + 1)]
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, b.barr, b.sky, pr.coh, clus=k)
    pw, iw = ref.clevmar(pblk, pr.x, md, 4, linsolv=linsolv, os_=os_)
    pg, ig = orc.lm_chunk(k, 0, pr.tilesz, pblk, pr.x, 4, linsolv=linsolv, os_=os_)
    assert relerr(pg, pw) < 1e-8
    assert np.allclose(ig[:2], iw[:2], rtol=1e-8)
    assert ig[5] == iw[5] and ig[6] == iw[6]


def test_update_w_and_nu(ref):
    rng = np.random.default_rng(5)
    ed = rng.standard_t(3, 4000) * 0.3
    w_ref = np.zeros_like(ed)
    from sagecal_b200.dirac_api import dptr
    nu_ref = ref.lib.update_w_and_nu(5.0, dptr(w_ref), dptr(ed.copy()), len(ed), 4, 2.0, 30.0)
    orc = orcdirac.Oracle(small_problem().pr)
    nu, w = orc.update_w_and_nu(5.0, ed)
    assert nu == nu_ref
    assert relerr(w, w_ref) < 1e-15


@pytest.mark.parametrize("os_", [False, True], ids=["rlm", "osrlm"])
def test_robust_lm_chunk(ref, os_):
    b = small_problem(N=8, M=2, tilesz=20, seed=52, outliers=0.03)
    pr = b.pr
    orc = orcdirac.Oracle(pr)
    k = 0
    pblk = pr.pp0[:8 * pr.N]
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, b.barr, b.sky, pr.coh, clus=k, robust_nu=2.0)
    pw, iw, nuw = ref.rlevmar(pblk, pr.x, md, 3, os_=os_)
    pg, ig, nug = orc.rlm_chunk(k, 0, pr.tilesz, pblk, pr.x, 3, os_=os_, nu0=2.0)
    assert nug == nuw
    assert relerr(pg, pw) < 1e-8
    assert np.allclose(ig[:2], iw[:2], rtol=1e-7)


SAGE = [
    ("lm", dict(N=8, M=2, tilesz=10, seed=20260922), dict(solver_mode=1, max_iter=5)),
    ("oslm", dict(N=8, M=3, tilesz=20, seed=33, kmean=1.0), dict(solver_mode=0, max_iter=4)),
    ("rlm", dict(N=8, M=2, tilesz=10, seed=34, outliers=0.02), dict(solver_mode=2, max_iter=3)),
    ("osrlm", dict(N=8, M=2, tilesz=20, seed=35, outliers=0.02), dict(solver_mode=3, max_iter=3)),
    ("hybrid", dict(N=8, M=3, tilesz=10, seed=36, nchunk=[1, 2, 5]), dict(solver_mode=1, max_iter=3)),
    # edge cases (the same ones the CUDA path is held to, tests/test_gpu_solvers.py)
    ("heavy-flags", dict(N=10, M=2, tilesz=10, seed=51, flag_frac=0.3, uvcut_frac=0.02),
     dict(solver_mode=1, max_iter=3)),
    ("one-slot", dict(N=9, M=2, tilesz=1, seed=52, uvcut_frac=0.0), dict(solver_mode=1, max_iter=3)),
    ("n264", dict(N=33, M=3, tilesz=4, seed=55, kmean=1.0), dict(solver_mode=1, max_iter=2)),
]


@pytest.mark.parametrize("name,prob,args", SAGE, ids=[c[0] for c in SAGE])
def test_sagefit(ref, name, prob, args):
    b = small_problem(**prob)
    pr = b.pr
    kw = dict(max_emiter=3, max_lbfgs=6, lbfgs_m=5)
    kw.update(args)
    xr, ppr = pr.x.copy(), pr.pp0.copy()
    rr = ref.sagefit_visibilities(pr.u, pr.v, pr.w, xr, pr.N, pr.Nbase, pr.tilesz, b.fresh_barr(),
                                  b.sky, pr.coh, ppr, randomize=0, **kw)
    xo, ppo = pr.x.copy(), pr.pp0.copy()
    ro = orcdirac.Oracle(pr).sagefit(xo, ppo, **kw)
    assert rr[0] == ro[0]
    assert abs(rr[1] - ro[1]) < 1e-9                      # mean nu
    assert abs(rr[2] - ro[2]) <= 1e-12 * rr[2]
    assert relerr(ppo, ppr) < 1e-6, relerr(ppo, ppr)
    assert abs(rr[3] - ro[3]) <= 1e-6 * rr[3]


@pytest.mark.parametrize("mode,nu", [(1, 2.0), (2, 4.0)], ids=["gauss", "robust"])
def test_bfgsfit(ref, mode, nu):
    b = small_problem(N=8, M=3, tilesz=8, seed=41, kmean=1.0, outliers=0.02 if mode == 2 else 0.0)
    pr = b.pr
    xr, ppr = pr.x.copy(), pr.pp0.copy()
    rr = ref.bfgsfit_visibilities(pr.u, pr.v, pr.w, xr, pr.N, pr.Nbase, pr.tilesz, b.fresh_barr(),
                                  b.sky, pr.coh, ppr, max_lbfgs=6, lbfgs_m=5, solver_mode=mode,
                                  mean_nu=nu)
    xo, ppo = pr.x.copy(), pr.pp0.copy()
    ro = orcdirac.Oracle(pr).bfgsfit(xo, ppo, max_lbfgs=6, lbfgs_m=5, solver_mode=mode, mean_nu=nu)
    assert relerr(ppo, ppr) < 1e-6
    assert abs(rr[2] - ro[2]) <= 1e-6 * rr[2]


def test_coherencies_and_multifreq(ref):
    b = small_problem(N=9, M=3, tilesz=4, seed=22, kmean=2.0, gaussian_frac=0.4)
    pr = b.pr
    for cl in pr.clusters:
        K = len(cl["ll"])
        cl["spec_idx"] = np.where(np.arange(K) % 2 == 0, -0.7, 0.0)
        cl["spec_idx1"] = np.full(K, 0.05)
        cl["spec_idx2"] = np.full(K, -0.01)
        cl["f0"] = np.full(K, 140e6)
    from sagecal_b200.dirac_api import SkyModel
    sky = SkyModel(pr.clusters, pr.N)
    osky = orcdirac.OracleSky(pr.clusters)
    barr = b.fresh_barr()
    want = ref.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, barr, sky, pr.freq0,
                                        pr.fdelta, uvmin=30.0, uvmax=1e5)
    fl = pr.flag.copy()
    got = osky.coherencies(pr.u, pr.v, pr.w, pr.freq0, pr.fdelta, 30.0, 1e5, fl)
    assert relerr(got, want) < 1e-13
    assert np.array_equal(fl, barr_to_numpy(barr, pr.Nbase1)[2])
    freqs = np.array([145e6, 150e6, 155e6])
    for add in (1, 2):
        rng = np.random.default_rng(2)
        x0 = rng.normal(0, 1, 8 * pr.Nbase1 * 3)
        xa, xb = x0.copy(), x0.copy()
        ref.predict_visibilities_multifreq(pr.u, pr.v, pr.w, xa, pr.N, pr.Nbase, pr.tilesz, barr,
                                           sky, freqs, pr.fdelta * 3, add_to_data=add)
        osky.predict_multifreq(pr.u, pr.v, pr.w, freqs, pr.fdelta * 3, add, xb)
        assert relerr(xb, xa) < 1e-13


@pytest.mark.parametrize("T", [12, 15, 25, 33])
@pytest.mark.parametrize("robust", [False, True], ids=["oslm", "osrlm"])
def test_os_subsets_with_the_reference_pairing(ref, T, robust):
    """tile counts that are not a multiple of the 10 ordered subsets: the reference pairs Jacobian rows
    with residuals / weights of other tiles and cuts the Jacobian (clmfit.c:1313-1413,
    robustlm.c:2835-2935); the restatement reproduces that literally"""
    b = small_problem(N=8, M=2, tilesz=T, seed=40 + T, outliers=0.02 if robust else 0.0)
    pr = b.pr
    orc = orcdirac.Oracle(pr)
    k, n8 = 0, 8 * pr.N
    pp = pr.pp0.copy()
    xd = pr.x - orc.predict_full(pp) + orc.predict_cluster(k, pp)
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, b.barr, b.sky, pr.coh, clus=k, robust_nu=2.0)
    if robust:
        pw, iw, nuw = ref.rlevmar(pp[:n8], xd, md, 3, os_=True)
        pg, ig, nug = orc.rlm_chunk(k, 0, pr.tilesz, pp[:n8], xd, 3, os_=True, nu0=2.0)
        assert nug == nuw
    else:
        pw, iw = ref.clevmar(pp[:n8], xd, md, 3, os_=True)
        pg, ig = orc.lm_chunk(k, 0, pr.tilesz, pp[:n8], xd, 3, os_=True)
    assert relerr(pg, pw) < 1e-9

"""GPU parity of the individual E-step passes against the compiled reference CPU code.
Tolerances: fp64 arithmetic on both sides; differences come from FMA contraction and summation
order only."""
import numpy as np
import pytest

from util import small_problem, perturbed_jones, relerr, known
from sagecal_b200 import lib as blib

pytestmark = pytest.mark.gpu

CASES = [
    dict(N=8, M=2, tilesz=10, seed=11),
    dict(N=13, M=5, tilesz=7, seed=12, kmean=2.0),
    dict(N=35, M=6, tilesz=9, seed=13, kmean=1.0),          # two q-blocks, partial tiles
    dict(N=20, M=4, tilesz=10, seed=14, nchunk=[1, 2, 1, 5]),  # hybrid chunks
    dict(N=9, M=3, tilesz=10, seed=15, nchunk=[3, 1, 4]),     # nchunk does not divide tilesz
]


@pytest.fixture(params=range(len(CASES)), ids=lambda i: "case%d" % i)
def bound(request):
    return small_problem(**CASES[request.param])


def test_predict_full(api, ref, bound):
    pr = bound.pr
    pp = perturbed_jones(pr)
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh)
    want = ref.predict_full(pp, md, bound.n)
    with blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, pr.x) as dp:
        _, got = dp.predict(pp, out_mode=2)
        c, res = dp.predict(pp, out_mode=1, cost_mode=1)
    assert relerr(got, want) < 1e-13
    assert relerr(res, pr.x - want) < 1e-13
    assert abs(c - ref.cost(pp, pr.x, md)) <= 1e-12 * c
    # flagged rows carry no model (lmfit.c:78-81)
    assert np.all(got.reshape(-1, 8)[pr.flag != 0] == 0.0)


@pytest.mark.parametrize("robust", [False, True])
def test_cost_and_grad(api, ref, bound, robust):
    pr = bound.pr
    pp = perturbed_jones(pr, seed=5)
    nu = 3.5
    md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, robust_nu=nu)
    cw = ref.cost(pp, pr.x, md, robust=robust)
    gw = ref.grad(pp, pr.x, md, robust=robust)
    with blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, pr.x) as dp:
        c = dp.cost(pp, robust=robust, nu=nu)
        g = dp.grad(pp, robust=robust, nu=nu)
    assert abs(c - cw) <= 1e-12 * abs(cw)
    assert relerr(g, gw) < 1e-11


def test_normal_equations(api, ref, bound):
    """J^T J, J^T e, ||e||^2 of every (cluster, chunk) against the reference's dense Jacobian"""
    pr = bound.pr
    pp = perturbed_jones(pr, seed=7)
    rng = np.random.default_rng(1)
    xd = pr.x + 0.01 * rng.normal(0, 1, pr.x.shape)
    xd.reshape(-1, 8)[pr.flag == 1] = 0.0
    with blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, pr.x) as dp:
        off = 0
        for k in range(pr.M):
            nch = pr.nchunk[k]
            tilechunk = (pr.tilesz + nch - 1) // nch
            for ck in range(nch):
                t0 = min(ck * tilechunk, pr.tilesz)
                t1 = min(t0 + tilechunk, pr.tilesz)
                pblk = pp[off:off + 8 * pr.N].copy()
                off += 8 * pr.N
                if t1 <= t0:
                    continue
                md = ref.me_data(pr.N, pr.Nbase, t1 - t0, bound.barr, bound.sky, pr.coh, clus=k,
                                 tileoff=t0)
                nn = 8 * (t1 - t0) * pr.Nbase
                xs = xd[8 * t0 * pr.Nbase: 8 * t1 * pr.Nbase]
                ee, JTe_ref, JTJ_ref = ref.normal_eq(pblk, xs, md)
                c, JTJ, JTe = dp.normal_eq(k, ck, pblk, xd)
                assert abs(c - ee) <= 1e-12 * ee
                assert relerr(JTe, JTe_ref) < 1e-11
                assert relerr(JTJ, JTJ_ref) < 1e-11
                assert np.array_equal(JTJ, JTJ.T)


def test_weighted_normal_equations(api, ref, bound):
    """robust LM system: J <- wt.J, e <- wt.e (robustlm.c:2298-2316) against the dense reference J"""
    pr = bound.pr
    pp = perturbed_jones(pr, seed=8)
    rng = np.random.default_rng(4)
    wt = rng.uniform(0.2, 1.3, pr.x.shape)
    with blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, bound.barr, bound.sky, pr.coh, pr.x) as dp:
        off = 0
        for k in range(pr.M):
            nch = pr.nchunk[k]
            tilechunk = (pr.tilesz + nch - 1) // nch
            for ck in range(nch):
                t0 = min(ck * tilechunk, pr.tilesz)
                t1 = min(t0 + tilechunk, pr.tilesz)
                pblk = pp[off:off + 8 * pr.N].copy()
                off += 8 * pr.N
                if t1 <= t0:
                    continue
                md = ref.me_data(pr.N, pr.Nbase, t1 - t0, bound.barr, bound.sky, pr.coh, clus=k,
                                 tileoff=t0)
                nn = 8 * (t1 - t0) * pr.Nbase
                sl = slice(8 * t0 * pr.Nbase, 8 * t1 * pr.Nbase)
                ee, JTe_ref, JTJ_ref = ref.normal_eq(pblk, pr.x[sl], md, wt[sl])
                c, JTJ, JTe = dp.normal_eq_weighted(k, ck, pblk, pr.x, wt)
                assert abs(c - ee) <= 1e-12 * ee
                assert relerr(JTe, JTe_ref) < 1e-11
                assert relerr(JTJ, JTJ_ref) < 1e-11
                assert relerr(JTJ, JTJ.T) < 1e-13


def test_coherencies_device(api, ref):
    b = small_problem(N=12, M=4, tilesz=6, seed=21, kmean=2.0, gaussian_frac=0.5)
    pr = b.pr
    barr1 = b.fresh_barr()
    want = ref.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, barr1, b.sky, pr.freq0,
                                        pr.fdelta, uvmin=30.0, uvmax=1e5)
    barr2 = b.fresh_barr()
    got = api.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, barr2, b.sky, pr.freq0,
                                       pr.fdelta, uvmin=30.0, uvmax=1e5)
    from sagecal_b200.dirac_api import barr_to_numpy
    assert np.array_equal(barr_to_numpy(barr1, pr.Nbase1)[2], barr_to_numpy(barr2, pr.Nbase1)[2])
    assert relerr(got, want) < 1e-11
    # resident variant
    barr3 = b.fresh_barr()
    with blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, barr3, b.sky, None, pr.x) as dp:
        dp.precalculate(pr.u, pr.v, pr.w, pr.freq0, pr.fdelta, uvmin=30.0, uvmax=1e5, barr=barr3)
        got2 = dp.get_coherencies()
    assert relerr(got2, want) < 1e-11
    assert np.array_equal(barr_to_numpy(barr1, pr.Nbase1)[2], barr_to_numpy(barr3, pr.Nbase1)[2])


def _extended_sky(pr, seed=5):
    """turn some sources of a problem's clusters into disks, rings and shapelets (orders 1-9, with
    and without the projection to the source's tangent plane)"""
    rng = np.random.default_rng(seed)
    cnt = 0
    for k, cl in enumerate(pr.clusters):
        K = len(cl["ll"])
        st = np.array(cl.get("stype", np.zeros(K)), dtype=np.uint8)
        disk, shp = {}, {}
        for s in range(K):
            if st[s] != 0:
                continue
            kind = cnt % 4  # point, disk, ring, shapelet in turn
            cnt += 1
            xi, phi = rng.uniform(0, 2 * np.pi), rng.uniform(0, 0.2)
            proj = (np.cos(xi), np.sin(xi), np.cos(phi), np.sin(phi))
            if kind in (1, 2):
                st[s] = 1 + kind  # disk / ring
                disk[s] = (np.deg2rad(rng.uniform(1.0, 4.0) / 60.0),) + proj + (1,)
            elif kind == 3:
                st[s] = 4
                n0 = int(rng.integers(1, 10))
                shp[s] = dict(n0=n0, beta=np.deg2rad(rng.uniform(0.5, 2.0) / 60.0),
                              modes=rng.normal(0, 1, n0 * n0) / n0, eX=rng.uniform(0.7, 1.5),
                              eY=rng.uniform(0.7, 1.5), eP=rng.uniform(0, np.pi), cxi=proj[0],
                              sxi=proj[1], cphi=proj[2], sphi=proj[3], use_projection=int(s % 2))
        cl["stype"] = st
        cl["disk"] = disk
        cl["shapelet"] = shp
    from sagecal_b200.dirac_api import SkyModel
    return SkyModel(pr.clusters, pr.N)


def test_coherencies_extended_sources(api, ref):
    """disks, rings and shapelets (shapelet.c:50-190) in the device coherency kernel"""
    b = small_problem(N=10, M=4, tilesz=4, seed=23, kmean=6.0, gaussian_frac=0.3)
    pr = b.pr
    sky = _extended_sky(pr)
    ntypes = set(int(t) for cl in pr.clusters for t in cl["stype"])
    assert ntypes >= {0, 2, 3, 4}
    want = ref.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(), sky,
                                        pr.freq0, pr.fdelta, uvmin=30.0, uvmax=1e5)
    got = api.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(), sky,
                                       pr.freq0, pr.fdelta, uvmin=30.0, uvmax=1e5)
    assert relerr(got, want) < 1e-11
    freqs = np.array([146e6, 152e6])
    xa = np.zeros(8 * pr.Nbase1 * len(freqs))
    xb = xa.copy()
    ref.predict_visibilities_multifreq(pr.u, pr.v, pr.w, xa, pr.N, pr.Nbase, pr.tilesz, b.barr, sky,
                                       freqs, pr.fdelta * 2, add_to_data=1)
    api.predict_visibilities_multifreq(pr.u, pr.v, pr.w, xb, pr.N, pr.Nbase, pr.tilesz, b.barr, sky,
                                       freqs, pr.fdelta * 2, add_to_data=1)
    assert relerr(xb, xa) < 1e-11


@pytest.mark.parametrize("add", [1, 2, 0])  # SIMUL_ONLY=1 clears, others accumulate
def test_predict_multifreq(api, ref, add):
    b = small_problem(N=10, M=3, tilesz=5, seed=22, kmean=2.0, gaussian_frac=0.3)
    pr = b.pr
    for cl in pr.clusters:  # give half of the sources a spectral index
        K = len(cl["ll"])
        cl["spec_idx"] = np.where(np.arange(K) % 2 == 0, -0.7, 0.0)
        cl["spec_idx1"] = np.full(K, 0.05)
        cl["spec_idx2"] = np.full(K, -0.01)
        cl["f0"] = np.full(K, 140e6)
    from sagecal_b200.dirac_api import SkyModel
    sky = SkyModel(pr.clusters, pr.N)
    freqs = np.array([145e6, 150e6, 155e6])
    rng = np.random.default_rng(2)
    x0 = rng.normal(0, 1, 8 * pr.Nbase1 * len(freqs))
    xa = x0.copy()
    xb = x0.copy()
    ref.predict_visibilities_multifreq(pr.u, pr.v, pr.w, xa, pr.N, pr.Nbase, pr.tilesz, b.barr, sky,
                                       freqs, pr.fdelta * 3, add_to_data=add)
    api.predict_visibilities_multifreq(pr.u, pr.v, pr.w, xb, pr.N, pr.Nbase, pr.tilesz, b.barr, sky,
                                       freqs, pr.fdelta * 3, add_to_data=add)
    assert relerr(xb, xa) < 1e-11


@pytest.mark.parametrize("ccid,nchunk,phase_only", [(-99999, None, 0), (1, None, 0), (2, [1, 2, 3], 0),
                                                    (1, None, 1), (2, [1, 2, 3], 1)],
                         ids=["no-correction", "correct-by-1", "hybrid-correct-by-2",
                              "phase-only-1", "phase-only-hybrid-2"])
def test_calculate_residuals_multifreq(api, ref, ccid, nchunk, phase_only):
    """full-resolution residual with the solved Jones and the optional correction by one cluster's
    inverse Jones (SURVEY.md 8f-2) against the compiled reference (residual.c:940-1061)"""
    from util import perturbed_jones
    b = small_problem(N=9, M=3, tilesz=6, seed=23, kmean=2.0, gaussian_frac=0.3, nchunk=nchunk)
    pr = b.pr
    for k, cl in enumerate(pr.clusters):
        K = len(cl["ll"])
        cl["spec_idx"] = np.where(np.arange(K) % 2 == 0, -0.7, 0.0)
        cl["spec_idx1"] = np.full(K, 0.05)
        cl["spec_idx2"] = np.full(K, -0.01)
        cl["f0"] = np.full(K, 140e6)
        cl["id"] = k if k != 0 else -1          # a negative id: predicted but not subtracted
    from sagecal_b200.dirac_api import SkyModel
    sky = SkyModel(pr.clusters, pr.N)
    freqs = np.array([146e6, 150e6, 154e6, 158e6])
    rng = np.random.default_rng(4)
    x0 = rng.normal(0, 1, 8 * pr.Nbase1 * len(freqs))
    pp = perturbed_jones(pr, amp=0.2)
    xa, xb = x0.copy(), x0.copy()
    ra = ref.calculate_residuals_multifreq(pr.u, pr.v, pr.w, pp.copy(), xa, pr.N, pr.Nbase, pr.tilesz,
                                           b.fresh_barr(), sky, freqs, pr.fdelta * 4, ccid=ccid, rho=1e-9,
                                           phase_only=phase_only)
    rb = api.calculate_residuals_multifreq(pr.u, pr.v, pr.w, pp.copy(), xb, pr.N, pr.Nbase, pr.tilesz,
                                           b.fresh_barr(), sky, freqs, pr.fdelta * 4, ccid=ccid, rho=1e-9,
                                           phase_only=phase_only)
    assert ra == rb == 0
    # (phase_only: the correction goes through a joint diagonalisation by Jacobi rotations,
    # manifold_average.c:399-610, restated on the host with its own 3x3 eigen-solver)
    assert relerr(xb, xa) < (1e-9 if phase_only else 1e-11)
    k = known(xa)
    assert relerr(xa[k], x0[k]) > 1e-3   # something was subtracted

"""GPU parity of the station-beam variants of the coherency / prediction calls (SURVEY.md 8f-4):
precalculate_coherencies_withbeam, predict_visibilities_multifreq_withbeam,
calculate_residuals_multifreq_withbeam against the compiled reference (predict_withbeam.c,
stationbeam.c, elementbeam.c): array factor of single and tile beam-formers, element beam, both,
narrow- and wide-band.  The element coefficient tables come from the REFERENCE library's
set_elementcoeffs (this library only evaluates them)."""
import ctypes as C

import numpy as np
import pytest

from util import small_problem, relerr, perturbed_jones, known
from sagecal_b200.dirac_api import BeamSetup, SkyModel, elementcoeff, dptr

pytestmark = pytest.mark.gpu

DOBEAM = {"array": 1, "full": 2, "element": 3, "array_wb": 4, "full_wb": 5, "element_wb": 6}


def beam_problem(ref, mode, tile, seed=31, freqs=(150e6,), tilesz=5):
    b = small_problem(N=9, M=3, tilesz=tilesz, seed=seed, kmean=2.0, gaussian_frac=0.3)
    pr = b.pr
    rng = np.random.default_rng(seed)
    ra0, dec0 = 1.2, np.deg2rad(58.0)
    for k, cl in enumerate(pr.clusters):   # sources a few degrees around the phase centre
        K = len(cl["ll"])
        cl["ra"] = ra0 + np.deg2rad(rng.uniform(-4, 4, K))
        cl["dec"] = dec0 + np.deg2rad(rng.uniform(-4, 4, K))
    pr.clusters[-1]["dec"][0] = np.deg2rad(-60.0)   # one source below the horizon: zero gain
    sky = SkyModel(pr.clusters, pr.N)
    lon = np.deg2rad(6.87 + rng.uniform(-0.5, 0.5, pr.N))
    lat = np.deg2rad(52.9 + rng.uniform(-0.3, 0.3, pr.N))
    t = 2456789.3 + np.arange(pr.tilesz) * 10.0 / 86400.0
    elems = []
    for n in range(pr.N):
        if tile:   # 16 dipoles of a 4 x 4 tile, then 20-24 tile centroids
            g = (np.arange(4) - 1.5) * 1.25
            dip = np.array([[x, y, 0.0] for x in g for y in g])
            cen = np.c_[rng.uniform(-15, 15, (20 + n % 5, 2)), rng.normal(0, 0.05, 20 + n % 5)]
            elems.append(np.vstack([dip, cen]))
        else:
            K = 40 + 3 * n
            elems.append(np.c_[rng.uniform(-40, 40, (K, 2)), rng.normal(0, 0.1, K)])
    ec = None
    if "element" in mode or "full" in mode:
        ec = elementcoeff()
        if mode.endswith("_wb"):
            f = np.ascontiguousarray(freqs, dtype=np.float64)
            ref.lib.set_elementcoeffs_wb(1 if tile else 0, dptr(f), len(f), C.byref(ec))
        else:
            ref.lib.set_elementcoeffs(1 if tile else 0, C.c_double(float(np.mean(freqs))),
                                      C.byref(ec))
    beam = BeamSetup(2 if tile else 1, ra0 + 0.01, dec0 - 0.01, ra0, dec0, 148e6, lon, lat, t, elems,
                     ec, DOBEAM[mode])
    return b, sky, beam


CASES = [("array", False), ("array", True), ("element", False), ("full", True), ("full_wb", False),
         ("array_wb", True), ("element_wb", True)]


@pytest.mark.parametrize("mode,tile", CASES, ids=["%s-%s" % (m, "tile" if t else "single")
                                                   for m, t in CASES])
def test_coherencies_withbeam(api, ref, mode, tile):
    b, sky, beam = beam_problem(ref, mode, tile)
    pr = b.pr
    want = ref.precalculate_coherencies_withbeam(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(),
                                                 sky, pr.freq0, pr.fdelta, beam, uvmin=30.0,
                                                 uvmax=1e5)
    got = api.precalculate_coherencies_withbeam(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(),
                                                sky, pr.freq0, pr.fdelta, beam, uvmin=30.0,
                                                uvmax=1e5)
    assert np.max(np.abs(want[known(want)])) > 0
    assert relerr(got, want) < 1e-10, relerr(got, want)
    # the beam matters: the result differs from the beam-less coherencies
    plain = ref.precalculate_coherencies(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(), sky,
                                         pr.freq0, pr.fdelta, uvmin=30.0, uvmax=1e5)
    k = known(want) & known(plain)
    assert relerr(want[k], plain[k]) > 1e-3


@pytest.mark.parametrize("mode,tile", [("full", False), ("full_wb", True), ("array", True)],
                         ids=["full-single", "full_wb-tile", "array-tile"])
def test_predict_and_residual_withbeam(api, ref, mode, tile):
    freqs = np.array([146e6, 152e6])
    b, sky, beam = beam_problem(ref, mode, tile, seed=37, freqs=freqs)
    pr = b.pr
    xa = np.zeros(8 * pr.Nbase1 * len(freqs))
    xb = xa.copy()
    ref.predict_visibilities_multifreq_withbeam(pr.u, pr.v, pr.w, xa, pr.N, pr.Nbase, pr.tilesz,
                                                b.barr, sky, freqs, pr.fdelta * 2, beam)
    api.predict_visibilities_multifreq_withbeam(pr.u, pr.v, pr.w, xb, pr.N, pr.Nbase, pr.tilesz,
                                                b.barr, sky, freqs, pr.fdelta * 2, beam)
    assert relerr(xb, xa) < 1e-10, relerr(xb, xa)
    # full-resolution residual with solutions and the correction by cluster 1
    pp = perturbed_jones(pr, seed=4, amp=0.1)
    rng = np.random.default_rng(2)
    x0 = xb + rng.normal(0, 0.01, xb.shape)   # (xa may be a stored sample of the reference's)
    ra, rb = x0.copy(), x0.copy()
    ref.calculate_residuals_multifreq_withbeam(pr.u, pr.v, pr.w, pp, ra, pr.N, pr.Nbase, pr.tilesz,
                                               b.barr, sky, freqs, pr.fdelta * 2, beam, ccid=1)
    api.calculate_residuals_multifreq_withbeam(pr.u, pr.v, pr.w, pp, rb, pr.N, pr.Nbase, pr.tilesz,
                                               b.barr, sky, freqs, pr.fdelta * 2, beam, ccid=1)
    assert relerr(rb, ra) < 1e-9, relerr(rb, ra)


def test_coherencies_multifreq(api, ref):
    """precalculate_coherencies_multifreq: the [chan][row][cluster][4] coherencies the minibatch
    drivers feed bfgsfit_minibatch_* (predict.c:745-816), flags included (uvmin at the first
    channel, uvmax at the last)"""
    from sagecal_b200.dirac_api import barr_to_numpy
    freqs = np.array([144e6, 150e6, 157e6])
    b, sky, _ = beam_problem(ref, "array", False, seed=41, freqs=freqs)
    pr = b.pr
    uvd = np.sqrt(pr.u ** 2 + pr.v ** 2) * freqs[0]
    uvmin, uvmax = float(np.quantile(uvd, 0.1)), float(np.quantile(uvd, 0.93))
    ba, bb = b.fresh_barr(), b.fresh_barr()
    want = ref.precalculate_coherencies_multifreq(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, ba, sky, freqs,
                                                  pr.fdelta * 3, None, uvmin=uvmin, uvmax=uvmax)
    got = api.precalculate_coherencies_multifreq(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, bb, sky, freqs,
                                                 pr.fdelta * 3, None, uvmin=uvmin, uvmax=uvmax)
    assert relerr(got, want) < 1e-10, relerr(got, want)
    fa, fb = barr_to_numpy(ba, pr.Nbase1)[2], barr_to_numpy(bb, pr.Nbase1)[2]
    assert np.array_equal(fa, fb) and np.sum(fa == 2) > 0


@pytest.mark.parametrize("mode,tile", [("full_wb", True), ("array", False), ("element", True)],
                         ids=["full_wb-tile", "array-single", "element-tile"])
def test_coherencies_multifreq_withbeam(api, ref, mode, tile):
    """precalculate_coherencies_multifreq_withbeam.  The reference's CPU implementation of THIS call
    cannot serve as the pin: it strides its channels by the baselines of one timeslot although the
    rows span all timeslots (chanoff = 4 M N(N-1)/2, predict_withbeam.c:281,787) and reads the beam
    tables without their channel index (:337-338,382-383), so every channel gets the first channel's
    beam and the channels overlap.  What this library computes is the evident meaning -- channel c =
    the single-channel call at freqs[c] with the smearing width fdelta / Nchan -- and that is what is
    compared: against the reference's single-channel precalculate_coherencies_withbeam per channel."""
    import ctypes as C
    from sagecal_b200.dirac_api import barr_to_numpy, elementcoeff
    freqs = np.array([144e6, 150e6, 157e6])
    b, sky, beam = beam_problem(ref, mode, tile, seed=41, freqs=freqs)
    pr = b.pr
    got = api.precalculate_coherencies_multifreq(pr.u, pr.v, pr.w, pr.N, pr.Nbase1, b.fresh_barr(),
                                                 sky, freqs, pr.fdelta * 3, beam, uvmin=30.0,
                                                 uvmax=1e5)
    n = 4 * sky.M * pr.Nbase1
    for c, f in enumerate(freqs):
        one = beam
        if mode.endswith("_wb") and beam.ecoeff is not None:  # this channel's coefficient set
            ec = elementcoeff()
            fc = np.array([f])
            ref.lib.set_elementcoeffs_wb(1 if tile else 0, dptr(fc), 1, C.byref(ec))
            one = BeamSetup(beam.bf_type, beam.s[0].value, beam.s[1].value, beam.s[2].value,
                            beam.s[3].value, beam.s[4].value, beam.lon, beam.lat, beam.t,
                            [e.T for e in beam.xyz], ec, beam.doBeam)
        want = ref.precalculate_coherencies_withbeam(pr.u, pr.v, pr.w, pr.N, pr.Nbase1,
                                                     b.fresh_barr(), sky, f, pr.fdelta, one,
                                                     uvmin=30.0, uvmax=1e5)
        assert relerr(got[c * n:(c + 1) * n], want) < 1e-10, (c, relerr(got[c * n:(c + 1) * n], want))

"""helpers shared by the tests: problems in API layout bound to ctypes structures"""
import numpy as np

import refgolden

from sagecal_b200 import synth
from sagecal_b200.dirac_api import SkyModel, make_barr


class Bound:
    """a synthetic problem plus the ctypes objects both libraries take"""

    def __init__(self, pr: synth.Problem):
        self.pr = pr
        self.barr = make_barr(pr.sta1, pr.sta2, pr.flag)
        self.sky = SkyModel(pr.clusters, pr.N)
        self.n = 8 * pr.Nbase1
        self.m = 8 * pr.N * pr.Mt

    def fresh_barr(self):
        return make_barr(self.pr.sta1, self.pr.sta2, self.pr.flag)


def small_problem(N=8, M=2, tilesz=10, seed=11, **kw):
    return Bound(synth.make_problem(N=N, M=M, tilesz=tilesz, seed=seed, **kw))


def perturbed_jones(pr, seed=3, amp=0.1):
    rng = np.random.default_rng(seed)
    return pr.pp0 + amp * rng.normal(0, 1, pr.pp0.shape)


def known(ref_out):
    """the entries of a reference output that are known: all of them, except while recorded reference
    results are replayed (refgolden.py), where an output stored as a sample is NaN elsewhere"""
    ref_out = np.asarray(ref_out)
    if refgolden.replaying():
        return ~np.isnan(ref_out)
    return np.ones(ref_out.shape, dtype=bool)


def relerr(a, b):
    """max |a - b| / max |b|; while reference results are replayed, over the known entries of b only
    (a NaN in a where b is known still fails)"""
    a = np.asarray(a)
    b = np.asarray(b)
    k = known(b)
    if a.shape == b.shape and not k.all():
        a, b = a[k], b[k]
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-300))

"""TEST INFRASTRUCTURE ONLY.  ctypes access to the compiled reference CPU hot path
(`oracle/_ref/libdirac_ref.so`, built by oracle/Makefile from the sources under /root/reference)
including the file-static callbacks exported by the shims (ref_shim_*.c).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from sagecal_b200.dirac_api import (DiracAPI, SkyModel, baseline_t, clus_source_t, c_double_p,
                                    dptr, cptr)

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_PATH = os.path.join(_HERE, "_ref", "libdirac_ref.so")
# same object code, except that the robust RTR / NSD solvers run their threads synchronously
# (ref_shim_rtr_serial.c): the deterministic pin of solver_mode 5 and 6
SERIAL_PATH = os.path.join(_HERE, "_ref", "libdirac_ref_serial.so")


def available() -> bool:
    return os.path.exists(REF_PATH)


class RefDirac(DiracAPI):
    def __init__(self, path: str = REF_PATH):
        super().__init__(path)
        L = self.lib
        i, d, dp, vp = C.c_int, C.c_double, c_double_p, C.c_void_p
        L.ref_sizeof_me_data.restype = C.c_size_t
        L.ref_fill_me_data.argtypes = [vp, i, i, i, i, C.POINTER(baseline_t),
                                       C.POINTER(clus_source_t), i, i, dp, i, dp, i, d]
        L.ref_get_robust_nu.restype = d
        L.ref_get_robust_nu.argtypes = [vp]
        for name in ("ref_mylm_fit_single_pth", "ref_mylm_fit_single_pth0",
                     "ref_mylm_jac_single_pth", "minimize_viz_full_pth"):
            getattr(L, name).argtypes = [dp, dp, i, i, vp]
            getattr(L, name).restype = None
        for name in ("ref_cost_func", "ref_robust_cost_func"):
            getattr(L, name).restype = d
            getattr(L, name).argtypes = [dp, i, dp, i, vp]
        for name in ("ref_grad_func", "ref_robust_grad_func"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [dp, dp, i, dp, i, vp]
        fn = C.CFUNCTYPE(None, dp, dp, i, i, vp)
        self._fn = fn
        L.clevmar_der_single_nocuda.restype = i
        L.clevmar_der_single_nocuda.argtypes = [vp, vp, dp, dp, i, i, i, dp, dp, i, vp]
        L.oslevmar_der_single_nocuda.restype = i
        L.oslevmar_der_single_nocuda.argtypes = [vp, vp, dp, dp, i, i, i, dp, dp, i, i, vp]
        L.rlevmar_der_single_nocuda.restype = i
        L.rlevmar_der_single_nocuda.argtypes = [vp, vp, dp, dp, i, i, i, dp, dp, i, i, d, d, vp]
        L.osrlevmar_der_single_nocuda.restype = i
        L.osrlevmar_der_single_nocuda.argtypes = [vp, vp, dp, dp, i, i, i, dp, dp, i, i, d, d, i,
                                                  vp]
        L.rtr_solve_nocuda.restype = i
        L.rtr_solve_nocuda.argtypes = [dp, dp, i, i, i, i, d, d, dp, vp]
        L.rtr_solve_nocuda_robust.restype = i
        L.rtr_solve_nocuda_robust.argtypes = [dp, dp, i, i, i, i, d, d, d, d, dp, vp]
        L.nsd_solve_nocuda_robust.restype = i
        L.nsd_solve_nocuda_robust.argtypes = [dp, dp, i, i, i, d, d, dp, vp]
        L.rtr_solve_nocuda_robust_admm.restype = i
        L.rtr_solve_nocuda_robust_admm.argtypes = [dp, dp, dp, dp, i, i, i, i, d, d, d, d, d, dp, vp]
        L.update_w_and_nu.restype = d
        L.update_w_and_nu.argtypes = [d, dp, dp, i, i, d, d]

    # ---- me_data_t -------------------------------------------------------------------------
    def me_data(self, N, Nbase, tilesz, barr, sky: SkyModel, coh, clus=-1, tileoff=0, Nt=4,
                robust_nu=2.0, freq0=150e6):
        buf = C.create_string_buffer(self.lib.ref_sizeof_me_data())
        f0 = np.array([freq0])
        self.lib.ref_fill_me_data(buf, clus, Nbase, tilesz, N, barr, sky.arr, sky.M, sky.Mt,
                                  dptr(f0), Nt, cptr(coh), tileoff, robust_nu)
        buf._keep = (f0, barr, sky, coh)
        return buf

    # ---- predict / cost / gradient ---------------------------------------------------------
    def predict_full(self, pp, md, n):
        """minimize_viz_full_pth, lmfit.c:692"""
        x = np.zeros(n)
        self.lib.minimize_viz_full_pth(dptr(pp), dptr(x), len(pp), n, md)
        return x

    def predict_cluster(self, pp, md, n):
        """mylm_fit_single_pth (md.clus selects the cluster), lmfit.c:137"""
        x = np.zeros(n)
        self.lib.ref_mylm_fit_single_pth(dptr(pp), dptr(x), len(pp), n, md)
        return x

    def lm_func(self, pblk, md, n):
        x = np.zeros(n)
        self.lib.ref_mylm_fit_single_pth0(dptr(pblk), dptr(x), len(pblk), n, md)
        return x

    def lm_jac(self, pblk, md, n):
        """dense Jacobian [n, 8N] (row major), lmfit.c:484"""
        m = len(pblk)
        jac = np.zeros(n * m)
        self.lib.ref_mylm_jac_single_pth(dptr(pblk), dptr(jac), m, n, md)
        return jac.reshape(n, m)

    def normal_eq(self, pblk, xs, md, wt=None):
        """(e.e, J^T e, J^T J) of one (cluster, chunk) from the dense Jacobian and the model, with
        J <- wt.J and e <- wt.e when weights are given (robustlm.c:2298-2316)"""
        n = len(xs)
        J = self.lm_jac(pblk, md, n)
        e = xs - self.lm_func(pblk, md, n)
        if wt is not None:
            J = J * wt[:, None]
            e = wt * e
        return e @ e, J.T @ e, J.T @ J

    def cost(self, pp, x, md, robust=False):
        f = self.lib.ref_robust_cost_func if robust else self.lib.ref_cost_func
        return f(dptr(pp), len(pp), dptr(x), len(x), md)

    def grad(self, pp, x, md, robust=False):
        g = np.zeros(len(pp))
        f = self.lib.ref_robust_grad_func if robust else self.lib.ref_grad_func
        f(dptr(pp), dptr(g), len(pp), dptr(x), len(x), md)
        return g

    # ---- LM on one (cluster, chunk) --------------------------------------------------------
    def clevmar(self, pblk, xd, md, itmax, linsolv=0, opts=(1e-3, 1e-15, 1e-15, 1e-20, -1e-6),
                os_=False, randomize=0):
        """clevmar_der_single_nocuda / oslevmar_der_single_nocuda on hidden data xd (clmfit.c:29,1074)"""
        pblk = np.ascontiguousarray(pblk, dtype=np.float64).copy()
        info = np.zeros(10)
        o = np.array(opts, dtype=np.float64)
        f = C.cast(self.lib.ref_mylm_fit_single_pth0, C.c_void_p)
        j = C.cast(self.lib.ref_mylm_jac_single_pth, C.c_void_p)
        if os_:
            self.lib.oslevmar_der_single_nocuda(f, j, dptr(pblk), dptr(xd), len(pblk), len(xd),
                                                itmax, dptr(o), dptr(info), linsolv, randomize, md)
        else:
            self.lib.clevmar_der_single_nocuda(f, j, dptr(pblk), dptr(xd), len(pblk), len(xd),
                                               itmax, dptr(o), dptr(info), linsolv, md)
        return pblk, info

    def rlevmar(self, pblk, xd, md, itmax, linsolv=0, nulow=2.0, nuhigh=30.0, Nt=4, os_=False,
                randomize=0):
        """rlevmar_der_single_nocuda / osrlevmar_der_single_nocuda (robustlm.c:2008,2607)"""
        pblk = np.ascontiguousarray(pblk, dtype=np.float64).copy()
        info = np.zeros(10)
        f = C.cast(self.lib.ref_mylm_fit_single_pth0, C.c_void_p)
        j = C.cast(self.lib.ref_mylm_jac_single_pth, C.c_void_p)
        if os_:
            self.lib.osrlevmar_der_single_nocuda(f, j, dptr(pblk), dptr(xd), len(pblk), len(xd),
                                                 itmax, None, dptr(info), linsolv, Nt, nulow,
                                                 nuhigh, randomize, md)
        else:
            self.lib.rlevmar_der_single_nocuda(f, j, dptr(pblk), dptr(xd), len(pblk), len(xd),
                                               itmax, None, dptr(info), linsolv, Nt, nulow, nuhigh,
                                               md)
        return pblk, info, self.lib.ref_get_robust_nu(md)


    def rtr(self, pblk, xd, md, N, nrows, kind, itmax_a, itmax_b, nulow=2.0, nuhigh=30.0):
        """rtr_solve_nocuda (kind 4, rtr_solve.c:1207), rtr_solve_nocuda_robust (5,
        rtr_solve_robust.c:1440), nsd_solve_nocuda_robust (6, :1877) on hidden data xd; md carries
        the cluster, the tile range and robust_nu (in/out)"""
        p = np.ascontiguousarray(pblk, dtype=np.float64).copy()
        info = np.zeros(10)
        xd = np.ascontiguousarray(xd, dtype=np.float64).copy()
        if kind == 4:
            self.lib.rtr_solve_nocuda(dptr(p), dptr(xd), N, nrows, itmax_a, itmax_b, 0.01,
                                      0.01 * 0.125, dptr(info), md)
        elif kind == 5:
            self.lib.rtr_solve_nocuda_robust(dptr(p), dptr(xd), N, nrows, itmax_a, itmax_b, 0.01,
                                             0.01 * 0.125, nulow, nuhigh, dptr(info), md)
        else:
            self.lib.nsd_solve_nocuda_robust(dptr(p), dptr(xd), N, nrows, itmax_a, nulow, nuhigh,
                                             dptr(info), md)
        return p, info, self.lib.ref_get_robust_nu(md)

    def rtr_admm(self, pblk, Y, BZ, xd, md, N, nrows, itmax_a, itmax_b, rho, nulow=2.0, nuhigh=30.0):
        """rtr_solve_nocuda_robust_admm (rtr_solve_robust_admm.c:1424) on hidden data xd"""
        p = np.ascontiguousarray(pblk, dtype=np.float64).copy()
        info = np.zeros(10)
        xd = np.ascontiguousarray(xd, dtype=np.float64).copy()
        Y = np.ascontiguousarray(Y, dtype=np.float64).copy()
        BZ = np.ascontiguousarray(BZ, dtype=np.float64).copy()
        self.lib.rtr_solve_nocuda_robust_admm(dptr(p), dptr(Y), dptr(BZ), dptr(xd), N, nrows, itmax_a,
                                              itmax_b, 2.0, 0.25, rho, nulow, nuhigh, dptr(info), md)
        return p, info, self.lib.ref_get_robust_nu(md)


_ref = None
_ser = None


def load_serial() -> RefDirac:
    global _ser
    if _ser is None:
        _ser = RefDirac(SERIAL_PATH)
    return _ser


def load() -> RefDirac:
    global _ref
    if _ref is None:
        _ref = RefDirac()
    return _ref

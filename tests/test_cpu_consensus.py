"""CPU: the consensus (ADMM over subbands) pieces that need no GPU.
 - frequency basis and per-cluster pseudo-inverse of the product library (host arithmetic in
   csrc/consensus.cu) against the compiled reference (consensus_poly.c: setup_polynomials,
   find_prod_inverse_full);
 - the fused exchange formula (every rank forms B_f Bi z itself from the all-reduced z) against the
   reference's master-side update_global_z followed by B_f Z, under gloo with world_size 2."""
import ctypes as C
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from sagecal_b200 import consensus as cons
from sagecal_b200.dirac_api import dptr


def vptr(a):
    """a void * to the array that keeps the array with it (numpy's data_as)"""
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope="module")
def capi():
    from sagecal_b200 import lib
    return lib.load()


@pytest.mark.parametrize("ptype", [0, 1, 2, 3])
def test_basis_matches_reference(capi, ref, ptype):
    freqs = np.linspace(115e6, 185e6, 8)
    for Npoly in (2, 3, 4):
        B = cons.basis(capi, freqs, 150e6, Npoly, ptype)
        Br = np.zeros((8, Npoly))
        ref.lib.setup_polynomials.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_int]
        ref.lib.setup_polynomials(vptr(Br), Npoly, 8, vptr(freqs), 150e6, ptype)
        assert np.allclose(B, Br, rtol=1e-14, atol=1e-300)


def test_prod_inverse_matches_reference(capi, ref):
    rng = np.random.default_rng(2)
    freqs = np.linspace(115e6, 185e6, 8)
    for Npoly, ptype in ((3, 1), (4, 2), (2, 0)):
        B = cons.basis(capi, freqs, 150e6, Npoly, ptype)
        M = 5
        rho = rng.uniform(0.5, 20.0, (8, M))
        Bi = cons.prod_inverse(capi, B, rho)
        Bir = np.zeros((M, Npoly, Npoly))
        ref.lib.find_prod_inverse_full.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                   C.c_void_p, C.c_int]
        Bc = np.ascontiguousarray(B)
        ref.lib.find_prod_inverse_full(vptr(Bc), vptr(Bir), Npoly, 8, M, vptr(rho), 2)
        assert np.max(np.abs(Bi - Bir)) <= 1e-9 * np.max(np.abs(Bir))


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import torch
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import refdirac
    from sagecal_b200 import lib
    api = lib.load()
    N, M, Npoly = 5, 3, 3
    m = 8 * N * M
    freqs = np.array([140e6, 160e6])
    rng = np.random.default_rng(7)                       # same numbers on both ranks
    Jall = rng.normal(0, 1, (world, m))
    Yall = rng.normal(0, 0.1, (world, m))
    rho = np.array([5.0, 2.0, 9.0])
    B = cons.basis(api, freqs, 150e6, Npoly, 1)
    Bi = cons.prod_inverse(api, B, np.tile(rho, (world, 1)))
    clus_of = np.repeat(np.arange(M), 8 * N)
    rho_i = rho[clus_of]

    def allreduce(z):
        t = torch.from_numpy(z)
        dist.all_reduce(t)

    Ynew, bz, pr, du = cons.step_numpy(Jall[rank], Yall[rank], np.zeros(m), rho_i, B[rank], Bi, clus_of,
                                       allreduce)
    ok = True
    if refdirac.available():
        # what the reference's master does: z = sum_f B_f (x) (Y_f + rho J_f) in its own ordering
        # (z[np][cluster][8N]), Z = update_global_z(z, Bi), then B_f Z for this subband
        ref = refdirac.load()
        z = np.zeros((Npoly, m))
        for f in range(world):
            z += B[f][:, None] * (Yall[f] + rho_i * Jall[f])[None, :]
        Z = np.zeros((M, Npoly, 8 * N))
        # update_global_z takes ONE Bi (Npoly x Npoly): call it per cluster with that cluster's Bi
        for k in range(M):
            zk = np.ascontiguousarray(z[:, k * 8 * N:(k + 1) * 8 * N]).reshape(-1)
            Zk = np.zeros(Npoly * 8 * N)
            ref.lib.update_global_z.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            Bik = np.ascontiguousarray(Bi[k])
            ref.lib.update_global_z(Zk.ctypes.data, N, 1, Npoly, zk.ctypes.data, Bik.ctypes.data)
            Z[k] = Zk.reshape(Npoly, 8 * N)
        bz_ref = np.concatenate([B[rank] @ Z[k] for k in range(M)])
        ok = ok and np.max(np.abs(bz - bz_ref)) <= 1e-12 * np.max(np.abs(bz_ref))
        ok = ok and np.allclose(Ynew, Yall[rank] + rho_i * (Jall[rank] - bz_ref), rtol=1e-12, atol=1e-14)
    out[rank] = 1 if ok else 0
    dist.destroy_process_group()


def test_consensus_exchange_gloo_world2():
    world = 2
    port = 29700 + (os.getpid() % 2000)
    with mp.Manager() as mgr:
        out = mgr.dict()
        mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
        assert dict(out) == {0: 1, 1: 1}

#!/usr/bin/env python
"""bench.py — baseline-visibilities/s through predict+Jacobian (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (own arm, hand-written sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K ...  (the reference's CPU path, bounded sample)

One "step" = one complete direction-dependent solve of the workload on device-resident inputs:
`max_emiter` SAGE sweeps over all M clusters (per cluster: hidden data, J^T e, J^T J, damped solve,
trial cost, Jones update) followed by `max_lbfgs` LBFGS iterations over all clusters (cost +
gradient passes).  Units per step = rows x clusters x (SAGE sweeps + LBFGS gradient evaluations
actually performed): every baseline-visibility of every direction goes through predict + Jacobian
once per sweep.  `value` = units / time on resident data, `e2e` = the same solve through the
drop-in C entry point `sagefit_visibilities` with pinned HOST buffers (upload of coherencies and
data, download of residual and Jones inside the timed region).  The K timed steps run without any
per-kernel instrumentation; the same K steps are then repeated with a CUDA-event pair around every
kernel of the path, which is where `roofline` (dominant streaming kernel) and `roofline.solver` /
`roofline.kernels` (shares of the step) come from.

Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "baseline_visibilities_per_sec_predict_jacobian"
UNIT = "baseline-visibilities/s"

SOLVE = dict(max_emiter=3, max_iter=2, max_lbfgs=10, lbfgs_m=7, linsolv=0, solver_mode=1,
             nulow=2.0, nuhigh=30.0, randomize=0)
#: bounded CPU sample of the same workload (dense Jacobian + dgemm make the full shape infeasible:
#: 7.2 GB and ~0.9 PFLOP per cluster-iteration at N=62,T=120; SURVEY.md 8d)
CPU_SAMPLE = dict(N=62, M=4, tilesz=4)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4",
                    help="C4 (512 stations, 32 clusters per GPU, 120 slots: the workload BASELINE.json's "
                         "metric is quoted on, 256 clusters on 8 GPUs) | C2 (62 st, 64 clusters) | C3 "
                         "(robust) | C1 | custom N,M,T e.g. 62,16,30")
    ap.add_argument("--only", action="store_true", help="one GPU: do not append the C2 and C3 lines")
    ap.add_argument("--profile-run", action="store_true",
                    help="for runs UNDER ncu only: 1 warm-up, no instrumented repeat, no e2e, no CPU leg "
                         "(a number printed by such a run is never a bench value)")
    ap.add_argument("--devgen", action="store_true", help="generate the coherencies on the device "
                    "(always for C4)")
    ap.add_argument("--c4-clusters-per-gpu", type=int, default=32)
    ap.add_argument("--c5-solver", default="lm", choices=["rtr", "lm"],
                    help="J-update of the consensus workload: lm = this library's LM on the augmented "
                         "cost (default: it keeps improving from a good starting point), rtr = the "
                         "reference's robust Riemannian trust-region solver on the same cost "
                         "(admm_solve.c:331-352; what sagefit_visibilities_admm runs): it keeps a "
                         "visit only if the WEIGHTED final cost beats the UNWEIGHTED entry cost, and "
                         "its weights exceed 1, so after the plain first iteration of this synthetic "
                         "workload it discards every visit (DESIGN.md 9b)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (solved Jones, return code, mean nu, "
                         "initial and final residual) as DIR/<workload>_<name>.npy, float64, so two "
                         "builds can be compared output for output on the same seeded inputs (the "
                         "reference arm: DIR/reference_<workload>_<name>.npy)")
    return ap.parse_args()


def dump_outputs(args, name, arrays):
    """rank 0 only: the arrays a caller of the timed path receives, one .npy per array"""
    if not args.dump_outputs:
        return
    os.makedirs(args.dump_outputs, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(args.dump_outputs, "%s_%s.npy" % (name, k)),
                np.asarray(a, dtype=np.float64))


def solve_args(name):
    """solver settings of a workload: C3 is the robust configuration (robust LM in the last sweep +
    Student's-t LBFGS, SURVEY.md 8d); everything else plain LM + LBFGS"""
    a = dict(SOLVE)
    if name == "C3":
        a["solver_mode"] = 2
    elif name == "C3os":
        a["solver_mode"] = 3
    elif name == "C2rtr":      # RSD + RTR per cluster (rtr_solve.c), plain LBFGS
        a["solver_mode"] = 4
    elif name in ("C3rtr", "C4rtr"):   # robust RTR: the reference driver's default -j 5 (data.cpp:69)
        a["solver_mode"] = 5
    elif name == "C3nsd":      # Nesterov's accelerated descent
        a["solver_mode"] = 6
    return a


def golden_parity(name, pr, pp, res):
    """solved Jones of one step against the committed golden of the CPU restatement at the FULL
    shape (tests/golden/full/*.npz, generator tests/golden/make_golden_full.py; the restatement is
    pinned to the compiled reference at the reduced shape).  Checker only, outside every timed region."""
    path = os.path.join(ROOT, "tests", "golden", "full", name + ".npz")
    if not os.path.exists(path):
        return {"checked": False, "why": "no golden for workload %s" % name}
    g = np.load(path)
    fp = np.array([np.sum(pr.x), np.sum(np.abs(pr.x)), np.sum(pr.coh.real), np.sum(pr.coh.imag),
                   np.sum(np.abs(pr.coh)), float(np.sum(pr.flag)), np.sum(pr.u), np.sum(pr.w)])
    same_inputs = bool(np.allclose(fp, g["fingerprint"], rtol=1e-10, atol=0))
    want = g["out_scalars"]
    err = float(np.max(np.abs(pp - g["out_pp"])) / np.max(np.abs(g["out_pp"])))
    return {"checked": True, "against": "oracle/liboracle.so golden tests/golden/full/%s.npz" % name,
            "same_inputs": same_inputs, "jones_max_relerr": err, "tolerance": 1e-5,
            "ok": bool(same_inputs and err < 1e-5),
            "res_0": [res[2], float(want[2])], "res_1": [res[3], float(want[3])],
            "mean_nu": [res[1], float(want[1])]}


def workload_shape(name):
    from sagecal_b200 import synth
    if name in ("C3os", "C3rtr", "C3nsd"):
        name = "C3"
    if name == "C2rtr":
        name = "C2"
    if name == "C4rtr":
        name = "C4"
    if name in synth.CONFIGS:
        c = synth.CONFIGS[name]
        return dict(N=c["N"], M=c["M"], tilesz=c["tilesz"], radius=c["radius"], seed=c["seed"],
                    kmean=c["kmean"], outliers=c.get("outliers", 0.0))
    N, M, T = (int(v) for v in name.split(","))
    return dict(N=N, M=M, tilesz=T, radius=40e3, seed=20260921 + 2, kmean=2.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload="C2"):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            t = json.load(f)
        if workload in ("C3rtr", "C3nsd"):
            return t.get("k_rtr_stats_dram_bytes_per_launch_C3")
        return t.get("k_cluster_pass_dram_bytes_per_launch_" + workload,
                     t.get("k_cluster_pass_dram_bytes_per_launch") if workload == "C2" else None)
    return None


# ---------------------------------------------------------------------------------------------
# reference (CPU) arm — the only place besides tests/ and smoke() that may execute oracle/
# ---------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, seed, outputs=None):
    """times the reference's own sagefit_visibilities (oracle/_ref) on a bounded sample of the
    workload with every host thread; returns (units/s, seconds per step, description).  `outputs`,
    if given, receives what the last step returned (solved Jones and result values)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refdirac
    from sagecal_b200 import synth
    from sagecal_b200.dirac_api import SkyModel, make_barr
    if not refdirac.available():
        return None, None, "oracle/_ref/libdirac_ref.so not built"
    ref = refdirac.load()
    # the reference spawns Nt pthreads per predict/Jacobian call AND lets OpenBLAS thread its dgemm;
    # beyond ~32 threads each the sample only gets slower (oversubscription), so cap there
    cores = min(os.cpu_count() or 1, 32)
    try:
        ref.lib.openblas_set_num_threads(cores)
    except AttributeError:
        pass
    pr = synth.make_problem(radius=40e3, seed=seed, kmean=2.0, **CPU_SAMPLE)
    barr = make_barr(pr.sta1, pr.sta2, pr.flag)
    sky = SkyModel(pr.clusters, pr.N)
    sweeps = SOLVE["max_emiter"] + SOLVE["max_lbfgs"] + 1
    units = pr.Nbase1 * pr.M * sweeps
    ts = []
    for it in range(warmup + steps):
        x = pr.x.copy()
        pp = pr.pp0.copy()
        t0 = time.perf_counter()
        res = ref.sagefit_visibilities(pr.u, pr.v, pr.w, x, pr.N, pr.Nbase, pr.tilesz, barr, sky,
                                       pr.coh, pp, Nt=cores, **SOLVE)
        t1 = time.perf_counter()
        if it >= warmup:
            ts.append(t1 - t0)
    if outputs is not None:
        outputs.update(jones=pp, result=res)
    sec = float(np.mean(ts))
    desc = ("reference sagefit_visibilities (oracle/_ref, gcc -O2, OpenBLAS %d threads, Nt=%d) on "
            "N=%d M=%d tilesz=%d, %d steps" % (cores, cores, pr.N, pr.M, pr.tilesz, steps))
    return units / sec, sec, desc


def cpu_stage_timings(seed):
    """SURVEY.md 8d: the reference's own CPU stages timed beside the GPU ones, at the largest shape
    its dense Jacobian allows (62 stations, 8 clusters, 10 timeslots): P1 full predict
    (minimize_viz_full_pth), one cost + one gradient (the LBFGS callbacks), one LM iteration of one
    cluster (clevmar_der_single_nocuda, itmax=1: dense J + dgemm, that IS the reference's cost).
    OpenBLAS pinned to 1 thread as the reference driver does (fullbatch_mode.cpp:85) and with all
    threads; Nt = cores pthreads in both."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import refdirac
    from sagecal_b200 import synth
    from sagecal_b200.dirac_api import SkyModel, make_barr
    if not refdirac.available():
        return None
    ref = refdirac.load()
    cores = min(os.cpu_count() or 1, 32)
    pr = synth.make_problem(N=62, M=8, tilesz=10, radius=40e3, seed=seed, kmean=2.0)
    barr = make_barr(pr.sta1, pr.sta2, pr.flag)
    sky = SkyModel(pr.clusters, pr.N)
    n = 8 * pr.Nbase1
    rows = pr.Nbase1
    out = {"shape": "N=62, M=8, tilesz=10 (%d rows)" % rows, "Nt": cores, "unit": UNIT}
    rng = np.random.default_rng(1)
    pp = pr.pp0 + 0.05 * rng.normal(0, 1, pr.pp0.shape)

    def timed(f, reps=1):
        t0 = time.perf_counter()
        for _ in range(reps):
            f()
        return (time.perf_counter() - t0) / reps

    for label, nth in (("openblas_1_thread", 1), ("openblas_all_threads", cores)):
        try:
            ref.lib.openblas_set_num_threads(nth)
        except AttributeError:
            pass
        md = ref.me_data(pr.N, pr.Nbase, pr.tilesz, barr, sky, pr.coh, Nt=cores)
        md0 = ref.me_data(pr.N, pr.Nbase, pr.tilesz, barr, sky, pr.coh, clus=0, Nt=cores)
        t_p1 = timed(lambda: ref.predict_full(pp, md, n), 5)
        t_cost = timed(lambda: ref.cost(pp, pr.x, md), 3)
        t_grad = timed(lambda: ref.grad(pp, pr.x, md), 1)
        t_lm = timed(lambda: ref.clevmar(pp[:8 * pr.N], pr.x, md0, 1), 1)
        if nth == cores:
            # SURVEY.md 8d: C4 on the CPU is feasible for P1 only, at tilesz = 2 (512 stations, 8 clusters)
            try:
                p4 = synth.make_problem(N=512, M=8, tilesz=2, radius=75e3, seed=seed + 1, kmean=1.0)
                b4 = make_barr(p4.sta1, p4.sta2, p4.flag)
                s4 = SkyModel(p4.clusters, p4.N)
                md4 = ref.me_data(p4.N, p4.Nbase, p4.tilesz, b4, s4, p4.coh, Nt=cores)
                t4 = timed(lambda: ref.predict_full(p4.jones_true, md4, 8 * p4.Nbase1), 3)
                out["C4_P1_full_predict_tilesz2"] = {"shape": "N=512, M=8, tilesz=2 (%d rows)" % p4.Nbase1,
                                                     "seconds": t4, "value": p4.Nbase1 * p4.M / t4}
            except Exception as e:
                out["C4_P1_full_predict_tilesz2"] = {"error": repr(e)}
        out[label] = {
            "P1_full_predict": {"seconds": t_p1, "value": rows * pr.M / t_p1},
            "cost_plus_grad": {"seconds": t_cost + t_grad, "value": rows * pr.M / (t_cost + t_grad)},
            "one_LM_iteration_one_cluster": {"seconds": t_lm, "value": rows / t_lm},
        }
    return out


def cpu_baseline_object(seed):
    v, sec, desc = cpu_reference_run(1, 0, seed)
    cores = min(os.cpu_count() or 1, 32)
    cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "sample": desc}
    if v is not None:
        cpu["seconds_per_step"] = sec
        try:
            cpu["stages"] = cpu_stage_timings(seed)
        except Exception as e:  # the stage timings are a report, never a reason to lose the line
            cpu["stages"] = {"error": repr(e)}
    return cpu


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    shape = workload_shape(args.workload)
    steps, warm = args.steps, args.warmup
    outputs = {}
    v, sec, desc = cpu_reference_run(steps, warm, shape["seed"], outputs)
    cores = min(os.cpu_count() or 1, 32)
    if v is None:
        emit({"impl": "reference", "unavailable": desc})
        return
    dump_outputs(args, "reference_" + args.workload, outputs)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s (N=%d, M=%d, tilesz=%d) sampled as N=%d M=%d tilesz=%d"
                   % (args.workload, shape["N"], shape["M"], shape["tilesz"], CPU_SAMPLE["N"],
                      CPU_SAMPLE["M"], CPU_SAMPLE["tilesz"]), "solve": SOLVE},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
                         "sample": desc, "stages": cpu_stage_timings(shape["seed"])},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# own arm
# ---------------------------------------------------------------------------------------------
def n512_parity(api, variant="lm"):
    """reduced-interval problem at the station count of C4 (512 stations, 2 timeslots, 2 clusters)
    against the committed golden of the CPU restatement (tests/golden/n512): the parity evidence for
    the 8N = 4096 code paths next to a C4 bench line (no CPU code can produce a full-shape C4 golden)"""
    path = os.path.join(ROOT, "tests", "golden", "n512", variant + ".npz")
    if not os.path.exists(path):
        return {"checked": False, "why": "tests/golden/n512/%s.npz missing" % variant}
    import ast
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden_n512 as gen
    from sagecal_b200.dirac_api import SkyModel, make_barr
    g = np.load(path)
    pr = gen.build()
    same_inputs = bool(np.allclose(gen.fingerprint(pr), g["fingerprint"], rtol=1e-10, atol=0))
    kw = ast.literal_eval(str(g["args"]))
    x, pp = pr.x.copy(), pr.pp0.copy()
    out = api.sagefit_visibilities(pr.u, pr.v, pr.w, x, pr.N, pr.Nbase, pr.tilesz,
                                   make_barr(pr.sta1, pr.sta2, pr.flag), SkyModel(pr.clusters, pr.N),
                                   pr.coh, pp, **kw)
    want = g["out_scalars"]
    err = float(np.max(np.abs(pp - g["out_pp"])) / np.max(np.abs(g["out_pp"])))
    return {"checked": True, "against": "oracle/liboracle.so golden tests/golden/n512/%s.npz "
                                        "(N=512, 2 clusters, 2 timeslots)" % variant,
            "same_inputs": same_inputs, "jones_max_relerr": err, "tolerance": 1e-5,
            "ok": bool(same_inputs and err < 1e-5), "res_1": [out[3], float(want[3])]}


def run_workload(name, args, ctx, with_cpu=True):
    """one workload through the own arm; returns the JSON line (dict) on rank 0, None elsewhere"""
    import torch
    import torch.distributed as dist
    from sagecal_b200 import lib as blib
    from sagecal_b200 import dist as sdist
    from sagecal_b200 import synth
    from sagecal_b200.dirac_api import SkyModel, make_barr
    api, stream, rank, world, local = ctx["api"], ctx["stream"], ctx["rank"], ctx["world"], ctx["local"]
    shape = dict(workload_shape(name))
    SOLVE_W = solve_args(name)

    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()

    # C4 (512 stations): the coherencies of one GPU's 32 clusters are 32 GB (257 GB for all 256
    # clusters) and never exist on the host: they are generated on the device from the sky model
    # (dirac_b200_precalculate, the device-side precalculate_coherencies), as SURVEY.md 8e prescribes
    is_c4 = name in ("C4", "C4rtr")
    devgen = is_c4 or args.devgen
    if is_c4:
        shape["M"] = args.c4_clusters_per_gpu
    coh_h = None
    if world == 1 and not devgen:
        pr = synth.make_problem(**shape)
        barr = make_barr(pr.sta1, pr.sta2, pr.flag)
        sky = SkyModel(pr.clusters, pr.N)
        coh_t, coh_h = pinned(pr.coh.view(np.float64))
        coh_h = coh_h.view(np.complex128)
    else:
        # weak scaling over directions: every GPU owns shape["M"] clusters of a sky with
        # M*world clusters; data, residual and Jones are replicated (DESIGN.md §9).  Each rank
        # generates only its own coherencies; the data is the all-reduced model + seeded noise.
        shape["M"] = shape["M"] * world
        pr = synth.make_problem(with_data=False, **shape)
        barr = make_barr(pr.sta1, pr.sta2, pr.flag)
        sky = SkyModel(pr.clusters, pr.N) if world == 1 else None
        k0, k1 = sdist.partition_clusters(pr.M, world)[rank]
        if not devgen:
            coh_local = synth.coherencies(pr.u, pr.v, pr.w, pr.clusters[k0:k1], pr.freq0, pr.fdelta)
            coh_t, coh_h = pinned(coh_local.view(np.float64))
            coh_h = coh_h.view(np.complex128)
        pr.x = np.zeros(8 * pr.Nbase1)

    def make_resident():
        if world == 1:
            dpx = blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, barr, sky, coh_h, pr.x)
            if devgen:
                dpx.precalculate(pr.u, pr.v, pr.w, pr.freq0, pr.fdelta)
            return dpx
        spx = sdist.ShardedProblem(api, pr, barr, rank, world, coh_local=coh_h)
        if devgen:
            spx.precalculate(pr.u, pr.v, pr.w, pr.freq0, pr.fdelta)
        return spx

    if world > 1 or devgen:
        with torch.cuda.stream(stream):
            sp0 = make_resident()
            model = np.zeros(8 * pr.Nbase1)
            api.lib.dirac_b200_predict(sp0.h, blib.dptr(pr.jones_true), blib.dptr(model), 2, 0, 0.0)
            sp0.close()
        rng = np.random.default_rng(shape["seed"] + 17)
        sigma = 1e-2 * np.median(np.abs(model[:: max(1, len(model) // 4000000)]))
        pr.x = model + rng.normal(0, sigma, model.shape)
        del model
        pr.x.reshape(pr.Nbase1, 8)[pr.flag == 1] = 0.0
    R, M = pr.Nbase1, pr.M
    x_t, x_h = pinned(pr.x)
    pr.x = x_h
    pp_t, pp_h = pinned(pr.pp0)
    coh_bytes = coh_h.nbytes if coh_h is not None else 64 * R * (M // world)

    K, W = args.steps, max(args.warmup, 3)
    if args.profile_run:
        K, W = 1, 1
    clocks = ClockSampler(local)

    # ---------------- resident-data throughput (`value`) ----------------
    with torch.cuda.stream(stream):
        dp = make_resident()
        res = None
        parity = None
        for it in range(W):
            pp = pr.pp0.copy()
            res = dp.sagefit(pp, None, **SOLVE_W)
            if it == 0 and world == 1 and rank == 0 and not is_c4:
                parity = golden_parity(name, pr, pp, res)
                if name == "C2" and parity.get("checked") and os.path.exists(
                        os.path.join(ROOT, "tests", "golden", "full", "C2lm.npz")):
                    # the Gaussian LBFGS stage differentiates the cost numerically with a step of
                    # 1e-9..1e-6 (lbfgs.c:546): its iterates carry the rounding of a 1.8-million-term
                    # sum (the restatement moves its OWN answer by 5e-5 when compiled with another
                    # summation order, DESIGN.md 6.1).  What is reproducible is pinned separately: the
                    # Jones after the SAGE stage (golden C2lm, untimed extra solve) and the final cost.
                    pp2 = pr.pp0.copy()
                    kw2 = dict(SOLVE_W)
                    kw2["max_lbfgs"] = 0
                    res2 = dp.sagefit(pp2, None, **kw2)
                    lm = golden_parity("C2lm", pr, pp2, res2)
                    parity["sage_stage"] = {k: lm[k] for k in ("against", "jones_max_relerr", "ok")}
                    r1 = parity["res_1"]
                    parity["res_1_relerr"] = abs(r1[0] - r1[1]) / r1[1]
                    parity["ok_criterion"] = ("SAGE-stage Jones < 1e-5 AND final residual within 1e-6 "
                                              "(LBFGS-stage Jones reported, not gated: numerical "
                                              "differentiation in the reference's line search)")
                    parity["ok"] = bool(parity["same_inputs"] and lm["ok"]
                                        and parity["res_1_relerr"] < 1e-6)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        g0 = api.kernel_count(1)
        l0 = api.launch_count()
        api.host_stats(reset=True)
        clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(K):
            pp = pr.pp0.copy()
            res = dp.sagefit(pp, None, **SOLVE_W)
        e1.record(stream)
        torch.cuda.synchronize()
        if rank == 0:
            dump_outputs(args, name, {"jones": pp, "result": res})
        if world > 1:
            dist.barrier()
        clk = clocks.stop()
        hstat = api.host_stats()
        ms_total = e0.elapsed_time(e1)
        launches = api.launch_count() - l0
        ngrad = (api.kernel_count(1) - g0) / K
        # the same K steps once more with a CUDA-event pair around every kernel of the path: the
        # per-kernel durations behind `roofline` (the ~4000 extra event records per step cost a few
        # per cent, so they stay out of the region `value` is taken from)
        api.profile_enable(True)
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(stream)
        for _ in range(0 if args.profile_run else K):
            pp = pr.pp0.copy()
            res = dp.sagefit(pp, None, **SOLVE_W)
        p1.record(stream)
        torch.cuda.synchronize()
        ms_profiled = p0.elapsed_time(p1) / K
        prof = {k: api.profile_read(k) for k in range(11)}
        api.profile_enable(False)
    sweeps = SOLVE_W["max_emiter"] + ngrad
    units_step = R * M * sweeps
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / K
    value = units_step / (ms_step * 1e-3)  # M already counts the clusters of all ranks

    # ---------------- end to end through the drop-in C entry point (`e2e`) ----------------
    e2e = None
    dp.close()
    if not args.no_e2e and not args.profile_run:
        if devgen:
            # u, v, w, data, Jones, flags up; the coherencies are generated on the device
            h2d = 3 * 8 * R + x_h.nbytes + pp_h.nbytes + R
        else:
            h2d = coh_h.nbytes + x_h.nbytes + pp_h.nbytes + R  # coherencies, data, Jones, flags
        d2h = x_h.nbytes + pp_h.nbytes
        with torch.cuda.stream(stream):
            dropin = world == 1 and not devgen
            # the drop-in entry point overwrites x with the residual (lmfit.c:1039-1040): its input
            # is restored before every step; the device layer leaves x alone and writes the residual
            # to a second pinned buffer
            x_keep = np.array(x_h) if dropin else None
            xo_t, xo = (None, None) if dropin else pinned(np.zeros_like(x_h))

            def one():
                pp_h[:] = pr.pp0
                if dropin:
                    x_h[:] = x_keep
                    return api.sagefit_visibilities(pr.u, pr.v, pr.w, x_h, pr.N, pr.Nbase,
                                                    pr.tilesz, barr, sky, coh_h, pp_h, **SOLVE_W)
                # sharded / device-generated public path: upload (or generate) this rank's shard,
                # solve, download, free
                sp = make_resident()
                rr = sp.sagefit(pp_h, xo, **SOLVE_W)
                sp.close()
                return rr
            one()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for _ in range(K):
                one()
            f1.record(stream)
            torch.cuda.synchronize()
            if dropin:
                x_h[:] = x_keep
        te = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        ms_e2e = float(te.item()) / K
        e2e = {"value": units_step / (ms_e2e * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": ms_e2e,
               "path": ("dirac_b200_create + dirac_b200_precalculate (device) + dirac_b200_sagefit + "
                        "destroy, host buffers" if (devgen or world > 1) else
                        "sagefit_visibilities (drop-in entry point), host buffers")}

    if rank != 0:
        return None

    # ---------------- roofline of the dominant own kernel ----------------
    peak, peak_src = measured_peaks()
    names = ["k_predict_full", "k_grad_full", "k_cluster_pass", "k_coh_gram", "assemble",
             "damped_solve", "k_weighted_jtj", "k_line_setup", "k_cluster_pass_addsub",
             "k_rtr_stats", "k_rtr_eval"]
    shares = {}
    for k in range(11):
        n, ms, by = prof[k]
        shares[names[k]] = {"launches_per_step": n / K, "ms_per_step": ms / K,
                            "share_of_step": (ms / K) / ms_profiled if ms_profiled else None,
                            "GBps": (by / (ms * 1e-3)) / 1e9 if ms > 0 and by > 0 else None}
    # `roofline` is quoted for the dominant HBM-streaming kernel.  The damped solves take a large
    # share of the step, are latency (N=62: a chain of 496 pivots on a 16-CTA cluster) or FP64 bound
    # (N=512: 23 GFLOP per factorisation), not HBM or tensor bound: reported next to it.
    # (k_rtr_eval, the O(Nbase) evaluation of the RTR family, is latency bound like the solves: it
    # works on 512 bytes per BASELINE, not on the rows)
    own = {k: v for k, v in shares.items() if not k.startswith("damped") and k != "k_rtr_eval"}
    dom = max(own, key=lambda k: own[k]["ms_per_step"])
    n8 = 8 * pr.N
    sv = shares["damped_solve"]
    flop = n8 ** 3 / 3.0 + 2.0 * n8 * n8
    solver = {"kernels": ("k_chol_solve (factor+solve), k_tri_solve (solve on batch-prefactored "
                          "systems), cusolverDnDpotrfBatched (one batch per sweep)") if n8 <= 512 else
                         "cusolverDnDpotrf + Dpotrs (8N > 512)",
              "bound": "latency (pivot chain)" if n8 <= 512 else "fp64",
              "launches_per_step": sv["launches_per_step"],
              "ms_per_step": sv["ms_per_step"], "share_of_step": sv["share_of_step"],
              "flop_per_factor_solve": flop,
              "TFLOPs": (flop * sv["launches_per_step"] / (sv["ms_per_step"] * 1e-3) / 1e12)
              if sv["ms_per_step"] else None}
    n, ms, by = prof[names.index(dom)]
    achieved = (by / (ms * 1e-3)) / 1e9 if ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu_traffic(name), "peak_source": peak_src,
                "launches_in_timed_region": n, "avg_launch_us": 1e3 * ms / n if n else None,
                "algorithmic_bytes_per_launch": by / n if n else None,
                "profiled_ms_per_step": ms_profiled,
                "dominant_by_time": max(shares, key=lambda k: shares[k]["ms_per_step"]),
                "solver": solver, "kernels": shares}

    cpu = None
    if with_cpu and not args.no_cpu_baseline and not args.profile_run:
        cpu = cpu_baseline_object(shape["seed"])

    if world > 1:
        par = {"checked": True, "sharded_vs_single_gpu": ctx.get("shard_check"),
               "ok": bool(ctx.get("shard_check") and ctx["shard_check"]["ok"])}
        if is_c4:
            par["n512_reduced"] = ctx.get("n512")
            par["ok"] = bool(par["ok"] and ctx.get("n512", {}).get("ok"))
    elif is_c4:
        par = ctx.get("n512")
    else:
        par = parity
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: N=%d stations, %d baselines, M=%d clusters (%d per GPU), "
                               "tilesz=%d, rows=%d per GPU" % (name, pr.N, pr.Nbase, M, M // world,
                                                              pr.tilesz, R),
                   "solve": SOLVE_W, "sweeps_per_step": sweeps,
                   "units_per_step": "rows*clusters*(em_sweeps+lbfgs_grad_evals)",
                   "l2": "inputs (%.0f MB coherencies per GPU) larger than the 126 MB L2, no flush needed"
                         % (coh_bytes / 1e6),
                   "coherencies": "generated on the device (dirac_b200_precalculate)" if devgen
                                  else "host array uploaded",
                   "parallelism": ("clusters sharded over %d GPUs (%d per GPU), ONE NCCL all-reduce "
                                   "(residual delta | Jones delta | nerr) per SAGE sweep, called from "
                                   "C" % (world, M // world)) if world > 1 else "1 GPU",
                   "final_res": [res[2], res[3]] if res else None},
        "clocks": clk, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "parity": par,
        # where a step goes on rank 0 (timed region, per step): kernels by CUDA events (instrumented
        # repeat), host blocked in stream/event waits, host enqueueing collectives; the remainder is
        # host-side solver logic and launch overhead
        "breakdown": {"ms_per_step": ms_step,
                      "kernels_ms": sum(v["ms_per_step"] for v in shares.values()),
                      "host_syncs_per_step": hstat["host_syncs"] / K,
                      "host_wait_ms": 1e3 * hstat["host_wait_s"] / K,
                      "collectives_per_step": hstat["collectives"] / K,
                      "collective_MB_per_step": hstat["collective_bytes"] / K / 1e6,
                      "collective_enqueue_ms": 1e3 * hstat["collective_enqueue_s"] / K},
    }
    return line


def run_consensus(args, ctx):
    """BASELINE.json config 5: 62 stations x `world` frequency subbands (one per GPU), 128 clusters,
    consensus (ADMM) calibration; one step = `ADMM` iterations, each a SAGE sweep with the consensus
    terms in every cluster's cost followed by ONE all-reduce of Npoly*8*N*Mt doubles"""
    import torch
    import torch.distributed as dist
    from sagecal_b200 import lib as blib
    from sagecal_b200 import synth, consensus as cons
    from sagecal_b200.dirac_api import SkyModel, make_barr
    api, stream, rank, world, local = ctx["api"], ctx["stream"], ctx["rank"], ctx["world"], ctx["local"]
    c = synth.CONFIGS["C5"]
    ADMM, NPOLY, RHO = 5, 3, 5.0
    # SAGE sweeps per J-update.  The reference's robust RTR J-update restarts nu at nulow in the first
    # sweep of every call (admm_solve.c:333-335); its row weights (nu+2)/(nu+e^2) are then ~2 and a
    # visit is only kept if it halves the cost, so a one-sweep J-update stalls near the solution; the
    # driver's default of 3 sweeps (data.cpp:61) lets the later sweeps run with the updated nu.
    EMIT = 3 if args.c5_solver == "rtr" else 1
    freqs = np.linspace(115e6, 185e6, 8)[:max(world, 1)] if world <= 8 else np.linspace(115e6, 185e6, world)
    f = float(freqs[rank])
    pr = synth.make_problem(N=c["N"], M=c["M"], tilesz=c["tilesz"], radius=c["radius"], seed=c["seed"],
                            kmean=c["kmean"], freq0=f, with_data=False)
    barr = make_barr(pr.sta1, pr.sta2, pr.flag)
    sky = SkyModel(pr.clusters, pr.N)
    # Jones smooth in frequency: linear around 150 MHz
    rng = np.random.default_rng(c["seed"] + 99)
    slope = 0.2 * rng.normal(0, 1, pr.jones_true.shape)
    jt = pr.jones_true + slope * (f - 150e6) / 150e6
    pr.x = np.zeros(8 * pr.Nbase1)
    R, M = pr.Nbase1, pr.M

    def make_resident():
        dpx = blib.DeviceProblem(api, pr.N, pr.Nbase, pr.tilesz, barr, sky, None, pr.x)
        dpx.precalculate(pr.u, pr.v, pr.w, f, pr.fdelta)
        return dpx

    with torch.cuda.stream(stream):
        dp = make_resident()
        _, model = dp.predict(jt, out_mode=2)
        sig = 1e-2 * np.median(np.abs(model))
        pr.x = model + np.random.default_rng(c["seed"] + 17 + rank).normal(0, sig, model.shape)
        pr.x.reshape(R, 8)[pr.flag == 1] = 0.0
        dp.set_data(pr.x)
        rho = np.full(M, RHO)

        def solve(dpx):
            sb = cons.ConsensusSubband(api, dpx, rank, freqs, 150e6, min(NPOLY, max(1, world - 1)) if world > 1 else 1,
                                       rho, ptype=1)
            pp = pr.pp0.copy()
            return sb, pp, sb.run(pp, admm_iters=ADMM, max_emiter=EMIT, max_iter=2,
                                  solver=args.c5_solver)

        K, W = args.steps, max(args.warmup, 3)
        hist = None
        for _ in range(W):
            sb, pp, hist = solve(dp)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        l0 = api.launch_count()
        api.host_stats(reset=True)
        clocks = ClockSampler(local)
        clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            sb, pp, hist = solve(dp)
        e1.record(stream)
        torch.cuda.synchronize()
        if rank == 0:
            dump_outputs(args, "C5", {"jones": pp, "history": hist})
        if world > 1:
            dist.barrier()
        clk = clocks.stop()
        hstat = api.host_stats()
        launches = api.launch_count() - l0
        ms_total = e0.elapsed_time(e1)
        dp.close()
        # end to end: upload + device coherencies + solve per step
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(K):
            dpe = make_resident()
            solve(dpe)
            dpe.close()
        f1.record(stream)
        torch.cuda.synchronize()
    t = torch.tensor([ms_total, f0.elapsed_time(f1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, ms_e2e = float(t[0].item()) / K, float(t[1].item()) / K
    units = R * M * ADMM * EMIT * world
    if rank != 0:
        return None
    return {
        "metric": METRIC, "value": units / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "C5: N=%d stations x %d subbands (one per GPU), M=%d clusters, tilesz=%d; "
                               "%d ADMM iterations (%d SAGE sweep(s) each; J-update: %s), Npoly=%d, rho=%g"
                               % (pr.N, world, M, pr.tilesz, ADMM, EMIT,
                                  "robust RTR on the augmented cost as in the reference "
                                  "(rtr_solve_nocuda_robust_admm), max_iter=2" if args.c5_solver == "rtr"
                                  else "LM on the augmented cost, 2 iterations", sb.Npoly, RHO),
                   "units_per_step": "rows*clusters*SAGE sweeps*ADMM iterations*subbands",
                   "parallelism": "one subband per GPU, ONE all-reduce of Npoly*8*N*Mt doubles per ADMM "
                                  "iteration, called from C",
                   "coherencies": "generated on the device (dirac_b200_precalculate)"},
        "clocks": clk, "gpu_launches": int(launches),
        "e2e": {"value": units / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(3 * 8 * R + 64 * R + R + 8 * len(pr.pp0)),
                "d2h_bytes_per_step": int(8 * len(pr.pp0) * 3 * ADMM)},
        "parity": {"checked": True, "what": "primal residual ||J - B Z|| and data residual per ADMM iteration; "
                                            "exchange and J-update are pinned by tests/test_gpu_consensus.py, "
                                            "tests/consensus_check.py, tests/test_cpu_consensus.py",
                   "primal": [h[2] for h in hist], "res_1": [h[1] for h in hist],
                   "ok": bool(world == 1 or hist[-1][2] < hist[0][2])},
        "breakdown": {"ms_per_step": ms_step, "host_syncs_per_step": hstat["host_syncs"] / K,
                      "host_wait_ms": 1e3 * hstat["host_wait_s"] / K,
                      "collectives_per_step": hstat["collectives"] / K,
                      "collective_MB_per_step": hstat["collective_bytes"] / K / 1e6},
    }


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: every other writer to fd 1 (the NCCL version banner, library
    chatter of any rank) is sent to stderr; the JSON line goes out through a private duplicate"""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from sagecal_b200 import lib as blib
    from sagecal_b200 import dist as sdist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        # keep stdout to the ONE JSON line: NCCL prints its version banner there otherwise
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api = blib.load()
    stream = torch.cuda.Stream()
    api.set_stream(stream.cuda_stream)
    ctx = dict(api=api, stream=stream, rank=rank, world=world, local=local)
    # checks that run before anything is timed
    with torch.cuda.stream(stream):
        if world > 1:
            # prove the sharded path right on this very box (small problem, sharded vs single GPU
            # on every rank; sagecal_b200.dist.verify_sharding)
            ctx["shard_check"] = sdist.verify_sharding(api, rank, world)
        if args.workload in ("C4", "C4rtr") and rank == 0:
            ctx["n512"] = n512_parity(api, "rtr" if args.workload == "C4rtr" else "lm")
    if world > 1:
        dist.barrier()

    if args.workload == "C5":
        if world > 1:
            sdist.init_nccl(api, rank, world)
        line = run_consensus(args, ctx)
        if rank == 0:
            emit(line)
        if world > 1:
            api.lib.dirac_b200_nccl_finalize()
            dist.destroy_process_group()
        return
    line = run_workload(args.workload, args, ctx)
    # one GPU: the two 62-station configurations of BASELINE.json ride along, and C3 once more under
    # the reference driver's default solver (solver_mode 5, robust RTR) (their own parity
    # against the full-shape goldens, value, roofline), so that one driver run covers C2, C3 and C4
    if world == 1 and rank == 0 and args.workload == "C4" and not args.only and not args.profile_run:
        others = {}
        for w in ("C2", "C3", "C3rtr"):
            o = run_workload(w, args, ctx, with_cpu=False)
            others[w] = {k: o[k] for k in ("value", "ms_per_step", "config", "e2e", "gpu_launches",
                                           "parity", "breakdown")}
            others[w]["roofline"] = {k: o["roofline"][k] for k in
                                     ("kernel", "achieved", "peak", "frac", "avg_launch_us", "solver")}
            others[w]["kernels"] = o["roofline"]["kernels"]
        line["other_workloads"] = others
    if rank == 0:
        emit(line)
    if world > 1:
        api.lib.dirac_b200_nccl_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

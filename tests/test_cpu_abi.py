"""CPU: the C-ABI library loads and exports every symbol include/dirac_b200.h declares; host-only
helpers (index / flag work) are bit-exact against the reference.  No compute calls."""
import json
import os
import re

import numpy as np
import pytest

from sagecal_b200 import lib as blib
from sagecal_b200.dirac_api import barr_to_numpy
from util import known

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SIGNATURES = os.path.join(ROOT, "tests", "golden", "ref_signatures.json")


@pytest.fixture(scope="module")
def product():
    if not os.path.exists(blib.LIB_PATH):
        pytest.skip("libdirac_b200.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    return blib.load()


def test_header_symbols_exported(product):
    hdr = open(os.path.join(ROOT, "include", "dirac_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    ctypes_ = {"void", "int", "double", "long", "char", "unsigned", "defined", "extern"}
    declared = set(re.findall(r"\b([a-z_0-9]+)\s*\(", hdr)) - ctypes_
    declared = {d for d in declared if not d.startswith("__")}
    assert declared, "no declarations parsed"
    for sym in sorted(declared):
        assert hasattr(product.lib, sym), "include/dirac_b200.h declares %s, not exported" % sym
    assert declared == set(blib.EXPORTED), declared ^ set(blib.EXPORTED)


def test_generate_baselines_bit_exact(product, ref):
    for N, T in ((8, 10), (5, 3), (33, 2), (62, 2)):
        Nbase = N * (N - 1) // 2
        a = barr_to_numpy(ref.generate_baselines(Nbase, T, N), Nbase * T)
        g = barr_to_numpy(product.generate_baselines(Nbase, T, N), Nbase * T)
        assert np.array_equal(a[0], g[0]) and np.array_equal(a[1], g[1])
        from sagecal_b200 import synth
        p, q = synth.baseline_pairs(N)
        assert np.array_equal(np.tile(p, T), g[0]) and np.array_equal(np.tile(q, T), g[1])


def test_preset_flags_bit_exact(product, ref):
    rng = np.random.default_rng(0)
    n = 257
    flag = (rng.uniform(0, 1, n) < 0.3).astype(np.float64) * rng.integers(1, 3, n)
    xs = rng.normal(0, 1, 8 * n)
    res = []
    for lib in (ref, product):
        barr = lib.generate_baselines(n, 1, 24)
        x = xs.copy()
        lib.preset_flags_and_data(flag.copy(), barr, x)
        res.append((barr_to_numpy(barr, n)[2], x))
    k = known(res[0][1])
    assert np.array_equal(res[0][0], res[1][0])
    assert np.array_equal(res[0][1][k], res[1][1][k])


def test_whiten_data_bit_exact(product, ref):
    """uv taper (driver option -W): host arithmetic, same libm -> identical bits; threaded and not"""
    rng = np.random.default_rng(3)
    for n, Nt in ((1001, 3), (70001, 4), (70001, 1)):
        # |(u,v)| f0 spread around the 400-wavelength cut-off, some rows exactly beyond it
        u = rng.normal(0, 1.2e-6, n)
        v = rng.normal(0, 1.2e-6, n)
        xs = rng.normal(0, 1, 8 * n)
        out = []
        for lib in (ref, product):
            x = xs.copy()
            lib.whiten_data(x, u, v, 150e6, Nt)
            out.append(x)
        k = known(out[0])
        assert np.array_equal(out[0][k], out[1][k])
        d = np.hypot(u, v) * 150e6
        assert (d > 400).any() and (d < 400).any()
        untouched = np.repeat(d > 400, 8)
        assert np.array_equal(out[1][untouched], xs[untouched])
        assert (np.abs(out[1][~untouched]) < np.abs(xs[~untouched])).all()


def test_barr_from_hbb_inverts_the_reference_rearrangement(product, ref):
    """the GPU-build argument list of the minibatch drivers: rows come as `short hbb[2]` written by
    the reference's rearrange_baselines (baseline_utils.c:145); the library rebuilds baseline_t rows"""
    import ctypes as C
    from sagecal_b200.dirac_api import baseline_t
    rng = np.random.default_rng(5)
    N, T = 13, 4
    Nbase = N * (N - 1) // 2
    R = Nbase * T
    barr = ref.generate_baselines(Nbase, T, N)
    flags = rng.choice([0, 0, 0, 1, 2], R).astype(np.uint8)
    for r in range(R):
        barr[r].flag = int(flags[r])
    hbb = np.zeros(2 * R, dtype=np.int16)
    sp = C.POINTER(C.c_short)
    ref.lib.rearrange_baselines.argtypes = [C.c_int, C.POINTER(baseline_t), sp, C.c_int]
    ref.lib.rearrange_baselines(R, barr, hbb.ctypes.data_as(sp), 3)
    out = (baseline_t * R)()
    product.lib.dirac_b200_barr_from_hbb.argtypes = [C.c_int, C.c_int, C.c_int, sp, C.POINTER(baseline_t)]
    assert product.lib.dirac_b200_barr_from_hbb(N, Nbase, T, hbb.ctypes.data_as(sp), out) == 0
    a, g = barr_to_numpy(barr, R), barr_to_numpy(out, R)
    assert np.array_equal(a[0], g[0]) and np.array_equal(a[1], g[1])
    assert np.array_equal(g[2], (flags != 0).astype(g[2].dtype))
    # a row out of the canonical order is refused
    k = int(np.flatnonzero(flags == 0)[3])
    hbb[2 * k + 1] += 1
    assert product.lib.dirac_b200_barr_from_hbb(N, Nbase, T, hbb.ctypes.data_as(sp), out) == -1


def _c_declarations(path):
    """{function name: [parameter type lists]} of a C header (comments stripped, names dropped)"""
    t = open(path).read()
    t = re.sub(r"/\*.*?\*/", "", t, flags=re.S)
    t = re.sub(r"//[^\n]*", "", t)
    out = {}
    for m in re.finditer(r"\b([a-z_0-9]+)\s*\(([^()]*)\)\s*;", t):
        types = []
        for a in m.group(2).replace("\n", " ").split(","):
            a = re.sub(r"\s+", " ", a.strip().replace("complex double", "double").replace("const ", ""))
            mm = re.match(r"(.*?)([A-Za-z_0-9]+)$", a)
            types.append((mm.group(1) if mm else a).replace(" ", ""))
        out.setdefault(m.group(1), []).append(types)
    return out


def _reference_declarations(names):
    """{entry point: [parameter type lists]} of the reference's Dirac.h, Dirac_common.h and
    Dirac_radio.h for the given names: parsed where the reference sources are (DIRAC_REFERENCE),
    else read back from tests/golden/ref_signatures.json (stored by a run with
    DIRAC_REF_GOLDEN=record)"""
    if not os.environ.get("DIRAC_REFERENCE"):
        with open(REF_SIGNATURES) as f:
            return json.load(f)
    refroot = os.path.join(os.environ["DIRAC_REFERENCE"], "src", "lib")
    ref = {}
    for h in ("Dirac/Dirac.h", "Dirac/Dirac_common.h", "Radio/Dirac_radio.h"):
        for k, v in _c_declarations(os.path.join(refroot, h)).items():
            ref.setdefault(k, []).extend(v)
    ref = {k: v for k, v in ref.items() if k in names}
    if os.environ.get("DIRAC_REF_GOLDEN") == "record":
        with open(REF_SIGNATURES, "w") as f:
            json.dump(ref, f, indent=1, sort_keys=True)
            f.write("\n")
    return ref


def test_signatures_equal_the_reference_headers():
    """every reference-named entry point is declared with the reference's own parameter type list
    (complex double * spelled double *); the *_hbb pair carries the HAVE_CUDA variant of its name"""
    ours = _c_declarations(os.path.join(ROOT, "include", "dirac_b200.h"))
    bases = {n[:-4] if n.endswith("_hbb") else n for n in ours if not n.startswith("dirac_b200")}
    ref = _reference_declarations(bases)
    checked = 0
    for name, sigs in ours.items():
        if name.startswith("dirac_b200"):
            continue
        base = name[:-4] if name.endswith("_hbb") else name
        assert base in ref, "%s is not a reference entry point" % name
        assert sigs[0] in ref[base], (name, sigs[0], ref[base])
        if name.endswith("_hbb"):  # ... and it is the OTHER variant of the name
            assert sigs[0] != ours[base][0] and len(ref[base]) == 2
        checked += 1
    assert checked >= 30


def test_no_oracle_in_product():
    """the product package must not import, link or execute anything under oracle/"""
    pkg = os.path.join(ROOT, "sagecal_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".c", ".cpp")) or f == "Makefile":
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                for bad in ("import refdirac", "import orcdirac", "liboracle", "libdirac_ref",
                            "dirac_oracle"):
                    assert bad not in src, "%s references %s" % (os.path.join(dirpath, f), bad)


def test_extract_phases_matches_reference(ref):
    """host arithmetic of the phase_only correction (joint diagonalisation by Jacobi rotations,
    manifold_average.c:399-610) against the compiled reference; runs without a GPU"""
    import ctypes as C
    from sagecal_b200 import lib as blib
    from sagecal_b200.dirac_api import dptr
    L = C.CDLL(blib.LIB_PATH)
    rng = np.random.default_rng(5)
    for N in (3, 8, 62):
        # a common unitary ambiguity on top of nearly diagonal Jones
        D = np.zeros((N, 2, 2), dtype=complex)
        D[:, 0, 0] = np.exp(1j * rng.uniform(-3, 3, N)) * rng.uniform(0.5, 1.5, N)
        D[:, 1, 1] = np.exp(1j * rng.uniform(-3, 3, N)) * rng.uniform(0.5, 1.5, N)
        D += 0.05 * (rng.normal(0, 1, D.shape) + 1j * rng.normal(0, 1, D.shape))
        th, ph = 0.7, 0.4
        U = np.array([[np.cos(th), -np.sin(th) * np.exp(1j * ph)],
                      [np.sin(th) * np.exp(-1j * ph), np.cos(th)]])
        J = D @ U
        p = np.zeros(8 * N)
        p[0::8], p[1::8] = J[:, 0, 0].real, J[:, 0, 0].imag
        p[2::8], p[3::8] = J[:, 0, 1].real, J[:, 0, 1].imag
        p[4::8], p[5::8] = J[:, 1, 0].real, J[:, 1, 0].imag
        p[6::8], p[7::8] = J[:, 1, 1].real, J[:, 1, 1].imag
        want, got = np.zeros(8 * N), np.zeros(8 * N)
        ref.lib.extract_phases(dptr(p.copy()), dptr(want), N, 10)
        L.dirac_b200_extract_phases(dptr(p), dptr(got), N, 10)
        k = known(want)
        assert np.max(np.abs(got - want)[k]) < 1e-10, np.max(np.abs(got - want)[k])

"""The compiled reference (oracle/_ref), recorded.

Tests that compare with the reference call it through the `ref` / `refser` fixtures.  Where the
reference library is built those calls run it; with DIRAC_REF_GOLDEN=record they also store, per test
and per call, what the call returned and which of its array arguments it wrote
(tests/golden/ref/<test module>.npz), with a fingerprint of its inputs.  Where the library is not
built (or with DIRAC_REF_GOLDEN=replay) the same calls are answered from that store: the stored
results are written back into the test's arrays, so every comparison a test makes stays as it is.
A call whose inputs no longer match what was recorded fails the test; re-record on a machine
that has the reference sources (make -C oracle, then the tests with DIRAC_REF_GOLDEN=record).

Outputs of more than SAMPLE_ABOVE elements are stored as a fixed, seeded sample of SAMPLE_SIZE of
their entries (the same entries for outputs of one size), plus their last SAMPLE_TAIL entries (the
last rows, where tail handling lives) and the entry of largest magnitude.  The others replay as NaN;
while results are replayed, `util.relerr` compares on the stored entries only."""
import ctypes as C
import json
import os
import zlib

import numpy as np

from sagecal_b200.dirac_api import baseline_t, elementcoeff

GOLDEN_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
SAMPLE_ABOVE = 1024
SAMPLE_SIZE = 512
SAMPLE_TAIL = 64
_CTYPES = {"baseline_t": baseline_t}


_replaying = False


def replaying():
    """True once a test of this process has been handed recorded reference results"""
    return _replaying


def mode(available):
    m = os.environ.get("DIRAC_REF_GOLDEN", "")
    if m in ("record", "replay"):
        return m
    return "live" if available else "replay"


def _test_id():
    """(module file stem, test name with parameters) of the running test"""
    cur = os.environ["PYTEST_CURRENT_TEST"].rsplit(" ", 1)[0]
    path, name = cur.split("::", 1)
    return os.path.splitext(os.path.basename(path))[0], name


def _as_array(v):
    """the numpy array behind an argument, if any (numpy's data_as pointers keep it as _arr)"""
    if isinstance(v, np.ndarray):
        return v
    a = getattr(v, "_arr", None)
    return a if isinstance(a, np.ndarray) else None


def _fingerprint(v):
    a = _as_array(v)
    if a is not None:
        f = np.asarray(a, dtype=np.complex128 if np.iscomplexobj(a) else np.float64).view(np.float64)
        return ["a", int(a.size), float(np.sum(f)), float(np.sum(np.abs(f)))]
    if isinstance(v, (bool, int, float, np.integer, np.floating)):
        return ["s", float(v)]
    if isinstance(v, (C.c_double, C.c_int)):
        return ["s", float(v.value)]
    if isinstance(v, C.Array) and issubclass(v._type_, C.Structure):
        return ["b", zlib.crc32(bytes(v))]
    return None


def _same(fp, want):
    if fp is None or want is None:
        return fp is None and want is None
    if fp[0] != want[0] or len(fp) != len(want):
        return False
    if fp[0] == "b":
        return fp == want
    return np.allclose(fp[1:], want[1:], rtol=1e-9, atol=1e-300)


def _pack(f):
    """{key: array} -> one array per dtype plus a JSON index (few, large members compress well)"""
    index, blobs = {}, {}
    for k in sorted(f):
        a = np.ascontiguousarray(f[k])
        parts = blobs.setdefault(a.dtype.str, [])
        off = sum(p.size for p in parts)
        parts.append(a.reshape(-1))
        index[k] = [a.dtype.str, list(a.shape), off]
    out = {"d" + dt: np.concatenate(parts) for dt, parts in blobs.items()}
    out["index"] = np.frombuffer(json.dumps(index).encode(), dtype=np.uint8)
    return out


def _unpack(z):
    blobs = {k[1:]: z[k] for k in z.files if k != "index"}
    f = {}
    for k, (dt, shape, off) in json.loads(z["index"].tobytes().decode()).items():
        n = int(np.prod(shape))
        f[k] = blobs[dt][off:off + n].reshape(shape)
    return f


class _Handle:
    """stands in for an opaque reference object (a me_data_t) during replay"""

    def __init__(self, k):
        self.k = k


class _Store:
    def __init__(self):
        self.files = {}      # module -> {key: array}
        self.dirty = set()
        self.counter = {}    # (module, test) -> next call index
        self.handles = {}    # id(obj) -> (handle number, obj) while recording
        self.written = {}    # id(array) -> (module, key, contents) of arrays a call wrote

    def _file(self, mod):
        if mod not in self.files:
            p = os.path.join(GOLDEN_REF, mod + ".npz")
            self.files[mod] = _unpack(np.load(p)) if os.path.exists(p) else {}
        return self.files[mod]

    def next_call(self, fresh):
        mod, test = _test_id()
        key = (mod, test)
        if key not in self.counter:
            self.counter[key] = 0
            if fresh:     # recording this test again: drop what was stored for it before
                f = self._file(mod)
                for k in [k for k in f if k.split("|", 1)[0] == test]:
                    del f[k]
        i = self.counter[key]
        self.counter[key] = i + 1
        return mod, "%s|%d" % (test, i)

    def save(self):
        os.makedirs(GOLDEN_REF, exist_ok=True)
        for mod in sorted(self.dirty):
            np.savez_compressed(os.path.join(GOLDEN_REF, mod + ".npz"), **_pack(self.files[mod]))
        self.dirty.clear()

    # ---- values -> stored form --------------------------------------------------------------
    def put_array(self, f, key, a):
        a = np.asarray(a)
        if a.size > SAMPLE_ABOVE and a.dtype.kind in "fc":
            flat = a.reshape(-1)
            rng = np.random.default_rng(flat.size)   # same entries for outputs of one size
            idx = np.union1d(rng.choice(flat.size, SAMPLE_SIZE, replace=False),
                             np.r_[flat.size - SAMPLE_TAIL:flat.size, np.argmax(np.abs(flat))])
            f[key + "|idx"] = idx.astype(np.uint16 if flat.size <= 65536 else np.uint32)
            f[key] = flat[idx]
            f[key + "|shape"] = np.array(a.shape, dtype=np.int64)
        else:
            f[key] = a.copy()

    def get_array(self, f, key):
        if key + "|idx" not in f:
            return f[key].copy()
        v = f[key]
        out = np.full(int(np.prod(f[key + "|shape"])), np.nan, dtype=v.dtype)
        out[f[key + "|idx"]] = v
        return out.reshape(tuple(f[key + "|shape"]))

    def enc(self, f, key, v):
        if v is None or isinstance(v, (bool, int, float, str)):
            return {"v": v}
        if isinstance(v, (np.integer, np.floating)):
            return {"v": v.item()}
        if isinstance(v, np.ndarray):
            self.put_array(f, key, v)
            return {"a": key}
        if isinstance(v, (tuple, list)):
            return {"t": [self.enc(f, "%s.%d" % (key, j), e) for j, e in enumerate(v)]}
        if isinstance(v, C.Array) and issubclass(v._type_, C.Structure):
            f[key] = np.frombuffer(bytes(v), dtype=np.uint8).copy()
            return {"c": key, "type": v._type_.__name__, "n": len(v)}
        if isinstance(v, C.Structure):
            f[key] = np.frombuffer(bytes(v), dtype=np.uint8).copy()
            return {"s": key}
        if isinstance(v, (C.c_double, C.c_int)):
            return {"v": v.value}
        # an opaque object the caller only hands back to the reference (me_data_t)
        k = self.handles.setdefault(id(v), (len(self.handles), v))[0]
        return {"h": k}

    def dec(self, f, d, restype=None):
        if "v" in d:
            return d["v"]
        if "a" in d:
            return self.get_array(f, d["a"])
        if "t" in d:
            return tuple(self.dec(f, e) for e in d["t"])
        if "c" in d:
            return (_CTYPES[d["type"]] * d["n"]).from_buffer_copy(f[d["c"]].tobytes())
        if "s" in d:
            return restype.from_buffer_copy(f[d["s"]].tobytes())
        return _Handle(d["h"])


_store = _Store()


def save():
    _store.save()


def _args(args, kw):
    return list(enumerate(args)) + sorted(kw.items())


def _ecoeff_arrays(ec):
    """the three tables an elementcoeff points to (Dirac_common.h: complex patterns per mode and
    frequency, one preamble per mode)"""
    n = 2 * ec.Nmodes * max(ec.Nf, 1)
    dp = C.POINTER(C.c_double)
    return [np.ctypeslib.as_array(C.cast(getattr(ec, nm), dp), shape=(m,)).copy()
            for nm, m in (("pattern_phi", n), ("pattern_theta", n), ("preamble", ec.Nmodes))]


def _record_call(name, fn, args, kw):
    mod, key = _store.next_call(fresh=True)
    f = _store._file(mod)
    items = _args(args, kw)
    fps = [_fingerprint(v) for _, v in items]
    before = {}
    for pos, v in items:
        a = _as_array(v)
        if a is not None:
            before[pos] = a.copy()
        elif isinstance(v, C.Array) and issubclass(v._type_, C.Structure):
            before[pos] = bytes(v)
    # handles passed in are identified by number
    for j, (_, v) in enumerate(items):
        if id(v) in _store.handles:
            fps[j] = ["h", _store.handles[id(v)][0]]
    for _, v in items:
        # an array a reference call wrote, handed back unchanged to a later one (an iterate): its
        # replayed value feeds the product's side of the comparison too, so it is stored in full
        a = _as_array(v)
        w = _store.written.get(id(a)) if a is not None else None
        if w is not None and w[0] == mod and np.array_equal(a, w[2]):
            g = _store._file(w[0])
            g.pop(w[1] + "|idx", None)
            g.pop(w[1] + "|shape", None)
            g[w[1]] = w[2]
    ret = fn(*args, **kw)
    muts = []
    for j, (pos, v) in enumerate(items):
        a = _as_array(v)
        mk = "%s|m%d" % (key, j)
        if a is not None:
            if not np.array_equal(a, before[pos], equal_nan=True):
                _store.put_array(f, mk, a)
                _store.written[id(a)] = (mod, mk, a.copy())
                muts.append([j, "a"])
        elif isinstance(v, C.Array) and issubclass(v._type_, C.Structure):
            if bytes(v) != before[pos]:
                f[mk] = np.frombuffer(bytes(v), dtype=np.uint8).copy()
                muts.append([j, "c"])
        elif type(v).__name__ == "CArgObject" and isinstance(v._obj, elementcoeff):
            ec = v._obj
            f[mk + "|hdr"] = np.array([ec.M, ec.Nmodes, ec.Nf, ec.beta])
            for t, arr in enumerate(_ecoeff_arrays(ec)):
                f["%s|%d" % (mk, t)] = arr
            muts.append([j, "ec"])
    meta = {"name": name, "fp": fps, "mut": muts, "ret": _store.enc(f, key + "|r", ret)}
    f[key] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    _store.dirty.add(mod)
    return ret


def _replay_call(name, args, kw, restype=None):
    mod, key = _store.next_call(fresh=False)
    f = _store._file(mod)
    if key not in f:
        raise AssertionError("no recorded reference call %s (%s) in tests/golden/ref/%s.npz"
                             % (key, name, mod))
    meta = json.loads(f[key].tobytes().decode())
    assert meta["name"] == name, ("reference calls out of the recorded order", key, name,
                                  meta["name"])
    items = _args(args, kw)
    assert len(items) == len(meta["fp"]), (key, name, "argument count")
    for j, (_, v) in enumerate(items):
        fp = ["h", v.k] if isinstance(v, _Handle) else _fingerprint(v)
        assert _same(fp, meta["fp"][j]), ("input differs from the recorded reference call", key,
                                          name, j, fp, meta["fp"][j])
    for j, kind in meta["mut"]:
        v = items[j][1]
        mk = "%s|m%d" % (key, j)
        if kind == "a":
            np.copyto(_as_array(v), _store.get_array(f, mk))
        elif kind == "c":
            C.memmove(v, f[mk].tobytes(), len(f[mk]))
        else:
            ec = v._obj
            M, Nmodes, Nf, beta = f[mk + "|hdr"]
            ec.M, ec.Nmodes, ec.Nf, ec.beta = int(M), int(Nmodes), int(Nf), float(beta)
            keep = [np.ascontiguousarray(f["%s|%d" % (mk, t)]) for t in range(3)]
            ec.pattern_phi, ec.pattern_theta, ec.preamble = [a.ctypes.data for a in keep]
            ec._keep = keep
    return _store.dec(f, meta["ret"], restype)


class _Fn:
    """one entry point of the reference library (ref.lib.<name>)"""

    def __init__(self, name, real, record):
        self.__dict__.update(_name=name, _real=real, _record=record, _attrs={})

    def __setattr__(self, k, v):      # argtypes / restype
        self._attrs[k] = v
        if self._real is not None:
            setattr(self._real, k, v)

    def __getattr__(self, k):
        if k in self._attrs:
            return self._attrs[k]
        if self._real is not None:
            return getattr(self._real, k)
        raise AttributeError(k)

    def __call__(self, *args, **kw):
        if self._record:
            return _record_call(self._name, self._real, args, kw)
        return _replay_call(self._name, args, kw, self._attrs.get("restype"))


class _Lib:
    def __init__(self, real, record):
        self._real, self._record, self._fns = real, record, {}

    def __getattr__(self, name):
        if name not in self._fns:
            self._fns[name] = _Fn("lib." + name, getattr(self._real, name) if self._real else None,
                                  self._record)
        return self._fns[name]


class GoldenRef:
    """the reference's Python interface (refdirac.RefDirac), recording or replaying"""

    def __init__(self, tag, real=None):
        global _replaying
        self._tag, self._real = tag, real
        self.lib = _Lib(real.lib if real is not None else None, real is not None)
        _replaying = _replaying or real is None

    def __getattr__(self, name):
        if self._real is not None:
            fn = getattr(self._real, name)
            return lambda *a, **k: _record_call("%s.%s" % (self._tag, name), fn, a, k)
        return lambda *a, **k: _replay_call("%s.%s" % (self._tag, name), a, k)

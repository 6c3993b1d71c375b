"""ctypes binding of the CPU oracle (oracle/dbl_oracle.c).  TEST INFRASTRUCTURE ONLY.

Imported only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
The product package (dblink_b200/) never imports this module.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

PCG_I, PCG_II, GIBBS, GIBBS_SEQ = 0, 1, 2, 3
SAMPLERS = {"PCG-I": PCG_I, "PCG-II": PCG_II, "Gibbs": GIBBS, "Gibbs-Sequential": GIBBS_SEQ}

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
c_dp = C.POINTER(C.c_double)


def build(force=False, native=False):
    """liboracle.so (portable flags).  native=True: the -march=native build of the same sources, made on the machine
    that runs it (bench.py's CPU legs) in a temporary directory removed at exit, so that nothing is written into a
    tree that may be read-only; returns the portable library when that build is not possible."""
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("dbl_oracle.c", "dbl_oracle.h", "dbl_oracle_priv.h", "dbl_refsweep.c", "Makefile")]
    srcs = [s for s in srcs if os.path.exists(s)]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    if native:
        try:
            tmp = tempfile.mkdtemp(prefix="dbl_oracle_")
            atexit.register(shutil.rmtree, tmp, True)  # a loaded library stays mapped after its file is removed
            subprocess.run(["make", "-C", _HERE, "-s", "native", "NATIVE_DIR=" + tmp], check=True, capture_output=True)
            nso = os.path.join(tmp, "liboracle.so")
            if os.path.exists(nso):
                return nso
        except Exception:
            pass
    return so


BUILD_FLAGS = {"portable": "-O3 -march=x86-64-v3 -ffp-contract=off", "native": "-O3 -march=native -ffp-contract=off"}
_NATIVE = False


def use_native():
    """bench.py only: load the -march=native build (must be called before the first lib())."""
    global _NATIVE
    _NATIVE = True


def flags():
    native = _LIB is not None and _LIB._name != os.path.join(_HERE, "liboracle.so")
    return BUILD_FLAGS["native" if native else "portable"]


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    L = C.CDLL(build(native=_NATIVE))
    vp = C.c_void_p

    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    sig("orc_philox4x32_10", None, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32))
    sig("orc_uniform2", None, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, c_dp)
    sig("orc_levenshtein", C.c_int, C.c_char_p, C.c_char_p)
    sig("orc_lev_similarity", C.c_double, C.c_char_p, C.c_char_p, C.c_double, C.c_double)
    sig("orc_index_build", vp, C.POINTER(C.c_char_p), c_dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int)
    sig("orc_index_from_tables", vp, C.c_int, C.c_int, c_dp, c_i32p, c_i32p, c_dp, C.c_int)
    sig("orc_index_free", None, vp)
    for n in ("num_values", "is_const", "nnz", "kmax"):
        sig("orc_index_" + n, C.c_int, vp)
    sig("orc_index_value_id", C.c_int, vp, C.c_char_p)
    sig("orc_index_value", C.c_char_p, vp, C.c_int)
    for n in ("phi", "norm", "invnorm", "expsim", "pk", "cdf"):
        sig("orc_index_" + n, c_dp, vp)
    for n in ("rowptr", "col"):
        sig("orc_index_" + n, c_i32p, vp)
    sig("orc_index_exp_sim_of", C.c_double, vp, C.c_int, C.c_int)
    sig("orc_kdtree_fit", vp, c_i32p, C.c_int64, C.c_int, C.c_int, c_i32p, C.c_int)
    sig("orc_kdtree_from_arrays", vp, C.c_int, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p)
    sig("orc_kdtree_free", None, vp)
    for n in ("num_nodes", "num_leaves", "set_len"):
        sig("orc_kdtree_" + n, C.c_int, vp)
    sig("orc_kdtree_export", None, vp, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p)
    sig("orc_kdtree_leaf", C.c_int, vp, c_i32p)
    sig("orc_model_create", vp, C.c_int, C.c_int, C.POINTER(vp), c_dp, c_dp, vp, C.c_uint64)
    sig("orc_model_free", None, vp)
    sig("orc_state_init", vp, vp, C.c_int64, c_i32p, c_i32p, C.c_int64)
    sig("orc_state_from_arrays", vp, vp, C.c_int64, C.c_int64, c_i32p, c_i32p, c_u8p, c_i32p, c_i32p, c_dp, C.c_int64)
    sig("orc_state_free", None, vp)
    for n in ("R", "E", "iteration"):
        sig("orc_state_" + n, C.c_int64, vp)
    for n in ("y", "link", "block"):
        sig("orc_state_" + n, c_i32p, vp)
    sig("orc_state_z", c_u8p, vp)
    sig("orc_state_theta", c_dp, vp)
    sig("orc_state_summary", None, vp, C.c_void_p, c_i64p, c_i64p)
    sig("orc_state_sweep", C.c_int, vp, C.c_int)
    sig("orc_draw_theta", None, vp, c_i64p, c_i64p, C.c_uint32, c_dp)
    sig("orc_det_log", C.c_double, C.c_double)
    sig("orc_det_exp", C.c_double, C.c_double)
    sig("orc_rest_of_sweep_timed", None, vp, C.c_int, C.c_int, c_dp)
    sig("orc_draw_index", C.c_int, c_dp, C.c_int64, C.c_double, C.POINTER(C.c_int))
    sig("orc_invcdf", C.c_int, c_dp, C.c_int, C.c_double)
    sig("orc_ref_link_weights", None, vp, C.c_int64, C.c_int, c_i32p, C.c_int64, c_dp)
    sig("orc_link_weights", None, vp, C.c_int64, C.c_int, c_i32p, C.c_int64, c_dp)
    sig("orc_ref_value_pmf", None, vp, C.c_int64, C.c_int, C.c_int, c_dp)
    sig("orc_value_draw", C.c_int, vp, C.c_int64, C.c_int, C.c_int, C.c_double, C.c_double)
    sig("orc_ref_dist_prob", C.c_double, vp, C.c_int64, C.c_int)
    sig("orc_alias_build", C.c_int, c_dp, C.c_int, c_dp, c_i32p)
    sig("orc_alias_sample", C.c_int, c_dp, c_i32p, C.c_int, C.c_double)
    if hasattr(L, "orc_refsweep_run"):
        sig("orc_refsweep_run", C.c_double, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, c_i64p)
    _LIB = L
    return L


def _p(a, t):
    return a.ctypes.data_as(t)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32_10(c, k, o)
    return list(o)


def uniform2(seed, phase, it, idx, sub):
    u = (C.c_double * 2)()
    lib().orc_uniform2(seed, phase, it, idx, sub, u)
    return u[0], u[1]


def levenshtein(a, b):
    return lib().orc_levenshtein(a.encode(), b.encode())


def lev_similarity(a, b, threshold=7.0, max_sim=10.0):
    return lib().orc_lev_similarity(a.encode(), b.encode(), threshold, max_sim)


class Index:
    """AttributeIndex restatement (AttributeIndex.scala:107-245)."""

    def __init__(self, handle):
        self.h = handle
        L = lib()
        self.V = L.orc_index_num_values(handle)
        self.is_const = bool(L.orc_index_is_const(handle))
        self.kmax = L.orc_index_kmax(handle)
        self.nnz = L.orc_index_nnz(handle)
        V, K = self.V, self.kmax
        self.phi = np.ctypeslib.as_array(L.orc_index_phi(handle), (V,)).copy()
        self.norm = np.ctypeslib.as_array(L.orc_index_norm(handle), (V,)).copy()
        self.invnorm = np.ctypeslib.as_array(L.orc_index_invnorm(handle), (V,)).copy()
        self.rowptr = np.ctypeslib.as_array(L.orc_index_rowptr(handle), (V + 1,)).copy()
        n = max(self.nnz, 1)
        self.col = np.ctypeslib.as_array(L.orc_index_col(handle), (n,)).copy()[: self.nnz]
        self.expsim = np.ctypeslib.as_array(L.orc_index_expsim(handle), (n,)).copy()[: self.nnz]
        self.pk = np.ctypeslib.as_array(L.orc_index_pk(handle), (K + 1, V)).copy()
        self.cdf = np.ctypeslib.as_array(L.orc_index_cdf(handle), (K + 1, V)).copy()

    @classmethod
    def build(cls, values_weights, is_const, threshold=7.0, max_sim=10.0, kmax=10):
        vals = list(values_weights.keys())
        arr = (C.c_char_p * len(vals))(*[v.encode() for v in vals])
        w = _f64([values_weights[v] for v in vals])
        h = lib().orc_index_build(arr, _p(w, c_dp), len(vals), int(is_const), threshold, max_sim, kmax)
        return cls(h)

    @classmethod
    def from_tables(cls, phi, rowptr, col, expsim, is_const, kmax=10):
        phi = _f64(phi)
        rowptr, col, expsim = _i32(rowptr), _i32(col if len(col) else [0]), _f64(expsim if len(expsim) else [0.0])
        h = lib().orc_index_from_tables(len(phi), int(is_const), _p(phi, c_dp), _p(rowptr, c_i32p), _p(col, c_i32p),
                                        _p(expsim, c_dp), kmax)
        return cls(h)

    def value_id(self, s):
        return lib().orc_index_value_id(self.h, s.encode())

    def value(self, v):
        r = lib().orc_index_value(self.h, v)
        return r.decode() if r is not None else None

    def exp_sim_of(self, v1, v2):
        if not (0 <= v1 < self.V and 0 <= v2 < self.V):
            raise IndexError("valueId is not in the index")  # AttributeIndex.scala:137,184
        return lib().orc_index_exp_sim_of(self.h, v1, v2)

    def sim_values_of(self, v):
        if not 0 <= v < self.V:
            raise IndexError("valueId is not in the index")
        lo, hi = self.rowptr[v], self.rowptr[v + 1]
        return {int(c): float(e) for c, e in zip(self.col[lo:hi], self.expsim[lo:hi])}


class KDTree:
    def __init__(self, handle):
        self.h = handle
        L = lib()
        self.n_nodes = L.orc_kdtree_num_nodes(handle)
        self.n_leaves = L.orc_kdtree_num_leaves(handle)
        n, sl = self.n_nodes, L.orc_kdtree_set_len(handle)
        self.attr = np.zeros(n, np.int32)
        self.kind = np.zeros(n, np.int32)
        self.split = np.zeros(n, np.int32)
        self.set_ptr = np.zeros(n + 1, np.int32)
        self.set_val = np.zeros(max(sl, 1), np.int32)
        self.leaf_no = np.zeros(n, np.int32)
        L.orc_kdtree_export(handle, _p(self.attr, c_i32p), _p(self.kind, c_i32p), _p(self.split, c_i32p),
                            _p(self.set_ptr, c_i32p), _p(self.set_val, c_i32p), _p(self.leaf_no, c_i32p))
        self.set_val = self.set_val[:sl]

    @classmethod
    def fit(cls, y, num_levels, attr_ids):
        y = _i32(y)
        attr_ids = _i32(attr_ids if len(attr_ids) else [0])
        return cls(lib().orc_kdtree_fit(_p(y, c_i32p), y.shape[0], y.shape[1], num_levels, _p(attr_ids, c_i32p),
                                        len(attr_ids)))

    @classmethod
    def from_arrays(cls, attr, kind, split, set_ptr, set_val, leaf_no):
        a, k, s, sp, lv = _i32(attr), _i32(kind), _i32(split), _i32(set_ptr), _i32(leaf_no)
        sv = _i32(set_val if len(set_val) else [0])
        return cls(lib().orc_kdtree_from_arrays(len(a), _p(a, c_i32p), _p(k, c_i32p), _p(s, c_i32p), _p(sp, c_i32p),
                                                _p(sv, c_i32p), _p(lv, c_i32p)))

    def leaf(self, yrow):
        yrow = _i32(yrow)
        return lib().orc_kdtree_leaf(self.h, _p(yrow, c_i32p))


class Model:
    def __init__(self, indexes, alpha, beta, tree, seed, F=1):
        self.indexes = list(indexes)
        self.A = len(self.indexes)
        self.F = F
        self.alpha = _f64(alpha)
        self.beta = _f64(beta)
        self.tree = tree
        self.seed = int(seed)
        arr = (C.c_void_p * self.A)(*[ix.h for ix in self.indexes])
        self.h = lib().orc_model_create(self.A, F, arr, _p(self.alpha, c_dp), _p(self.beta, c_dp),
                                        tree.h if tree is not None else None, self.seed)


class SummaryHead(C.Structure):
    _fields_ = [("iteration", C.c_int64), ("num_isolates", C.c_int64), ("log_likelihood", C.c_double)]


class State:
    def __init__(self, model, handle, x, file):
        self.model = model
        self.h = handle
        self.x = x
        self.file = file

    @classmethod
    def init(cls, model, x, file, pop_size=0):
        x, file = _i32(x), _i32(file)
        h = lib().orc_state_init(model.h, x.shape[0], _p(x, c_i32p), _p(file, c_i32p), pop_size)
        return cls(model, h, x, file)

    @classmethod
    def from_arrays(cls, model, x, file, z, link, y, theta, iteration=0):
        x, file, link, y = _i32(x), _i32(file), _i32(link), _i32(y)
        z = np.ascontiguousarray(z, dtype=np.uint8)
        theta = _f64(theta)
        h = lib().orc_state_from_arrays(model.h, x.shape[0], y.shape[0], _p(x, c_i32p), _p(file, c_i32p), _p(z, c_u8p),
                                        _p(link, c_i32p), _p(y, c_i32p), _p(theta, c_dp), iteration)
        return cls(model, h, x, file)

    @property
    def R(self):
        return lib().orc_state_R(self.h)

    @property
    def E(self):
        return lib().orc_state_E(self.h)

    @property
    def iteration(self):
        return lib().orc_state_iteration(self.h)

    @property
    def y(self):
        return np.ctypeslib.as_array(lib().orc_state_y(self.h), (self.E, self.model.A)).copy()

    @property
    def link(self):
        return np.ctypeslib.as_array(lib().orc_state_link(self.h), (self.R,)).copy()

    @property
    def z(self):
        return np.ctypeslib.as_array(lib().orc_state_z(self.h), (self.R, self.model.A)).copy()

    @property
    def block(self):
        return np.ctypeslib.as_array(lib().orc_state_block(self.h), (self.E,)).copy()

    @property
    def theta(self):
        return np.ctypeslib.as_array(lib().orc_state_theta(self.h), (self.model.A, self.model.F)).copy()

    def summary(self):
        head = SummaryHead()
        agg = np.zeros((self.model.A, self.model.F), np.int64)
        rec = np.zeros(self.model.A + 1, np.int64)
        lib().orc_state_summary(self.h, C.byref(head), _p(agg, c_i64p), _p(rec, c_i64p))
        return {"iteration": head.iteration, "num_isolates": head.num_isolates, "log_likelihood": head.log_likelihood,
                "agg_dist": agg, "rec_dist": rec}

    def sweep(self, sampler=PCG_I, n=1):
        st = 0
        for _ in range(n):
            st |= lib().orc_state_sweep(self.h, sampler)
            if st:  # an abandoned sweep leaves the state as it was: later sweeps would fail the same way
                break
        return st

    def link_weights(self, r, sampler, cand, literal=False):
        cand = _i32(cand)
        w = np.zeros(len(cand), np.float64)
        f = lib().orc_ref_link_weights if literal else lib().orc_link_weights
        f(self.h, r, sampler, _p(cand, c_i32p), len(cand), _p(w, c_dp))
        return w

    def ref_value_pmf(self, e, a, sampler):
        pmf = np.zeros(self.model.indexes[a].V, np.float64)
        lib().orc_ref_value_pmf(self.h, e, a, sampler, _p(pmf, c_dp))
        return pmf

    def value_draw(self, e, a, sampler, u0, u1):
        return lib().orc_value_draw(self.h, e, a, sampler, u0, u1)

    def ref_dist_prob(self, r, a):
        return lib().orc_ref_dist_prob(self.h, r, a)


def draw_index(w, u):
    w = _f64(w)
    st = C.c_int(0)
    j = lib().orc_draw_index(_p(w, c_dp), len(w), u, C.byref(st))
    return j, st.value


def draw_theta(model, agg_dist, file_sizes, it):
    agg = np.ascontiguousarray(agg_dist, dtype=np.int64)
    fs = np.ascontiguousarray(file_sizes, dtype=np.int64)
    out = np.zeros((model.A, model.F), np.float64)
    lib().orc_draw_theta(model.h, _p(agg, c_i64p), _p(fs, c_i64p), it, _p(out, c_dp))
    return out


def alias_build(w):
    w = _f64(w)
    prob = np.zeros(len(w), np.float64)
    alias = np.zeros(len(w), np.int32)
    rc = lib().orc_alias_build(_p(w, c_dp), len(w), _p(prob, c_dp), _p(alias, c_i32p))
    if rc == -1:
        raise ValueError("invalid weight encountered")  # AliasSampler.scala:58-61
    if rc == -2:
        raise ValueError("zero probability mass")
    return prob, alias


def alias_sample(prob, alias, u):
    return lib().orc_alias_sample(_p(prob, c_dp), _p(alias, c_i32p), len(prob), u)

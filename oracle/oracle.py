"""ctypes binding of the CPU oracle (oracle/dzo_oracle.c -> oracle/_build/libdzo_oracle.so).

TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  Never imported by the product package.
"""
import ctypes as C
import importlib.util
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libdzo_oracle.so")

# the signature table is shared with the product binding (same argument meaning by design)
_spec = importlib.util.spec_from_file_location(
    "_dzo_capi", os.path.join(_HERE, "..", "dzoptimization.jl_b200", "_capi.py"))
_capi = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(_capi)

OBJ_ROSENBROCK, OBJ_RIESZ = 1, 2
CONSTRAINT_NONE, CONSTRAINT_SPHERE = 0, 1
SEQ, TREE, TREE_BLOCKED = 0, 1, 2

_lib = None


def build(force=False):
    src = os.path.join(_HERE, "dzo_oracle.c")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = _capi.bind(C.CDLL(LIB_PATH), cpu=True)
    return _lib


NATIVE_FLAGS = "-O3 -march=native -ffp-contract=off -fno-fast-math -fopenmp -fPIC -std=gnu11"


def use_native_build():
    """bench.py's CPU arm: the same source compiled for THIS host's cores (-O3 -march=native, still no contraction
    and no reassociation, so every bit stays the same -- tests/test_oracle.py asserts it).  Compiled at run time for the
    host that runs it, into a temporary directory so that the source tree may be read-only; must be called before the
    first oracle call of the process."""
    global _lib
    if _lib is not None and getattr(_lib, "_dzo_native", False):
        return NATIVE_FLAGS
    with tempfile.TemporaryDirectory(prefix="dzo_oracle_native_") as tmp:
        out = os.path.join(tmp, "libdzo_oracle_native.so")
        subprocess.run(["gcc"] + NATIVE_FLAGS.split() + ["-shared", "-o", out, os.path.join(_HERE, "dzo_oracle.c"), "-lm"],
                       check=True, capture_output=True)
        _lib = _capi.bind(C.CDLL(out), cpu=True)      # stays mapped after the file is removed
    _lib._dzo_native = True
    return NATIVE_FLAGS


def use_default_build():
    global _lib
    _lib = None
    return lib()


class OracleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"oracle error {code}: {msg}")
        self.code = code


def _check(rc):
    if rc != 0:
        raise OracleError(rc, lib().dzo_cpu_last_error().decode())


def _dp(a):
    return a.ctypes.data_as(_capi.c_double_p)


def pcg_fill(count, seed):
    """PCG.random_fill!(zeros(count), seed) -- legacy/PCG.jl:15-22"""
    out = np.empty(int(count), dtype=np.float64)
    _check(lib().dzo_cpu_pcg_fill(_dp(out), int(count), C.c_uint64(seed % (1 << 64))))
    return out


class _Base:
    _prefix = ""

    def _vec(self, name):
        out = np.empty((self.batch, self.n), dtype=np.float64)
        _check(getattr(lib(), f"dzo_cpu_{self._prefix}_{name}")(self._h, _dp(out)))
        return out

    def _scal(self, name, dtype=np.float64, ptr=None):
        out = np.empty(self.batch, dtype=dtype)
        _check(getattr(lib(), f"dzo_cpu_{self._prefix}_{name}")(
            self._h, out.ctypes.data_as(ptr or _capi.c_double_p)))
        return out

    point = property(lambda s: s._vec("get_point"))
    gradient = property(lambda s: s._vec("get_gradient"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    direction = property(lambda s: s._vec("get_direction"))
    objective = property(lambda s: s._scal("get_objective"))
    step_length = property(lambda s: s._scal("get_step_length"))
    iteration_count = property(lambda s: s._scal("get_iteration_count", np.int64, _capi.c_i64_p))
    terminated = property(lambda s: s._scal("get_terminated", np.uint8, _capi.c_u8_p).astype(bool))

    def step(self, k=1):
        _check(getattr(lib(), f"dzo_cpu_{self._prefix}_step")(self._h, int(k)))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            getattr(lib(), f"dzo_cpu_{self._prefix}_destroy")(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BFGS(_Base):
    """x0: (batch, n) C-order == n x batch column-major."""
    _prefix = "bfgs"

    def __init__(self, objective, x0, step, order=SEQ, constraint=CONSTRAINT_NONE, dim=0, nthreads=1):
        a = np.ascontiguousarray(np.atleast_2d(x0), dtype=np.float64)
        self.batch, self.n = a.shape
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_cpu_bfgs_create(C.byref(h), objective, constraint, dim, self.n, self.batch,
                                         _dp(a), float(step), order, nthreads))
        self._h = h

    step_type = property(lambda s: s._scal("get_step_type", np.int32, _capi.c_i32_p))

    def inverse_hessian(self, problem=0):
        out = np.empty((self.n, self.n), dtype=np.float64)
        _check(lib().dzo_cpu_bfgs_get_inverse_hessian(self._h, int(problem), _dp(out)))
        return out.T  # out is column-major; .T[i, j] = H[i, j]

    def count_active(self):
        c = C.c_int64()
        _check(lib().dzo_cpu_bfgs_count_active(self._h, C.byref(c)))
        return c.value

    def set_state(self, point, H, dx, dg, L, stype, it):
        f64 = lambda v: np.ascontiguousarray(v, dtype=np.float64)
        Hc = np.ascontiguousarray(np.swapaxes(f64(H).reshape((-1, self.n, self.n)), 1, 2))
        t = np.ascontiguousarray(np.atleast_1d(stype), dtype=np.int32)
        i = np.ascontiguousarray(np.atleast_1d(it), dtype=np.int64)
        _check(lib().dzo_cpu_bfgs_set_state(self._h, _dp(f64(point)), _dp(Hc), _dp(f64(dx)), _dp(f64(dg)),
                                            _dp(f64(np.atleast_1d(L))), t.ctypes.data_as(_capi.c_i32_p),
                                            i.ctypes.data_as(_capi.c_i64_p)))
        return self


class GD(_Base):
    _prefix = "gd"

    def __init__(self, objective, x0, step, order=SEQ, constraint=CONSTRAINT_NONE, dim=0,
                 max_increases=0, nthreads=1):
        a = np.ascontiguousarray(np.atleast_2d(x0), dtype=np.float64)
        self.batch, self.n = a.shape
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_cpu_gd_create(C.byref(h), objective, constraint, dim, self.n, self.batch,
                                       _dp(a), float(step), max_increases, order, nthreads))
        self._h = h

    delta_objective = property(lambda s: s._scal("get_delta_objective"))


def objective(obj, x, order=SEQ, constraint=CONSTRAINT_NONE, dim=0):
    a = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
    f = np.empty(a.shape[0])
    _check(lib().dzo_cpu_objective(obj, constraint, dim, order, a.shape[1], a.shape[0], _dp(a), _dp(f)))
    return f


def gradient(obj, x, order=SEQ, constraint=CONSTRAINT_NONE, dim=0):
    a = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
    g = np.empty_like(a)
    _check(lib().dzo_cpu_gradient(obj, constraint, dim, order, a.shape[1], a.shape[0], _dp(a), _dp(g)))
    return g


def dot(v, w, order=SEQ):
    v = np.ascontiguousarray(v, dtype=np.float64); w = np.ascontiguousarray(w, dtype=np.float64)
    out = C.c_double()
    _check(lib().dzo_cpu_dot(order, v.size, _dp(v), _dp(w), C.byref(out)))
    return out.value


def gemv(H, v, order=SEQ, nthreads=1):
    """H: (n, n) numpy with H[i, j]; returns H @ v in the oracle's summation order."""
    n = H.shape[0]
    Hc = np.ascontiguousarray(H.T, dtype=np.float64)  # column-major buffer
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.empty(n)
    _check(lib().dzo_cpu_gemv(order, n, _dp(Hc), _dp(v), _dp(out), nthreads))
    return out


def update_inverse_hessian(H, step_length, d, dg, next_g=None, order=SEQ, nthreads=1):
    """update_inverse_hessian! (:864-889).  Returns (H_new, d_scaled, scratch, next_d|None)."""
    n = H.shape[0]
    Hc = np.ascontiguousarray(H.T, dtype=np.float64)
    d = np.array(d, dtype=np.float64); dg = np.ascontiguousarray(dg, dtype=np.float64)
    scratch = np.empty(n)
    if next_g is None:
        _check(lib().dzo_cpu_update_inverse_hessian(order, n, _dp(Hc), float(step_length), _dp(d), _dp(dg),
                                                    _dp(scratch), None, None, nthreads))
        nd = None
    else:
        ng = np.ascontiguousarray(next_g, dtype=np.float64); nd = np.empty(n)
        _check(lib().dzo_cpu_update_inverse_hessian(order, n, _dp(Hc), float(step_length), _dp(d), _dp(dg),
                                                    _dp(scratch), _dp(ng), _dp(nd), nthreads))
    return Hc.T, d, scratch, nd


def line_search(obj, x, direction, f0, t1, order=SEQ, constraint=CONSTRAINT_NONE, dim=0):
    x = np.ascontiguousarray(x, dtype=np.float64); d = np.ascontiguousarray(direction, dtype=np.float64)
    tb, fb = C.c_double(), C.c_double()
    _check(lib().dzo_cpu_line_search(obj, constraint, dim, order, x.size, _dp(x), _dp(d), float(f0),
                                     float(t1), C.byref(tb), C.byref(fb)))
    return tb.value, fb.value


# ---------------------------------------------------------------------------------------------
# pairwise radial kernels of the live package (src/ExampleFunctions.jl:117-468), Lennard-Jones
POT_LJ = 1


def _v(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def pairwise_energy(x, y, z, order=SEQ):
    """(point_energies, energy) -- :117-173"""
    x, y, z = _v(x), _v(y), _v(z)
    pe = np.empty(x.size); e = C.c_double()
    _check(lib().dzo_cpu_pairwise_energy(POT_LJ, order, x.size, _dp(x), _dp(y), _dp(z), _dp(pe), C.byref(e)))
    return pe, e.value


def pairwise_gradient(x, y, z, order=SEQ):
    """(gx, gy, gz) -- :224-294"""
    x, y, z = _v(x), _v(y), _v(z)
    g = [np.empty(x.size) for _ in range(3)]
    _check(lib().dzo_cpu_pairwise_gradient(POT_LJ, order, x.size, _dp(x), _dp(y), _dp(z), _dp(g[0]), _dp(g[1]), _dp(g[2])))
    return g


def pairwise_hvp(x, y, z, u, v, w, order=SEQ):
    """(px, py, pz) -- :367-468"""
    x, y, z, u, v, w = map(_v, (x, y, z, u, v, w))
    p = [np.empty(x.size) for _ in range(3)]
    _check(lib().dzo_cpu_pairwise_hvp(POT_LJ, order, x.size, _dp(x), _dp(y), _dp(z), _dp(u), _dp(v), _dp(w),
                                      _dp(p[0]), _dp(p[1]), _dp(p[2])))
    return p


class LBFGS:
    """live LBFGSOptimizer (src/DZOptimization.jl:321-509), one problem; x0: (n,)"""

    def __init__(self, objective, x0, step, history_length, order=TREE):
        a = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1)
        self.n = a.size
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_cpu_lbfgs_create(C.byref(h), objective, CONSTRAINT_NONE, 0, self.n, _dp(a), float(step),
                                          int(history_length), order))
        self._h = h

    def _vec(self, name):
        out = np.empty(self.n)
        _check(getattr(lib(), "dzo_cpu_lbfgs_" + name)(self._h, _dp(out)))
        return out

    def _sc(self, name, ctype=C.c_double):
        v = ctype()
        _check(getattr(lib(), "dzo_cpu_lbfgs_" + name)(self._h, C.byref(v)))
        return v.value

    point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    direction = property(lambda s: s._vec("get_direction"))
    objective = property(lambda s: s._sc("get_objective"))
    delta_objective = property(lambda s: s._sc("get_delta_objective"))
    iteration_count = property(lambda s: s._sc("get_iteration_count", C.c_int64))
    stuck = property(lambda s: bool(s._sc("get_stuck", C.c_uint8)))

    @property
    def rho_history(self):
        cnt = C.c_int64(); rho = np.zeros(64)
        _check(lib().dzo_cpu_lbfgs_get_rho_history(self._h, C.byref(cnt), _dp(rho)))
        return rho[:cnt.value].copy()

    def step(self, k=1):
        _check(lib().dzo_cpu_lbfgs_step(self._h, int(k)))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().dzo_cpu_lbfgs_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class AdGD:
    """live AdGDOptimizer (src/DZOptimization.jl:179-312), one problem"""

    def __init__(self, objective, x0, step, order=TREE):
        a = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1)
        self.n = a.size
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_cpu_adgd_create(C.byref(h), objective, CONSTRAINT_NONE, 0, self.n, _dp(a), float(step), order))
        self._h = h

    def _vec(self, name):
        out = np.empty(self.n)
        _check(getattr(lib(), "dzo_cpu_adgd_" + name)(self._h, _dp(out)))
        return out

    point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))

    @property
    def scalars(self):
        """(f, df, current_step_size, previous_step_size, iteration_count, is_stuck)"""
        out = np.empty(6)
        _check(lib().dzo_cpu_adgd_get_scalars(self._h, _dp(out)))
        return out

    def step(self, k=1):
        _check(lib().dzo_cpu_adgd_step(self._h, int(k)))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().dzo_cpu_adgd_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


DECOR_NONE, DECOR_L2, DECOR_BOX = 0, 1, 2


class LegacyLBFGS:
    """legacy LBFGSOptimizer (legacy/DZOptimization.jl:458-695) with the optional L2 / box decorators
    (:222-296), one problem; x0: (n,)"""

    _PFX = "dzo_cpu_legacy_lbfgs_"

    def __init__(self, objective, x0, step, history_length, max_increases=0, l2_lambda=None, box=None, order=TREE):
        a = np.ascontiguousarray(x0, dtype=np.float64).reshape(-1)
        self.n, self.m = a.size, int(history_length)
        self._h = None
        h = C.c_void_p()
        decor = (DECOR_L2 if l2_lambda is not None else 0) | (DECOR_BOX if box is not None else 0)
        lo, hi = box if box is not None else (0.0, 0.0)
        _check(lib().dzo_cpu_legacy_lbfgs_create(C.byref(h), objective, CONSTRAINT_NONE, 0, self.n, _dp(a), float(step),
                                                 self.m, int(max_increases), decor,
                                                 float(l2_lambda if l2_lambda is not None else 0.0), float(lo), float(hi), order))
        self._h = h

    def _vec(self, name):
        out = np.empty(self.n)
        _check(getattr(lib(), self._PFX + name)(self._h, _dp(out)))
        return out

    point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    direction = property(lambda s: s._vec("get_direction"))

    @property
    def scalars(self):
        """(f, df, last_step_length, iteration_count, has_terminated, _history_count)"""
        out = np.empty(6)
        _check(getattr(lib(), self._PFX + "get_scalars")(self._h, _dp(out)))
        return out

    @property
    def history(self):
        """(_rho, _alpha), physical column order"""
        rho, alpha = np.zeros(self.m), np.zeros(self.m)
        _check(getattr(lib(), self._PFX + "get_history")(self._h, _dp(rho), _dp(alpha)))
        return rho, alpha

    def step(self, k=1):
        _check(getattr(lib(), self._PFX + "step")(self._h, int(k)))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            getattr(lib(), self._PFX + "destroy")(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def line_search_evaluate(objective, x, f_old, direction, overlap, step_size, compute_gradient, order=TREE):
    """live LineSearchEvaluator call (src/DZOptimization.jl:66-92) -> (trial_point, trial_gradient | None,
    (f_new, improvement_ratio, slope_ratio))"""
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1)
    d = np.ascontiguousarray(direction, dtype=np.float64).reshape(-1)
    tp, tg, res = np.empty(x.size), np.empty(x.size), np.empty(3)
    _check(lib().dzo_cpu_line_search_evaluate(objective, CONSTRAINT_NONE, 0, order, x.size, _dp(x), float(f_old), _dp(d),
                                              float(overlap), float(step_size), 1 if compute_gradient else 0, _dp(tp),
                                              _dp(tg), _dp(res)))
    return tp, (tg if compute_gradient else None), res

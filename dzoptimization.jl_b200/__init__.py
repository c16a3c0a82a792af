"""dzoptimization.jl_b200 -- host-side mirror of DZOptimization.jl's optimizer API over the
sm_100a CUDA library ``csrc/libdzopt_b200.so`` (C ABI: ``include/dzopt.h``).

The reference is Julia; Julia is not installed where this is built or run, so the host
side above the C ABI is Python with the reference's names, argument order and error
behaviour (the Julia ``ccall`` wrapper a maintainer would ship is ``julia/DZOptimizationB200.jl``).

    reference (README.md:33-41)                      this module
    -------------------------------------------     -------------------------------------------
    opt = BFGSOptimizer(f, g!, x0, 1.0)             opt = BFGSOptimizer(f, g_, x0, 1.0)
    while !opt.has_converged[]                      while not opt.has_converged[()]:
        step!(opt)                                      step_(opt)
    opt.current_objective_value[]                   opt.current_objective_value[()]
    opt.current_point                               opt.current_point

Julia closures cannot run on the device: ``f``/``g_``/constraint are the *device versions* of
``legacy/ExampleFunctions.jl`` exported from :mod:`ExampleFunctions` below (tokens that select
a compiled device objective).  Passing an arbitrary Python callable raises ``TypeError``.

There is no CPU fallback: importing works anywhere, constructing an optimizer without the
CUDA library or without a GPU raises.
"""
from __future__ import annotations

import ctypes as C
import os
from types import SimpleNamespace

import numpy as np

from . import _capi
from .pcg import pcg_fill  # noqa: F401  (legacy/PCG.jl:7-22, the input generator of bench.py and the tools)

__all__ = [
    "LBFGSOptimizer", "AdGDOptimizer", "LegacyLBFGSOptimizer", "LineSearchEvaluator",
    "L2RegularizationWrapper", "L2GradientWrapper", "UniformBoxConstraint", "UniformBoxGradientWrapper",
    "accelerated_pairwise_radial_energy", "accelerated_pairwise_radial_gradient_", "accelerated_pairwise_radial_hvp_",
    "BFGSOptimizer", "GradientDescentOptimizer", "QuadraticLineSearch", "step_",
    "ExampleFunctions", "NULL_CONSTRAINT", "SPHERE_CONSTRAINT", "StepType",
    "DZOptError", "lib", "lib_path", "pcg_fill",
]

_HERE = os.path.dirname(os.path.abspath(__file__))
#: DZOPT_B200_LIB selects another build of the same library (A/B measurements of compile-time variants)
lib_path = os.environ.get("DZOPT_B200_LIB") or os.path.join(_HERE, "csrc", "libdzopt_b200.so")
_lib = None

# include/dzopt.h constants
OBJ_ROSENBROCK, OBJ_RIESZ = 1, 2
CONSTRAINT_NONE, CONSTRAINT_SPHERE = 0, 1
ORDER_SEQUENTIAL, ORDER_TREE = 0, 1
SMALL_N_MAX = 32


class DZOptError(RuntimeError):
    """A negative status from the C ABI (the reference raises AssertionError for the same
    conditions: legacy/DZOptimization.jl:771,773)."""

    def __init__(self, code, msg):
        super().__init__(f"dzopt error {code}: {msg}")
        self.code = code


def lib():
    """Load (once) and return the CUDA library.  Fails loudly when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(lib_path):
            raise DZOptError(-6, f"{lib_path} not built; run `python __graft_entry__.py build` "
                                 "(there is no CPU fallback)")
        raw = C.CDLL(lib_path, mode=C.RTLD_GLOBAL)
        _lib = _capi.bind(_capi._DevAlias(raw), cpu=False)
    return _lib


def _check(rc):
    if rc != 0:
        raise DZOptError(rc, lib().dzo_last_error().decode())


def set_tuning(key: str, value: int):
    _check(lib().dzo_set_tuning(key.encode(), int(value)))


def _dp(a):
    return a.ctypes.data_as(_capi.c_double_p)


# ------------------------------------------------------------------------------------------
# Device objectives: tokens standing for legacy/ExampleFunctions.jl functions.
class _DeviceFunction:
    def __init__(self, name, objective, role):
        self.name, self.objective, self.role = name, objective, role

    def __repr__(self):
        return f"<device {self.role} {self.name}>"


class _Constraint:
    def __init__(self, name, cid):
        self.name, self.cid = name, cid

    def __repr__(self):
        return f"<device constraint {self.name}>"


#: ``x -> true`` (the reference's NULL_CONSTRAINT, legacy/DZOptimization.jl:384,759)
NULL_CONSTRAINT = _Constraint("NULL_CONSTRAINT", CONSTRAINT_NONE)
#: normalise every point to the unit sphere (SURVEY.md 8.0 [GLUE]); selects the tangent
#: projection of the gradient (legacy/ExampleFunctions.jl:361-374)
SPHERE_CONSTRAINT = _Constraint("SPHERE_CONSTRAINT", CONSTRAINT_SPHERE)

ExampleFunctions = SimpleNamespace(
    #: legacy/ExampleFunctions.jl:10-15; for n > 2 the extended (pairwise) form
    rosenbrock_function=_DeviceFunction("rosenbrock_function", OBJ_ROSENBROCK, "objective"),
    #: legacy/ExampleFunctions.jl:17-24
    rosenbrock_gradient_=_DeviceFunction("rosenbrock_gradient!", OBJ_ROSENBROCK, "gradient"),
    #: legacy/ExampleFunctions.jl:30-45
    riesz_energy=_DeviceFunction("riesz_energy", OBJ_RIESZ, "objective"),
    #: legacy/ExampleFunctions.jl:47-83
    riesz_gradient_=_DeviceFunction("riesz_gradient!", OBJ_RIESZ, "gradient"),
)


class _RadialFunction:
    def __init__(self, name, potential, derivative):
        self.name, self.potential, self.derivative = name, potential, derivative

    def __repr__(self):
        return f"<device radial function {self.name}>"


POT_LENNARD_JONES = 1
#: src/ExampleFunctions.jl:16-72 of the live package
ExampleFunctions.lj_energy = _RadialFunction("lj_energy", POT_LENNARD_JONES, 0)
ExampleFunctions.lj_first_derivative = _RadialFunction("lj_first_derivative", POT_LENNARD_JONES, 1)
ExampleFunctions.lj_second_derivative = _RadialFunction("lj_second_derivative", POT_LENNARD_JONES, 2)


def _radial(fn, derivative):
    if not isinstance(fn, _RadialFunction) or fn.derivative != derivative:
        want = ("lj_energy", "lj_first_derivative", "lj_second_derivative")[derivative]
        raise TypeError(f"expected the device radial function ExampleFunctions.{want}")
    return fn.potential


def _is_cuda_tensor(a):
    return hasattr(a, "is_cuda") and a.is_cuda


def _axes_check(arrays):
    n = arrays[0].shape[0]
    for a in arrays:
        if tuple(a.shape) != (n,):                       # @assert (Base.OneTo(n),) == axes(.)  src/...:160-162
            raise AssertionError("all particle arrays must be vectors of one length")
    return n


def accelerated_pairwise_radial_energy(energy_function, x, y, z, order=ORDER_SEQUENTIAL, workgroupsize=256):
    """src/ExampleFunctions.jl:152-173.  numpy arrays (host) or CUDA torch tensors (device, asynchronous
    launch on the current torch stream; the scalar read at the end synchronises like the reference's sum)."""
    pot = _radial(energy_function, 0)
    if _is_cuda_tensor(x):
        import torch
        n = _axes_check([x, y, z])
        pe = torch.empty_like(x); out = torch.empty(1, dtype=torch.float64, device=x.device)
        _check(lib().dzo_pairwise_energy_device(torch.cuda.current_stream().cuda_stream, pot, order, n, x.data_ptr(),
                                                y.data_ptr(), z.data_ptr(), pe.data_ptr(), out.data_ptr(), None))
        return float(out.item())
    x, y, z = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, z))
    n = _axes_check([x, y, z])
    e = C.c_double()
    _check(lib().dzo_pairwise_energy(pot, order, n, _dp(x), _dp(y), _dp(z), None, C.byref(e), 0))
    return e.value


def accelerated_pairwise_radial_gradient_(gx, gy, gz, energy_first_derivative, x, y, z, order=ORDER_SEQUENTIAL,
                                          workgroupsize=256):
    """src/ExampleFunctions.jl:265-294; writes gx, gy, gz in place and returns None (asynchronously for
    CUDA tensors, like the reference launcher)."""
    pot = _radial(energy_first_derivative, 1)
    if _is_cuda_tensor(x):
        import torch
        n = _axes_check([gx, gy, gz, x, y, z])
        _check(lib().dzo_pairwise_gradient_device(torch.cuda.current_stream().cuda_stream, pot, order, n, x.data_ptr(),
                                                  y.data_ptr(), z.data_ptr(), gx.data_ptr(), gy.data_ptr(), gz.data_ptr(), None))
        return None
    n = _axes_check([gx, gy, gz, x, y, z])
    x, y, z = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, z))
    _check(lib().dzo_pairwise_gradient(pot, order, n, _dp(x), _dp(y), _dp(z), _dp(gx), _dp(gy), _dp(gz), 0))
    return None


def accelerated_pairwise_radial_hvp_(px, py, pz, energy_first_derivative, energy_second_derivative, x, y, z, u, v, w,
                                     order=ORDER_SEQUENTIAL, workgroupsize=256):
    """src/ExampleFunctions.jl:427-468"""
    pot = _radial(energy_first_derivative, 1)
    if _radial(energy_second_derivative, 2) != pot:
        raise TypeError("first and second derivative belong to different potentials")
    if _is_cuda_tensor(x):
        import torch
        n = _axes_check([px, py, pz, x, y, z, u, v, w])
        _check(lib().dzo_pairwise_hvp_device(torch.cuda.current_stream().cuda_stream, pot, order, n, x.data_ptr(),
                                             y.data_ptr(), z.data_ptr(), u.data_ptr(), v.data_ptr(), w.data_ptr(),
                                             px.data_ptr(), py.data_ptr(), pz.data_ptr(), None))
        return None
    n = _axes_check([px, py, pz, x, y, z, u, v, w])
    x, y, z, u, v, w = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, z, u, v, w))
    _check(lib().dzo_pairwise_hvp(pot, order, n, _dp(x), _dp(y), _dp(z), _dp(u), _dp(v), _dp(w), _dp(px), _dp(py), _dp(pz), 0))
    return None


class StepType:
    """@enum StepType, legacy/DZOptimization.jl:727-731"""
    NullStep, GradientDescentStep, BFGSStep = 0, 1, 2


class QuadraticLineSearch:
    """legacy/DZOptimization.jl:181-188"""

    def __init__(self, max_increases: int = 0):
        self.max_increases = int(max_increases)


def _resolve(objective_function, gradient_function_, constraint_function_):
    if not isinstance(objective_function, _DeviceFunction) or objective_function.role != "objective":
        raise TypeError("objective_function must be a device objective from ExampleFunctions "
                        "(host callables cannot run inside the CUDA step!)")
    if not isinstance(gradient_function_, _DeviceFunction) or gradient_function_.role != "gradient":
        raise TypeError("gradient_function! must be a device gradient from ExampleFunctions")
    if objective_function.objective != gradient_function_.objective:
        raise TypeError("objective and gradient belong to different example functions")
    if not isinstance(constraint_function_, _Constraint):
        raise TypeError("constraint_function! must be NULL_CONSTRAINT or SPHERE_CONSTRAINT")
    return objective_function.objective, constraint_function_.cid


def _layout(initial_point, objective, batched):
    """numpy (C order) -> the reference's column-major layout.

    Julia ``x0::Array{T,N}`` column-major <-> numpy C-order with reversed axes:
      Rosenbrock vector of n          : shape (n,)            batch of them: (batch, n)
      Riesz ``dim x N`` Matrix         : shape (N, dim)        batch of them: (batch, N, dim)
    """
    a = np.ascontiguousarray(initial_point, dtype=np.float64)
    base_ndim = 2 if objective == OBJ_RIESZ else 1
    if batched:
        if a.ndim != base_ndim + 1:
            raise ValueError(f"batched initial point must have {base_ndim + 1} dimensions")
        batch = a.shape[0]
        pshape = a.shape[1:]
    else:
        if a.ndim != base_ndim:
            raise ValueError(f"initial point must have {base_ndim} dimension(s)")
        batch = 1
        pshape = a.shape
    n = int(np.prod(pshape))
    dim = int(pshape[-1]) if objective == OBJ_RIESZ else 0
    return a, n, batch, pshape, dim


# Page-locking host memory costs milliseconds (tens of them on a virtualised host), so page-locked field
# buffers are recycled process-wide instead of being freed with the optimizer that used them.
_PINNED_FREE = {}


def _pinned_take(nbytes):
    free = _PINNED_FREE.get(nbytes)
    if free:
        return free.pop()
    ptr = C.c_void_p()
    _check(lib().dzo_host_alloc(C.byref(ptr), nbytes))
    return ptr


def _pinned_give(nbytes, ptr):
    _PINNED_FREE.setdefault(nbytes, []).append(ptr)


def release_pinned_buffers():
    """cudaFreeHost every recycled page-locked buffer (optional; they are reused otherwise)."""
    for free in _PINNED_FREE.values():
        while free:
            lib().dzo_host_free(free.pop())


class _Optimizer:
    _prefix = ""
    _cache = None

    def reuse_host_buffers(self, enable: bool = True):
        """Like the Julia wrapper's cached host Arrays: every field read fills (and returns) ONE
        page-locked host buffer per field instead of a fresh pageable array, so the device->host
        copy is a straight DMA.  The returned arrays are overwritten by the next read of that field."""
        self._release_cache()
        self._cache = {} if enable else None
        return self

    def _release_cache(self):
        for arr, ptr in (self._cache or {}).values():
            _pinned_give(max(arr.nbytes, 8), ptr)
        self._cache = None

    def _out(self, getter, shape, dtype):
        if self._cache is None:
            return np.empty(shape, dtype=dtype)
        hit = self._cache.get(getter)
        if hit is None:
            nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
            ptr = _pinned_take(max(nbytes, 8))
            raw = (C.c_char * max(nbytes, 8)).from_address(ptr.value)
            hit = (np.frombuffer(raw, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape), ptr)
            self._cache[getter] = hit
        return hit[0]

    def _vec(self, getter):
        out = self._out(getter, (self._batch,) + self._pshape if self._batched else self._pshape, np.float64)
        _check(getattr(lib(), f"dzo_{self._prefix}_{getter}")(self._h, _dp(out)))
        return out

    def _scalar(self, getter, dtype=np.float64, ptr=_capi.c_double_p):
        out = self._out(getter, self._batch, dtype)
        _check(getattr(lib(), f"dzo_{self._prefix}_{getter}")(self._h, out.ctypes.data_as(ptr)))
        # reference scalars are 0-dim Arrays read with `[]`; numpy 0-dim arrays read with `[()]`
        return out if self._batched else out.reshape(())

    # fields shared by both optimizers
    @property
    def current_point(self): return self._vec("get_point")
    @property
    def current_gradient(self): return self._vec("get_gradient")
    @property
    def delta_point(self): return self._vec("get_delta_point")
    @property
    def delta_gradient(self): return self._vec("get_delta_gradient")
    @property
    def next_step_direction(self): return self._vec("get_direction")
    @property
    def current_objective_value(self): return self._scalar("get_objective")
    @property
    def last_step_length(self): return self._scalar("get_step_length")
    @property
    def iteration_count(self): return self._scalar("get_iteration_count", np.int64, _capi.c_i64_p)
    @property
    def has_terminated(self):
        return self._scalar("get_terminated", np.uint8, _capi.c_u8_p).view(np.bool_)
    #: README.md:38 spelling of has_terminated
    has_converged = has_terminated

    def set_stream(self, cuda_stream: int | None):
        _check(getattr(lib(), f"dzo_{self._prefix}_set_stream")(self._h, C.c_void_p(cuda_stream or 0)))

    def step(self, k: int = 1):
        _check(getattr(lib(), f"dzo_{self._prefix}_step")(self._h, int(k)))
        return self

    def step_async(self, k: int = 1):
        _check(getattr(lib(), f"dzo_{self._prefix}_step_async")(self._h, int(k)))
        return self

    def sync(self):
        _check(getattr(lib(), f"dzo_{self._prefix}_sync")(self._h))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._release_cache()
            getattr(lib(), f"dzo_{self._prefix}_destroy")(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BFGSOptimizer(_Optimizer):
    """struct BFGSOptimizer, legacy/DZOptimization.jl:733-751.

    ``BFGSOptimizer(f, g_, x0, step)`` (:753-760) or ``BFGSOptimizer(f, g_, c_, x0, step)``
    (:762-810).  ``batched=True`` treats the leading axis of x0 as independent problems
    (README.md:12 "run multiple optimizers in parallel").  ``shard=(rank, nranks, nccl_id)``
    row-shards one large-n inverse Hessian over GPUs (one process per GPU).
    """
    _prefix = "bfgs"

    def __init__(self, objective_function, gradient_function_, *args, batched=False, device=0,
                 shard=None):
        if len(args) == 2:
            constraint_function_, (initial_point, initial_step_length) = NULL_CONSTRAINT, args
        elif len(args) == 3:
            constraint_function_, initial_point, initial_step_length = args
        else:
            raise TypeError("BFGSOptimizer(f, g!, [c!,] x0, initial_step_length)")
        obj, cid = _resolve(objective_function, gradient_function_, constraint_function_)
        a, n, batch, pshape, dim = _layout(initial_point, obj, batched)
        self._batched, self._batch, self._pshape, self._n = batched, batch, pshape, n
        self._h = None
        h = C.c_void_p()
        if shard is None:
            _check(lib().dzo_bfgs_create(C.byref(h), obj, cid, dim, n, batch, _dp(a),
                                         float(initial_step_length), int(device)))
        else:
            rank, nranks, nccl_id = shard
            if batched:
                raise ValueError("row sharding applies to a single large-n problem")
            idbuf = C.create_string_buffer(bytes(nccl_id), 128)
            _check(lib().dzo_bfgs_create_sharded(C.byref(h), obj, cid, dim, n, _dp(a),
                                                 float(initial_step_length), int(device),
                                                 int(rank), int(nranks), idbuf))
        self._h = h

    @property
    def last_step_type(self): return self._scalar("get_step_type", np.int32, _capi.c_i32_p)

    def reuse_host_buffers(self, enable: bool = True):
        """Cached page-locked field buffers (see _Optimizer).  For a batched optimizer the two fields of the README loop
        -- ``has_converged[]`` and ``current_objective_value[]`` -- additionally become ZERO-COPY MIRRORS
        (dzo_bfgs_mirror_fields): the step kernel itself stores them into the cached host arrays while it runs, and
        reading them only synchronises."""
        self._unmirror()
        super().reuse_host_buffers(enable)
        if enable and self._batched:
            f = self._out("get_objective", self._batch, np.float64)
            t = self._out("get_terminated", self._batch, np.uint8)
            rc = lib().dzo_bfgs_mirror_fields(self._h, _dp(f), t.ctypes.data_as(_capi.c_u8_p))
            if rc != -5:                 # DZO_ERR_UNSUPPORTED (generic batched kernel): ordinary copies into the cache
                _check(rc)
            self._mirrored = (rc == 0)
        return self

    def _unmirror(self):
        if getattr(self, "_mirrored", False) and getattr(self, "_h", None):
            lib().dzo_bfgs_mirror_fields(self._h, None, None)      # before the buffers go back to the recycling pool
        self._mirrored = False

    def _release_cache(self):
        self._unmirror()
        super()._release_cache()

    def inverse_hessian(self, problem: int = 0):
        """approximate_inverse_hessian (:746) of one problem as an (n, n) array.  It is bitwise
        symmetric, so the column-major device matrix and this C-order view coincide."""
        r0, r1 = self.row_range
        out = np.empty((self._n, r1 - r0), dtype=np.float64)  # column-major rows x n
        _check(lib().dzo_bfgs_get_inverse_hessian(self._h, int(problem), _dp(out)))
        return out.T  # (rows, n): out.T[i, j] = H[r0 + i, j]

    @property
    def approximate_inverse_hessian(self): return self.inverse_hessian(0)

    @property
    def row_range(self):
        r0, r1 = C.c_int64(), C.c_int64()
        _check(lib().dzo_bfgs_info(self._h, None, None, None, C.byref(r0), C.byref(r1)))
        return r0.value, r1.value

    @property
    def summation_order(self):
        o = C.c_int()
        _check(lib().dzo_bfgs_info(self._h, None, None, C.byref(o), None, None))
        return o.value

    @property
    def gather_mode(self):
        """0 = not sharded, 1 = fused peer-memory gathers, 2 = ncclAllGather"""
        m = C.c_int()
        _check(lib().dzo_bfgs_gather_mode(self._h, C.byref(m)))
        return m.value

    def step_log(self):
        """(calls, kinds) -- kinds[c % 64] is the StepType of step! call c (large-n handles)."""
        calls = C.c_int64()
        kinds = np.zeros(64, dtype=np.uint8)
        _check(lib().dzo_bfgs_get_step_log(self._h, C.byref(calls), kinds.ctypes.data_as(_capi.c_u8_p)))
        return calls.value, kinds

    def count_active(self) -> int:
        c = C.c_int64()
        _check(lib().dzo_bfgs_count_active(self._h, C.byref(c)))
        return c.value

    STEP_KINDS = ("bfgs_read_h", "bfgs_identity_h", "gradient_descent", "terminate", "idle", "idle_warp")

    def step_kind_counts(self, reset: bool = False) -> dict:
        """What the step! calls of a batched optimizer did, counted on the device (dzo_bfgs_get_step_kind_counts):
        BFGS-type steps that read H from HBM / whose H was an implicit identity, gradient-descent steps (:962-986),
        terminations (:988-990), step! calls on terminated problems (:893).  Running totals."""
        c = np.zeros(8, dtype=np.int64)
        _check(lib().dzo_bfgs_get_step_kind_counts(self._h, c.ctypes.data_as(_capi.c_i64_p), int(bool(reset))))
        return {k: int(v) for k, v in zip(self.STEP_KINDS, c)}

    def set_state(self, point, inverse_hessian, delta_point, delta_gradient, last_step_length,
                  last_step_type, iteration_count):
        """Resume from saved fields (README.md:11); semantics of the rebuilding constructor
        legacy/DZOptimization.jl:819-862 (f, g and H*g are recomputed)."""
        f64 = lambda v: np.ascontiguousarray(v, dtype=np.float64)
        x, Hm, dx, dg = f64(point), f64(inverse_hessian), f64(delta_point), f64(delta_gradient)
        # numpy (n,n) C-order of a symmetric matrix == column-major; for generality transpose
        Hm = np.ascontiguousarray(np.swapaxes(Hm.reshape((-1, self._n, self._n)), 1, 2))
        L = f64(np.atleast_1d(last_step_length))
        t = np.ascontiguousarray(np.atleast_1d(last_step_type), dtype=np.int32)
        it = np.ascontiguousarray(np.atleast_1d(iteration_count), dtype=np.int64)
        _check(lib().dzo_bfgs_set_state(self._h, _dp(x), _dp(Hm), _dp(dx), _dp(dg), _dp(L),
                                        t.ctypes.data_as(_capi.c_i32_p),
                                        it.ctypes.data_as(_capi.c_i64_p)))
        return self


class GradientDescentOptimizer(_Optimizer):
    """struct GradientDescentOptimizer, legacy/DZOptimization.jl:305-327.

    ``GradientDescentOptimizer(f, g_, line_search, x0, step)`` (:377-390) or
    ``GradientDescentOptimizer(c_, f, g_, line_search, x0, step)`` (:330-337; note the
    constraint comes FIRST in this constructor, unlike BFGSOptimizer)."""
    _prefix = "gd"

    def __init__(self, *args, batched=False, device=0):
        if len(args) == 5:
            constraint_function_ = NULL_CONSTRAINT
            objective_function, gradient_function_, line_search, initial_point, step = args
        elif len(args) == 6:
            constraint_function_, objective_function, gradient_function_, line_search, initial_point, step = args
        else:
            raise TypeError("GradientDescentOptimizer([c!,] f, g!, line_search!, x0, initial_step_length)")
        if not isinstance(line_search, QuadraticLineSearch):
            raise TypeError("line_search_function! must be a QuadraticLineSearch")
        obj, cid = _resolve(objective_function, gradient_function_, constraint_function_)
        a, n, batch, pshape, dim = _layout(initial_point, obj, batched)
        self._batched, self._batch, self._pshape, self._n = batched, batch, pshape, n
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_gd_create(C.byref(h), obj, cid, dim, n, batch, _dp(a), float(step),
                                   line_search.max_increases, int(device)))
        self._h = h

    @property
    def delta_objective_value(self): return self._scalar("get_delta_objective")

    def evaluation_count(self) -> int:
        """objective evaluations so far (constructor + line-search probes); one-problem handles"""
        c = C.c_int64()
        _check(lib().dzo_gd_get_evaluation_count(self._h, C.byref(c)))
        return c.value


class LBFGSOptimizer:
    """struct LBFGSOptimizer of the LIVE package, src/DZOptimization.jl:321-344.

    ``LBFGSOptimizer(c_, f, g_, x0, initial_step_length, history_length)`` (:400-427); ``c_`` is ``None``
    (Julia ``nothing``) or NULL_CONSTRAINT.  Fields as in the reference: ``is_stuck`` (the live spelling of
    has_terminated), ``iteration_count``, ``current_point``, ``delta_point``, ``current_objective_value``,
    ``delta_objective_value``, ``current_gradient``, ``delta_gradient``, ``step_direction``, ``rho_history``.

    ``batched=True`` treats the leading axis of x0 as independent problems (README.md:12), like
    ``BFGSOptimizer(batched=True)``: x0 has shape (batch, n), vector fields come back as (batch, n), scalar fields as
    (batch,), ``rho_history`` as a list of ``batch`` arrays (each newest first); sums in DZO_ORDER_SEQUENTIAL."""

    def __init__(self, constraint_function_, objective_function, gradient_function_, initial_point,
                 initial_step_length, history_length, batched=False, device=0):
        c = NULL_CONSTRAINT if constraint_function_ is None else constraint_function_
        obj, cid = _resolve(objective_function, gradient_function_, c)
        a = np.ascontiguousarray(initial_point, dtype=np.float64)
        if a.ndim != (2 if batched else 1):
            raise ValueError("batched initial point must have shape (batch, n)" if batched else "initial point must be a vector")
        if not initial_step_length > 0:
            raise AssertionError("initial_step_length > 0")              # @assert :375
        self._batched = bool(batched)
        self._batch, self._n = a.shape if batched else (1, a.size)
        self._h = None
        h = C.c_void_p()
        if batched:
            _check(lib().dzo_lbfgs_create_batched(C.byref(h), obj, cid, 0, self._n, self._batch, _dp(a),
                                                  float(initial_step_length), int(history_length), int(device)))
        else:
            _check(lib().dzo_lbfgs_create(C.byref(h), obj, cid, 0, self._n, _dp(a), float(initial_step_length),
                                          int(history_length), int(device)))
        self._h = h
        self.history_length = int(history_length)

    def _vec(self, name):
        out = np.empty((self._batch, self._n) if self._batched else self._n)
        _check(getattr(lib(), "dzo_lbfgs_" + name)(self._h, _dp(out)))
        return out

    def _sc(self, name, ctype, dtype):
        if self._batched:
            out = np.empty(self._batch, dtype=np.dtype(ctype))
            _check(getattr(lib(), "dzo_lbfgs_" + name)(self._h, out.ctypes.data_as(C.POINTER(ctype))))
            return out.astype(dtype, copy=False)
        v = ctype()
        _check(getattr(lib(), "dzo_lbfgs_" + name)(self._h, C.byref(v)))
        return np.array(v.value, dtype=dtype)

    current_point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    current_gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    step_direction = property(lambda s: s._vec("get_direction"))
    current_objective_value = property(lambda s: s._sc("get_objective", C.c_double, np.float64))
    delta_objective_value = property(lambda s: s._sc("get_delta_objective", C.c_double, np.float64))
    iteration_count = property(lambda s: s._sc("get_iteration_count", C.c_int64, np.int64))
    is_stuck = property(lambda s: s._sc("get_stuck", C.c_uint8, np.bool_))
    has_converged = is_stuck

    @property
    def rho_history(self):
        cnt = np.zeros(self._batch, dtype=np.int64); rho = np.zeros((self._batch, 64))
        _check(lib().dzo_lbfgs_get_rho_history(self._h, cnt.ctypes.data_as(_capi.c_i64_p), _dp(rho)))
        if self._batched:
            return [rho[p, :cnt[p]].copy() for p in range(self._batch)]
        return rho[0, :cnt[0]].copy()

    @property
    def summation_order(self):
        o = C.c_int()
        _check(lib().dzo_lbfgs_info(self._h, None, C.byref(o), None))
        return o.value

    def set_stream(self, cuda_stream):
        _check(lib().dzo_lbfgs_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def step(self, k: int = 1):
        _check(lib().dzo_lbfgs_step(self._h, int(k)))
        return self

    def step_async(self, k: int = 1):
        _check(lib().dzo_lbfgs_step_async(self._h, int(k)))
        return self

    def sync(self):
        _check(lib().dzo_lbfgs_sync(self._h))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().dzo_lbfgs_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class AdGDOptimizer:
    """struct AdGDOptimizer of the LIVE package, src/DZOptimization.jl:179-198;
    ``AdGDOptimizer(c_, f, g_, x0, initial_step_length)`` (:252-271)."""

    def __init__(self, constraint_function_, objective_function, gradient_function_, initial_point,
                 initial_step_length, device=0):
        c = NULL_CONSTRAINT if constraint_function_ is None else constraint_function_
        obj, cid = _resolve(objective_function, gradient_function_, c)
        a = np.ascontiguousarray(initial_point, dtype=np.float64)
        if a.ndim != 1:
            raise ValueError("initial point must be a vector")
        if not initial_step_length > 0:
            raise AssertionError("initial_step_length > 0")              # @assert :232
        self._n = a.size
        self._h = None
        h = C.c_void_p()
        _check(lib().dzo_adgd_create(C.byref(h), obj, cid, 0, self._n, _dp(a), float(initial_step_length), int(device)))
        self._h = h

    def _vec(self, name):
        out = np.empty(self._n)
        _check(getattr(lib(), "dzo_adgd_" + name)(self._h, _dp(out)))
        return out

    def _scalars(self):
        out = np.empty(6)
        _check(lib().dzo_adgd_get_scalars(self._h, _dp(out)))
        return out

    current_point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    current_gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    current_objective_value = property(lambda s: np.array(s._scalars()[0]))
    delta_objective_value = property(lambda s: np.array(s._scalars()[1]))
    current_step_size = property(lambda s: np.array(s._scalars()[2]))
    previous_step_size = property(lambda s: np.array(s._scalars()[3]))
    iteration_count = property(lambda s: np.array(int(s._scalars()[4])))
    is_stuck = property(lambda s: np.array(bool(s._scalars()[5])))
    has_converged = is_stuck

    def step(self, k: int = 1):
        _check(lib().dzo_adgd_step(self._h, int(k)))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().dzo_adgd_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------
# legacy decorators (legacy/DZOptimization.jl:222-296) and the legacy L-BFGS (:458-695)
DECOR_L2, DECOR_BOX = 1, 2


class L2RegularizationWrapper:
    """legacy/DZOptimization.jl:228-234: ``f(x) + lambda * norm2(x)`` around a device objective."""

    def __init__(self, objective_function, lambda_):
        self.objective_function, self.lambda_ = objective_function, float(lambda_)


class L2GradientWrapper:
    """legacy/DZOptimization.jl:237-251: ``g += (lambda + lambda) * x`` after a device gradient."""

    def __init__(self, gradient_function_, lambda_):
        self.gradient_function_, self.lambda_ = gradient_function_, float(lambda_)


class UniformBoxConstraint:
    """legacy/DZOptimization.jl:257-272: clamp every coordinate to [lower_bound, upper_bound]; returns true."""

    def __init__(self, lower_bound, upper_bound):
        self.lower_bound, self.upper_bound = float(lower_bound), float(upper_bound)


class UniformBoxGradientWrapper:
    """legacy/DZOptimization.jl:275-296: zero the gradient entries that point out of the box at an active bound."""

    def __init__(self, gradient_function_, lower_bound, upper_bound):
        self.gradient_function_ = gradient_function_
        self.lower_bound, self.upper_bound = float(lower_bound), float(upper_bound)


def _resolve_decorated(constraint_function_, objective_function, gradient_function_):
    """Peel the legacy wrappers off the three callables; the device applies them in the fixed order
    gradient! = Box(L2(g!)) (include/dzopt.h).  Inconsistent wrappers raise TypeError."""
    lam_f = lam_g = None
    box_c = box_g = None
    if isinstance(objective_function, L2RegularizationWrapper):
        lam_f, objective_function = objective_function.lambda_, objective_function.objective_function
    if isinstance(gradient_function_, UniformBoxGradientWrapper):
        box_g = (gradient_function_.lower_bound, gradient_function_.upper_bound)
        gradient_function_ = gradient_function_.gradient_function_
    if isinstance(gradient_function_, L2GradientWrapper):
        lam_g, gradient_function_ = gradient_function_.lambda_, gradient_function_.gradient_function_
    if isinstance(gradient_function_, UniformBoxGradientWrapper):
        raise TypeError("device composition order is UniformBoxGradientWrapper(L2GradientWrapper(g!, lambda), lo, hi)")
    if isinstance(constraint_function_, UniformBoxConstraint):
        box_c = (constraint_function_.lower_bound, constraint_function_.upper_bound)
        constraint_function_ = NULL_CONSTRAINT
    if constraint_function_ is None:
        constraint_function_ = NULL_CONSTRAINT
    if lam_f != lam_g:
        raise TypeError("L2RegularizationWrapper and L2GradientWrapper must be used together with one lambda")
    if box_c != box_g:
        raise TypeError("UniformBoxConstraint and UniformBoxGradientWrapper must be used together with the same bounds")
    obj, cid = _resolve(objective_function, gradient_function_, constraint_function_)
    return obj, cid, lam_f, box_c


class LegacyLBFGSOptimizer:
    """struct LBFGSOptimizer of the LEGACY file, legacy/DZOptimization.jl:458-486.

    ``LegacyLBFGSOptimizer(c_, f, g_, linesearch, x0, initial_step_length, history_length)`` (:489-548) or the
    6-argument form without a constraint (:551-562).  ``linesearch`` is a :class:`QuadraticLineSearch`;
    ``f`` / ``g_`` / ``c_`` may carry the L2 / uniform-box wrappers.  (The live package's optimizer of the
    same Julia name is :class:`LBFGSOptimizer`.)"""

    def __init__(self, *args, device=0):
        if len(args) == 7:
            c, f, g, ls, x0, L0, m = args
        elif len(args) == 6:
            f, g, ls, x0, L0, m = args
            c = NULL_CONSTRAINT
        else:
            raise TypeError("LegacyLBFGSOptimizer([c!,] f, g!, linesearch, x0, initial_step_length, history_length)")
        if not isinstance(ls, QuadraticLineSearch):
            raise TypeError("line_search_function! must be a QuadraticLineSearch")
        obj, cid, lam, box = _resolve_decorated(c, f, g)
        a = np.ascontiguousarray(x0, dtype=np.float64)
        if a.ndim != 1:
            raise ValueError("initial point must be a vector")
        if not int(m) > 0:
            raise AssertionError("history_length > 0")                   # @assert :528
        self._n, self.history_length = a.size, int(m)
        self._h = None
        h = C.c_void_p()
        decor = (DECOR_L2 if lam is not None else 0) | (DECOR_BOX if box is not None else 0)
        lo, hi = box if box is not None else (0.0, 0.0)
        _check(lib().dzo_legacy_lbfgs_create(C.byref(h), obj, cid, 0, self._n, _dp(a), float(L0), int(m), ls.max_increases,
                                             decor, float(lam if lam is not None else 0.0), lo, hi, int(device)))
        self._h = h

    def _vec(self, name):
        out = np.empty(self._n)
        _check(getattr(lib(), "dzo_legacy_lbfgs_" + name)(self._h, _dp(out)))
        return out

    def _scalars(self):
        out = np.empty(6)
        _check(lib().dzo_legacy_lbfgs_get_scalars(self._h, _dp(out)))
        return out

    current_point = property(lambda s: s._vec("get_point"))
    delta_point = property(lambda s: s._vec("get_delta_point"))
    current_gradient = property(lambda s: s._vec("get_gradient"))
    delta_gradient = property(lambda s: s._vec("get_delta_gradient"))
    next_step_direction = property(lambda s: s._vec("get_direction"))
    current_objective_value = property(lambda s: np.array(s._scalars()[0]))
    delta_objective_value = property(lambda s: np.array(s._scalars()[1]))
    last_step_length = property(lambda s: np.array(s._scalars()[2]))
    iteration_count = property(lambda s: np.array(int(s._scalars()[3])))
    has_terminated = property(lambda s: np.array(bool(s._scalars()[4])))
    has_converged = has_terminated
    _history_count = property(lambda s: np.array(int(s._scalars()[5])))

    def _history(self):
        rho, alpha = np.zeros(self.history_length), np.zeros(self.history_length)
        _check(lib().dzo_legacy_lbfgs_get_history(self._h, _dp(rho), _dp(alpha)))
        return rho, alpha

    _rho = property(lambda s: s._history()[0])
    _alpha = property(lambda s: s._history()[1])

    def set_stream(self, cuda_stream):
        _check(lib().dzo_legacy_lbfgs_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def step(self, k: int = 1):
        _check(lib().dzo_legacy_lbfgs_step(self._h, int(k)))
        return self

    def step_async(self, k: int = 1):
        _check(lib().dzo_legacy_lbfgs_step_async(self._h, int(k)))
        return self

    def sync(self):
        _check(lib().dzo_legacy_lbfgs_sync(self._h))
        return self

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().dzo_legacy_lbfgs_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LineSearchEvaluator:
    """struct LineSearchEvaluator of the LIVE package, src/DZOptimization.jl:12-26.

    ``LineSearchEvaluator(c_, f, g_, initial_point, initial_objective_value, initial_gradient, step_direction,
    overlap)`` (:29-63); calling ``lse(step_size, compute_gradient)`` (:66-92) fills ``trial_point``,
    ``trial_objective_value``, ``improvement_ratio`` and, with ``compute_gradient``, ``trial_gradient`` and
    ``slope_ratio``, and returns the trial objective value.  One cluster launch per call."""

    def __init__(self, constraint_function_, objective_function, gradient_function_, initial_point,
                 initial_objective_value, initial_gradient, step_direction, overlap, device=0):
        c = NULL_CONSTRAINT if constraint_function_ is None else constraint_function_
        self._obj, self._cid = _resolve(objective_function, gradient_function_, c)
        self.current_point = np.ascontiguousarray(initial_point, dtype=np.float64)
        self.current_gradient = np.ascontiguousarray(initial_gradient, dtype=np.float64)
        self.step_direction = np.ascontiguousarray(step_direction, dtype=np.float64)
        if not (self.current_point.shape == self.current_gradient.shape == self.step_direction.shape):
            raise AssertionError("point_axes == axes(initial_gradient) == axes(step_direction)")   # @assert :41-43
        self.current_objective_value = np.array(float(initial_objective_value))
        self.overlap = np.array(float(overlap))
        self.trial_point = np.empty_like(self.current_point)
        self.trial_gradient = np.empty_like(self.current_point)
        self.trial_objective_value = np.array(np.nan)
        self.improvement_ratio = np.array(np.nan)
        self.slope_ratio = np.array(np.nan)
        self._device = int(device)

    def __call__(self, step_size, compute_gradient):
        res = np.empty(3)
        _check(lib().dzo_line_search_evaluate(self._obj, self._cid, 0, ORDER_TREE, self.current_point.size,
                                              _dp(self.current_point), float(self.current_objective_value[()]),
                                              _dp(self.step_direction), float(self.overlap[()]), float(step_size),
                                              1 if compute_gradient else 0, _dp(self.trial_point),
                                              _dp(self.trial_gradient), _dp(res), self._device))
        self.trial_objective_value[()] = res[0]
        self.improvement_ratio[()] = res[1]
        if compute_gradient:
            self.slope_ratio[()] = res[2]
        return float(res[0])


def step_(opt):
    """step!(opt) -- legacy/DZOptimization.jl:393, :891.  Returns opt (:448, :993)."""
    return opt.step(1)

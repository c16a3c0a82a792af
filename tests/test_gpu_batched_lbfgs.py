"""Batched live LBFGSOptimizer (dzo_lbfgs_create_batched, csrc/batched_lbfgs.cuh): `batch` problems in one handle, one
device thread per problem, compared bit for bit with one oracle DZO_ORDER_SEQUENTIAL handle per problem after the
constructor and after every checked launch -- point, delta_point, gradient, delta_gradient, direction, objective,
delta_objective, iteration_count, is_stuck and the rho history with its count.  The CPU tests at the top check the
argument validation, which runs before any CUDA call."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_bitwise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEQ = 0
VECS = (("current_point", "point"), ("delta_point", "delta_point"), ("current_gradient", "gradient"),
        ("delta_gradient", "delta_gradient"), ("step_direction", "direction"))


# ----------------------------------------------------------------------------- CPU: validation before any CUDA call
def test_batched_lbfgs_argument_validation_needs_no_gpu(dz):
    lib = dz.lib()
    x = np.zeros(34 * 4)
    dp = x.ctypes.data_as(dz._capi.c_double_p)
    h = C.c_void_p()
    create = lambda obj, prm, n, batch, m, xp=dp, out=C.byref(h): lib.dzo_lbfgs_create_batched(out, obj, 0, prm, n, batch, xp,
                                                                                                1.0, m, 0)
    assert create(1, 0, 3, 4, 10) == -1 and b"even n" in lib.dzo_last_error()             # odd n
    assert create(1, 0, 34, 4, 10) == -5 and b"n <= 32" in lib.dzo_last_error()           # n > DZO_SMALL_N_MAX
    assert create(2, 2, 4, 4, 10) == -5 and b"DZO_OBJ_ROSENBROCK" in lib.dzo_last_error()  # Riesz
    assert create(1, 0, 4, 4, 0) == -1 and b"history_length" in lib.dzo_last_error()
    assert create(1, 0, 4, 4, 65) == -1 and b"history_length" in lib.dzo_last_error()
    assert create(1, 0, 4, 0, 10) == -1 and b"batch" in lib.dzo_last_error()
    assert create(1, 0, 4, 4, 10, xp=None) == -1 and b"null pointer" in lib.dzo_last_error()
    assert create(1, 0, 4, 4, 10, out=None) == -1 and b"null pointer" in lib.dzo_last_error()
    assert lib.dzo_lbfgs_create_batched(C.byref(h), 1, 0, 0, 4, 4, dp, 0.0, 10, 0) == -1   # initial_step_length (:375)
    assert lib.dzo_lbfgs_info(None, None, None, None) == -1


def test_batched_lbfgs_without_a_device_fails_loudly():
    child = "\n".join([
        "import sys",
        "sys.path.insert(0, %r)" % ROOT,
        "import numpy as np",
        "import dzopt_b200 as dz",
        "EF = dz.ExampleFunctions",
        "try:",
        "    dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros((5, 4)), 1.0, 3, batched=True)",
        "    print('computed')",
        "except dz.DZOptError as e:",
        "    print(e.code)",
    ])
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == ["-6"], r.stdout


def test_batched_lbfgs_python_shapes(dz):
    EF = dz.ExampleFunctions
    with pytest.raises(ValueError):
        dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros(4), 1.0, 3, batched=True)
    with pytest.raises(ValueError):
        dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros((2, 4)), 1.0, 3)


# ----------------------------------------------------------------------------- GPU
def _make(dz, x0, m, step=1.0):
    EF = dz.ExampleFunctions
    opt = dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, step, m, batched=True)
    order, ctas = C.c_int(), C.c_int()
    assert dz.lib().dzo_lbfgs_info(opt._h, None, C.byref(order), C.byref(ctas)) == 0
    assert order.value == SEQ and ctas.value >= -(-x0.shape[0] // 256)
    return opt


def _rho(dz, opt):
    """(count[batch], rho[batch, 64]) in one call"""
    cnt = np.zeros(opt._batch, dtype=np.int64)
    rho = np.zeros((opt._batch, 64))
    assert dz.lib().dzo_lbfgs_get_rho_history(opt._h, cnt.ctypes.data_as(dz._capi.c_i64_p),
                                              rho.ctypes.data_as(dz._capi.c_double_p)) == 0, dz.lib().dzo_last_error()
    return cnt, rho


def _device_state(dz, opt, idx):
    st = {k: getattr(opt, a)[idx] for a, k in VECS}
    st["objective"] = opt.current_objective_value[idx]
    st["delta_objective"] = opt.delta_objective_value[idx]
    st["iteration_count"] = opt.iteration_count[idx]
    st["stuck"] = opt.is_stuck[idx]
    cnt, rho = _rho(dz, opt)
    st["count"], st["rho"] = cnt[idx], rho[idx]
    return st


def _oracle_state(refs):
    st = {k: np.array([getattr(r, k) for r in refs]) for _, k in VECS}
    st["objective"] = np.array([r.objective for r in refs])
    st["delta_objective"] = np.array([r.delta_objective for r in refs])
    st["iteration_count"] = np.array([r.iteration_count for r in refs], dtype=np.int64)
    st["stuck"] = np.array([r.stuck for r in refs])
    rho = np.zeros((len(refs), 64))
    cnt = np.zeros(len(refs), dtype=np.int64)
    for i, r in enumerate(refs):
        h = r.rho_history
        cnt[i] = h.size
        rho[i, :h.size] = h
    st["count"], st["rho"] = cnt, rho
    return st


def _compare(dz, opt, refs, idx, what):
    dev, ref = _device_state(dz, opt, idx), _oracle_state(refs)
    for k in ("point", "delta_point", "gradient", "delta_gradient", "direction", "objective", "delta_objective", "rho"):
        assert_bitwise(dev[k], ref[k], f"{what}: {k}")
    for k in ("iteration_count", "stuck", "count"):
        assert np.array_equal(dev[k], ref[k]), f"{what}: {k} {dev[k]} vs {ref[k]}"
    return dev


def _endless(x, d):
    """Rows on which the reference's backtracking loop never ends: a trial point is never isequal to the point when the
    direction is not finite (a NaN or Inf from rho = 0 or an overflowing gradient) or when a -0.0 coordinate moves by
    +0.0.  The device caps those searches (the oracle, like the reference, would loop forever), so a problem the device
    left stuck with such a direction is retired from the oracle comparison."""
    negzero_up = np.signbit(x) & (x == 0) & ~np.signbit(d) & (d == 0)
    return ~np.isfinite(d).all(axis=1) | negzero_up.any(axis=1)


def _step_all(dz, opt, refs, idx, active, k, what):
    """one launch of step(k); the oracle handles of the still active problems follow.  Returns the new active mask."""
    before = _device_state(dz, opt, idx)
    opt.step(k)
    after = _device_state(dz, opt, idx)
    capped = active & after["stuck"] & _endless(after["point"], after["direction"]) & (k > 0)
    if k == 1:      # capped in this very step: the not-accepted branch
        for j in np.flatnonzero(capped & ~before["stuck"]):
            assert_bitwise(after["point"][j], before["point"][j], f"{what}: capped point")
            assert_bitwise(after["delta_point"][j], before["point"][j], f"{what}: capped delta_point")
            assert after["iteration_count"][j] == before["iteration_count"][j]
    active = active & ~capped
    for j in np.flatnonzero(active):
        refs[j].step(k)
    _compare(dz, opt, [refs[j] for j in np.flatnonzero(active)], idx[active], what)
    return active


def _oracles(orc, x0, m, idx, step=1.0):
    return [orc.LBFGS(orc.OBJ_ROSENBROCK, x0[p], step, m, order=orc.SEQ) for p in idx]


def _run(dz, orc, x0, m, launches, idx=None):
    idx = np.arange(x0.shape[0]) if idx is None else idx
    opt = _make(dz, x0, m)
    refs = _oracles(orc, x0, m, idx)
    _compare(dz, opt, refs, idx, "constructor")
    active = np.ones(idx.size, dtype=bool)
    for i, k in enumerate(launches):
        active = _step_all(dz, opt, refs, idx, active, k, f"after launch {i} (step({k}))")
    assert active.mean() > 0.9, "too few problems left to compare"
    return opt, _device_state(dz, opt, idx)


def _x0(orc, batch, n, seed):
    return (4.0 * orc.pcg_fill(batch * n, seed) - 2.0).reshape(batch, n)


N_ALL = list(range(2, 33, 2))


# A: every even n with m in {1, 3, 10} on a batch that leaves a partial warp; 997 problems (partial last CTA); batch 1
@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 3, 10])
@pytest.mark.parametrize("n", N_ALL)
def test_batched_lbfgs_every_n(gpu, orc, n, m):
    _run(gpu, orc, _x0(orc, 67, n, 100 + n), m, [1, 1, 1, 2, 5])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 16, 32])
def test_batched_lbfgs_partial_last_cta(gpu, orc, n):
    _run(gpu, orc, _x0(orc, 997, n, 200 + n), 10, [1, 1, 3, 5])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 32])
def test_batched_lbfgs_batch_of_one(gpu, orc, n):
    _run(gpu, orc, _x0(orc, 1, n, 300 + n), 10, [1, 1, 3, 5])


# B: the history ring wraps around (m + 6 single steps)
@pytest.mark.gpu
@pytest.mark.parametrize("m", [1, 2, 64])
@pytest.mark.parametrize("n", [2, 16])
def test_batched_lbfgs_ring_wraps(gpu, orc, n, m):
    x0 = 25.0 * _x0(orc, 67, n, 400 + n)                      # far out: problems stay live past m + 6 steps
    opt, dev = _run(gpu, orc, x0, m, [1] * (m + 6))
    assert (dev["iteration_count"] > m).any() and (dev["count"] == m).any()


# C: stuck at construction, converging at different steps, and cap-bounded searches inside the same warps as live problems
def _mixed_x0(orc, n):
    batch = 64
    x0 = _x0(orc, batch, n, 500 + n)
    u = 2.0 * orc.pcg_fill(batch * n, 77).reshape(batch, n) - 1.0
    near = np.array([3, 4, 6, 10, 11, 13, 17, 20, 22, 36, 37, 40, 45, 50])
    scales = np.array([1e-15, 1e-12, 1e-9, 1e-6] * 4)[:near.size, None]
    x0[near] = 1.0 + scales * u[near]
    at_min = np.array([0, 5, 33])
    x0[at_min] = 1.0                                          # gradient 0: stuck at construction (:377)
    nan_dir = np.array([7, 38])
    x0[nan_dir] = 1e200                                       # x^2 overflows: gradient +-Inf, direction NaN
    neg_zero = np.array([9, 42])
    x0[neg_zero, 0::2] = -0.0                                 # |g|^2 overflows: direction +-0.0, and +0.0 at the -0.0 coordinates
    x0[neg_zero, 1::2] = 1e156
    return x0, near, at_min, np.concatenate([nan_dir, neg_zero])


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 16])
def test_batched_lbfgs_mixed_states_in_a_warp(gpu, orc, n):
    dz = gpu
    x0, near, at_min, capped = _mixed_x0(orc, n)
    assert np.signbit(x0[capped[2:], 0]).all()
    live = np.setdiff1d(np.arange(x0.shape[0]), capped)
    opt = _make(dz, x0, 5)
    refs = _oracles(orc, x0, 5, live)
    _compare(dz, opt, refs, live, "constructor")
    before = _device_state(dz, opt, capped)
    assert not before["stuck"].any() and np.isinf(before["objective"]).all()
    assert np.isnan(before["direction"][:2]).any()
    active = np.ones(live.size, dtype=bool)
    for i, k in enumerate([1] * 10 + [5] * 6):
        active = _step_all(dz, opt, refs, live, active, k, f"after launch {i}")
        dev = _device_state(dz, opt, live)
        # the cap: point unchanged, delta_point = the point, is_stuck, everything else as before the first step
        cap = _device_state(dz, opt, capped)
        assert cap["stuck"].all()
        assert_bitwise(cap["point"], before["point"], "capped point")
        assert_bitwise(cap["delta_point"], before["point"], "capped delta_point")
        for k2 in ("gradient", "delta_gradient", "direction", "objective", "delta_objective", "rho"):
            assert_bitwise(cap[k2], before[k2], f"capped {k2}")
        assert (cap["iteration_count"] == 0).all() and (cap["count"] == 0).all()
    pos = {p: j for j, p in enumerate(live)}
    stuck_at = dev["iteration_count"][[pos[p] for p in near]][dev["stuck"][[pos[p] for p in near]]]
    assert len(set(stuck_at.tolist())) >= 2, stuck_at               # converged at different steps
    assert dev["stuck"][[pos[p] for p in at_min]].all() and (dev["iteration_count"][[pos[p] for p in at_min]] == 0).all()
    assert (~dev["stuck"]).any()                                    # and live neighbours


# D: step(k) in one launch, and step_async + sync, equal k single steps
@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 1, 7, 25])
def test_batched_lbfgs_k_steps_per_launch(gpu, orc, k):
    dz = gpu
    x0 = _x0(orc, 67, 16, 600)
    one = _make(dz, x0, 5)
    many = _make(dz, x0, 5)
    asy = _make(dz, x0, 5)
    refs = _oracles(orc, x0, 5, range(67))
    idx = np.arange(67)
    active = np.ones(67, dtype=bool)
    for i in range(k):
        active = _step_all(dz, one, refs, idx, active, 1, f"single step {i}")
    many.step(k)
    asy.step_async(k).sync()
    for opt, what in ((many, "step(k)"), (asy, "step_async(k) + sync")):
        dev, ref = _device_state(dz, opt, idx), _device_state(dz, one, idx)
        for key in dev:
            assert np.array_equal(np.asarray(dev[key]).view(np.uint8), np.asarray(ref[key]).view(np.uint8)), f"{what}: {key}"


@pytest.mark.gpu
def test_batched_lbfgs_rho_history_list(gpu, orc):
    x0 = _x0(orc, 37, 6, 700)
    opt, _ = _run(gpu, orc, x0, 3, [1, 1, 1, 1])
    hist = opt.rho_history
    assert isinstance(hist, list) and len(hist) == 37
    for p in (0, 17, 36):
        r = orc.LBFGS(orc.OBJ_ROSENBROCK, x0[p], 1.0, 3, order=orc.SEQ).step(4)
        assert_bitwise(hist[p], r.rho_history, f"rho_history[{p}]")
    assert opt.current_point.shape == (37, 6) and opt.current_objective_value.shape == (37,)


def _sample(batch, count, seed):
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([rng.choice(batch, count - 2, replace=False), [0, batch - 1]]))


# E: bench-sized batch, 1 M problems x n = 16 x m = 10, a seeded sample after steps 1, 5 and 20
@pytest.mark.gpu
def test_batched_lbfgs_one_million(gpu, orc):
    dz = gpu
    batch, n, m = 1_000_000, 16, 10
    x0 = (4.0 * dz.pcg_fill(batch * n, 2024) - 2.0).reshape(batch, n)
    idx = _sample(batch, 4096, 1)
    opt = _make(dz, x0, m)
    refs = _oracles(orc, x0, m, idx)
    _compare(dz, opt, refs, idx, "constructor")
    active = np.ones(idx.size, dtype=bool)
    for k in (1, 4, 15):                     # checked after steps 1, 5 and 20
        active = _step_all(dz, opt, refs, idx, active, k, f"after step({k})")
    assert active.mean() > 0.99


# F: m * n * batch > 2^31 (64-bit indexing of the history): m = 64, n = 32, 1.1 M problems (about 40 GB)
@pytest.mark.gpu
def test_batched_lbfgs_history_beyond_2_pow_31(gpu, orc):
    dz = gpu
    batch, n, m = 1_100_000, 32, 64
    assert m * n * batch > 2 ** 31
    x0 = (4.0 * dz.pcg_fill(batch * n, 9) - 2.0).reshape(batch, n)
    idx = _sample(batch, 2048, 2)
    _run(dz, orc, x0, m, [1, 1, 2], idx=idx)

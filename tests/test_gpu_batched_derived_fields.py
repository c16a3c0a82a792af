"""GPU parity tests of the two layouts of the batched small-n BFGS kernel (Tuning::batched_derived), against the CPU oracle.

batched_derived = 1: a move writes its new point into the other of two point buffers and stores no gradient, delta_point
or delta_gradient; the getters recompute them from the two points (explicit dx / dg after the constructor and set_state).
batched_derived = 0: every field is stored.  Both layouts must give the same bits as the oracle, after every launch:
  - every even n <= 32 under tiles 32 and 27, with k > 1 steps in one launch, problems that terminate beside live ones,
    and a batch resumed through set_state from the getters' own output (the forced-tile run of
    test_gpu_batched_dispatch.py);
  - set_state with delta_point / delta_gradient that are not differences of anything, read back, stepped, read again;
  - a start point whose gradient overflows to +-Inf (the derived delta_gradient would be NaN; the explicit zeros win).
Each test forces the layout it covers through the knob, restores the default, and asserts through
dzo_bfgs_batched_layout that every handle it checks was created with that layout.
"""
import contextlib

import numpy as np
import pytest

from conftest import assert_bitwise
from test_gpu_batched_dispatch import _oracle_trajectory, _run_forced
from test_gpu_bfgs import ROSEN, _compare_state, _sym, _x0

pytestmark = pytest.mark.gpu

LAYOUTS = (0, 1)
DEFAULTS = {"batched_tile": 0, "batched_derived": -1}    # host_common.h, Tuning (-1: derived for n > 8)


@contextlib.contextmanager
def _knobs(dz, **knobs):
    """Knobs for the handles created inside (both are read when a handle is created); the defaults come back whatever
    happens."""
    try:
        for key, value in knobs.items():
            dz.set_tuning(key, value)
        yield
    finally:
        for key in knobs:
            dz.set_tuning(key, DEFAULTS[key])


def _assert_layout(dz, opt, derived):
    import ctypes as C
    lazy, got = C.c_int(-1), C.c_int(-1)
    assert dz.lib().dzo_bfgs_batched_layout(opt._h, C.byref(lazy), C.byref(got)) == 0, dz.lib().dzo_last_error().decode()
    assert (lazy.value, got.value) == (1, derived), "layout of the handle"


@pytest.mark.parametrize("derived", LAYOUTS)
@pytest.mark.parametrize("tile", (32, 27))
@pytest.mark.parametrize("n", range(2, 33, 2))
def test_layout_every_field_every_launch(gpu, orc, n, tile, derived):
    """Every field after 12 single-step launches and one 30-step launch; then the batch is resumed through set_state
    from the getters' output (point, delta_point, delta_gradient) and stepped again."""
    dz = gpu
    EF = dz.ExampleFunctions
    tr = _oracle_trajectory(orc, n)
    tag = f"n={n} tile={tile} derived={derived}"
    with _knobs(dz, batched_tile=tile, batched_derived=derived):
        opt, H = _run_forced(dz, tr, tag, tile=tile)
        _assert_layout(dz, opt, derived)
        b = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, tr.x0, 1.0, batched=True)
        _assert_layout(dz, b, derived)
        b.set_state(opt.current_point, H, opt.delta_point, opt.delta_gradient, opt.last_step_length,
                    opt.last_step_type, opt.iteration_count)
        _compare_state(b, tr.resumed[0], True, f"{tag}: after set_state")
        for i, k in enumerate((1, 1, 6)):
            b.step(k)
            _compare_state(b, tr.resumed[i + 1], True, f"{tag}: resumed launch {i} (k={k})")
        b.close()
        opt.close()


@pytest.mark.parametrize("derived", LAYOUTS)
@pytest.mark.parametrize("n", (2, 16, 32))
def test_set_state_with_arbitrary_deltas(gpu, orc, n, derived):
    """set_state stores the caller's delta_point / delta_gradient as given (random values, not differences of points):
    they read back unchanged, and after one step they are the differences of that step for every problem that moved
    and stay the caller's values for every problem that did not."""
    dz = gpu
    EF = dz.ExampleFunctions
    batch = 300
    x0 = _x0(orc, n * batch, 5100 + n).reshape(batch, n)
    x0[7] = 1.0                                       # at the minimiser: never moves
    dxs = _x0(orc, n * batch, 5200 + n).reshape(batch, n)
    dgs = 1e3 * _x0(orc, n * batch, 5300 + n).reshape(batch, n)
    H = np.stack([_sym(orc, n, 5400 + n + p) for p in range(batch)])
    L = np.full(batch, 0.5)
    ty = np.where(np.arange(batch) % 2, 2, 1).astype(np.int32)
    it = np.arange(batch, dtype=np.int64)
    ref = orc.BFGS(ROSEN, x0, 1.0, order=orc.SEQ, nthreads=8)
    ref.set_state(x0, H, dxs, dgs, L, ty, it)
    with _knobs(dz, batched_derived=derived):
        opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
        try:
            _assert_layout(dz, opt, derived)
            opt.set_state(x0, H, dxs, dgs, L, ty, it)
            assert_bitwise(opt.delta_point, dxs, "delta_point after set_state")
            assert_bitwise(opt.delta_gradient, dgs, "delta_gradient after set_state")
            _compare_state(opt, ref, True, f"n={n} derived={derived}: after set_state")
            opt.step(1)
            ref.step(1)
            _compare_state(opt, ref, True, f"n={n} derived={derived}: after one step")
            assert opt.iteration_count[7] == it[7]
            assert_bitwise(opt.delta_point[7], dxs[7], "unmoved problem keeps the caller's delta_point")
            opt.step(3)
            ref.step(3)
            _compare_state(opt, ref, True, f"n={n} derived={derived}: after 3 more steps in one launch")
        finally:
            opt.close()
            ref.close()


@pytest.mark.parametrize("derived", LAYOUTS)
def test_gradient_overflow_at_construction(gpu, orc, derived):
    """x0 whose gradient overflows to +-Inf (objective +Inf): the constructor's delta_gradient is
    zero (the derived difference would be Inf - Inf = NaN), before and after steps that terminate those problems while
    their neighbours keep moving."""
    dz = gpu
    EF = dz.ExampleFunctions
    n, batch = 16, 200
    x0 = _x0(orc, n * batch, 5500).reshape(batch, n)
    x0[3, 0] = 1e103                                  # 400 * x * (y - x^2) overflows
    x0[5, 1] = -1e307                                 # 200 * (y - x^2) overflows
    x0[9] = 1e200
    ref = orc.BFGS(ROSEN, x0, 1.0, order=orc.SEQ, nthreads=8)
    assert not np.isfinite(ref.gradient[[3, 5, 9]]).all()
    with _knobs(dz, batched_derived=derived):
        opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
        try:
            _assert_layout(dz, opt, derived)
            _compare_state(opt, ref, True, f"derived={derived}: after construction")
            assert (opt.delta_gradient[[3, 5, 9]] == 0).all()
            for i in range(3):
                dz.step_(opt)
                ref.step(1)
                _compare_state(opt, ref, True, f"derived={derived}: step {i}")
            opt.step(5)
            ref.step(5)
            _compare_state(opt, ref, True, f"derived={derived}: after 5 steps in one launch")
            assert opt.has_converged[9]
        finally:
            opt.close()
            ref.close()


def test_terminated_problems_keep_their_last_deltas(gpu, orc):
    """Problems that terminate after moving, inside a launch of many steps, while neighbours keep moving: their deltas
    stay those of their last move in both layouts (the points of that move stay in the two buffers)."""
    dz = gpu
    tr = _oracle_trajectory(orc, 16)
    last = tr.snaps[-1]
    moved_then_done = last.terminated & (last.iteration_count > 0)
    assert moved_then_done.sum() > 0 and (~last.terminated).sum() > 0
    assert np.abs(last.delta_point[moved_then_done]).sum() > 0
    for derived in LAYOUTS:
        with _knobs(dz, batched_tile=32, batched_derived=derived):
            opt, _ = _run_forced(dz, tr, f"derived={derived}")
            _assert_layout(dz, opt, derived)
            assert_bitwise(opt.delta_point[moved_then_done], last.delta_point[moved_then_done], "delta_point")
            assert_bitwise(opt.delta_gradient[moved_then_done], last.delta_gradient[moved_then_done], "delta_gradient")
            opt.close()


@pytest.mark.parametrize("n", (2, 8, 10, 16, 32))
def test_default_layout_and_status_of_other_handles(gpu, orc, n):
    """By default the derived layout is taken for n > 8 and the stored one for n <= 8; dzo_bfgs_batched_layout answers
    for handles of the small-n step kernel only."""
    dz = gpu
    EF = dz.ExampleFunctions
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, _x0(orc, 4 * n, 5600).reshape(4, n), 1.0,
                           batched=True)
    _assert_layout(dz, opt, int(n > 8))
    opt.close()
    big = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, _x0(orc, 64, 5601), 1.0)
    assert dz.lib().dzo_bfgs_batched_layout(big._h, None, None) == -5     # DZO_ERR_UNSUPPORTED: the large-n path
    big.close()

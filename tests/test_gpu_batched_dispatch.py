"""GPU parity tests of the batched BFGS kernels in every variant the dispatcher can pick, against the CPU oracle.

A batched handle picks its kernel variant when it is created: the problems per warp ("tile") of the small-n kernel
(batched_hybrid.cuh) from the batch size and the SM count, and the n^2 sweeps of a medium-n batch from n and the batch
size.  The batches of test_gpu_bfgs.py are small enough that the small-n kernel gets one problem per warp, so here
  A  every tile size is forced through the batched_tile knob at every even n <= 32, on a batch with partial tiles and
     terminated problems beside live ones;
  B  the knobs that only change scheduling (prefetch distance, implicit identities) run under the full and a partial tile;
  C  the automatic tile policy is run at the batch sizes where it picks the full 32-problem tile and 27, and on the
     1 M-problem batch of bench.py;
  D  medium-n batches run on the one-warp-per-problem sweeps and on the tiled sweeps with 128 threads per CTA.
Every field is compared bit for bit, and every test asserts the variant it covers, so that a change of a dispatch
policy cannot quietly turn it into a test of another variant.
"""
import contextlib
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import assert_bitwise
from test_gpu_bfgs import FIELDS, ROSEN, _compare_state, _oracle_kinds, _x0

pytestmark = pytest.mark.gpu

KINDS = ("bfgs_read_h", "bfgs_identity_h", "gradient_descent", "terminate")
DEFAULTS = {"batched_tile": 0, "batched_prefetch": 3, "batched_lazy": 1, "small_sweeps": 1}   # host_common.h, Tuning


@contextlib.contextmanager
def _tuning(dz, **knobs):
    """Knobs for the handles created and stepped inside (the tile and lazy knobs are read when a handle is created, the
    prefetch distance at every launch); the defaults come back whatever happens."""
    try:
        for key, value in knobs.items():
            dz.set_tuning(key, value)
        yield
    finally:
        for key in knobs:
            dz.set_tuning(key, DEFAULTS[key])


def _snap(ref):
    """the oracle's fields at one point of its trajectory, readable by _compare_state like the oracle handle itself"""
    return SimpleNamespace(**{k: getattr(ref, k) for k in FIELDS + ("step_type", "iteration_count", "terminated")})


def _replay(ref, k):
    """k single oracle steps, the model of ONE device launch of k steps: (which problems had terminated before each step,
    shape (k, batch); the step kinds of _oracle_kinds summed over the k steps)"""
    done, total = [], dict.fromkeys(KINDS + ("idle",), 0)
    for _ in range(k):
        done.append(ref.terminated)
        for key, v in _oracle_kinds(ref, 1)[0].items():
            total[key] += v
    return np.stack(done), total


def _idle_split(done, tile):
    """(idle, idle_warp) as the batched kernel counts them in one launch with `tile` problems per warp: a warp whose
    problems have all terminated leaves the launch and counts them as idle_warp for every remaining step; terminated
    problems of any other warp count as idle.  Which problems share a warp depends on the tile alone, so the split
    pins the tile the kernel ran with."""
    k, batch = done.shape
    pad = -batch % tile
    d = np.concatenate([done, np.ones((k, pad), dtype=bool)], axis=1).reshape(k, -1, tile)
    size = np.full(d.shape[1], tile)
    size[-1] -= pad
    count = d.sum(axis=2)
    count[:, -1] -= pad
    whole = d.all(axis=2)           # a problem never leaves the terminated state, so neither does a whole tile
    return int(count[~whole].sum()), int((whole * size).sum())


def _expected_counts(launches, tile):
    want = dict.fromkeys(KINDS + ("idle", "idle_warp"), 0)
    for done, kinds in launches:
        for key in KINDS:
            want[key] += kinds[key]
        idle, idle_warp = _idle_split(done, tile)
        want["idle"] += idle
        want["idle_warp"] += idle_warp
    return want


def _all_h(opt, batch):
    return np.stack([opt.inverse_hessian(p) for p in range(batch)])


# ----------------------------------------------------------------------------- A, B: forced tiles
BATCH_A = 997                        # prime: the last warp's tile and the last 4-warp CTA are partial for every tile size
TILES = (32, 31, 27, 16, 5, 2, 1)
IDLE_BLOCK = slice(64, 128)          # problems at the minimiser: whole warps of every tile size <= 32 go idle
SINGLE_A, FUSED_A, RESUME_A = 12, 30, (1, 1, 6)


def _mixed_x0(orc, n, batch, seed):
    """PCG start points with problems that terminate at their first step sitting in tiles beside live ones: at the
    minimiser (zero gradient, no probe), at 1e200 (objective +Inf; also the last problem, in the last partial tile),
    and rows of the special values of test_batched_awkward_inputs (signed zeros, tiny and huge coordinates)."""
    x0 = _x0(orc, n * batch, seed).reshape(batch, n)
    x0[IDLE_BLOCK] = 1.0
    x0[3] = 1.0
    x0[30] = 1e200
    x0[batch - 1] = 1e200
    special = np.array([0.0, -0.0, 1.0, -1.0, 1e-8, -1e-8, 1e6, -1e6, 1e-160, 1e150])
    pick = (orc.pcg_fill(8 * n, seed + 1) * 14).astype(int).reshape(8, n)
    x0[40:48] = np.where(pick < 10, special[np.minimum(pick, 9)], x0[40:48])
    return x0


_trajectory = {}


def _oracle_trajectory(orc, n):
    """The oracle's run of the forced-tile batch at this n, computed once per n (the tests are ordered n-major): the
    fields after every launch, the launches themselves (for the step-kind counters), every final inverse Hessian, and
    a run resumed through set_state from the final fields."""
    if n not in _trajectory:
        _trajectory.clear()
        x0 = _mixed_x0(orc, n, BATCH_A, 3300 + n)
        ref = orc.BFGS(ROSEN, x0, 1.0, order=orc.SEQ, nthreads=8)
        launches, snaps = [], []
        for k in (1,) * SINGLE_A + (FUSED_A,):
            launches.append(_replay(ref, k))
            snaps.append(_snap(ref))
        H = _all_h(ref, BATCH_A)
        rb = orc.BFGS(ROSEN, x0, 1.0, order=orc.SEQ, nthreads=8)
        rb.set_state(ref.point, H, ref.delta_point, ref.delta_gradient, ref.step_length, ref.step_type, ref.iteration_count)
        resumed = [_snap(rb)]
        for k in RESUME_A:
            rb.step(k)
            resumed.append(_snap(rb))
        _trajectory[n] = SimpleNamespace(x0=x0, launches=launches, snaps=snaps, H=H, resumed=resumed)
    return _trajectory[n]


def _run_forced(dz, tr, tag, tile=None, mirrors=False):
    """Steps a new handle through the trajectory: every field after each launch, every inverse Hessian at the end.
    With `tile`, the step-kind counters after each launch as well (their idle / idle_warp split witnesses the tile)."""
    EF = dz.ExampleFunctions
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, tr.x0, 1.0, batched=True)
    if mirrors:
        opt.reuse_host_buffers(True)
        assert opt._mirrored
    f_copy, t_copy = np.empty(BATCH_A), np.empty(BATCH_A, dtype=np.uint8)
    for i, ((done, _), want) in enumerate(zip(tr.launches, tr.snaps)):
        k = done.shape[0]
        if k == 1:
            dz.step_(opt)
        else:
            opt.step(k)                 # k steps in one launch: phase 1 restages the tile from phase 2's stores
        _compare_state(opt, want, True, f"{tag} launch {i} (k={k})")
        if tile is not None:
            assert opt.step_kind_counts() == _expected_counts(tr.launches[:i + 1], tile), f"{tag} launch {i}: step kinds"
        if mirrors:                     # the step kernel's zero-copy stores vs ordinary copies of the device fields
            f_mirror, t_mirror = opt.current_objective_value, opt.has_converged
            assert dz.lib().dzo_bfgs_get_objective(opt._h, f_copy.ctypes.data_as(dz._capi.c_double_p)) == 0
            assert dz.lib().dzo_bfgs_get_terminated(opt._h, t_copy.ctypes.data_as(dz._capi.c_u8_p)) == 0
            assert_bitwise(f_mirror, f_copy, f"{tag} launch {i}: mirrored objective")
            assert np.array_equal(t_mirror.view(np.uint8), t_copy), f"{tag} launch {i}: mirrored has_terminated"
    H = _all_h(opt, BATCH_A)
    assert_bitwise(H, tr.H, f"{tag}: inverse Hessians")
    return opt, H


@pytest.mark.parametrize("tile", TILES)
@pytest.mark.parametrize("n", range(2, 33, 2))
def test_forced_tile(gpu, orc, n, tile):
    """bfgs_batched_hybrid_kernel with `tile` problems per warp: the fixed full tile (<N, false>, the instantiation behind
    large batches and bench.py) and run-time tiles (<N, true>), with partial tiles, lanes past the tile, phase-2 rounds
    that mix live and terminated problems, warps that go idle, and k steps in one launch.  Tiles 32 and 27 also run
    with the zero-copy field mirrors and resume the whole batch through set_state."""
    dz = gpu
    EF = dz.ExampleFunctions
    tr = _oracle_trajectory(orc, n)
    want = _expected_counts(tr.launches, tile)
    assert want["bfgs_read_h"] > 0 and want["bfgs_identity_h"] > 0 and want["gradient_descent"] > 0
    assert want["terminate"] > 0 and want["idle_warp"] > 0 and (want["idle"] > 0 or tile == 1)   # tiles mixing both
    extra = tile in (32, 27)
    with _tuning(dz, batched_tile=tile):
        opt, H = _run_forced(dz, tr, f"n={n} tile={tile}", tile=tile, mirrors=extra)
        if extra:
            b = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, tr.x0, 1.0, batched=True)
            b.set_state(opt.current_point, H, opt.delta_point, opt.delta_gradient, opt.last_step_length,
                        opt.last_step_type, opt.iteration_count)
            _compare_state(b, tr.resumed[0], True, f"n={n} tile={tile}: after set_state")
            for i, k in enumerate(RESUME_A):
                b.step(k)
                _compare_state(b, tr.resumed[i + 1], True, f"n={n} tile={tile}: resumed launch {i} (k={k})")
            b.close()
        opt.close()


@pytest.mark.parametrize("tile", (32, 27))
@pytest.mark.parametrize("n", (2, 6, 14, 4, 16, 32))
def test_tile_scheduling_knobs_change_no_bit(gpu, orc, n, tile):
    """The L2 prefetch distance (0 = none) and the implicit identities (batched_lazy = 0: H = I is written to HBM) only
    change scheduling and traffic.  n = 2, 6, 14: a problem's inverse Hessian straddles 128-byte lines (the line-wise
    prefetch of a whole round); n = 4, 16, 32: it fills whole lines (the prefetch of live problems only)."""
    dz = gpu
    tr = _oracle_trajectory(orc, n)
    for prefetch in (0, 3, 5):
        for lazy in (0, 1):
            with _tuning(dz, batched_tile=tile, batched_prefetch=prefetch, batched_lazy=lazy):
                opt, _ = _run_forced(dz, tr, f"n={n} tile={tile} prefetch={prefetch} lazy={lazy}",
                                     tile=tile if lazy else None)
                opt.close()


# ----------------------------------------------------------------------------- C: the automatic tile policy
def _policy_tile(n, batch, sms):
    """Problems per warp the batched kernel gets by default; mirrors the batched_tile == 0 branch of create_common
    (csrc/dzopt_bfgs.cu): a batch that fills the resident warps at most three times over is spread evenly over that
    many full waves, a larger one gets full 32-problem tiles."""
    slots = sms * (16 if n <= 16 else 8)           # hybrid_warps_per_sm (batched_hybrid.cuh)
    waves = -(-(-(-batch // 32)) // slots)
    if waves > 3:
        return 32
    return min(32, max(1, -(-batch // (waves * slots))))


AUTO = {   # case: (n, batch from the resident warp slots of the GPU, the tile it is meant to cover)
    "n16_first_full_tiles": (16, lambda slots: 96 * slots + 37, 32),
    "n32_first_full_tiles": (32, lambda slots: 96 * slots + 37, 32),
    "n16_tile27": (16, lambda slots: 26 * slots + slots // 2, 27),
    "n16_bench_1M": (16, lambda slots: 1_000_000, 32),
}


@pytest.mark.parametrize("case", list(AUTO))
def test_automatic_tile(gpu, orc, case):
    """The tile create_common picks at the batch sizes users run: just above the switch to full tiles (n = 16 and 32:
    one warp per 32 problems, the <N, false> kernel), about 62.5 k problems at n = 16 (27 per warp), and bench.py's
    1 M problems of n = 16 (its PCG seed 2024; 64 of them moved to the minimiser so that whole warps go idle and the
    device's idle_warp counter shows the tile)."""
    import torch
    dz = gpu
    EF = dz.ExampleFunctions
    n, batch_of, tile = AUTO[case]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    batch = batch_of(sms * (16 if n <= 16 else 8))
    assert _policy_tile(n, batch, sms) == tile
    x0 = _x0(orc, n * batch, 2024).reshape(batch, n)
    x0[IDLE_BLOCK] = 1.0
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
    ref = orc.BFGS(ROSEN, x0, 1.0, order=orc.SEQ, nthreads=8)
    del x0
    try:
        launches = []
        for it in range(3):
            dz.step_(opt)
            launches.append(_replay(ref, 1))
            _compare_state(opt, ref, True, f"{case} (batch {batch}) iter {it}")
        opt.step(10)
        launches.append(_replay(ref, 10))
        _compare_state(opt, ref, True, f"{case} (batch {batch}) after 10 steps in one launch")
        want = _expected_counts(launches, tile)
        assert want["idle_warp"] > 0 and want["gradient_descent"] > 0
        assert opt.step_kind_counts() == want, "step kinds"
        for p in np.unique(np.linspace(0, batch - 1, 2000).astype(np.int64)):
            assert_bitwise(opt.inverse_hessian(p), ref.inverse_hessian(p), f"{case}: H[{p}]")
    finally:
        opt.close()
        ref.close()


# ----------------------------------------------------------------------------- D: medium-n batches
def _small_sweeps_run(n, batch, knob):
    """whether the n^2 sweeps of a batch run on one warp per problem (small_sweeps.cuh); mirrors large_step_once in
    csrc/dzopt_bfgs.cu (with the O(n) stage on one warp per problem too, the default for n <= 512)"""
    return bool(knob) and batch > 1 and n <= 64


def _sweep_threads(n, batch):
    """threads per CTA of the tiled n^2 sweeps; mirrors sweep_threads in csrc/dzopt_bfgs.cu (kSweepThreads = 128,
    DZO_GEMV_CHUNK = 1024 columns, 4 tiles per SM of a 148-SM GPU)"""
    nchunks = -(-n // 1024)
    t = 128
    while t > 64 and -(-n // (2 * t)) * nchunks * batch < 4 * 148:
        t //= 2
    while t > 64 and t > n:
        t //= 2
    return t


def _medium_x0(orc, n, batch):
    x0 = _x0(orc, n * batch, 4400 + n).reshape(batch, n)
    x0[1] = 1.0                       # at the minimiser: terminates at the first step
    x0[batch - 1] = 1e200             # objective +Inf: terminates at the first step
    return x0


def _medium_run(dz, orc, n, batch, steps, fused, h_problems, tag):
    EF = dz.ExampleFunctions
    x0 = _medium_x0(orc, n, batch)
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
    ref = orc.BFGS(ROSEN, x0, 1.0, order=orc.TREE, nthreads=8)
    try:
        assert opt.summation_order == orc.TREE
        kinds = set()
        for it in range(steps):
            before = opt.iteration_count
            dz.step_(opt)
            ref.step(1)
            _compare_state(opt, ref, True, f"{tag} iter {it}")
            kinds |= set(opt.last_step_type[opt.iteration_count > before].tolist())
        if fused:
            opt.step(fused)
            ref.step(fused)
            _compare_state(opt, ref, True, f"{tag} after {fused} steps in one call")
        # a GD-type step makes the update sweep write identity_matrix! (:981), a BFGS-type step the rank-2 update
        assert {dz.StepType.BFGSStep, dz.StepType.GradientDescentStep} <= kinds
        assert opt.has_converged[1] and opt.has_converged[batch - 1] and opt.count_active() == ref.count_active()
        for p in h_problems:
            assert_bitwise(opt.inverse_hessian(p), ref.inverse_hessian(p), f"{tag}: H[{p}]")
    finally:
        opt.close()
        ref.close()


@pytest.mark.parametrize("n,batch,small_sweeps,warp_sweeps",
                         [(n, b, s, s == 1) for n in (34, 40, 62, 64) for b in (37, 517) for s in (1, 0)] +
                         [(66, 37, 1, False), (66, 517, 1, False)])
def test_medium_n_small_sweeps(gpu, orc, n, batch, small_sweeps, warp_sweeps):
    """Batches of 32 < n <= 64 on the one-warp-per-problem sweeps (small_sweeps = 1) and on the tiled sweeps
    (small_sweeps = 0); n = 66 is the first size past the switch.  The batches are not multiples of the 4 problems
    of a CTA."""
    dz = gpu
    assert _small_sweeps_run(n, batch, small_sweeps) == warp_sweeps
    with _tuning(dz, small_sweeps=small_sweeps):
        _medium_run(dz, orc, n, batch, 10, 10, range(batch), f"n={n} batch={batch} small_sweeps={small_sweeps}")


@pytest.mark.parametrize("n,batch", [(130, 600), (1026, 300), (2050, 40)])
def test_medium_n_128_thread_sweeps(gpu, orc, n, batch):
    """Batches that give the tiled n^2 sweeps 128 threads per CTA, with blockIdx.z > 0 serving the later problems:
    n = 130 (O(n) stage on one warp per problem), 1026 (two column chunks) and 2050 (three, the last 2 columns wide;
    O(n) stage on one 1024-thread CTA per problem)."""
    dz = gpu
    assert _sweep_threads(n, batch) == 128
    _medium_run(dz, orc, n, batch, 8, 0, (0, batch // 2, batch - 1), f"n={n} batch={batch}")

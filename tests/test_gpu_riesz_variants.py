"""GPU parity tests of the cooperative Riesz kernel (riesz_gd_kernel<DIM, NT>, csrc/gd_kernels.cuh) in every dimension,
CTA size and variant, against the CPU oracle.

The kernel runs the GradientDescentOptimizer step! (modes 0 and 1), the search stage of a BFGSOptimizer step! (modes 5
and 6) and the kernel-level objective, gradient and line search (modes 2-4).  Its variant is picked when a handle is
created, from the tuning knobs riesz_threads, riesz_esplit, riesz_gvariant, riesz_pair and riesz_bar, none of which may
change a bit of the results.  Here
  A  every variant runs a GD trace in dims 1-4, on the shapes where the work split changes: partial row blocks, one-source
     segments, rows that wrap the 4096-wide canonical tree, more items than the grid has warps, and clouds that run away
     (non-finite values inside the search, termination inside a k-step launch);
  B  bench.py's Riesz configuration runs its 3 + 20 steps under the default and three other variants;
  C  the search's edge branches: a start step so small that the point does not move, clouds whose pair distances
     straddle the range of the fast sqrt / reciprocal paths, and a capped bracket that leaves the speculative probe unused;
  D  runs to termination inside 64-step launches, and starts with a coincident pair (terminated at construction);
  E  BFGSOptimizer with the Riesz objective, odd n included (the scalar fallbacks of the n^2 sweeps, the partial last
     pair of cluster_delta_kernel), with cluster and single-CTA delta kernels.
Every field is compared bit for bit after every launch (NaN payloads aside where a trajectory produces NaN), and every
test asserts through dzo_gd_riesz_info which variant it ran, so that a change of the dispatch cannot quietly turn it into
a test of another variant.
"""
import contextlib
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from conftest import assert_bitwise
from test_gpu_gd import GD_FIELDS, NONE, RIESZ, SPHERE, TREE, _compare_gd, line_points, sphere_points

pytestmark = pytest.mark.gpu

DEFAULTS = {"riesz_threads": 512, "riesz_esplit": 1, "riesz_gvariant": 0, "riesz_pair": 1, "riesz_bar": 0,
            "search_variant": 0}   # host_common.h, Tuning

# name: (knobs, (threads per CTA, lanes per energy row, paired probes, gradient tiles, flag barrier))
VARIANTS = {
    "default": ({}, (512, 1, 1, 0, 0)),
    "single_probe": ({"riesz_pair": 0}, (512, 1, 0, 0, 0)),
    "esplit2": ({"riesz_esplit": 2}, (512, 2, 0, 0, 0)),           # two lanes per row turn pairing off
    "t1024": ({"riesz_threads": 1024}, (1024, 1, 1, 0, 0)),
    "t1024_single": ({"riesz_threads": 1024, "riesz_pair": 0}, (1024, 1, 0, 0, 0)),
    "tiles": ({"riesz_gvariant": 1}, (1024, 1, 1, 1, 0)),          # the tile gradient is written for 32 warps
    "tiles_esplit2": ({"riesz_gvariant": 1, "riesz_esplit": 2}, (1024, 2, 0, 1, 0)),
    "bar": ({"riesz_bar": 1}, (512, 1, 1, 0, 1)),
    "bar_t1024_single": ({"riesz_bar": 1, "riesz_threads": 1024, "riesz_pair": 0}, (1024, 1, 0, 0, 1)),
}
SEG = 128                                    # DZO_RIESZ_SEG: sources per segment


@contextlib.contextmanager
def _tuning(dz, **knobs):
    """Knobs for the handles created and stepped inside; the defaults come back whatever happens."""
    try:
        for key, value in knobs.items():
            dz.set_tuning(key, value)
        yield
    finally:
        for key in knobs:
            dz.set_tuning(key, DEFAULTS[key])


def _riesz_info(dz, opt):
    v = [C.c_int(-1) for _ in range(6)]
    assert dz.lib().dzo_gd_riesz_info(opt._h, *[C.byref(x) for x in v]) == 0, dz.lib().dzo_last_error().decode()
    threads, ctas, lanes, paired, tiles, bar = (x.value for x in v)
    return (threads, lanes, paired, tiles, bar), ctas


def _assert_variant(dz, opt, variant):
    import torch
    got, ctas = _riesz_info(dz, opt)
    assert got == VARIANTS[variant][1], f"{variant}: the handle runs (threads, lanes, paired, tiles, bar) = {got}"
    assert ctas == torch.cuda.get_device_properties(0).multi_processor_count


def _energy_items(N, rows):
    """(row block, segment) energy items with at least one pair i < j; mirrors energy_items in csrc/dzopt_gd.cu"""
    count = 0
    for rb in range(-(-N // rows)):
        jmax = min(N, rb * rows + rows) - 1
        count += -(-jmax // SEG)
    return count


def _gradient_items(N):
    """(32 rows x 128 sources) gradient items of gradient_segments: every row block against every segment"""
    return -(-N // 32) * -(-N // SEG)


def _constraint(dz, constraint):
    return dz.SPHERE_CONSTRAINT if constraint == SPHERE else dz.NULL_CONSTRAINT


def _start(orc, dim, N, seed, scale=1.0):
    """dim 1: distinct points on a line; dims 2-4: points on the unit sphere; times `scale`"""
    x = line_points(orc, N, seed) if dim == 1 else sphere_points(orc, N, dim, seed)
    return x * scale


def _snap(ref, fields):
    return SimpleNamespace(**{k: getattr(ref, k) for k in fields})


GD_SNAP = GD_FIELDS + ("iteration_count", "terminated")
BFGS_FIELDS = ("point", "gradient", "delta_point", "delta_gradient", "direction", "objective", "step_length")
BFGS_SNAP = BFGS_FIELDS + ("step_type", "iteration_count", "terminated")

_trajectory = {}


def _cached(key, build):
    """one oracle trajectory at a time: the tests of a section are ordered case-major, every variant of a case in a row"""
    if key not in _trajectory:
        _trajectory.clear()
        _trajectory[key] = build()
    return _trajectory[key]


def _gd_trajectory(orc, x, L0, constraint, dim, launches, max_increases=0):
    """the oracle's fields at construction and after each launch of `launches` steps"""
    ref = orc.GD(RIESZ, x.reshape(1, -1), L0, order=orc.TREE, constraint=constraint, dim=dim, max_increases=max_increases)
    snaps = [_snap(ref, GD_SNAP)]
    for k in launches:
        ref.step(k)
        snaps.append(_snap(ref, GD_SNAP))
    ref.close()
    return SimpleNamespace(x=x, L0=L0, constraint=constraint, dim=dim, launches=launches, snaps=snaps,
                           max_increases=max_increases, evals=None)


def _run_gd(dz, tr, variant, tag, nan_canon=False):
    """a new handle under the variant's knobs through the trajectory's launches, every field after each; the evaluation
    count must be the same for every variant (a variant may change scheduling, never the probes the search consumes)"""
    EF = dz.ExampleFunctions
    with _tuning(dz, **VARIANTS[variant][0]):
        opt = dz.GradientDescentOptimizer(_constraint(dz, tr.constraint), EF.riesz_energy, EF.riesz_gradient_,
                                          dz.QuadraticLineSearch(tr.max_increases), tr.x, tr.L0)
        try:
            _assert_variant(dz, opt, variant)
            _compare_gd(opt, tr.snaps[0], f"{tag}: ctor", nan_canon)
            for i, k in enumerate(tr.launches):
                if k == 1:
                    dz.step_(opt)
                else:
                    opt.step(k)
                _compare_gd(opt, tr.snaps[i + 1], f"{tag}: launch {i} (k={k})", nan_canon)
            evals = opt.evaluation_count()
        finally:
            opt.close()
    if tr.evals is None:
        tr.evals = evals
    assert evals == tr.evals, f"{tag}: {evals} objective evaluations, {tr.evals} under the first variant run"


# ----------------------------------------------------------------------------- A: GD traces, every shape x every variant
SHAPES_A = {   # name: (dim, N, constraint, scale, runs away)
    "d1_N33": (1, 33, NONE, 1.0, False),          # first cooperative size: the second row block has one row
    "d1_N129": (1, 129, NONE, 1.0, False),        # the last segment has one source
    "d1_N4097": (1, 4097, NONE, 1.0, False),      # rows wrap the canonical tree
    "d2_N17": (2, 17, SPHERE, 1.0, False),        # one partial row block, one segment
    "d2_N257": (2, 257, SPHERE, 1.0, False),      # one-source segment; 257 mod 16 = 1 for two lanes per row
    "d2_N257_runaway": (2, 257, NONE, 1.3, True),
    "d3_N11": (3, 11, SPHERE, 1.0, False),        # n = 33
    "d3_N129": (3, 129, SPHERE, 1.0, False),
    "d3_N700": (3, 700, SPHERE, 1.0, False),
    "d3_N6200": (3, 6200, SPHERE, 1.0, False),    # every variant's items outnumber the grid's warps
    "d4_N9": (4, 9, SPHERE, 1.0, False),          # n = 36
    "d4_N31": (4, 31, SPHERE, 1.0, False),        # N < 32: a single partial row block
    "d4_N160_runaway": (4, 160, NONE, 1.3, True),
    "d4_N513": (4, 513, SPHERE, 1.0, False),
}
SINGLE_A, FUSED_A = 6, 8


def _trajectory_a(orc, shape):
    dim, N, constraint, scale, runaway = SHAPES_A[shape]

    def build():
        # the runaway clouds terminate inside the first launch; single step! calls then must change nothing
        launches = (FUSED_A,) + (1,) * SINGLE_A if runaway else (1,) * SINGLE_A + (FUSED_A,)
        x = _start(orc, dim, N, 5 if runaway else 41, scale)
        tr = _gd_trajectory(orc, x, 1e-3, constraint, dim, launches)
        flat = x.reshape(1, -1)
        tr.f0 = orc.objective(RIESZ, flat, orc.TREE, constraint, dim)
        tr.g0 = orc.gradient(RIESZ, flat, orc.TREE, constraint, dim)
        return tr

    return _cached(("A", shape), build)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("shape", list(SHAPES_A))
def test_gd_trace_every_variant(gpu, orc, shape, variant):
    """6 single step! calls and one launch of 8 steps (the runaway clouds: the launch first), then the kernel-level
    objective and gradient (modes 2 and 3) of the start point under the same knobs."""
    import dev
    import torch
    dz = gpu
    dim, N, constraint, _, runaway = SHAPES_A[shape]
    assert dim * N > 32                              # n <= 32 runs on the one-thread-per-problem kernel
    tr = _trajectory_a(orc, shape)
    last = tr.snaps[-1]
    assert int(last.iteration_count[0]) > 0
    if runaway:
        fused = tr.snaps[1]
        assert fused.terminated[0] and 0 < int(fused.iteration_count[0]) < FUSED_A
        assert int(last.iteration_count[0]) == int(fused.iteration_count[0])
    else:
        assert not tr.snaps[SINGLE_A].terminated[0]
        assert int(last.iteration_count[0]) > SINGLE_A
    if N == 6200:
        warps = torch.cuda.get_device_properties(0).multi_processor_count * (1024 // 32)
        assert min(_energy_items(N, 32), _energy_items(N, 16), _gradient_items(N)) > warps
    _run_gd(dz, tr, variant, f"{shape} {variant}", nan_canon=runaway)
    with _tuning(dz, **VARIANTS[variant][0]):
        flat = tr.x.reshape(1, -1)
        assert_bitwise(dev.objective(RIESZ, flat, TREE, constraint, dim), tr.f0, f"{shape} {variant}: objective")
        assert_bitwise(dev.gradient(RIESZ, flat, TREE, constraint, dim), tr.g0, f"{shape} {variant}: gradient")


def test_energy_item_counts_of_the_wrapping_shape():
    """the mirror of energy_items against the item counts of N = 6200 and bench.py's N = 4096"""
    assert (_energy_items(6200, 32), _energy_items(6200, 16), _gradient_items(6200)) == (4802, 9604, 9506)
    assert (_energy_items(4096, 32), _gradient_items(4096)) == (2112, 4096)


# ----------------------------------------------------------------------------- B: bench.py's configuration
@pytest.mark.parametrize("variant", ["default", "single_probe", "t1024", "bar"])
def test_bench_configuration(gpu, orc, variant):
    """bench_riesz: N = 4096 points of PCG seed 3 on the sphere, L0 = 1e-3, step(3) and then 20 steps in one launch."""
    dz = gpu
    EF = dz.ExampleFunctions
    N = 4096
    assert_bitwise(dz.pcg_fill(3 * N, 3), orc.pcg_fill(3 * N, 3), "pcg_fill")
    tr = _cached(("B",), lambda: _gd_trajectory(orc, sphere_points(orc, N, 3, 3), 1e-3, SPHERE, 3, (3, 20)))
    assert int(tr.snaps[-1].iteration_count[0]) == 23 and not tr.snaps[-1].terminated[0]
    with _tuning(dz, **VARIANTS[variant][0]):
        opt = dz.GradientDescentOptimizer(dz.SPHERE_CONSTRAINT, EF.riesz_energy, EF.riesz_gradient_,
                                          dz.QuadraticLineSearch(0), tr.x, 1e-3)
        try:
            _assert_variant(dz, opt, variant)
            _compare_gd(opt, tr.snaps[0], f"bench {variant}: ctor")
            opt.step(3)
            _compare_gd(opt, tr.snaps[1], f"bench {variant}: step(3)")
            opt.step_async(20)
            opt.sync()
            _compare_gd(opt, tr.snaps[2], f"bench {variant}: 20 steps in one launch")
            assert int(opt.iteration_count[()]) == 23
            evals = opt.evaluation_count()
        finally:
            opt.close()
    if tr.evals is None:
        tr.evals = evals
    assert evals == tr.evals


# ----------------------------------------------------------------------------- C: the search's edge branches
def _cloud(orc, dim, side):
    """clouds whose squared pair distances straddle the fast-path range [2^-500, 2^500) of ieee_fast.cuh.  The tiny dim-1
    cloud is a jittered lattice: with random points on a line the closest pair makes |g|^2 overflow, the direction 0
    and the first step! terminate without a probe."""
    if side == "tiny":
        if dim == 1:
            h = 5e-77
            return ((np.arange(40) + 0.3 * orc.pcg_fill(40, 23)) * h).reshape(40, 1), h
        return sphere_points(orc, 40, dim, 23) * 3e-76, 3e-76
    return _start(orc, dim, 40, 23, 1e76), 1e76


CASES_C = ("tiny_L0", "tiny_cloud", "huge_cloud", "max_increases_2")
LAUNCHES_C = (1, 1, 1, 1, 6)


def _trajectory_c(orc, case, dim):
    def build():
        constraint = NONE if dim == 1 else SPHERE
        mi = 0
        if case == "tiny_L0":              # x + t*d == x at t = 1: the doubling loop and the `small` branch (:91-123)
            x, L0 = _start(orc, dim, 300 if dim == 1 else 200, 23), 1e-300
        elif case == "max_increases_2":    # expanding searches stop after two doublings, before the paired probe is used
            x, L0, mi = _start(orc, dim, 300 if dim == 1 else 200, 23), 1e-9, 2
        else:
            x, scale = _cloud(orc, dim, case.split("_")[0])
            L0, constraint = 1e-3 * scale, NONE
        return _gd_trajectory(orc, x, L0, constraint, dim, LAUNCHES_C, max_increases=mi)

    return _cached(("C", case, dim), build)


@pytest.mark.parametrize("variant", ["default", "esplit2", "tiles"])
@pytest.mark.parametrize("dim", [1, 3])
@pytest.mark.parametrize("case", CASES_C)
def test_search_edge_branches(gpu, orc, case, dim, variant):
    tr = _trajectory_c(orc, case, dim)
    assert int(tr.snaps[-1].iteration_count[0]) >= 1
    if case.endswith("cloud"):
        x = tr.x
        d2 = ((x[:, None, :] - x[None, :, :]) ** 2).sum(axis=-1)[np.triu_indices(len(x), 1)]
        fast = (d2 >= 2.0 ** -500) & (d2 < 2.0 ** 500)
        assert fast.any() and not fast.all(), "the start's pair distances straddle the fast-path range"
    if case == "tiny_L0":
        x = tr.x.reshape(-1)
        assert np.array_equal(x + tr.snaps[0].direction[0], x), "the first trial step leaves the point unchanged"
    _run_gd(gpu, tr, variant, f"{case} dim {dim} {variant}", nan_canon=case.endswith("cloud"))


# ----------------------------------------------------------------------------- D: termination, non-finite starts
SHAPES_D = {"d2_N17": (2, 17, 102), "d3_N11": (3, 11, 504), "d4_N12": (4, 12, 320)}   # (dim, N, oracle's last step)
K_D = 64


def _trajectory_d(orc, shape):
    dim, N, _ = SHAPES_D[shape]

    def build():
        ref = orc.GD(RIESZ, sphere_points(orc, N, dim, 8).reshape(1, -1), 1e-2, order=orc.TREE, constraint=SPHERE, dim=dim)
        launches = []
        while not ref.terminated[0]:
            assert len(launches) < 20
            ref.step(K_D)
            launches.append(K_D)
        ref.close()
        return _gd_trajectory(orc, sphere_points(orc, N, dim, 8), 1e-2, SPHERE, dim, tuple(launches) + (1,))

    return _cached(("D", shape), build)


@pytest.mark.parametrize("variant", ["default", "t1024", "bar"])
@pytest.mark.parametrize("shape", list(SHAPES_D))
def test_terminates_inside_a_k_step_launch(gpu, orc, shape, variant):
    """launches of 64 steps until the run terminates, which happens inside the last one; one more step! changes
    nothing.  The flag barrier is the k-step mode's."""
    dim, N, last_step = SHAPES_D[shape]
    tr = _trajectory_d(orc, shape)
    its = [int(s.iteration_count[0]) for s in tr.snaps]
    assert its[-1] == its[-2] == last_step and tr.snaps[-2].terminated[0] and not tr.snaps[-3].terminated[0]
    assert its[-2] - its[-3] < K_D
    _run_gd(gpu, tr, variant, f"{shape} {variant}")


COINCIDENT = {1: 40, 2: 20, 3: 12, 4: 9}   # dim: N, with dim * N > 32


@pytest.mark.parametrize("variant", ["default", "t1024"])
@pytest.mark.parametrize("dim", list(COINCIDENT))
def test_coincident_start_is_terminated(gpu, orc, dim, variant):
    """A start with a coincident pair has energy +Inf: the handle is terminated at construction (:364-366) with the
    oracle's fields, and step! leaves it alone.  dim 1 on the sphere: every point is +-1."""
    dz = gpu
    EF = dz.ExampleFunctions
    N = COINCIDENT[dim]
    x = sphere_points(orc, N, dim, 61)
    if dim > 1:
        x[7] = x[2]
    ref = orc.GD(RIESZ, x.reshape(1, -1), 1e-2, order=orc.TREE, constraint=SPHERE, dim=dim)
    assert ref.terminated[0] and np.isinf(ref.objective[0])
    with _tuning(dz, **VARIANTS[variant][0]):
        opt = dz.GradientDescentOptimizer(dz.SPHERE_CONSTRAINT, EF.riesz_energy, EF.riesz_gradient_,
                                          dz.QuadraticLineSearch(0), x, 1e-2)
        try:
            _assert_variant(dz, opt, variant)
            _compare_gd(opt, ref, f"dim {dim} {variant}: ctor", nan_canon=True)
            dz.step_(opt)
            ref.step(1)
            _compare_gd(opt, ref, f"dim {dim} {variant}: step!", nan_canon=True)
            assert int(opt.iteration_count[()]) == 0
        finally:
            opt.close()
            ref.close()


# ----------------------------------------------------------------------------- E: BFGSOptimizer with the Riesz objective
SHAPES_E = {   # name: (dim, N)
    "d1_N33": (1, 33),        # n = 33
    "d2_N17": (2, 17),        # n = 34
    "d3_N129": (3, 129),      # n = 387
    "d3_N343": (3, 343),      # n = 1029: odd, two column chunks, the last 5 wide
    "d4_N513": (4, 513),      # n = 2052: three chunks
}
VARIANTS_E = ["default", "esplit2", "t1024", "tiles", "single_probe"]
CASES_E = [(shape, v) for shape, (dim, N) in SHAPES_E.items()
           for v in VARIANTS_E + (["single_cta_delta"] if dim * N % 2 else [])]
LAUNCHES_E = (1,) * 8 + (5,)


def _trajectory_e(orc, shape):
    dim, N = SHAPES_E[shape]

    def build():
        constraint = NONE if dim == 1 else SPHERE
        x = _start(orc, dim, N, 17)
        ref = orc.BFGS(RIESZ, x.reshape(1, -1), 1e-3, order=orc.TREE, constraint=constraint, dim=dim)
        snaps, kinds = [_snap(ref, BFGS_SNAP)], set()
        for k in LAUNCHES_E:
            for _ in range(k):
                ref.step(1)
                kinds.add(int(ref.step_type[0]))
            snaps.append(_snap(ref, BFGS_SNAP))
        H = ref.inverse_hessian(0)
        ref.close()
        return SimpleNamespace(x=x, constraint=constraint, snaps=snaps, kinds=kinds, H=H)

    return _cached(("E", shape), build)


def _compare_bfgs(opt, snap, tag):
    got = {"point": opt.current_point, "gradient": opt.current_gradient, "delta_point": opt.delta_point,
           "delta_gradient": opt.delta_gradient, "direction": opt.next_step_direction,
           "objective": opt.current_objective_value, "step_length": opt.last_step_length}
    for name in BFGS_FIELDS:
        assert_bitwise(np.asarray(got[name]).reshape(-1), np.asarray(getattr(snap, name)[0]).reshape(-1), f"{tag}: {name}")
    assert int(opt.last_step_type[()]) == int(snap.step_type[0]), f"{tag}: step type"
    assert int(opt.iteration_count[()]) == int(snap.iteration_count[0]), f"{tag}: iteration count"
    assert bool(opt.has_converged[()]) == bool(snap.terminated[0]), f"{tag}: has_converged"


@pytest.mark.parametrize("shape,variant", CASES_E)
def test_bfgs_riesz_every_variant(gpu, orc, shape, variant):
    """8 single step! calls and one launch of 5: the search stage in the cooperative kernel (modes 5 and 6), the n^2
    sweeps after BFGS-type and gradient-descent steps (odd n: the scalar fallbacks of gemv_kernel, update_gemv_kernel and
    identity_tile).  single_cta_delta: vec_delta_kernel instead of the cluster one (search_variant = 1), at odd n."""
    dz = gpu
    EF = dz.ExampleFunctions
    tr = _trajectory_e(orc, shape)
    assert {dz.StepType.BFGSStep, dz.StepType.GradientDescentStep} <= tr.kinds
    assert not tr.snaps[-1].terminated[0]
    knobs, witness = ({"search_variant": 1}, "default") if variant == "single_cta_delta" else (VARIANTS[variant][0], variant)
    c = _constraint(dz, tr.constraint)
    with _tuning(dz, **knobs):
        # the BFGS handle's cooperative kernel comes from the same RieszWork::init as a GD handle's
        probe = dz.GradientDescentOptimizer(c, EF.riesz_energy, EF.riesz_gradient_, dz.QuadraticLineSearch(0), tr.x, 1e-3)
        try:
            _assert_variant(dz, probe, witness)
        finally:
            probe.close()
        opt = dz.BFGSOptimizer(EF.riesz_energy, EF.riesz_gradient_, c, tr.x, 1e-3)
        try:
            tag = f"{shape} {variant}"
            _compare_bfgs(opt, tr.snaps[0], f"{tag}: ctor")
            for i, k in enumerate(LAUNCHES_E):
                if k == 1:
                    dz.step_(opt)
                else:
                    opt.step(k)
                _compare_bfgs(opt, tr.snaps[i + 1], f"{tag}: launch {i} (k={k})")
            assert_bitwise(opt.inverse_hessian(), tr.H, f"{tag}: inverse Hessian")
        finally:
            opt.close()


def test_riesz_info_refuses_handles_without_the_cooperative_kernel(gpu, orc):
    """n <= 32 (one thread per problem) and Rosenbrock handles have no cooperative Riesz kernel"""
    dz = gpu
    EF = dz.ExampleFunctions
    small = dz.GradientDescentOptimizer(dz.SPHERE_CONSTRAINT, EF.riesz_energy, EF.riesz_gradient_,
                                        dz.QuadraticLineSearch(0), sphere_points(orc, 10, 3, 4), 1e-3)
    rosen = dz.GradientDescentOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, dz.QuadraticLineSearch(0),
                                        4.0 * orc.pcg_fill(64, 6) - 2.0, 1e-2)
    try:
        for opt in (small, rosen):
            t = C.c_int(-1)
            assert dz.lib().dzo_gd_riesz_info(opt._h, C.byref(t), None, None, None, None, None) == -5   # DZO_ERR_UNSUPPORTED
            assert t.value == -1
    finally:
        small.close()
        rosen.close()

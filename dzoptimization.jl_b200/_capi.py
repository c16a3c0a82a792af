"""ctypes signatures of include/dzopt.h.

One table serves both symbol families (``dzo_`` = CUDA library, ``dzo_cpu_`` = oracle):
the two have identical argument meaning by design (include/dzopt.h header comment).
"""
import ctypes as C

c_double_p = C.POINTER(C.c_double)
c_i64_p = C.POINTER(C.c_int64)
c_i32_p = C.POINTER(C.c_int32)
c_u8_p = C.POINTER(C.c_uint8)
c_int_p = C.POINTER(C.c_int)
c_float_p = C.POINTER(C.c_float)
H = C.c_void_p   # opaque handle
HP = C.POINTER(C.c_void_p)

# name -> (argtypes for the CUDA flavour, extra trailing args of the oracle flavour or None
#          if the symbol has no oracle twin, drop_device: CUDA flavour ends with `int device`)
_VEC_GETTERS_BFGS = ["get_point", "get_gradient", "get_delta_point", "get_delta_gradient",
                     "get_direction", "get_objective", "get_step_length"]
_VEC_GETTERS_GD = ["get_point", "get_delta_point", "get_gradient", "get_delta_gradient",
                   "get_direction", "get_objective", "get_delta_objective", "get_step_length"]


def bind(lib, cpu: bool):
    """Attach argtypes/restype for every symbol of include/dzopt.h that `lib` must export.

    Raises AttributeError naming the first missing symbol (the library must export ALL of
    its family)."""
    p = "dzo_cpu_" if cpu else "dzo_"
    I, I64, D = C.c_int, C.c_int64, C.c_double

    def sig(name, args, res=I):
        fn = getattr(lib, p + name)
        fn.argtypes = args
        fn.restype = res
        return fn

    sig("last_error", [], C.c_char_p)
    tail_create = [I, I] if cpu else [I]              # (order, nthreads) | (device)
    sig("bfgs_create", [HP, I, I, I64, I64, I64, c_double_p, D] + tail_create)
    sig("bfgs_step", [H, I])
    for g in _VEC_GETTERS_BFGS:
        sig("bfgs_" + g, [H, c_double_p])
    sig("bfgs_get_inverse_hessian", [H, I64, c_double_p])
    sig("bfgs_get_step_type", [H, c_i32_p])
    sig("bfgs_get_iteration_count", [H, c_i64_p])
    sig("bfgs_get_terminated", [H, c_u8_p])
    sig("bfgs_count_active", [H, c_i64_p])
    sig("bfgs_set_state", [H, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                           c_i32_p, c_i64_p])
    sig("bfgs_destroy", [H], None)

    tail_gd = [I, I, I] if cpu else [I, I]            # (max_inc, order, nthreads) | (max_inc, device)
    sig("gd_create", [HP, I, I, I64, I64, I64, c_double_p, D] + tail_gd)
    sig("gd_step", [H, I])
    for g in _VEC_GETTERS_GD:
        sig("gd_" + g, [H, c_double_p])
    sig("gd_get_iteration_count", [H, c_i64_p])
    sig("gd_get_terminated", [H, c_u8_p])
    sig("gd_destroy", [H], None)

    tail_lb = [I, I] if cpu else [I, I]               # (history_length, order) | (history_length, device)
    sig("lbfgs_create", [HP, I, I, I64, I64, c_double_p, D] + tail_lb)
    sig("lbfgs_step", [H, I])
    for g in ("get_point", "get_delta_point", "get_gradient", "get_delta_gradient", "get_direction",
              "get_objective", "get_delta_objective"):
        sig("lbfgs_" + g, [H, c_double_p])
    sig("lbfgs_get_iteration_count", [H, c_i64_p])
    sig("lbfgs_get_stuck", [H, c_u8_p])
    sig("lbfgs_get_rho_history", [H, c_i64_p, c_double_p])
    sig("lbfgs_destroy", [H], None)

    sig("adgd_create", [HP, I, I, I64, I64, c_double_p, D, I])      # last: order (oracle) | device (CUDA)
    sig("adgd_step", [H, I])
    for g in ("get_point", "get_delta_point", "get_gradient", "get_delta_gradient", "get_scalars"):
        sig("adgd_" + g, [H, c_double_p])
    sig("adgd_destroy", [H], None)

    # last: order (oracle) | device (CUDA)
    sig("legacy_lbfgs_create", [HP, I, I, I64, I64, c_double_p, D, I, I, I, D, D, D, I])
    sig("legacy_lbfgs_step", [H, I])
    for g in ("get_point", "get_delta_point", "get_gradient", "get_delta_gradient", "get_direction", "get_scalars"):
        sig("legacy_lbfgs_" + g, [H, c_double_p])
    sig("legacy_lbfgs_get_history", [H, c_double_p, c_double_p])
    sig("legacy_lbfgs_destroy", [H], None)

    dev = [] if cpu else [I]
    sig("objective", [I, I, I64, I, I64, I64, c_double_p, c_double_p] + dev)
    sig("gradient", [I, I, I64, I, I64, I64, c_double_p, c_double_p] + dev)
    sig("dot", [I, I64, c_double_p, c_double_p, c_double_p] + dev)
    sig("gemv", [I, I64, c_double_p, c_double_p, c_double_p] + ([I] if cpu else [I]))
    sig("update_inverse_hessian", [I, I64, c_double_p, D, c_double_p, c_double_p, c_double_p,
                                   c_double_p, c_double_p, I])
    sig("line_search", [I, I, I64, I, I64, c_double_p, c_double_p, D, D, c_double_p, c_double_p] + dev)

    sig("line_search_evaluate", [I, I, I64, I, I64, c_double_p, D, c_double_p, D, D, I, c_double_p, c_double_p, c_double_p] + dev)
    P = c_double_p
    sig("pairwise_energy", [I, I, I64, P, P, P, P, P] + dev)
    sig("pairwise_gradient", [I, I, I64, P, P, P, P, P, P] + dev)
    sig("pairwise_hvp", [I, I, I64, P, P, P, P, P, P, P, P, P] + dev)
    if cpu:
        sig("pcg_fill", [c_double_p, I64, C.c_uint64])
        sig("gemv_rows", [I, I64, I64, I64, c_double_p, c_double_p, c_double_p])
        sig("update_rows", [I64, I64, I64, c_double_p, D, c_double_p, c_double_p])
    else:
        # CUDA-only entry points (dzo_dev_* are spelled dzo_dev_ in the header; the kernel-level
        # names above are looked up through the alias table below)
        sig("nccl_get_unique_id", [C.c_void_p])
        sig("bfgs_create_sharded", [HP, I, I, I64, I64, c_double_p, D, I, I, I, C.c_void_p])
        sig("bfgs_set_stream", [H, C.c_void_p])
        sig("bfgs_step_async", [H, I])
        sig("bfgs_sync", [H])
        sig("bfgs_info", [H, c_i64_p, c_i64_p, c_int_p, c_i64_p, c_i64_p])
        sig("bfgs_get_step_log", [H, c_i64_p, c_u8_p])
        sig("bfgs_gather_mode", [H, c_int_p])
        sig("bfgs_get_step_kind_counts", [H, c_i64_p, I])
        sig("bfgs_mirror_fields", [H, c_double_p, c_u8_p])
        sig("lbfgs_set_stream", [H, C.c_void_p])
        sig("lbfgs_step_async", [H, I])
        sig("lbfgs_sync", [H])
        sig("lbfgs_info", [H, c_i64_p, c_int_p, c_int_p])
        sig("legacy_lbfgs_set_stream", [H, C.c_void_p])
        sig("legacy_lbfgs_step_async", [H, I])
        sig("legacy_lbfgs_sync", [H])
        sig("gd_set_stream", [H, C.c_void_p])
        sig("gd_step_async", [H, I])
        sig("gd_sync", [H])
        sig("gd_info", [H, c_i64_p, c_i64_p, c_int_p])
        sig("gd_riesz_info", [H, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p, c_int_p])
        sig("gd_get_evaluation_count", [H, c_i64_p])
        sig("gd_get_phase_log", [H, C.POINTER(C.c_uint64), I64, c_i64_p])
        sig("identity", [I64, c_double_p, I])
        sig("bench_kernel", [I, I64, I, I, c_float_p, I])
        sig("dev_selftest_ieee_fast", [C.c_uint64, C.c_uint64, C.POINTER(C.c_uint64), I])
        sig("set_tuning", [C.c_char_p, I])
        V = C.c_void_p
        sig("pairwise_workspace_bytes", [I64], C.c_uint64)
        sig("pairwise_energy_device", [V, I, I, I64, V, V, V, V, V, V])
        sig("pairwise_gradient_device", [V, I, I, I64, V, V, V, V, V, V, V])
        sig("pairwise_hvp_device", [V, I, I, I64, V, V, V, V, V, V, V, V, V, V])
        sig("host_register", [C.c_void_p, C.c_uint64])
        sig("host_unregister", [C.c_void_p])
        sig("host_alloc", [C.POINTER(C.c_void_p), C.c_uint64])
        sig("host_free", [C.c_void_p])
    return lib


class _DevAlias:
    """The header spells kernel-level CUDA entry points ``dzo_dev_<name>``; present them
    under the same short names the oracle uses (``dzo_cpu_<name>``) so bind() is uniform."""

    _DEV = {"objective", "gradient", "dot", "gemv", "update_inverse_hessian", "line_search", "line_search_evaluate",
            "identity", "pairwise_energy", "pairwise_gradient", "pairwise_hvp"}

    def __init__(self, lib):
        object.__setattr__(self, "_lib", lib)

    def __getattr__(self, name):
        if name.startswith("dzo_") and name[4:] in self._DEV:
            name = "dzo_dev_" + name[4:]
        return getattr(self._lib, name)

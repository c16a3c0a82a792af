"""CPU tests of the drop-in boundary: the C-ABI libraries load and export every symbol that
include/dzopt.h declares (no compute calls: there is no GPU here), and the host-side mirror of the
Julia API validates its arguments like the reference does."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "dzopt.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dzo_[a-z0-9_]+)\s*\(", src)))


def test_header_declares_both_families():
    syms = declared_symbols()
    assert "dzo_bfgs_step" in syms and "dzo_cpu_bfgs_step" in syms and "dzo_gd_step" in syms
    assert len(syms) > 80


def test_cuda_library_exports_every_declared_symbol(dz):
    lib = C.CDLL(dz.lib_path)
    missing = [s for s in declared_symbols() if not s.startswith("dzo_cpu_") and not hasattr(lib, s)]
    assert not missing, f"libdzopt_b200.so lacks: {missing}"


def test_oracle_library_exports_every_declared_symbol(orc):
    lib = C.CDLL(orc.LIB_PATH)
    missing = [s for s in declared_symbols() if s.startswith("dzo_cpu_") and not hasattr(lib, s)]
    assert not missing, f"libdzo_oracle.so lacks: {missing}"


def test_product_library_does_not_link_the_oracle(dz):
    """The product path must not route through the oracle (or any CPU fallback)."""
    import subprocess
    out = subprocess.run(["ldd", dz.lib_path], capture_output=True, text=True).stdout
    assert "dzo_oracle" not in out
    nm = subprocess.run(["nm", "-D", "--defined-only", dz.lib_path], capture_output=True, text=True).stdout
    assert "dzo_cpu_" not in nm
    pkg_dir = os.path.dirname(dz.lib_path)
    for root, _, files in os.walk(os.path.dirname(pkg_dir)):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".jl")):
                text = open(os.path.join(root, f)).read()
                assert "import oracle" not in text and "libdzo_oracle" not in text, f


def test_no_gpu_means_loud_failure_not_fallback(dz):
    """Without a CUDA device the constructor must raise DZO_ERR_NO_DEVICE (-6), never compute.  Runs in a child process
    with CUDA_VISIBLE_DEVICES="", which hides every device, so the check also runs on a machine that has GPUs."""
    import subprocess
    import sys
    child = "\n".join([
        "import sys",
        "sys.path.insert(0, %r)" % ROOT,
        "import numpy as np",
        "import dzopt_b200 as dz",
        "EF = dz.ExampleFunctions",
        "makers = [lambda: dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros(2), 1.0),",
        "          lambda: dz.GradientDescentOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_,",
        "                                              dz.QuadraticLineSearch(0), np.zeros(64), 1.0)]",
        "for make in makers:",
        "    try:",
        "        make()",
        "        print('computed')",
        "    except dz.DZOptError as e:",
        "        print(e.code)",
    ])
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.split() == ["-6", "-6"], r.stdout


def test_constructor_argument_validation(dz):
    EF = dz.ExampleFunctions
    with pytest.raises(TypeError):                                   # host closures cannot run in the CUDA step!
        dz.BFGSOptimizer(lambda x: 0.0, EF.rosenbrock_gradient_, np.zeros(2), 1.0)
    with pytest.raises(TypeError):                                   # objective / gradient of different functions
        dz.BFGSOptimizer(EF.rosenbrock_function, EF.riesz_gradient_, np.zeros(2), 1.0)
    with pytest.raises(TypeError):
        dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros(2))          # arity (:753-766)
    with pytest.raises(TypeError):
        dz.GradientDescentOptimizer(EF.riesz_energy, EF.riesz_gradient_, "not a line search", np.zeros((4, 3)), 1.0)
    with pytest.raises(ValueError):
        dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, np.zeros((3, 2)), 1.0)   # needs batched=True
    assert dz.StepType.NullStep == 0 and dz.StepType.GradientDescentStep == 1 and dz.StepType.BFGSStep == 2
    assert dz.QuadraticLineSearch().max_increases == 0


def test_layout_matches_julia_column_major(dz):
    a, n, batch, pshape, dim = dz._layout(np.zeros((5, 3)), dz.OBJ_RIESZ, False)   # Julia 3 x 5 Matrix
    assert (n, batch, pshape, dim) == (15, 1, (5, 3), 3)
    a, n, batch, pshape, dim = dz._layout(np.zeros((7, 16)), dz.OBJ_ROSENBROCK, True)
    assert (n, batch, pshape, dim) == (16, 7, (16,), 0)


def test_error_paths_need_no_gpu(dz):
    """argument validation happens before any CUDA call: null handles / pointers and bad shapes give
    DZO_ERR_INVALID_ARGUMENT (-1) with a message, on any machine"""
    lib = dz.lib()
    assert lib.dzo_bfgs_step(None, 1) == -1 and b"bad arguments" in lib.dzo_last_error()
    assert lib.dzo_gd_step(None, 1) == -1
    assert lib.dzo_lbfgs_step(None, 1) == -1
    assert lib.dzo_adgd_step(None, 1) == -1
    out = np.zeros(4)
    dp = out.ctypes.data_as(dz._capi.c_double_p)
    assert lib.dzo_bfgs_get_point(None, dp) == -1
    h = C.c_void_p()
    assert lib.dzo_bfgs_create(C.byref(h), 1, 0, 0, 3, 1, dp, 1.0, 0) == -1          # odd n for Rosenbrock
    assert b"even n" in lib.dzo_last_error()
    assert lib.dzo_bfgs_create(C.byref(h), 7, 0, 0, 4, 1, dp, 1.0, 0) == -1          # unknown objective id
    assert lib.dzo_bfgs_create(C.byref(h), 2, 0, 5, 4, 1, dp, 1.0, 0) == -1          # Riesz: n not a multiple of dim
    assert lib.dzo_lbfgs_create(C.byref(h), 1, 0, 0, 4, dp, 1.0, 0, 0) == -1         # history_length < 1
    assert lib.dzo_set_tuning(b"no_such_knob", 1) == -1
    assert lib.dzo_dot(0, 0, dp, dp, dp, 0) == -1                                     # n <= 0
    e = C.c_double()
    assert lib.dzo_pairwise_energy(9, 0, 4, dp, dp, dp, None, C.byref(e), 0) == -1    # unknown potential


@pytest.mark.parametrize("steps", [3, 27])
def test_bench_reference_arm_contract(steps):
    """bench.py --impl reference runs without a GPU and prints ONE JSON line with the contract's keys (27 steps: the timed
    region crosses into a second batch of the workload, bench.py STEPS_PER_BATCH = 25)."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", str(steps), "--warmup", "3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0
    assert d["steps"] == steps and ("%d batch(es)" % (-(-steps // 25))) in d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_product_pcg_generator_equals_the_oracle_and_the_golden_vectors(dz, orc):
    """dzoptimization.jl_b200/pcg.py (legacy/PCG.jl:7-22, numpy): the inputs of bench.py come from the product, not
    from oracle/; bit-identical to dzo_cpu_pcg_fill and to the committed golden vectors."""
    import json
    import os
    here = os.path.dirname(os.path.abspath(__file__))
    with open(os.path.join(here, "golden", "golden.json")) as f:
        golden = json.load(f)["pcg"]
    for seed, vals in golden.items():
        assert [float(v).hex() for v in dz.pcg_fill(8, int(seed))] == vals
    for count, seed in ((1, 0), (4095, 3), (4096, 2024), (4097, 5), (10000, 2 ** 63 + 5), (300000, 9)):
        assert np.array_equal(dz.pcg_fill(count, seed), orc.pcg_fill(count, seed))
    assert dz.pcg_fill(0, 1).size == 0


# ----------------------------------------------------------------------------- the Julia wrapper against the header
def _c_prototypes():
    """{symbol: (return type, [parameter types])} of include/dzopt.h, comments stripped, names dropped."""
    import re
    text = open(os.path.join(ROOT, "include", "dzopt.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    protos = {}
    for m in re.finditer(r"(?:^|[;}\n])\s*((?:const\s+)?[A-Za-z_][\w]*(?:\s*\*)?)\s+(dzo_\w+)\s*\(([^;{}]*?)\)\s*;", text, flags=re.S):
        ret, name, params = m.group(1), m.group(2), m.group(3)
        plist = []
        params = " ".join(params.split())
        if params and params != "void":
            for prm in params.split(","):
                prm = prm.strip()
                stars = prm.count("*")
                prm = prm.replace("*", " ")
                toks = [t for t in prm.split() if t != "const"]
                base = toks[0] if len(toks) <= 2 else " ".join(toks[:-1])
                if toks[0] == "unsigned" or toks[0] == "struct":
                    base = " ".join(toks[:2])
                plist.append(base + "*" * stars)
        protos[name] = (" ".join(ret.replace("const", "").split()).replace(" *", "*"), plist)
    return protos


# Julia ccall argument type -> the C parameter types it may bind to
_JL_TO_C = {
    "Cint": {"int", "int32_t"}, "Int64": {"int64_t"}, "UInt64": {"uint64_t"}, "Float64": {"double"}, "Cstring": {"char*"},
    "Ptr{Float64}": {"double*"}, "Ptr{Int64}": {"int64_t*"}, "Ref{Int64}": {"int64_t*"}, "Ptr{Int32}": {"int32_t*"},
    "Ptr{UInt8}": {"uint8_t*", "void*"}, "Ptr{UInt64}": {"uint64_t*"}, "Ref{UInt64}": {"uint64_t*"}, "Ref{Cint}": {"int*"},
    "Ptr{Cint}": {"int*"}, "Ref{Float64}": {"double*"}, "Ptr{Float32}": {"float*"}, "Ref{Float32}": {"float*"},
    "Ref{Ptr{Cvoid}}": {"HANDLE**", "void**"}, "Ptr{Cvoid}": {"HANDLE*", "void*", "double*", "uint8_t*"},
}
_HANDLES = {"dzo_bfgs", "dzo_gd", "dzo_lbfgs", "dzo_adgd", "dzo_legacy_lbfgs"}


def _c_kind(t):
    base = t.rstrip("*")
    if base in _HANDLES:
        return "HANDLE" + "*" * (len(t) - len(base))
    return t


def _split_top(s):
    out, depth, cur = [], 0, ""
    for ch in s:
        if ch in "({[":
            depth += 1
        elif ch in ")}]":
            depth -= 1
        if ch == "," and depth == 0:
            out.append(cur.strip()); cur = ""
        else:
            cur += ch
    if cur.strip():
        out.append(cur.strip())
    return out


def test_julia_wrapper_ccalls_match_the_header():
    """julia/DZOptimizationB200.jl cannot run here (no Julia), so its `ccall`s are checked statically: every symbol it
    names is declared in include/dzopt.h (and exported by the library), with the same number of arguments and C types the
    Julia argument tuple can bind to; the symbols passed to its generic (sym) helpers have the (handle, T*) shape."""
    import re
    protos = _c_prototypes()
    assert len(protos) > 100 and "dzo_bfgs_create" in protos and protos["dzo_bfgs_step"] == ("int", ["dzo_bfgs*", "int"])
    src = open(os.path.join(ROOT, "dzoptimization.jl_b200", "julia", "DZOptimizationB200.jl")).read()
    src_nc = "\n".join(line.split("#")[0] if "#=" not in line else line for line in src.split("\n"))
    lib = dz_lib_symbols()
    checked = 0
    for m in re.finditer(r"ccall\(\(\s*:(\w+)\s*,\s*libdzopt\s*\)\s*,", src_nc):
        name = m.group(1)
        # the balanced argument list of this ccall
        i = src_nc.index("(", m.start())          # '(' of ccall(
        depth, j = 0, i
        while True:
            depth += src_nc[j] == "("
            depth -= src_nc[j] == ")"
            if depth == 0:
                break
            j += 1
        parts = _split_top(src_nc[i + 1:j])
        ret, argt = parts[1], parts[2]
        assert argt.startswith("(") and argt.endswith(")"), (name, argt)
        jl_args = [a for a in _split_top(argt[1:-1]) if a]
        assert name in protos, f"ccall names {name}, which include/dzopt.h does not declare"
        assert name in lib, f"{name} is not exported by libdzopt_b200.so"
        cret, cargs = protos[name]
        assert len(parts) - 3 == len(jl_args), f"{name}: {len(jl_args)} argument types but {len(parts) - 3} values"
        assert len(jl_args) == len(cargs), f"{name}: Julia passes {len(jl_args)} arguments, the header declares {len(cargs)}: {cargs}"
        want_ret = {"Cint": "int", "Cvoid": "void", "Cstring": "char*", "UInt64": "uint64_t"}[ret]
        assert cret == want_ret, f"{name}: returns {cret}, Julia expects {ret}"
        for k, (ja, ca) in enumerate(zip(jl_args, cargs)):
            assert ja in _JL_TO_C, f"{name}: unknown Julia argument type {ja}"
            assert _c_kind(ca) in _JL_TO_C[ja], f"{name}: argument {k} is `{ca}` in the header, Julia passes {ja}"
        checked += 1
    assert checked >= 40
    # symbols handed to the generic helpers:  vecfield / vec -> (handle, double*),  scalarfield / sc -> (handle, T*)
    generic = 0
    for m in re.finditer(r"\b(vecfield|vec|scalarfield|sc)\(\s*(?:opt\s*,\s*)?:(dzo_\w+)\s*(?:,\s*(\w+))?\)", src_nc):
        helper, name, T = m.groups()
        assert name in protos and name in lib, f"{name} (used through {helper}) is not in the header / library"
        cret, cargs = protos[name]
        assert cret == "int" and len(cargs) == 2 and _c_kind(cargs[0]) == "HANDLE*", (name, cargs)
        if helper in ("vecfield", "vec"):
            assert cargs[1] == "double*", (name, cargs)
        else:
            assert cargs[1] == {"Float64": "double*", "Int64": "int64_t*", "Int32": "int32_t*", "UInt8": "uint8_t*"}[T], (name, T, cargs)
        generic += 1
    assert generic >= 30
    # and nothing else: every :dzo_ symbol literal of the file went through one of the two checks
    literals = set(re.findall(r":(dzo_\w+)", src_nc))
    assert literals <= set(protos), literals - set(protos)


def dz_lib_symbols():
    import subprocess
    import __graft_entry__ as ge
    out = subprocess.run(["nm", "-D", "--defined-only", ge.LIB], capture_output=True, text=True, check=True).stdout
    return {line.split()[-1] for line in out.splitlines() if line.strip()}

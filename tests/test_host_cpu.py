"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol that
include/jslp_b200.h declares, the product front end builds the same initial tableau as the
oracle's restatement on every golden fixture, and the product fails loudly without a GPU."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, load_bundle
from helpers import strip_timeouts

BUNDLE = load_bundle()


def test_library_exports_every_declared_symbol():
    from jslpsolver_b200 import _lib
    L = _lib.load()
    header = open(os.path.join(ROOT, "include", "jslp_b200.h")).read()
    declared = set(re.findall(r"\b(jslp_[a-z0-9_]+)\s*\(", header))
    declared -= {"jslp_ctx", "jslp_tab"}
    assert declared, "no declarations parsed"
    bound = {name for name, _, _ in _lib.SYMBOLS}
    assert declared == bound, (declared ^ bound)
    for name in declared:
        assert hasattr(L, name), name
    assert L.jslp_abi_version() == 2


def test_library_contains_sm100a_code():
    import subprocess
    from jslpsolver_b200 import _lib
    out = subprocess.run(["cuobjdump", "-lelf", _lib.lib_path()], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out


@pytest.mark.parametrize("fx", BUNDLE["fixtures"] + BUNDLE["readme"], ids=lambda f: f["file"])
def test_front_end_matches_oracle_front_end(fx, monkeypatch):
    """Row/column order decides every tie-break (SURVEY.md 3.10): the upload source must be
    identical, bit for bit, to the restated reference front end."""
    import jslpsolver_b200.tableau as T
    from jslpsolver_b200.model import Model, presolve
    from oracle import ref_model

    class NoDevice:  # the front end itself needs no GPU
        def __init__(self, *a, **k):
            pass
    monkeypatch.setattr(T, "GpuTableau", NoDevice)
    jm = strip_timeouts(fx["model"])
    m = Model().loadJson(jm)
    r = ref_model.RefModel().loadJson(jm)
    pm = presolve(m)
    inf, fixed = ref_model.presolve(r)
    assert pm.isInfeasible == inf
    assert sorted((v.id, float(x)) for v, x in pm.fixedVariables.items()) == sorted((v.id, float(x)) for v, x in fixed.items())
    it = m.initial_tableau()
    M, vr, vc, pr, rc = r.build_tableau()
    assert np.array_equal(it.matrix, M)
    assert np.array_equal(it.varIndexByRow, vr) and np.array_equal(it.varIndexByCol, vc)
    assert it.optionalPriorities == pr and np.array_equal(it.optionalCosts, rc)
    assert m.checkForCycles == r.checkForCycles and m.tolerance == r.tolerance
    assert [v.index for v in m.integerVariables] == [v.index for v in r.integerVariables]


def test_direct_tableau_equals_model_path(monkeypatch):
    import jslpsolver_b200.tableau as T
    from jslpsolver_b200 import problems
    from jslpsolver_b200.model import Model

    class NoDevice:
        def __init__(self, *a, **k):
            pass
    monkeypatch.setattr(T, "GpuTableau", NoDevice)
    it = Model().loadJson(problems.dense_packing_lp_model(7, 5, seed=3)).initial_tableau()
    direct = problems.dense_packing_lp_tableau(7, 5, seed=3)
    assert np.array_equal(it.matrix, direct.matrix)
    assert np.array_equal(it.varIndexByRow, direct.varIndexByRow)
    assert np.array_equal(it.varIndexByCol, direct.varIndexByCol)


def test_no_cpu_fallback():
    """Without a CUDA device the product path must raise, never compute."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import jslpsolver_b200 as J
    with pytest.raises(J.JslpError):
        J.Solve(BUNDLE["readme"][0]["model"])


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "jslpsolver_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("oracle/", "").lower() or f in (), (f, "mentions oracle")


def test_ctypes_structs_match_the_header(tmp_path):
    """sizeof/offsetof of every struct in include/jslp_b200.h, as gcc sees them, equal the ctypes mirrors."""
    import ctypes as C
    import subprocess
    from jslpsolver_b200 import _lib
    structs = {"jslp_lp_status": _lib.LpStatus, "jslp_cut": _lib.Cut, "jslp_bnb_opts": _lib.BnbOpts,
               "jslp_bnb_status": _lib.BnbStatus}
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{os.path.join(ROOT, "include", "jslp_b200.h")}"',
             "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["return 0; }"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(got[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


def test_frontier_heap_follows_the_reference_min_heap(tmp_path):
    """tests/cpp/frontier_test.cpp: the product's frontier (jslp_frontier.h, host-only) replays the ordering
    scenarios of the reference's min-heap.test.ts (best-first, LIFO on ties) and the all-gather record round trip."""
    import subprocess
    exe = tmp_path / "frontier_test"
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"),
                    "-I", os.path.join(ROOT, "jslpsolver_b200", "csrc"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "cpp", "frontier_test.cpp")], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and "FRONTIER OK" in out.stdout, out.stdout + out.stderr


def test_cycle_detectors_follow_the_reference_scan(tmp_path):
    """tests/cpp/cycles_test.cpp: the product's two host-side detectors (jslp_cycles.h) report exactly what a literal
    restatement of checkForCycles (simplex.ts:415-440) reports, push by push, on 4000 random pivot histories."""
    import subprocess
    exe = tmp_path / "cycles_test"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "jslpsolver_b200", "csrc"),
                    "-o", str(exe), os.path.join(ROOT, "tests", "cpp", "cycles_test.cpp")], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and "CYCLES OK" in out.stdout, out.stdout + out.stderr


def test_host_rounding_matches_the_oracle(tmp_path):
    """tests/cpp/hostmath_test.cpp: the product's Math.round / setEvaluation (jslp_hostmath.h) against the oracle's
    restatement (tableau.ts:420-430), bit for bit, on tie cases and random magnitudes."""
    import struct
    import subprocess
    from oracle import ref_model
    exe = tmp_path / "hostmath_test"
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(ROOT, "jslpsolver_b200", "csrc"),
                    "-o", str(exe), os.path.join(ROOT, "tests", "cpp", "hostmath_test.cpp")], check=True)
    rng = np.random.default_rng(7)
    xs = [0.0, -0.0, 0.5, -0.5, 1.5, 2.5, -2.5, 0.49999999999999994, 1e15 + 0.5, -1e15 - 0.5, 681907.6430000001,
          25432.999999995, -523.612072085, 1e-9, -1e-9, 5e-9, -5e-9, float("inf"), float("-inf")]
    xs += list(rng.normal(0, 1, 300) * 10.0 ** rng.integers(-9, 9, 300))
    xs += [float(k) + 0.5 * 1e-8 * s for k in range(-3, 4) for s in (-1, 1)]  # ties at the 1e-8 grid
    cases = [(x, p) for x in xs for p in (1e-8, 1e-9, 1e-6)]
    bits = lambda v: struct.unpack("<Q", struct.pack("<d", v))[0]
    stdin = "".join(f"{bits(x):x} {bits(p):x}\n" for x, p in cases)
    out = subprocess.run([str(exe)], input=stdin, capture_output=True, text=True, check=True).stdout.split()
    assert len(out) == 2 * len(cases)
    for k, (x, p) in enumerate(cases):
        coeff = ref_model.js_round(1 / p)
        want_r = ref_model.js_round(x)
        want_e = ref_model.js_round((2.220446049250313e-16 + x) * coeff) / coeff
        # the sign of a zero result is not compared: JS gives -0 on [-0.5, 0], observable nowhere in the reference
        same = lambda got, want: got == bits(float(want)) or (want == 0 and got in (0, 1 << 63))
        assert same(int(out[2 * k], 16), want_r), (x, "round")
        assert same(int(out[2 * k + 1], 16), want_e), (x, p, "evaluation")


def test_napi_addon_compiles_against_the_header(tmp_path):
    """binding/jslp_addon.cc (the N-API shim of north_star) is compiled -- -Wall -Wextra -Werror -- against the real
    include/jslp_b200.h and a stub node_api.h that carries Node's own prototypes for the N-API calls it makes; every
    jslp_* symbol the object file needs must be exported by libjslp_b200.so, every napi_* one declared by the stub."""
    import re
    import subprocess
    from jslpsolver_b200 import _lib
    obj = tmp_path / "jslp_addon.o"
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wextra", "-Werror", "-fPIC", "-c", "-I", os.path.join(ROOT, "tests", "stubs"),
                    "-I", os.path.join(ROOT, "include"), "-o", str(obj), os.path.join(ROOT, "binding", "jslp_addon.cc")], check=True)
    undef = subprocess.run(["nm", "-u", str(obj)], check=True, capture_output=True, text=True).stdout.split()
    need_jslp = {s for s in undef if s.startswith("jslp_")}
    need_napi = {s for s in undef if s.startswith("napi_")}
    assert len(need_jslp) >= 20 and len(need_napi) >= 30
    bound = {name for name, _, _ in _lib.SYMBOLS}
    assert need_jslp <= bound, need_jslp - bound
    L = _lib.load(build_if_missing=False)
    for s in need_jslp:
        assert hasattr(L, s), s
    stub = open(os.path.join(ROOT, "tests", "stubs", "node_api.h")).read()
    declared = set(re.findall(r"\b(napi_[a-z0-9_]+)\s*\(", stub))
    assert need_napi <= declared, need_napi - declared
    # the TypeScript glue names the same addon methods the shim defines
    ts = open(os.path.join(ROOT, "binding", "src", "tableau", "gpu-tableau.ts")).read()
    cc = open(os.path.join(ROOT, "binding", "jslp_addon.cc")).read()
    methods = set(re.findall(r'\{"([A-Za-z0-9]+)", nullptr, tab_', cc))
    used = set(re.findall(r"this\.tab\(\)\.([A-Za-z0-9]+)\(", ts))
    assert used and used <= methods, used - methods


def test_bench_output_dump_fits_its_budget_and_repeats(tmp_path, monkeypatch):
    """bench.py --dump-outputs: small arrays are written whole as float64, an array beyond the 64 MB budget becomes a
    fixed seeded sample of its elements with their flat indices, and the same arrays give the same files."""
    import sys
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)  # bench.py sets it on import
    import bench
    big = np.arange(3001 * 3001, dtype=np.float64).reshape(3001, 3001)  # 72 MB: each value is its flat index
    arrays = {"lp_matrix": big, "lp_var_index_by_row": np.arange(3001, dtype=np.int32), "lp_status": np.array([1, 1, -5.5])}
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["lp_matrix.npy", "lp_matrix_index.npy", "lp_status.npy", "lp_var_index_by_row.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f
        assert np.load(tmp_path / "a" / f).dtype == np.float64, f
    sample, idx = np.load(tmp_path / "a" / "lp_matrix.npy"), np.load(tmp_path / "a" / "lp_matrix_index.npy")
    assert len(sample) > 3_000_000 and np.array_equal(sample, idx) and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "lp_var_index_by_row.npy"), np.arange(3001))
    assert np.array_equal(np.load(tmp_path / "a" / "lp_status.npy"), [1, 1, -5.5])

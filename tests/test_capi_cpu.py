"""CPU tests of the boundary: the C-ABI library builds, loads and exports exactly what
include/minsnap_b200.h declares; argument errors come back as codes; and there is no CPU
fallback -- compute entry points fail loudly without a GPU."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "minsnap_b200.h")


def declared_functions():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"MINSNAP_API\s+[\w\s\*]+?\b(minsnap_\w+)\s*\(", text)))


def test_header_declares_expected_surface():
    names = declared_functions()
    for must in ("minsnap_reorder", "minsnap_solve", "minsnap_solve_standard", "minsnap_sample_uniform",
                 "minsnap_sample_at", "minsnap_evaluate_range", "minsnap_cost_sweep", "minsnap_solve_standard_host"):
        assert must in names
    assert len(names) >= 25


def test_library_exports_every_declared_symbol(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    out = subprocess.check_output(["nm", "-D", "--defined-only", capi.LIB_PATH]).decode()
    exported = {line.split()[-1] for line in out.splitlines() if " T " in line}
    declared = declared_functions()
    missing = [n for n in declared if n not in exported]
    assert not missing, missing
    # and nothing undeclared leaks out of the library
    extra = [n for n in exported if n.startswith("minsnap_") and n not in declared]
    assert not extra, extra
    # the ctypes table covers the same set
    assert sorted(capi.SIGNATURES) == declared


def test_abi_version_and_strings(ms):
    lib = ms.load()
    assert lib.minsnap_abi_version() == 1
    assert lib.minsnap_error_string(0) == b"ok"
    assert b"argument" in lib.minsnap_error_string(1)


def test_argument_errors_are_codes_not_crashes(ms):
    lib = ms.load()
    from mav_trajectory_generation_cmake_b200 import capi
    # unsupported N, K < 1, NULL pointers
    assert lib.minsnap_solve_workspace_bytes(7, 10) == 0
    assert lib.minsnap_solve_workspace_bytes(10, 10) > 0
    assert lib.minsnap_reorder(10, 0, 1, None, None, None, None) == capi.ERR_ARG
    assert lib.minsnap_solve(1, 10, 3, 10, 4, None, None, None, None, None, None, None, None, None, 0, None) == capi.ERR_ARG
    assert lib.minsnap_solve_standard(1, 10, 3, 10, 7, None, None, None, 0.0, 0.0, 0.0, None, None, None, None, None,
                                      None) == capi.ERR_ARG
    assert lib.minsnap_sample_uniform(1, 10, 3, 10, None, None, 10, 5, None, None, None) == capi.ERR_ARG
    assert lib.minsnap_fp64_peak(0, None) == capi.ERR_ARG


def test_evaluate_range_empty_batch_is_a_no_op(ms):
    """B = 0 reads no pointer, like every other batched entry; the shape is still checked."""
    lib = ms.load()
    from mav_trajectory_generation_cmake_b200 import capi
    args = (0.0, 1.0, 0.1, 0, 16, None, None, None, None)
    assert lib.minsnap_evaluate_range(0, 10, 3, 10, None, None, *args) == capi.OK
    assert lib.minsnap_evaluate_range(1, 10, 3, 10, None, None, *args) == capi.ERR_ARG
    assert lib.minsnap_evaluate_range(0, 10, 3, 7, None, None, *args) == capi.ERR_ARG
    assert lib.minsnap_evaluate_range(-1, 10, 3, 10, None, None, *args) == capi.ERR_ARG


def test_random_positions_match_oracle_generator(ms, oracle):
    lo, hi = [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0]
    got = ms.random_positions_host(33, 10, lo, hi, 12345)
    want = np.stack([oracle.create_random_positions(10, lo, hi, 12345 + b) for b in range(33)])
    assert np.array_equal(got, want)
    got1 = ms.random_positions_host(5, 100, [-50.0], [50.0], 0)
    want1 = np.stack([oracle.create_random_positions(100, [-50.0], [50.0], b) for b in range(5)])
    assert np.array_equal(got1, want1)


def test_no_cpu_fallback_without_gpu(ms):
    """Without a CUDA device every compute entry point must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is exercised on CPU-only machines")
    with pytest.raises(ms.MinsnapError) as ei:
        ms.device_info()
    assert ei.value.code in (2, 4)
    pos = np.zeros((2, 11, 3))
    pos[:, :, 0] = np.arange(11)
    with pytest.raises(ms.MinsnapError):
        ms.solve_standard_host(pos, times=np.ones((2, 10)))
    with pytest.raises(ms.MinsnapError):
        ms.segment_matrices_host([1.0, 2.0])
    with pytest.raises(ms.MinsnapError):
        ms.fp64_peak()


def test_product_package_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under the product package may reference it."""
    pkg = os.path.join(ROOT, "mav_trajectory_generation_cmake_b200")
    inc = os.path.join(ROOT, "include")
    offenders = []
    for base in (pkg, inc):
        for dirpath, _, files in os.walk(base):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                    text = open(os.path.join(dirpath, f), errors="ignore").read()
                    if re.search(r"oracle_py|liboracle|orc_\w+\(|from oracle|import oracle", text):
                        offenders.append(os.path.join(dirpath, f))
    assert not offenders, offenders


def test_generated_tables_are_in_sync_and_consistent(tmp_path, oracle):
    """csrc/minsnap_tables.h is what tools/gen_tables.py writes (exact rational arithmetic), and the two derived
    tables the kernels read -- the per-lane-role recovery constants and the packed cost form -- agree with A1inv and
    H1 as the oracle forms them (ref LIN.i:101-111, 132-169, 573-589)."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("gen_tables", os.path.join(root, "tools", "gen_tables.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    tracked = open(gen.OUT).read()
    gen.OUT = str(tmp_path / "minsnap_tables.h")
    gen.main()
    assert open(gen.OUT).read() == tracked, "run python tools/gen_tables.py"

    def table(name):
        m = re.search(name + r"\[\d+\] = \{(.*?)\};", tracked, re.S)
        return np.array([float(x) for x in m.group(1).replace("\n", " ").split(",") if x.strip()])

    a1 = table("kA1inv_N10").reshape(10, 10)
    h1 = table("kH1_N10_d4").reshape(10, 10)
    A = np.array(oracle.mapping_matrix(10, 1.0)).reshape(10, 10)
    assert np.abs(a1 @ A - np.eye(10)).max() <= 1e-9
    H = np.array(oracle.segment_hessian(10, 4, 1.0)).reshape(10, 10)
    assert np.abs(h1 - H).max() <= 1e-7 * np.abs(H).max()   # the oracle's A^-T Q A^-1 carries the cancellation
    roles = table("kRecoveryRoles_N10").reshape(2, 54)
    sign = np.array([-1.0, 1.0, -1.0, 1.0])
    for i in range(5, 10):
        for role in (0, 1):
            row = roles[role, (i - 5) * 9:(i - 4) * 9]
            assert row[0] == a1[i, 5]
            new_cols, old_cols = (a1[i, 6:10], a1[i, 1:5]) if role else (a1[i, 1:5], a1[i, 6:10])
            flip = sign if role else np.ones(4)
            assert np.array_equal(row[1:5], flip * new_cols) and np.array_equal(row[5:9], flip * old_cols)
    diag = np.array([a1[k, k] for k in range(1, 5)])
    assert np.array_equal(roles[0, 45:49], diag) and np.array_equal(roles[1, 49:53], sign * diag)
    assert not roles[0, 49:53].any() and not roles[1, 45:49].any()
    cost = table("kCostForm_N10_d4")
    rows = [5, 1, 2, 3, 4, 6, 7, 8, 9]
    u = np.random.default_rng(3).normal(size=9)
    packed = sum(u[r] * sum(cost[r * (r + 1) // 2 + s] * u[s] for s in range(r + 1)) for r in range(9))
    full = sum(h1[rows[r], rows[s]] * u[r] * u[s] for r in range(9) for s in range(9))
    assert abs(packed / full - 1.0) <= 1e-12

"""Dry run, on CPU, of the GPU test modules that were written after this round's GPU time was spent: the Python harness is pointed
at the CPU test double of the device entry points (tests/mock/sb200_cpu_double.cpp + the UNCHANGED host layer, as a shared library)
and every "device" tensor is a CPU tensor (tests/support/dry_run_gpu_tests.py).  This exercises the tests' and the harness's own
logic - ctypes signatures, argument order, sizes, the host orchestration in host/saddle.cpp - not the CUDA kernels."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = ["tests/mock/sb200_cpu_double.cpp", "spectral_petsc_b200/host/reference_api.cpp", "spectral_petsc_b200/host/petsc_shim.cpp",
       "spectral_petsc_b200/host/host_ilu.cpp", "spectral_petsc_b200/host/saddle.cpp", "spectral_petsc_b200/csrc/exact.cpp", "spectral_petsc_b200/csrc/cheb_matrix.cpp"]


@pytest.fixture(scope="module")
def libmock(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("mock") / "libsb200_cpu_double.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out] + [os.path.join(ROOT, s) for s in SRC])
    return out


@pytest.mark.parametrize("module,filters,expect", [
    ("test_zz1_gpu_saddle", [], 28),
    ("test_zz4_gpu_optins", [], 12),
    ("test_zz3_gpu_drivers", ["test_elliptic_config1_and_nonlinear", "test_stokes_continuation_and_vtk"], 2),
    ("test_gpu_solvers", [], 5),  # green on the B200 in round 1; kept here as the regression net of the Python solver orchestration
    # the row-wise bounds against oracle/highprec.py must also hold for the double's plain dense products: C is not too tight
    ("test_gpu_cheb", ["test_cheb_mult_matches_oracle", "test_misaligned_views"], 204),
    ("test_gpu_elliptic", ["test_function_and_matmult_match_oracle"], 25),
    ("test_gpu_stokes", ["test_shells_match_oracle"], 14),
])
def test_dry_run(libmock, module, filters, expect):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "support", "dry_run_gpu_tests.py"), libmock, module] + filters,
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "dry run: %d test invocations passed" % expect in r.stdout


def test_bench_extras_dry_run(libmock):
    """The per-P sweep and the KSP metric that bench.py runs in child processes: every row and key they are meant to produce."""
    import json

    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "support", "dry_run_bench_extras.py"), libmock], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    ops = [row["op"] for row in d["p_sweep"]]
    assert ops[:8] == ["StokesMatMult", "StokesMatMultVV", "StokesMatMultVP", "StokesMatMultPV", "StokesFunction", "StokesPCSetUp0 (device CSR)",
                       "StokesMatMult (evaluation switches off: three separate shells)", "StokesFunction (evaluation switches off: three separate shells)"]
    cfg = [(row["op"], row["dim"], row["launches"]) for row in d["p_sweep"] if "dim" in row]
    cfg = [c for c in cfg if not c[0].startswith("Stokes")]
    st20 = [row["op"] for row in d["p_sweep"] if row.get("dim") == "20x20x20"]
    assert st20 == ["StokesMatMult", "StokesMatMult (CUDA graph)", "StokesMatMultVV", "StokesMatMultVV (CUDA graph)", "StokesMatMultPV",
                    "StokesMatMultPV (CUDA graph)", "StokesMatMultVP", "StokesMatMultVP (CUDA graph)"]
    assert [c[:2] for c in cfg] == [("MatMult_Elliptic", "12x12x12x12x12"), ("FormFunction", "12x12x12x12x12"), ("MatMult_Elliptic (CUDA graph)", "12x12x12x12x12"),
                                    ("MatMult_Elliptic", "16x16x16"), ("FormFunction", "16x16x16"), ("MatMult_Elliptic (CUDA graph)", "16x16x16")]
    ell = [(row["P"], row["path"]) for row in d["p_sweep"] if row["op"] == "MatMult_Elliptic" and "P" in row]
    assert ell == [(16, "generic"), (17, "generic"), (32, "generic"), (32, "chain per axis"), (32, "persistent chain")]
    assert sum(row["op"] == "ChebMult" for row in d["p_sweep"]) == 6 and sum(row["op"].startswith("FormJacobian") for row in d["p_sweep"]) == 3
    k = d["ksp"]
    assert k["config1_elliptic16_exact2_pc_ilu2"]["iterations"] == 16 and k["config1_elliptic16_exact2_pc_lu"]["iterations"] == 13
    assert k["config1_elliptic16_exact2_pc_lu"]["norm_of_error"] < 1e-9 and k["fgmres30_cycle_128"]["iterations"] == 30
    dj = k["elliptic128_exact2_device_jacobi"]  # 16^3 in this dry run
    assert "error" not in dj and dj["reason"] == 2 and 20 < dj["iterations"] < 200 and dj["norm_of_error"] < 1e-8
    c4 = k["config4_stokes20_exact2_block_lu"]
    assert "error" not in c4 and c4["reason"] == 2 and abs(c4["iterations"] - 26) <= 1 and c4["norm_of_error_velocity"] < 1e-6  # 26: apps/stokes with ILU(2)
    assert c4["pc_host_standin_calls"] > 0 and c4["inner_iterations"]["velocity"] > 0 and c4["inner_iterations"]["schur"] > 0
    # the headline flow (bench.run_cuda at 16^3 over the double): every key of the JSON contract, both end-to-end legs
    line = d["line"]
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "roofline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["metric"] == "spectral MatMult GDOF/s (fp64)" and line["dtype"] == "f64" and line["value"] > 0 and line["warmup"] >= 3
    assert line["e2e"]["queued_equals_sync_call_bitwise"] is True and "submit" in line["e2e"]["api"]
    assert line["e2e"]["h2d_bytes_per_step"] == line["e2e"]["d2h_bytes_per_step"] == 8 * line["config"]["global_vec_len"]
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and line["roofline"]["traffic"] == 225293824


def test_smoke_dry_run(libmock):
    """__graft_entry__.smoke() with the harness pointed at the test double: the calls it makes and its oracle comparisons."""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "from support.dry_run_gpu_tests import patch\npatch(%r)\nimport __graft_entry__ as g\ng.smoke()\n") % (ROOT, os.path.join(ROOT, "tests"), libmock)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    assert "smoke ok" in r.stdout and "StokesMatMult" in r.stdout

"""bench.py's reference arm on CPU: one JSON line with the keys the driver reads (the CUDA arm needs a GPU and is exercised
on the B200 box); argument validation of the KSP / slab entry points that happens before any CUDA call."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_max

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "spectral MatMult GDOF/s (fp64)" and d["unit"] == "GDOF/s"
    assert d["higher_is_better"] is True and d["dtype"] == "f64" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "GDOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "128,128,128" in d["config"]["workload"]


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_result(tmp_path):
    """--dump-outputs DIR: the CUDA arm writes the MatMult_Elliptic result of its last timed step, float64 over the 126^3 interior
    nodes, and it is the oracle's MatMult_Elliptic of the benchmark's seeded state and input."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-extras",
                          "--no-ksp", "--no-stokes", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["parity"]["ok"]
    assert os.listdir(tmp_path) == ["matmult_elliptic.npy"]
    V = np.load(tmp_path / "matmult_elliptic.npy")
    assert V.dtype == np.float64 and V.shape == (126 ** 3,)
    sys.path.insert(0, ROOT)
    import bench

    O, U = bench.build_state_oracle(workers=os.cpu_count() or 1)
    assert rel_max(V, O.mat_mult(U)) < 1e-12


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_ksp_and_slab_argument_validation_before_cuda():
    import spectral_petsc_b200 as sp

    L = sp.lib()
    h = ctypes.c_void_p()
    assert L.sb200_ksp_create(ctypes.c_longlong(10), 0, ctypes.byref(h)) == 83      # restart out of range
    assert L.sb200_ksp_create(ctypes.c_longlong(10), 100, ctypes.byref(h)) == 83
    assert L.sb200_ksp_create(ctypes.c_longlong(-1), 30, ctypes.byref(h)) == 83
    dims = (ctypes.c_int * 3)(16, 16, 16)
    assert L.sb200_slab_geometry(3, dims, 0, 3, None, None, None, None, None, None) == 83  # 16 % 3 != 0
    assert b"divisible" in L.sb200_last_error()
    assert L.sb200_slab_geometry(3, dims, 0, 4, None, None, None, None, None, None) == 0
    assert L.sb200_ipc_handle_bytes() == 64


def test_secondary_measurements_are_isolated_in_child_processes(monkeypatch):
    """The per-P sweep and the KSP metric run as `bench.py --child NAME`; a child that fails (here: no CUDA device) or overruns its
    limit yields an error record for the JSON line instead of an exception in the process that holds the headline numbers."""
    sys.path.insert(0, ROOT)
    import bench

    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")  # the children inherit it: no device, on a GPU machine too
    r = bench.run_child("ksp", limit_s=300)
    assert set(r) == {"error"} and "no CUDA device" in r["error"]
    r = bench.run_child("p_sweep", limit_s=0.01)
    assert set(r) == {"error"} and "exceeded" in r["error"]

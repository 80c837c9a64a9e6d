#!/usr/bin/env python
"""bench.py - spectral MatMult throughput of the B200-native Chebyshev collocation operator.

Contract (see DESIGN.md "Measurement"):
  python bench.py --gpus N --steps K --warmup W            -> ONE JSON line (this repo's CUDA path)
  python bench.py --impl reference --gpus N --steps K ...   -> ONE JSON line (CPU restatement of the
                                                               reference's FFT path, all host cores)
  python bench.py ... --dump-outputs DIR                    -> also DIR/matmult_elliptic.npy, the last timed step's result
A "step" is one MatMult_Elliptic application (elliptic.C:297-339) on the 128^3 grid with a
variable-coefficient state (eta, deta, gradu populated by one FormFunction call, gamma=4, exponent=2),
on N(0,1) synthetic input (numpy default_rng(0)), SURVEY.md 8(d).
metric = "spectral MatMult GDOF/s (fp64)", N_dof = fields * prod(dim) = 2,097,152.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "spectral MatMult GDOF/s (fp64)"
UNIT = "GDOF/s"
DIM = [128, 128, 128]
GAMMA, EXPONENT = 4.0, 2.0
FP64_PEAK_FALLBACK_TFLOPS = 37.1  # round-1 measurement (profiles/r01_fp64_peak.jsonl); used only if the in-run measurement fails
WORKLOAD = "elliptic 3D -dim 128,128,128 MatMult_Elliptic, variable coefficients (gamma=4, exponent=2)"
PARITY_TOL = 1e-12  # BASELINE.json: MatMult output within 1e-12 relative (max norm) of the reference's FFT path


def sb200_env():
    """Every SB200_* variable the process sees (tuning / test hooks); recorded in the line so a run that set one says so."""
    return {k: v for k, v in sorted(os.environ.items()) if k.startswith("SB200_")}


def config_dict(world, extra=None):
    """The `config` object: identical keys in both arms (the driver compares them)."""
    m = int(np.prod(DIM))
    g = int(np.prod([p - 2 for p in DIM]))
    c = {"workload": WORKLOAD, "n_dof_per_step": m, "global_vec_len": g,
         "l2": "256 MiB flush between timed steps (per-step CUDA events, flush untimed)",
         "parallelism": ("slab%d: axis 0 cut over %d GPUs, axis-0 chain through NVLink peer memory inside the chain kernel" % (world, world)) if world > 1 else "single"}
    if extra:
        c.update(extra)
    return c


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def ncu_traffic():
    """DRAM bytes per step of the two persistent launches from the committed ncu --set full capture (None if absent)."""
    try:
        for name in ("r02_traffic.json", "r01_traffic.json"):
            f = os.path.join(ROOT, "profiles", name)
            if os.path.exists(f):
                d = json.load(open(f))
                return d["dram_bytes_per_step"], "profiles/%s (%s)" % (name, d.get("how", "ncu --set full, every launch of the step"))
    except Exception:
        pass
    return None, None


def alg_flops(dim):
    # SURVEY 8(d): 2*P flop per node per scalar axis-derivative, 2 derivatives per axis
    m = int(np.prod(dim))
    return sum(2 * (2 * p) for p in dim) * m


def alg_bytes(dim):
    # SURVEY 8(d): variable-coefficient MatMult_Elliptic = 8*(2g + (2+d)m)
    m = int(np.prod(dim))
    g = int(np.prod([p - 2 for p in dim]))
    return 8 * (2 * g + (2 + len(dim)) * m)


class ClockSampler:
    """Samples SM clock, power and throttle reasons through NVML every ~10 ms on a background thread for
    the whole measurement (the timed region is only milliseconds long, so nvidia-smi's 100 ms loop cannot
    see it).  Reports the median clock over the samples taken under load (GPU utilisation or power up)."""

    def __init__(self, gpu_index):
        import threading

        self.samples = []
        self.ok = False
        self._stop = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            # LOCAL_RANK indexes the visible devices; map through CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            try:
                phys = int(vis.split(",")[gpu_index]) if vis else gpu_index
            except (ValueError, IndexError):
                phys = gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.smax = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.ok:
            return out
        self._stop.set()
        self.t.join(timeout=2)
        nv = self.nv
        if not self.samples:
            return out
        pmax = max(p for _, p, _ in self.samples)
        pmin = min(p for _, p, _ in self.samples)
        thr = pmin + 0.5 * (pmax - pmin)
        load = [x for x in self.samples if x[1] >= thr] or self.samples
        out["sm_mhz"] = statistics.median(x[0] for x in load)
        out["sm_max_mhz"] = self.smax
        out["samples"] = len(self.samples)
        out["samples_under_load"] = len(load)
        out["power_w_max"] = pmax
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        seen = set()
        for _, _, rs in load:
            for k, bit in names.items():
                if rs & bit:
                    seen.add(k)
        out["reasons"] = sorted(seen)
        return out


def build_state_oracle(workers):
    """CPU restatement with the benchmark's synthetic state (used by cpu_baseline / --impl reference)."""
    from oracle.elliptic import MatElliptic

    O = MatElliptic(DIM, gamma=GAMMA, exponent=EXPONENT, workers=workers)
    Us = 0.1 * np.random.default_rng(1).standard_normal(O.g)
    O.form_function(Us)
    U = np.random.default_rng(0).standard_normal(O.g)
    return O, U


def _time_oracle(steps, warmup):
    """Times `steps` full MatMult_Elliptic applications of the oracle port on all host cores (after `warmup` untimed ones)."""
    cores = os.cpu_count() or 1
    O, U = build_state_oracle(workers=cores)
    for _ in range(warmup):
        O.mat_mult(U)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.mat_mult(U)
    dt = time.perf_counter() - t0
    return O.m * steps / dt / 1e9, dt / steps * 1e3, cores


def _oracle_child(steps, warmup):
    """Runs the oracle timing in a FRESH process whose environment lets scipy's FFT thread pool use every host core:
    torch.distributed.run exports OMP_NUM_THREADS=1 to its workers, which throttles the pool 3-4x (round 1's N>1 reference arm)."""
    cores = os.cpu_count() or 1
    env = dict(os.environ)
    env["OMP_NUM_THREADS"] = str(cores)
    env["SB200_REF_CHILD"] = "1"
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup)],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError("oracle child failed: " + (r.stderr or r.stdout)[-300:])
    d = json.loads(lines[-1])
    return d["value"], d["ms_per_step"], d["cores"]


def cpu_baseline(sample_steps=3):
    val, ms, cores = _oracle_child(sample_steps, 1)
    return {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d full MatMult_Elliptic applications at 128^3 by the numpy/scipy(pocketfft) restatement of the reference's FFT path "
                      "(FFTW/PETSc unavailable), scipy.fft workers=%d" % (sample_steps, cores),
            "ms_per_step": ms}


def run_reference(args):
    """The reference arm: the CPU restatement of the reference's FFT path (oracle/, the one other place bench.py may execute it),
    all host cores, each step one full MatMult_Elliptic at 128^3.  Under torchrun rank 0 alone measures."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if os.environ.get("SB200_REF_CHILD") == "1":
        val, ms, cores = _time_oracle(args.steps, args.warmup)
        print(json.dumps({"value": val, "ms_per_step": ms, "cores": cores}))
        return 0
    val, ms, cores = _oracle_child(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "each step = one full MatMult_Elliptic at 128^3 by the numpy/scipy(pocketfft) restatement of the reference's FFT path "
                                   "(a numpy port, not the reference binary: that cannot be built here - no FFTW/PETSc/MPI); timed in a child process "
                                   "with OMP_NUM_THREADS = host cores so that the launcher's thread limit does not apply"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def parity_check(G, U, V, torch, dist, world, rank, dev):
    """Hardware parity of the very vectors the timed loop used, at every N: V (the result of the last application) against the
    oracle's single-domain MatMult_Elliptic (computed once on rank 0 - the oracle is the checker here, nothing timed - and
    broadcast), max-norm relative error over all ranks; plus the count of device-side flag waits that timed out."""
    O_g = G.gtotal
    Vo = torch.empty(O_g, dtype=torch.float64, device=dev)
    if rank == 0:
        O, Uo = build_state_oracle(workers=os.cpu_count() or 1)
        Vo.copy_(torch.from_numpy(O.mat_mult(Uo)))
    if world > 1:
        dist.broadcast(Vo, src=0)
    sl = slice(G.goff, G.goff + G.g)
    err = float((V - Vo[sl]).abs().max()) if G.g else 0.0
    nonfinite = float((~torch.isfinite(V)).sum()) if G.g else 0.0
    tmo = float(G.slab_timeouts()) if world > 1 else 0.0
    t = torch.tensor([err, nonfinite, tmo], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    err, nonfinite, tmo = t.tolist()
    rel = err / float(Vo.abs().max())
    ok = bool(rel < PARITY_TOL and nonfinite == 0 and tmo == 0)
    return {"rel": rel, "tol": PARITY_TOL, "timeouts": int(tmo), "nonfinite": int(nonfinite), "ok": ok,
            "checked": "V of the last timed application on every rank vs the oracle's single-domain MatMult_Elliptic (max-norm relative, max over ranks)"}


STOKES_WORKLOAD = "stokes -rheology 1 -exponent 3 -eps 1e-4 at -dim 128,128,128: StokesMatMult (BASELINE config 5's operator)"


def stokes_secondary(sp, torch, dist, world, rank, dev, steps):
    """BASELINE config 5 at EVERY N (row g1 of the round-1 verdict): StokesMatMult (stokes.C:499-519) on the 128^3 grid with the
    power-law rheology state of one StokesFunction call, slab-partitioned over the N ranks; device-resident GDOF/s (4 DOF per node,
    per-step CUDA events, L2 flushed between steps, max over ranks) and hardware parity of the timed result against the oracle's
    single-domain StokesMatMult (rank 0 computes it once - the oracle is the checker, nothing timed - and broadcasts it).
    Every rank reaches every collective whatever fails locally (a failure is reported in the object, never raised)."""
    out = {"workload": STOKES_WORKLOAD, "n_gpus": world}
    dim, err, S = DIM, None, None
    m = int(np.prod(dim))
    gtot = 4 * int(np.prod([p - 2 for p in dim]))
    ms_local, rel_local, tmo_local = 1e30, 1e30, 0.0
    y = None
    try:
        S = sp.Stokes(dim, rheology=1, hardness=1.0, exponent=3.0, regularization=1e-4, gamma0=1.0, rank=rank, nranks=world)
        if world > 1:
            from spectral_petsc_b200 import dist as spd

            spd.attach_peers(S)
        S.set_dirichlet(torch.zeros(S.dv, dtype=torch.float64, device=dev))
        S.set_force(torch.zeros(S.g, dtype=torch.float64, device=dev))
        sl = slice(4 * S.goff, 4 * S.goff + S.g) if world > 1 else slice(0, S.g)
        xs = torch.from_numpy(0.1 * np.random.default_rng(1).standard_normal(gtot)[sl].copy()).to(dev)
        x = torch.from_numpy(np.random.default_rng(0).standard_normal(gtot)[sl].copy()).to(dev)
        y = torch.empty_like(x)
        S.function(xs, y)  # eta / deta / strain of the power-law state
        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        for _ in range(3):
            S.mat_mult(x, y)
        torch.cuda.synchronize()
    except Exception as e:
        err = "%s: %s" % (type(e).__name__, e)
    if world > 1:
        dist.barrier()
    if err is None:
        try:
            l0 = sp.launch_count()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for a, b in ev:
                flush.zero_()
                a.record()
                S.mat_mult(x, y)
                b.record()
            torch.cuda.synchronize()
            ms_local = sum(a.elapsed_time(b) for a, b in ev) / steps
            out["launches_per_step"] = (sp.launch_count() - l0) // steps
            tmo_local = float(S.slab_timeouts()) if world > 1 else 0.0
        except Exception as e:
            err = "%s: %s" % (type(e).__name__, e)
    # parity: the oracle's single-domain result of the same application
    yo = torch.zeros(gtot, dtype=torch.float64, device=dev)
    oerr = None
    if rank == 0:
        try:
            # in a fresh process whose environment lets the FFT thread pool use every host core (see _oracle_child)
            with tempfile.TemporaryDirectory() as td:
                f = os.path.join(td, "stokes_oracle.npy")
                env = dict(os.environ)
                env["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "stokes_oracle", "--out", f], capture_output=True, text=True,
                                   env=env, cwd=ROOT, timeout=600)
                if r.returncode != 0:
                    raise RuntimeError("oracle child failed: " + (r.stderr or r.stdout)[-300:])
                yo.copy_(torch.from_numpy(np.load(f)))
        except Exception as e:
            oerr = "%s: %s" % (type(e).__name__, e)
    if world > 1:
        dist.broadcast(yo, src=0)
    scale = float(yo.abs().max())
    if err is None and scale > 0:
        rel_local = float((y - yo[sl]).abs().max()) / scale if y.numel() else 0.0
        if not bool(torch.isfinite(y).all()):
            rel_local = 1e30
    t = torch.tensor([ms_local, rel_local, tmo_local, 1.0 if err else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, rel, tmo, bad = t.tolist()
    if S is not None:
        try:
            S.destroy()
        except Exception:
            pass
    if bad or oerr or scale == 0:
        out["error"] = err or oerr or "a rank failed (see its stderr)"
        return out
    fl = 24 * 2.0 * dim[0] * m  # SURVEY 8(d): 24 scalar axis-derivatives of 2P flop per node (18 executed: trace + folded pressure)
    out.update({"value": 4 * m / ms / 1e6, "unit": UNIT, "ms_per_step": ms, "steps": steps, "n_dof_per_step": 4 * m,
                "algorithmic_flops_per_step": fl, "achieved_tflops": fl / ms / 1e9,
                "parity": {"rel": rel, "tol": PARITY_TOL, "timeouts": int(tmo), "ok": bool(rel < PARITY_TOL and tmo == 0),
                           "checked": "y of the last timed StokesMatMult on every rank vs the oracle's single-domain StokesMatMult (max-norm relative, max over ranks)"}})
    return out


def ksp_secondary(sp, torch, dev, G128, U128):
    """Secondary metric of BASELINE.json: 'KSP time to rtol 1e-10'.
    (a) config 1, ./elliptic -dim 16,16,16 -exact 2 -ksp_rtol 1e-10: device FGMRES(30) on the MatShell; the preconditioning
        matrix is assembled on the device (FormJacobian = sb200_elliptic_jacobian_csr); the PC built from it is PETSc's own
        and out of scope, so a HOST stand-in applies it and its time is reported separately: ILU(2), what the reference sets
        in code (elliptic.C:183-184), and an exact LU;
    (b) 128^3: one full FGMRES(30) cycle (30 iterations, no PC) on the benchmark operator: operator time vs KSP vector work.
    Nothing here touches oracle/: exact solution and matrices come from the library itself."""
    import scipy.sparse as sps
    import scipy.sparse.linalg as spla

    out = {}
    dim = [16, 16, 16]
    u, u2, dirichlet = sp.elliptic_exact_solution(dim, 2)
    G = sp.Elliptic(dim, gamma=0.0)
    G.set_dirichlet(torch.from_numpy(dirichlet).to(dev))
    G.set_rhs(torch.from_numpy(u2).to(dev))
    F = G.form_function(torch.zeros(G.g, dtype=torch.float64, device=dev))
    rowptr, colidx, vals = [t.cpu().numpy() for t in G.jacobian_csr()]
    P = sps.csr_matrix((vals, colidx, rowptr), shape=(G.g, G.g))
    rhs = -F
    for name, solve in (("ilu2", sp.HostILU(P, 2).solve), ("lu", spla.splu(P.tocsc()).solve)):
        K = sp.KSP(G.g)
        K.set_operators(G, pc=lambda r, solve=solve: torch.from_numpy(solve(r.cpu().numpy())).to(dev))
        K.set_tolerances(rtol=1e-10)
        K.solve(rhs)  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dx = K.solve(rhs)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        r, t = K.result, K.times_ms
        out["config1_elliptic16_exact2_pc_%s" % name] = {
            "ksp_rtol": 1e-10, "pc": "host stand-in for PETSc's PC: " + ("ILU(2), the reference's in-code default" if name == "ilu2" else "exact LU (SuperLU)"),
            "iterations": r["its"], "reason": r["reason"], "time_ms_total": wall, "time_ms_operator": t["operator"], "time_ms_pc_host_standin": t["pc"],
            "time_ms_ksp_vector_work": t["ksp_vector_work"], "time_ms_without_pc": wall - t["pc"],
            "norm_of_error": float((dx.cpu() - torch.from_numpy(u)).abs().max())}
        K.destroy()
    G.destroy()
    try:
        out["config4_stokes20_exact2_block_lu"] = ksp_config4(sp, torch, dev)
    except Exception as e:  # written after the last GPU run of round 1: must not cost the figures above
        out["config4_stokes20_exact2_block_lu"] = {"error": "%s: %s" % (type(e).__name__, e)}
    try:
        out["elliptic128_exact2_device_jacobi"] = ksp_device_jacobi(sp, torch, dev, list(G128.dim))
    except Exception as e:  # written after the last GPU run of round 1: must not cost the figures above
        out["elliptic128_exact2_device_jacobi"] = {"error": "%s: %s" % (type(e).__name__, e)}
    for la, key in ((0, "fgmres30_cycle_128_no_lookahead"), (1, "fgmres30_cycle_128")):
        K = sp.KSP(G128.g)
        K.set_operators(G128)
        K.set_tolerances(rtol=1e-30, maxits=30)
        K.set_lookahead(la)
        K.solve(U128)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        K.solve(U128)
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        r, t = K.result, K.times_ms
        out[key] = {"iterations": r["its"], "time_ms_total": wall, "time_ms_operator": t["operator"], "time_ms_ksp_vector_work": t["ksp_vector_work"],
                    "ms_per_iteration": wall / max(r["its"], 1), "residual_reduction": r["rnorm"] / r["bnorm"],
                    "lookahead": la, "note": "sb200_ksp_set_lookahead(%d): %s" % (la, "step k+1 enqueued before the host reads the norm of step k (same iterates)" if la else "one host read per iteration before the next step is enqueued")}
        K.destroy()
    return out


def ksp_device_jacobi(sp, torch, dev, dim, maxits=3000):
    """'KSP time to rtol 1e-10' on the headline grid with NOTHING on the host: ./elliptic -dim 128,128,128 -exact 2 -ksp_rtol 1e-10
    -pc_type jacobi.  FGMRES(30) on the MatShell, the preconditioner the diagonal of the device-assembled finite-difference matrix
    (FormJacobian), applied on the device.  Jacobi is a weak PC (the reference's ILU(2) / hypre are PETSc's and out of scope), so the
    iteration count is large; what the figure shows is the cost per iteration of operator + Krylov vector work at this size."""
    u, u2, dirichlet = sp.elliptic_exact_solution(dim, 2)
    G = sp.Elliptic(dim, gamma=0.0)
    G.set_dirichlet(torch.from_numpy(dirichlet).to(dev))
    G.set_rhs(torch.from_numpy(u2).to(dev))
    F = G.form_function(torch.zeros(G.g, dtype=torch.float64, device=dev))
    rowptr, colidx, vals = G.jacobian_csr()
    counts = (rowptr[1:] - rowptr[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(G.g, device=rowptr.device), counts)
    diag = vals[colidx.long() == rows]
    assert diag.numel() == G.g
    del rows, counts, rowptr, colidx, vals
    K = sp.KSP(G.g)
    K.set_operators(G, pc=lambda r: r / diag)
    K.set_lookahead(1)  # (same iterates; the GPU does not idle on the host's per-iteration convergence read)
    rhs = -1.0 * F
    K.set_tolerances(rtol=1e-10, maxits=5)
    K.solve(rhs)  # warm-up: 5 iterations
    K.set_tolerances(rtol=1e-10, maxits=maxits)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dx = K.solve(rhs)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    r, t = K.result, K.times_ms
    res = {"dim": "x".join(str(p) for p in dim), "ksp_rtol": 1e-10, "pc": "Jacobi of the device-assembled FD matrix, applied on the device", "iterations": r["its"],
           "reason": r["reason"], "time_ms_total": wall, "ms_per_iteration": wall / max(r["its"], 1), "time_ms_operator": t["operator"], "time_ms_pc": t["pc"],
           "time_ms_ksp_vector_work": t["ksp_vector_work"], "residual_reduction": r["rnorm"] / r["bnorm"],
           "norm_of_error": float((dx.cpu() - torch.from_numpy(u)).abs().max())}
    K.destroy()
    G.destroy()
    return res


def ksp_config4(sp, torch, dev):
    """BASELINE config 4: ./stokes -dim 20,20,20 -exact 2 -ksp_type fgmres -ksp_rtol 1e-10, Schur block LU (README:44's inner
    settings -schur_ksp_max_it 3 -vel_ksp_max_it 4 -svel_ksp_type preonly).  Outer FGMRES and the whole saddle-point PC
    (StokesPCApply0: shells, three inner Krylov solves, scatters, null space) run on the device (sb200_ksp + sb200_saddle); the PC on
    MatVVPC is PETSc's (hypre in the README) and out of scope: a HOST ILU(2) of the device-assembled matrix stands in, timed separately."""
    import scipy.sparse as sps

    dim = [20, 20, 20]
    U, U2, dirichlet = sp.stokes_exact_solution(dim, 2)
    S = sp.Stokes(dim, rheology=0)
    S.set_dirichlet(torch.from_numpy(dirichlet.reshape(-1).copy()).to(dev))
    S.set_force(torch.from_numpy(U2).to(dev))
    F = S.function(torch.zeros(S.g, dtype=torch.float64, device=dev))
    rowptr, colidx, vals = [t.cpu().numpy() for t in S.pc_velocity_csr()]
    ilu = sp.HostILU(sps.csr_matrix((vals, colidx, rowptr), shape=(S.gv, S.gv)), 2)
    spent = {"s": 0.0, "calls": 0}

    def vpc(r):  # the stand-in: down, two triangular solves on the host, up (all of it counted as PC time)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        z = torch.from_numpy(ilu.solve(r.cpu().numpy())).to(dev)
        torch.cuda.synchronize()
        spent["s"] += time.perf_counter() - t0
        spent["calls"] += 1
        return z

    pc = sp.StokesSaddle(S, 0, velocity_pc=vpc, vel_max_it=4, schur_max_it=3, svel_preonly=True)
    K = sp.KSP(S.g)
    K.set_operators(S, pc=pc)
    K.set_tolerances(rtol=1e-10, maxits=400)
    rhs = -1.0 * F
    K.solve(rhs)  # warm-up
    spent["s"], spent["calls"] = 0.0, 0
    its0 = pc.inner_its
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dx = K.solve(rhs)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    r, its1 = K.result, pc.inner_its
    ve = torch.from_numpy(U).to(dev).reshape(-1, 4)[:, :3]
    res = {"ksp_rtol": 1e-10, "iterations": r["its"], "reason": r["reason"], "time_ms_total": wall, "time_ms_pc_host_standin": spent["s"] * 1e3,
           "pc_host_standin_calls": spent["calls"], "time_ms_without_pc_standin": wall - spent["s"] * 1e3, "time_ms_outer_operator": K.times_ms["operator"],
           "inner_iterations": {k: its1[k] - its0[k] for k in its1}, "norm_of_error_velocity": float((dx.reshape(-1, 4)[:, :3] - ve).abs().max()),
           "pc": "StokesPCApply0 on the device (sb200_saddle); velocity PC = host ILU(2) stand-in for PETSc's PC on MatVVPC"}
    K.destroy()
    pc.destroy()
    S.destroy()
    return res


def run_child(name, limit_s):
    """Run one of the secondary measurements (`bench.py --child NAME`) in its own process; returns its JSON or an error record."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", name], capture_output=True, text=True, timeout=limit_s, cwd=ROOT)
    except subprocess.TimeoutExpired:
        return {"error": "child '%s' exceeded %d s and was killed" % (name, limit_s)}
    except Exception as e:
        return {"error": "%s: %s" % (type(e).__name__, e)}
    lines = [l for l in r.stdout.splitlines() if l.startswith("{") or l.startswith("[")]
    if r.returncode != 0 or not lines:
        return {"error": "child '%s' exit %d: %s" % (name, r.returncode, (r.stderr or r.stdout).strip()[-400:])}
    try:
        return json.loads(lines[-1])
    except ValueError as e:
        return {"error": "child '%s' printed no JSON: %s" % (name, e)}


def child_main(name, out=None):
    """The body of `bench.py --child NAME` (N = 1 only): prints ONE JSON value."""
    if name == "stokes_oracle":
        # the checker of stokes_secondary: the oracle's single-domain StokesMatMult on the bench's synthetic vectors (CPU only)
        from oracle.stokes import StokesCtx

        gtot = 4 * int(np.prod([p - 2 for p in DIM]))
        O = StokesCtx(DIM, rheology=1, hardness=1.0, exponent=3.0, regularization=1e-4, gamma0=1.0, workers=os.cpu_count() or 1)
        O.function(0.1 * np.random.default_rng(1).standard_normal(gtot))
        np.save(out, O.mat_mult(np.random.default_rng(0).standard_normal(gtot)))
        return 0
    import torch

    import spectral_petsc_b200 as sp

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --child: no CUDA device")
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    if name == "p_sweep":
        from tools.p_sweep import config4_rows, config_rows, rows, stokes_rows

        flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        t_ex, extra = time.perf_counter(), []
        # one generator after the other, each in its own guard: an exception in one group of rows (the opt-in paths run here for the
        # first time on a GPU) keeps the rows measured so far and lets the next group run
        for gen in (stokes_rows, config_rows, config4_rows, rows):
            try:
                for row in gen(steps=5, dev=dev, flush=flush):
                    extra.append({k: (round(v, 6) if isinstance(v, float) else v) for k, v in row.items()})
                    if time.perf_counter() - t_ex > 90.0:
                        break
            except Exception as e:
                extra.append({"error": "%s: %s: %s" % (gen.__name__, type(e).__name__, e)})
            if time.perf_counter() - t_ex > 90.0:
                extra.append({"truncated": "90 s budget reached"})
                break
        print(json.dumps(extra))
    elif name == "ksp":
        G = sp.Elliptic(DIM, gamma=GAMMA, exponent=EXPONENT)
        G.form_function(torch.from_numpy(0.1 * np.random.default_rng(1).standard_normal(G.g)).to(dev))
        U = torch.from_numpy(np.random.default_rng(0).standard_normal(G.g)).to(dev)
        print(json.dumps(ksp_secondary(sp, torch, dev, G, U)))
    else:
        raise SystemExit("unknown child " + name)
    sys.stdout.flush()
    return 0


def dump_outputs(out_dir, V, G, torch, dist, world, rank, dev):
    """--dump-outputs DIR: what the last timed step returned to its caller, the MatMult_Elliptic result V over all interior
    nodes of the global grid, as DIR/matmult_elliptic.npy (float64, 126^3 values, 16 MB).  The inputs are seeded, so two
    builds run with the same arguments can be compared output for output."""
    if world > 1:  # each rank holds its slab of V: place it in a zero global vector and sum (exact, the slabs are disjoint)
        full = torch.zeros(G.gtotal, dtype=torch.float64, device=dev)
        full[G.goff:G.goff + G.g] = V
        dist.all_reduce(full)
        V = full
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "matmult_elliptic.npy"), V.cpu().numpy())


def run_cuda(args):
    import torch
    import torch.distributed as dist

    import spectral_petsc_b200 as sp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # N > 1: slab partition along axis 0, one rank per GPU; the axis-0 chain crosses NVLink through peer
    # memory inside the chain kernel (no NCCL call on the data path).  Vectors are the ranks' local parts.
    G = sp.Elliptic(DIM, gamma=GAMMA, exponent=EXPONENT, rank=rank, nranks=world)
    if world > 1:
        from spectral_petsc_b200 import dist as spd

        spd.attach_peers(G)
    if args.path is not None:
        G.set_path(args.path)
    sl = slice(G.goff, G.goff + G.g)
    Us = torch.from_numpy(0.1 * np.random.default_rng(1).standard_normal(G.gtotal)[sl].copy()).to(dev)
    G.form_function(Us)  # populates eta / deta / gradu
    U_host = torch.from_numpy(np.random.default_rng(0).standard_normal(G.gtotal)[sl].copy()).pin_memory()
    V_host = torch.empty(G.g, dtype=torch.float64).pin_memory()
    U = U_host.to(dev)
    V = torch.empty_like(U)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # 256 MiB > 126 MB L2
    m_global = int(np.prod(DIM))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        G.mat_mult(U, V)
    barrier()

    # ---- device-resident timing: per-step CUDA events, L2 flushed between steps ----------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    l0 = sp.launch_count()
    barrier()
    for a, b in ev:
        flush.zero_()
        a.record()
        G.mat_mult(U, V)
        b.record()
    barrier()
    launches = sp.launch_count() - l0
    dump_dir = getattr(args, "dump_outputs", None)
    V_last = V.clone() if dump_dir else None  # (the L2-warm loop below overwrites V)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = sum(step_ms)
    # back-to-back (L2-warm) figure for context
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    hot_steps = max(args.steps, 2000)  # >= 0.2 s under load so the clock sampler sees the loaded state
    e0.record()
    for _ in range(hot_steps):
        G.mat_mult(U, V)
    e1.record()
    barrier()
    hot_ms = e0.elapsed_time(e1) * args.steps / hot_steps
    clocks = sampler.stop() if sampler else None

    # ---- hardware parity of the timed vectors (every N) and the FP64 tensor-pipe peak, both outside the timed regions ----------
    parity = parity_check(G, U, V, torch, dist, world, rank, dev)
    import ctypes as _ct
    peak_tf, peak_ms = _ct.c_double(0.0), _ct.c_double(0.0)
    peak_rc = sp.lib().sb200_fp64_dmma_peak(_ct.c_double(50.0), _ct.byref(peak_tf), _ct.byref(peak_ms))
    fp64_peak = peak_tf.value if (peak_rc == 0 and peak_tf.value > 1.0) else FP64_PEAK_FALLBACK_TFLOPS
    fp64_peak_source = ("measured in this run: sb200_fp64_dmma_peak, register-resident mma.sync.m8n8k4.f64 on every SM for %.0f ms (rank 0's GPU)" % peak_ms.value
                        if fp64_peak == peak_tf.value else "fallback: round-1 measurement 37.1 TFLOP/s (the in-run measurement failed)")

    # ---- end-to-end through the host-buffer C-ABI calls (H2D + op + D2H every step, all inside the timed region) ----------
    # (1) one synchronous call per step (sb200_elliptic_matmult_host): copy in, run, copy out, synchronise;
    # (2) the queued form (sb200_elliptic_matmult_host_submit / _wait): the same per-step copies from / to pinned host
    #     buffers, up to SB200_HOST_QUEUE_DEPTH applications in flight so a step's copy-in overlaps its predecessors'
    #     kernels and copy-out (full-duplex PCIe).  Every step's result lands in host memory before the clock stops.
    Uh, Vh = U_host.numpy(), V_host.numpy()
    lib = sp.lib()
    import ctypes
    hp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    for _ in range(2):
        lib.sb200_elliptic_matmult_host(G._h, hp(Uh), hp(Vh))
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rc = lib.sb200_elliptic_matmult_host(G._h, hp(Uh), hp(Vh))
        assert rc == 0
    barrier()
    e2e_sync_s = time.perf_counter() - t0

    depth = G.HOST_QUEUE_DEPTH
    e2e_steps = max(args.steps, 200)  # >= ~60 ms so the figure is a steady-state throughput, not the pipeline fill
    queue_ok, queue_err, e2e_s, nbar = False, None, e2e_sync_s, 0
    try:
        Uq = [U_host.clone().pin_memory().numpy() for _ in range(depth)]
        Vq = [torch.empty(G.g, dtype=torch.float64).pin_memory().numpy() for _ in range(depth)]
        G.mat_mult_host_stream(Uq, Vq)  # warm-up: builds the queue's streams and device vectors
        queue_ok = all(np.array_equal(v, Vh) for v in Vq)  # reported, not asserted: a raise on one rank would hang the others' barrier
        barrier()
        nbar = 1
        t0 = time.perf_counter()
        G.mat_mult_host_stream((Uq[i % depth] for i in range(e2e_steps)), (Vq[i % depth] for i in range(e2e_steps)))
        barrier()
        nbar = 2
        e2e_s = (time.perf_counter() - t0) * args.steps / e2e_steps
    except Exception as e:  # every rank still takes part in both barriers and the reductions below; the blocking call's figure stands in
        queue_ok, queue_err = False, "%s: %s" % (type(e).__name__, e)
        for _ in range(2 - nbar):
            barrier()
    if not queue_ok:  # a queued result that differs from the blocking call's is not a measurement: report the blocking call
        e2e_s = e2e_sync_s

    t = torch.tensor([total_ms, hot_ms, e2e_s * 1e3, e2e_sync_s * 1e3, 0.0 if queue_ok else 1.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, hot_ms, e2e_ms, e2e_sync_ms, any_queue_bad = t.tolist()
    if any_queue_bad:  # some rank fell back: the job-wide figure is the blocking call's
        e2e_ms, queue_ok = e2e_sync_ms, False

    # ---- BASELINE config 5's operator at this N (after and outside the headline's timed regions; collective: every rank takes part) ----
    stokes = None
    if not getattr(args, "no_stokes", False):
        del flush
        torch.cuda.empty_cache()
        try:
            stokes = stokes_secondary(sp, torch, dist, world, rank, dev, max(args.steps // 2, 5))
        except Exception as e:  # (only a failure of a collective itself lands here)
            stokes = {"workload": STOKES_WORKLOAD, "error": "%s: %s" % (type(e).__name__, e)}

    if rank == 0:
        ndof = m_global  # one global operator application per step, whatever the number of ranks
        value = ndof * args.steps / (total_ms * 1e-3) / 1e9
        fl = alg_flops(DIM)
        achieved = fl * args.steps / (total_ms * 1e-3) / 1e12
        peaks = measured_peaks()
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_src = ncu_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world),  # identical in both arms (the driver compares them)
            "value_l2_warm": ndof * args.steps / (hot_ms * 1e-3) / 1e9,  # back-to-back figure (no L2 flush between steps), for context
            "parity": parity,
            "env": sb200_env(),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": fp64_peak * world, "unit": "TFLOP/s", "frac": achieved / (fp64_peak * world),
                         "traffic": traffic if world == 1 else None, "traffic_source": traffic_src if world == 1 else None,
                         "pipe": "fp64 DMMA", "peak_source": fp64_peak_source + "; MEASURED_PEAKS.json has no fp64 entry",
                         "algorithmic_flops_per_step": fl, "kernel": G.kernel_name(),
                         "hbm": {"achieved": alg_bytes(DIM) * args.steps / (total_ms * 1e-3) / 1e9, "peak": hbm_peak * world, "unit": "GB/s",
                                 "frac": alg_bytes(DIM) * args.steps / (total_ms * 1e-3) / 1e9 / (hbm_peak * world), "algorithmic_bytes_per_step": alg_bytes(DIM)}},
            "e2e": {"value": ndof * args.steps / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": G.gtotal * 8, "d2h_bytes_per_step": G.gtotal * 8,
                    "api": ("sb200_elliptic_matmult_host_submit / _wait (pinned host buffers, <= %d applications in flight, %d steps timed)" % (depth, e2e_steps))
                           if queue_ok else "sb200_elliptic_matmult_host (one blocking call per step; the queued form was not usable: %s)" % (queue_err or "result differs"),
                    "sync_call_value": ndof * args.steps / (e2e_sync_ms * 1e-3) / 1e9, "sync_call_api": "sb200_elliptic_matmult_host (one blocking call per step)",
                    "queued_equals_sync_call_bitwise": bool(queue_ok)},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if stokes is not None:
            if "value" in stokes:
                stokes["frac_of_fp64_roofline"] = stokes["achieved_tflops"] / (fp64_peak * world)
            line["stokes"] = stokes
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline()
        # The per-P table of SURVEY 8d + set-up kernels (tools/p_sweep.py) and the secondary KSP metric run AFTER and OUTSIDE every timed
        # region above, each in a child process with its own CUDA context and a wall-clock limit: a crash, a sticky CUDA error or a
        # hang there is recorded in the line and cannot cost the headline numbers.
        if world == 1 and not args.no_extras:
            line["p_sweep"] = run_child("p_sweep", limit_s=240)
        if world == 1 and not args.no_ksp:
            line["ksp"] = run_child("ksp", limit_s=240)
        print(json.dumps(line))
    if dump_dir:
        dump_outputs(dump_dir, V_last, G, torch, dist, world, rank, dev)
    if world > 1:
        dist.destroy_process_group()
    if not parity["ok"]:
        sys.stderr.write("bench.py: PARITY FAILURE: %s\n" % json.dumps(parity))
        return 1
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline figure (value, ms_per_step); the context figures time max(STEPS, 2000) (value_l2_warm), "
                         "max(STEPS, 200) (e2e) and max(STEPS // 2, 5) (stokes) steps so that each is a steady-state measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--path", type=int, default=None, help="kernel path override (1 generic, 2 fused)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-P sweep (ChebMult, MatMult_Elliptic on every path, device FormJacobian)")
    ap.add_argument("--no-ksp", action="store_true", help="skip the secondary 'KSP time to rtol 1e-10' measurement")
    ap.add_argument("--no-stokes", action="store_true", help="skip the StokesMatMult 128^3 object (BASELINE config 5's operator at this N, with its parity check)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/matmult_elliptic.npy (float64) after the run")
    ap.add_argument("--child", default=None, choices=["p_sweep", "ksp", "stokes_oracle"], help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.child:
        return child_main(args.child, args.out)
    if args.impl == "reference":
        return run_reference(args)
    return run_cuda(args)


if __name__ == "__main__":
    sys.exit(main())

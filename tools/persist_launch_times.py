"""Per-launch kernel times of MatMult_Elliptic at P^3 (default path) from torch.profiler: the L2 is flushed before every
application, as in bench.py, and each kernel name gets its median / min / max device duration over the profiled steps.
Prints one JSON line per kernel name; run it on its own (the profiler slows the host, not the kernels it times).

usage: python tools/persist_launch_times.py [P] [steps]
"""
import json
import os
import statistics
import sys

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spectral_petsc_b200 as sp  # noqa: E402


def main():
    P = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 50
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    G = sp.Elliptic([P] * 3, gamma=4.0, exponent=2.0)
    G.form_function(torch.from_numpy(0.1 * np.random.default_rng(1).standard_normal(G.g)).to(dev))
    U = torch.from_numpy(np.random.default_rng(0).standard_normal(G.g)).to(dev)
    V = torch.empty_like(U)
    for _ in range(5):
        G.mat_mult(U, V)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            flush.zero_()
            G.mat_mult(U, V)
        torch.cuda.synchronize()
    times = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "persist_kernel" in ev.name:
            times.setdefault(ev.name, []).append(ev.time_range.elapsed_us())
    for name, us in sorted(times.items()):
        print(json.dumps({"P": P, "kernel": name, "launches": len(us), "us_median": statistics.median(us), "us_min": min(us), "us_max": max(us)}))
    G.destroy()


if __name__ == "__main__":
    main()

"""Multigrid-preconditioned CG (MultiGrid3D*.pcg) against the stationary V-cycle solve (solve) to the same target.

For each configuration, one JSON line with the card's name and power limit (read in this process), from the same start
(init_problem), fp64, MG_CORRECTED, rtol 1e-9 on the 2-norm of the residual:
  solve_ms / pcg_ms  -- medians of --reps alternating solve() and pcg() calls, host clock around the call (both are
                        synchronous, both run their loop on the device as one CUDA graph);
  cycles / iters     -- V-cycles solve() took, PCG iterations (one V-cycle each);
  kernels            -- the three vector passes of a PCG iteration (csrc/mg3d_cg.cu): mean GPU time per launch from the
                        CUPTI kernel records of one warm pcg() under torch.profiler, the bytes the pass moves (one read
                        or write of each field it touches, points of the grid only) and the achieved GB/s and fraction of
                        the measured copy peak (6451.8 GB/s, DESIGN.md section 4).
Every key is warmed up first: the first solve()/pcg() of a key runs host-driven, the second builds the graph.

    python scripts/bench_pcg.py [--reps 5] [--only cube1025,box1025x513x257,...]
"""
import argparse
import json
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import pde_multigrid_b200 as mg  # noqa: E402

COPY_PEAK_GBS = 6451.8
# fields each pass reads or writes once per point (csrc/mg3d_cg.cu)
PASS_FIELDS = {"k_pcg_dots": 3, "k_pcg_dir": 3, "k_pcg_upd": 7}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        power = None
    return name, power


def configs():
    C, f64 = mg.MG_CORRECTED, np.float64

    def cube(n, smoother=None):
        def make():
            e = mg.MultiGrid3D(n, dtype=f64, residual_mode=C)
            if smoother is not None:
                e.set_smoother(smoother)
            return e
        return make
    return [
        ("cube1025", cube(1025), (2, 2), (1025,) * 3),
        ("cube257", cube(257), (2, 2), (257,) * 3),
        ("cube257_jacobi", cube(257, mg.MG_SMOOTHER_JACOBI), (2, 2), (257,) * 3),
        ("cube257_v21", cube(257), (2, 1), (257,) * 3),
        ("box1025x513x257", lambda: mg.MultiGrid3DBox((1025, 513, 257), dtype=f64, residual_mode=C), (2, 2), (1025, 513, 257)),
    ]


def kernel_times(eng, v1, v2, rtol, cap):
    import os
    import tempfile

    from torch.profiler import ProfilerActivity, profile
    eng.init_problem()
    eng.sync()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        eng.pcg(v1, v2, rtol=rtol, max_iters=cap)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path))["traceEvents"]
    out = {}
    for ev in events:
        if ev.get("ph") != "X" or ev.get("cat") != "kernel":
            continue
        for k in PASS_FIELDS:
            if k in ev.get("name", ""):
                t = out.setdefault(k, [0.0, 0])
                t[0] += ev["dur"] / 1e3
                t[1] += 1
    return out


def measure(eng, v1, v2, rtol, cap, reps, points):
    for _ in range(2):
        eng.init_problem()
        eng.solve(v1, v2, rtol=0.0, max_cycles=2)
        eng.init_problem()
        eng.pcg(v1, v2, rtol=0.0, max_iters=2)
    eng.init_problem()
    s = eng.solve(v1, v2, rtol=rtol, max_cycles=cap)
    eng.init_problem()
    p = eng.pcg(v1, v2, rtol=rtol, max_iters=cap)
    t_solve, t_pcg = [], []
    for _ in range(reps):
        eng.init_problem()
        eng.sync()
        t0 = time.perf_counter()
        rs = eng.solve(v1, v2, rtol=rtol, max_cycles=cap)
        t_solve.append((time.perf_counter() - t0) * 1e3)
        assert rs.cycles == s.cycles and np.array_equal(rs.history, s.history)
        eng.init_problem()
        eng.sync()
        t0 = time.perf_counter()
        rp = eng.pcg(v1, v2, rtol=rtol, max_iters=cap)
        t_pcg.append((time.perf_counter() - t0) * 1e3)
        assert rp.cycles == p.cycles and np.array_equal(rp.history, p.history)
    kt = kernel_times(eng, v1, v2, rtol, cap)
    kernels = {}
    for k, (ms, n) in kt.items():
        per = ms / max(n, 1)
        gbytes = PASS_FIELDS[k] * points * 8 / 1e9
        kernels[k] = dict(launches=n, ms=per, gbytes=gbytes, gbs=gbytes / (per / 1e3), frac_copy_peak=gbytes / (per / 1e3) / COPY_PEAK_GBS)
    solve_ms, pcg_ms = statistics.median(t_solve), statistics.median(t_pcg)
    return dict(cycles=s.cycles, iters=p.cycles, solve_converged=s.converged, pcg_converged=p.converged,
                solve_final_rel=float(s.history[-1][0] / s.history[0][0]), pcg_final_rel=float(p.history[-1][0] / p.history[0][0]),
                solve_ms=solve_ms, pcg_ms=pcg_ms, speedup=solve_ms / pcg_ms,
                solve_ms_per_cycle=solve_ms / max(s.cycles, 1), pcg_ms_per_iter=pcg_ms / max(p.cycles, 1),
                solve_ms_all=t_solve, pcg_ms_all=t_pcg, kernels=kernels)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_pcg: no CUDA device (there is no CPU path)")
    torch.cuda.init()
    name, power = card()
    only = set(filter(None, args.only.split(",")))
    rtol, cap = 1e-9, 200
    for tag, make, (v1, v2), shape in configs():
        if only and tag not in only:
            continue
        eng = make()
        res = measure(eng, v1, v2, rtol, cap, args.reps, int(np.prod(shape)))
        eng.close()
        print(json.dumps(dict(config=tag, shape=shape, v1=v1, v2=v2, rtol=rtol, dtype="float64", gpu=name, power_limit_w=power, **res)),
              flush=True)


if __name__ == "__main__":
    main()

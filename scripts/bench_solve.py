"""Cost of the tolerance-driven solve against the loop a caller writes by hand.

For each configuration, one JSON line with the card's name and power limit (read in this process) and three timings
of the same number of cycles K, from the same start (init_problem), each the median of --reps alternating runs:
  solve     -- MultiGrid*.solve: the device loop (one graph launch and one wait per solve), host clock around the call;
  loop      -- residual_norm, then K x (VCycle + residual_norm): one read-back and one host wait per cycle, host clock;
  vcycle    -- K x VCycle alone, CUDA events on the engine's stream (no norm, no wait);
  norm      -- one residual_norm call (norm pass + read-back + wait), host clock: solve ~ vcycle + norm per cycle.
K is what the solve took to reach its target (or its cycle cap).  Every key is warmed up first: the first solve of a
key runs host-driven and the second builds the graph; the first VCycle of a key runs eagerly, the second captures.

    python scripts/bench_solve.py [--reps 5] [--only 3d257,2d,...]
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
    C = mg.MG_CORRECTED
    f64 = np.float64
    return [
        ("3d1025", lambda: mg.MultiGrid3D(1025, dtype=f64, residual_mode=C), (2, 2), 1e-9, 100),
        ("3d257", lambda: mg.MultiGrid3D(257, dtype=f64, residual_mode=C), (2, 2), 1e-9, 100),
        ("3d129", lambda: mg.MultiGrid3D(129, dtype=f64, residual_mode=C), (2, 2), 1e-9, 100),
        ("box1025x513x257", lambda: mg.MultiGrid3DBox((1025, 513, 257), dtype=f64, residual_mode=C), (2, 2), 1e-9, 100),
        ("2d1025", lambda: mg.MultiGrid2D(1025, dtype=f64), (2, 2), 1e-6, 200),
        ("1d1025_v1000", lambda: mg.MultiGrid1D(1025, dtype=f64, residual_mode=C), (1000, 1000), 1e-6, 100),
        ("1d1025_v2", lambda: mg.MultiGrid1D(1025, dtype=f64, residual_mode=C), (2, 2), 1e-6, 50),
    ]


def measure(eng, v1, v2, rtol, cap, reps):
    # warm-up: solve key (host-driven, then graph build + replay), cycle graph
    eng.solve(v1, v2, rtol=0.0, max_cycles=2)
    eng.solve(v1, v2, rtol=0.0, max_cycles=2)
    eng.init_problem()
    r = eng.solve(v1, v2, rtol=rtol, max_cycles=cap)
    K = r.cycles
    stream = torch.cuda.ExternalStream(eng.stream)
    t_solve, t_loop, t_vc, t_norm = [], [], [], []
    for _ in range(reps):
        eng.init_problem()
        eng.sync()
        t0 = time.perf_counter()
        rr = eng.solve(v1, v2, rtol=rtol, max_cycles=cap)
        t_solve.append((time.perf_counter() - t0) * 1e3)
        assert rr.cycles == K and np.array_equal(rr.history, r.history)

        eng.init_problem()
        eng.sync()
        t0 = time.perf_counter()
        eng.residual_norm(0)
        for _ in range(K):
            eng.VCycle(0, v1, v2)
            eng.residual_norm(0)
        t_loop.append((time.perf_counter() - t0) * 1e3)

        eng.init_problem()
        eng.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(K):
            eng.VCycle(0, v1, v2)
        e1.record(stream)
        eng.sync()
        t_vc.append(e0.elapsed_time(e1))

        t0 = time.perf_counter()
        eng.residual_norm(0)
        t_norm.append((time.perf_counter() - t0) * 1e3)
    per = lambda ts: statistics.median(ts) / max(K, 1)  # noqa: E731
    return dict(cycles=K, converged=r.converged, final_l2=float(r.history[-1][0]), l2_0=float(r.history[0][0]),
                solve_ms_per_cycle=per(t_solve), loop_ms_per_cycle=per(t_loop), vcycle_ms_per_cycle=per(t_vc),
                norm_ms=statistics.median(t_norm),
                solve_ms=statistics.median(t_solve), loop_ms=statistics.median(t_loop), vcycle_ms=statistics.median(t_vc),
                solve_ms_all=t_solve, loop_ms_all=t_loop)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_solve: no CUDA device (there is no CPU path)")
    torch.cuda.init()
    name, power = card()
    only = set(filter(None, args.only.split(",")))
    for tag, make, (v1, v2), rtol, cap in configs():
        if only and tag not in only:
            continue
        eng = make()
        res = measure(eng, v1, v2, rtol, cap, args.reps)
        eng.close()
        print(json.dumps(dict(config=tag, v1=v1, v2=v2, rtol=rtol, max_cycles=cap, dtype="float64", gpu=name, power_limit_w=power,
                              **res)), flush=True)


if __name__ == "__main__":
    main()

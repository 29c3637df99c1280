#!/usr/bin/env python3
"""tests/golden/make_level_paths.py -- the kernels each operator of a cubic 3D handle launches (test data).

Every case of CASES is one MultiGrid3D handle (smoother, size, dtype, range, arithmetic, MG_B200_FULL_CORRECTION) that runs the
calls of CALLS on level 0 in that order, each under its own torch.profiler session with CUDA activities.  The record of a call is
the ordered list of the kernels CUPTI saw (names without their argument lists) and the handle's kernel_launches count for it.
Graphs are off (MG_B200_NO_GRAPH), so a V-cycle's kernels show one by one.  Every kernel path gives the same bits, so only this
record shows which one a level took: tests/test_level_path_gpu.py runs this script and demands tests/golden/level_paths.json.
Needs a GPU:   MG_B200_NO_GRAPH=1 python tests/golden/make_level_paths.py [--out FILE]
"""
import argparse
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
GOLDEN = os.path.join(HERE, "level_paths.json")

RANGES = {
    "unit": (0, 1, 0, 1, 0, 1),
    # hy = hz = 2 hx: every h^2 is a power of two and den = 6 * 2^e still holds (fast_den), only iso is false
    "aniso": (0, 1, 0, 2, 0, 2),
    # h = 3/(n-1): h^2 is not a power of two (no fast_den)
    "h2_not_pow2": (0, 3, 0, 3, 0, 3),
}
SMOOTHERS = ("AUTO", "COLOUR", "FUSED", "JACOBI", "TMA", "PIPE")


def _case(smoother, n, dtype, rng="unit", arith="exact", full_correction=False):
    name = "%s/%d/%s/%s/%s" % (smoother, n, dtype, rng, arith) + ("/full_correction" if full_correction else "")
    return name, dict(smoother=smoother, n=n, dtype=dtype, range=rng, arith=arith, full_correction=full_correction)


CASES = dict(
    [_case(s, n, dt) for s in SMOOTHERS for n in (33, 129, 257) for dt in ("f32", "f64")] + [
        _case("AUTO", 257, "f64", arith="fast"),
        _case("AUTO", 257, "f64", rng="aniso"),
        _case("PIPE", 257, "f32", rng="aniso"),
        _case("AUTO", 257, "f64", rng="h2_not_pow2"),
        _case("PIPE", 257, "f32", rng="h2_not_pow2"),
        _case("AUTO", 33, "f64", rng="h2_not_pow2"),
        _case("AUTO", 257, "f64", full_correction=True),
        _case("COLOUR", 129, "f32", full_correction=True),
    ])

CALLS = (
    ("Relax(0,1)", lambda e: e.Relax(0, 1)),
    ("Relax(0,2)", lambda e: e.Relax(0, 2)),
    ("Relax(0,3)", lambda e: e.Relax(0, 3)),
    ("residual_norm(0)", lambda e: e.residual_norm(0)),
    ("residual_restrict(0)", lambda e: e.residual_restrict(0)),
    ("interpolate_correct(0)", lambda e: e.interpolate_correct(0)),
    ("VCycle(0,1,1)", lambda e: e.VCycle(0, 1, 1)),
    ("VCycle(0,2,2)", lambda e: e.VCycle(0, 2, 2)),
    ("VCycle(0,3,3)", lambda e: e.VCycle(0, 3, 3)),
)


def short_name(name):
    """`void (anonymous namespace)::k<double, 0>(double*, int)` -> `k<double, 0>`"""
    if name.endswith(")"):
        depth = 0
        for i in range(len(name) - 1, -1, -1):
            depth += {")": 1, "(": -1}.get(name[i], 0)
            if depth == 0:
                name = name[:i]
                break
    name = name[5:] if name.startswith("void ") else name
    return name[23:] if name.startswith("(anonymous namespace)::") else name


def record():
    """{case: {call: {"launches": int, "kernels": [names]}}}; MG_B200_NO_GRAPH must be set before the first handle exists."""
    assert os.environ.get("MG_B200_NO_GRAPH"), "graphs would hide the kernels of a V-cycle: set MG_B200_NO_GRAPH=1"
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    import pde_multigrid_b200 as mg
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]):  # CUPTI set up before the first recorded call
        torch.zeros(1, device="cuda")
        torch.cuda.synchronize()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        trace = os.path.join(tmp, "trace.json")
        for name, c in CASES.items():
            if c["full_correction"]:
                os.environ["MG_B200_FULL_CORRECTION"] = "1"
            else:
                os.environ.pop("MG_B200_FULL_CORRECTION", None)
            eng = mg.MultiGrid3D(c["n"], RANGES[c["range"]], dtype=np.float32 if c["dtype"] == "f32" else np.float64,
                                 residual_mode=mg.MG_CORRECTED)
            eng.set_smoother(getattr(mg, "MG_SMOOTHER_" + c["smoother"]))
            eng.set_arith(mg.MG_ARITH_FAST if c["arith"] == "fast" else mg.MG_ARITH_EXACT)
            rec = {}
            for call, fn in CALLS:
                eng.sync()
                before = eng.kernel_launches
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    fn(eng)
                    eng.sync()
                prof.export_chrome_trace(trace)
                with open(trace) as fh:
                    ev = [e for e in json.load(fh)["traceEvents"] if e.get("ph") == "X" and e.get("cat") == "kernel"]
                ev.sort(key=lambda e: float(e["ts"]))
                rec[call] = {"launches": eng.kernel_launches - before, "kernels": [short_name(e["name"]) for e in ev]}
            eng.close()
            out[name] = rec
    os.environ.pop("MG_B200_FULL_CORRECTION", None)
    return out


def dump(res, path):
    """one line per call: a changed path shows as a changed line"""
    lines = []
    for name, rec in res.items():
        calls = ["  %s: %s" % (json.dumps(call), json.dumps(r)) for call, r in rec.items()]
        lines.append(" %s: {\n%s\n }" % (json.dumps(name), ",\n".join(calls)))
    with open(path, "w") as fh:
        fh.write("{\n" + ",\n".join(lines) + "\n}\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=GOLDEN)
    args = ap.parse_args()
    res = record()
    dump(res, args.out)
    print(len(res), "cases ->", args.out)


if __name__ == "__main__":
    sys.exit(main())

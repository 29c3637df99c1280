"""GPU: the multigrid-preconditioned conjugate-gradient solve (mg3d_pcg / mg3b_pcg, MultiGrid3D*.pcg).

The engine runs the schedule of tests/pcg_mirror.py: its iteration counts must be the mirror's, its history the mirror's
up to the order of the fp64 sums, history[0] the bits of residual_norm and of solve().history[0]; f of the level comes
back bit for bit; the device loop, the host-driven first call, MG_B200_NO_GRAPH and a profiled run give the same bits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from pcg_mirror import make_oracle, pcg as mirror_pcg
from util import assert_bits_equal

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def engine(mg, kind, shape, dtype, smoother=None, mode=None):
    mode = mg.MG_CORRECTED if mode is None else mode
    if kind == "box":
        return mg.MultiGrid3DBox(shape, dtype=dtype, residual_mode=mode)
    e = mg.MultiGrid3D(shape[0], dtype=dtype, residual_mode=mode)
    if smoother is not None:
        e.set_smoother(smoother)
    return e


def snapshot(e, level=0):
    return e.get_v(level).copy(), e.get_f(level).copy()


# (kind, shape, dtype, v1, v2, smoother name, rtol)
F64, F32 = np.float64, np.float32
CASES = [
    ("cube", (33,), F64, 2, 2, "default", 1e-9),
    ("cube", (65,), F64, 2, 1, "default", 1e-9),
    ("cube", (129,), F64, 1, 1, "colour", 1e-9),
    ("cube", (257,), F64, 2, 2, "default", 1e-9),
    ("cube", (65,), F64, 2, 2, "jacobi", 1e-9),
    ("cube", (33,), F32, 2, 2, "default", 1e-4),
    ("cube", (65,), F32, 2, 1, "colour", 1e-4),
    ("cube", (257,), F32, 2, 2, "default", 1e-4),
    ("box", (33, 17, 9), F64, 2, 2, "default", 1e-9),
    ("box", (65, 33, 17), F64, 2, 1, "default", 1e-9),
    ("box", (129, 65, 33), F64, 2, 2, "default", 1e-9),
    ("box", (65, 33, 17), F32, 2, 2, "default", 1e-4),
]


def _smoother(mg, name):
    return {"default": None, "colour": mg.MG_SMOOTHER_COLOUR, "jacobi": mg.MG_SMOOTHER_JACOBI}[name]


def _rule(hist, thr):
    for k, (l2, _) in enumerate(hist):
        if not np.isfinite(l2) or l2 <= thr:
            return k
    return None


@pytest.mark.parametrize("kind,shape,dtype,v1,v2,sm,rtol", CASES, ids=lambda c: str(getattr(c, "__name__", c)))
def test_pcg_matches_the_mirror(mg, kind, shape, dtype, v1, v2, sm, rtol):
    k, conv, mh, _ = mirror_pcg(make_oracle(kind, shape, dtype), v1, v2, rtol=rtol, max_iters=60, jacobi=sm == "jacobi")
    e = engine(mg, kind, shape, dtype, _smoother(mg, sm))
    r0 = np.array(e.residual_norm(0))
    v0, f0 = snapshot(e)
    s0 = e.solve(v1, v2, rtol=0.0, max_cycles=0).history[0]
    tol = 1e-9 if dtype == F64 else 1e-4
    for call in range(2):  # the first call of a key runs host-driven, the second on the device
        e.set_v(0, v0)
        r = e.pcg(v1, v2, rtol=rtol, max_iters=60)
        assert_bits_equal(r.history[0], r0, "history[0] vs residual_norm")
        assert_bits_equal(r.history[0], s0, "history[0] vs solve().history[0]")
        assert r.cycles == k and r.converged == conv, (call, r.cycles, k, r.converged, conv, r.history[:, 0] / r.history[0, 0])
        j = min(5, k) + 1
        np.testing.assert_allclose(r.history[:j], mh[:j], rtol=tol, atol=0)
        assert_bits_equal(e.get_f(0), f0, "f after pcg")
        if conv:  # the returned v has the residual the history reports, and it meets the target
            thr = rtol * r0[0]
            assert r.history[-1, 0] <= thr
            l2 = e.residual_norm(0)[0]
            assert abs(l2 - r.history[-1, 0]) <= 1e-12 * r.history[-1, 0], (l2, r.history[-1, 0])
            assert l2 <= thr * (1 + 1e-12)
        if call == 0:
            v_first, h_first = e.get_v(0).copy(), r.history
        else:
            assert_bits_equal(e.get_v(0), v_first, "v: device loop vs host-driven first call")
            assert_bits_equal(r.history, h_first, "history: device loop vs host-driven first call")
    # the iteration count the rule gives on the mirror's history, tolerances at geometric midpoints
    for it in range(1, min(k, 5) + 1):
        if not mh[it, 0] < 0.5 * mh[it - 1, 0]:
            continue
        rt = np.sqrt(mh[it - 1, 0] * mh[it, 0]) / mh[0, 0]
        e.set_v(0, v0)
        r = e.pcg(v1, v2, rtol=rt, max_iters=60)
        assert r.cycles == _rule(mh, rt * mh[0, 0]) == it, (it, r.cycles)
    e.close()


@pytest.mark.parametrize("kind,shape", [("cube", (65,)), ("box", (65, 33, 17))])
def test_no_iteration_leaves_v_and_f(mg, kind, shape):
    e = engine(mg, kind, shape, F64)
    e.VCycle(0, 1, 1)  # a start with a nonzero interior
    v0, f0 = snapshot(e)
    for kw in (dict(max_iters=0), dict(atol=1e30), dict(rtol=2.0)):
        for _ in range(2):
            r = e.pcg(2, 2, **kw)
            assert r.cycles == 0 and r.history.shape == (1, 2)
            assert_bits_equal(e.get_v(0), v0, "v %r" % kw)
            assert_bits_equal(e.get_f(0), f0, "f %r" % kw)
    e.close()


@pytest.mark.parametrize("n,sm", [(65, "default"), (257, "default"), (65, "jacobi")])
def test_later_calls_match_a_fresh_handle(mg, n, sm):
    """after a pcg, VCycle and solve on the handle give the bits of a fresh handle holding the same v and f"""
    a = engine(mg, "cube", (n,), F64, _smoother(mg, sm))
    for _ in range(2):
        a.init_problem()
        a.pcg(2, 1, rtol=1e-6, max_iters=3)
    b = engine(mg, "cube", (n,), F64, _smoother(mg, sm))
    b.set_v(0, a.get_v(0))
    b.set_f(0, a.get_f(0))
    for e in (a, b):
        e.VCycle(0, 2, 1)
    assert_bits_equal(a.get_v(0), b.get_v(0), "VCycle after pcg")
    ra, rb = a.solve(2, 1, rtol=1e-3, max_cycles=20), b.solve(2, 1, rtol=1e-3, max_cycles=20)
    assert_bits_equal(ra.history, rb.history, "solve history after pcg")
    assert_bits_equal(a.get_v(0), b.get_v(0), "solve v after pcg")
    a.close()
    b.close()


def test_pcg_needs_fewer_cycles_where_the_cycle_is_weak(mg):
    e = engine(mg, "box", (129, 65, 33), F64)
    s = e.solve(2, 2, rtol=1e-9, max_cycles=200)
    e.init_problem()
    p = e.pcg(2, 2, rtol=1e-9, max_iters=200)
    assert s.converged and p.converged and 2 * p.cycles <= s.cycles, (p.cycles, s.cycles)
    e.close()
    e = engine(mg, "cube", (65,), F64, mg.MG_SMOOTHER_JACOBI)
    s = e.solve(2, 2, rtol=1e-9, max_cycles=200)
    e.init_problem()
    p = e.pcg(2, 2, rtol=1e-9, max_iters=200)
    assert s.converged and p.converged and p.cycles < s.cycles, (p.cycles, s.cycles)
    e.close()


def test_errors_run_nothing(mg):
    from pde_multigrid_b200._lib import MGError, MG_ERR_ARG, MG_ERR_STATE
    for kind, shape in (("cube", (33,)), ("box", (33, 17, 9))):
        e = engine(mg, kind, shape, F64, mode=mg.MG_REF_COMPAT)
        v0, f0 = snapshot(e)
        with pytest.raises(MGError) as ex:
            e.pcg()
        assert ex.value.code == MG_ERR_STATE
        assert_bits_equal(e.get_v(0), v0, "v")
        assert_bits_equal(e.get_f(0), f0, "f")
        e.close()
        e = engine(mg, kind, shape, F64)
        v0, f0 = snapshot(e)
        for kw in (dict(v1=-1), dict(rtol=-1.0), dict(atol=float("nan")), dict(max_iters=-1), dict(level=99)):
            with pytest.raises(MGError) as ex:
                e.pcg(**kw)
            assert ex.value.code == MG_ERR_ARG, kw
        assert_bits_equal(e.get_v(0), v0, "v")
        assert_bits_equal(e.get_f(0), f0, "f")
        e.close()


@pytest.mark.parametrize("kind,shape", [("cube", (65,)), ("box", (33, 17, 9))])
def test_nan_in_f_stops_at_once(mg, kind, shape):
    e = engine(mg, kind, shape, F64)
    f = e.get_f(0).copy()
    f[tuple(s // 2 for s in f.shape)] = np.nan
    e.set_f(0, f)
    for _ in range(2):
        r = e.pcg(2, 2, rtol=1e-9, max_iters=10)
        assert r.cycles == 0 and not r.converged and np.isnan(r.history[0]).all(), r
        assert_bits_equal(e.get_f(0), f, "f")
    e.close()


def test_jacobi_weight_change_matches_a_new_handle(mg):
    a = engine(mg, "cube", (65,), F64, mg.MG_SMOOTHER_JACOBI)
    for _ in range(2):
        a.init_problem()
        a.pcg(2, 2, rtol=1e-9, max_iters=20)
    a.set_jacobi_weight(0.8)
    a.init_problem()
    ra = a.pcg(2, 2, rtol=1e-9, max_iters=20)
    b = engine(mg, "cube", (65,), F64, mg.MG_SMOOTHER_JACOBI)
    b.set_jacobi_weight(0.8)
    rb = b.pcg(2, 2, rtol=1e-9, max_iters=20)
    assert_bits_equal(ra.history, rb.history, "history")
    assert_bits_equal(a.get_v(0), b.get_v(0), "v")
    a.close()
    b.close()


CHILD = r'''
import json, os, sys, ctypes
sys.path.insert(0, ".")
import numpy as np
import torch
import pde_multigrid_b200 as mg
from torch.profiler import profile, ProfilerActivity
out = sys.argv[1]
torch.cuda.init()
eng = mg.MultiGrid3D(65, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
box = mg.MultiGrid3DBox((65, 33, 17), dtype=np.float64, residual_mode=mg.MG_CORRECTED)
if os.environ.get("PCG_PROFILE"):
    eng._call("profile", ctypes.c_int(1))
for _ in range(2):  # host-driven first call, then the graph is built
    eng.init_problem(); eng.pcg(2, 2, rtol=0.0, max_iters=3)
    box.init_problem(); box.pcg(2, 2, rtol=0.0, max_iters=3)
eng.init_problem(); box.init_problem()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    r = eng.pcg(2, 2, rtol=0.0, atol=0.0, max_iters=7)
prof.export_chrome_trace(out + ".trace.json")
ev = json.load(open(out + ".trace.json"))["traceEvents"]
def count(pred):
    return sum(1 for e in ev if e.get("ph") == "X" and pred(e.get("name", ""), e.get("cat", "")))
counts = dict(graph_launch=count(lambda n, c: "GraphLaunch" in n and c in ("cuda_runtime", "cuda_driver")),
              runtime=count(lambda n, c: c == "cuda_runtime"),
              kernels=count(lambda n, c: c == "kernel"))
rb = box.pcg(2, 2, rtol=0.0, atol=0.0, max_iters=7)
np.savez(out, hist=r.history, cycles=r.cycles, v=eng.get_v(0), f=eng.get_f(0), bhist=rb.history, bv=box.get_v(0))
print("COUNTS", json.dumps(counts))
'''


def _child(tmp_path, tag, **env):
    out = str(tmp_path / tag)
    p = subprocess.run([sys.executable, "-c", CHILD, out], cwd=ROOT, env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    counts = json.loads(p.stdout.split("COUNTS", 1)[1].strip().splitlines()[0])
    print(tag, counts)
    return np.load(out + ".npz"), counts


def test_device_loop_and_fallbacks_agree(mg, tmp_path):
    dev, cd = _child(tmp_path, "device")
    host, _ = _child(tmp_path, "nograph", MG_B200_NO_GRAPH="1")
    prof, _ = _child(tmp_path, "profiled", PCG_PROFILE="1")
    assert int(dev["cycles"]) == 7
    for other, tag in ((host, "MG_B200_NO_GRAPH"), (prof, "profiling")):
        for k in dev.files:
            assert_bits_equal(dev[k], other[k], "%s: %s" % (tag, k))
    assert cd["kernels"] > 0, cd
    if cd["runtime"] > 0:  # the runtime calls are visible when CUPTI sees the library's own runtime
        assert cd["graph_launch"] == 1, cd


def test_debug_bounds_build_runs_pcg(mg):
    from pde_multigrid_b200.build import SO_DEBUG, build_debug_bounds
    syms = subprocess.run(["nm", "-D", "--defined-only", SO_DEBUG], capture_output=True, text=True).stdout if os.path.exists(SO_DEBUG) else ""
    if "mg3b_pcg" not in syms:
        build_debug_bounds()
    code = ("import sys; sys.path.insert(0, '.'); import numpy as np, pde_multigrid_b200 as mg\n"
            "e = mg.MultiGrid3D(129, dtype=np.float64, residual_mode=mg.MG_CORRECTED)\n"
            "a = e.pcg(2, 1, rtol=1e-8, max_iters=30); e.init_problem(); a = e.pcg(2, 1, rtol=1e-8, max_iters=30)\n"
            "b = mg.MultiGrid3DBox((65, 33, 17), dtype=np.float32, residual_mode=mg.MG_CORRECTED)\n"
            "c = b.pcg(2, 2, rtol=1e-4, max_iters=30); b.init_problem(); c = b.pcg(2, 2, rtol=1e-4, max_iters=30)\n"
            "print('PCG', a.cycles, a.converged, c.cycles, c.converged)\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, MG_B200_LIB=SO_DEBUG), capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0 and "PCG" in p.stdout and "MG_DEBUG_BOUNDS" not in p.stdout + p.stderr, p.stdout[-2000:] + p.stderr[-2000:]

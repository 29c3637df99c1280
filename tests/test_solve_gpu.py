"""GPU: the tolerance-driven solve (mg?d_solve, MultiGrid*.solve).

The device loop (one CUDA graph with a WHILE node) must give the bits of the hand-written loop
`VCycle + residual_norm`, stop where the rule max(atol, rtol * ||r_0||) says, agree with the host-driven
fallback, and really run on the device: O(1) launches, waits and read-backs per solve."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import assert_bits_equal, oracles

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DTYPES = [np.float32, np.float64]


def hand_loop(eng, v1, v2, cycles, level=0):
    h = [eng.residual_norm(level)]
    for _ in range(cycles):
        eng.VCycle(level, v1, v2)
        h.append(eng.residual_norm(level))
    return np.array(h, dtype=np.float64)


def assert_same_v(a, b, what):
    for l in range(a.numGrids):
        assert_bits_equal(a.get_v(l), b.get_v(l), "%s: v level %d" % (what, l))


def rule_cycles(hist, rtol, atol, max_cycles):
    """The stopping rule restated on a history of (l2, linf)."""
    thr = max(atol, rtol * hist[0][0])
    for k in range(len(hist)):
        l2 = hist[k][0]
        if not np.isfinite(l2) or l2 <= thr or k == max_cycles:
            return k
    raise AssertionError("history too short for the rule")


def check_against_hand_loop(make, v1, v2, level=0, n_device=3):
    """a: a host-driven solve of 2 cycles (the first solve of a key warms it up), then a device solve of n_device cycles;
    b: the hand-written loop over the same 2 + n_device cycles.  Then one more VCycle on both: the host-side state the solve
    left behind (ping-pong buffers of the 3D smoother) must be what the loop left."""
    a, b = make(), make()
    r1 = a.solve(v1, v2, rtol=0.0, atol=0.0, max_cycles=2, level=level)
    r2 = a.solve(v1, v2, rtol=0.0, atol=0.0, max_cycles=n_device, level=level)
    assert (r1.cycles, r1.converged, r2.cycles, r2.converged) == (2, False, n_device, False)
    h = hand_loop(b, v1, v2, 2 + n_device, level)
    assert_bits_equal(r1.history, h[:3], "history of the host-driven solve")
    assert_bits_equal(r2.history, h[2:], "history of the device solve")
    assert_same_v(a, b, "after the solves")
    a.VCycle(level, v1, v2)
    b.VCycle(level, v1, v2)
    assert_same_v(a, b, "after one more VCycle")
    assert a.residual_norm(level) == b.residual_norm(level)
    a.close()
    b.close()


VS = [(2, 2), (1, 1), (2, 1), (1, 2)]


@pytest.mark.parametrize("v1,v2", VS)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [33, 65, 129, 257, 513])
def test_3d_matches_hand_loop(mg, n, dtype, v1, v2):
    check_against_hand_loop(lambda: mg.MultiGrid3D(n, dtype=dtype, residual_mode=mg.MG_CORRECTED), v1, v2)


@pytest.mark.parametrize("v1,v2", [(2, 2), (2, 1)])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [33, 129, 257])
def test_3d_jacobi_matches_hand_loop(mg, n, dtype, v1, v2):
    def make():
        e = mg.MultiGrid3D(n, dtype=dtype, residual_mode=mg.MG_CORRECTED)
        e.set_smoother(mg.MG_SMOOTHER_JACOBI)
        return e
    check_against_hand_loop(make, v1, v2)


def test_3d_coarser_level_matches_hand_loop(mg):
    check_against_hand_loop(lambda: mg.MultiGrid3D(257, dtype=np.float64, residual_mode=mg.MG_CORRECTED), 2, 1, level=1)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(33, 17, 9), (65, 33, 17)])
def test_box_matches_hand_loop(mg, shape, dtype):
    check_against_hand_loop(lambda: mg.MultiGrid3DBox(shape, dtype=dtype, residual_mode=mg.MG_CORRECTED), 2, 2)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [65, 1025])
def test_2d_matches_hand_loop(mg, n, dtype):
    check_against_hand_loop(lambda: mg.MultiGrid2D(n, dtype=dtype), 2, 2)


@pytest.mark.parametrize("v1,v2", [(1000, 1000), (2, 2)])
def test_1d_matches_hand_loop(mg, v1, v2):
    check_against_hand_loop(lambda: mg.MultiGrid1D(1025, dtype=np.float64, residual_mode=mg.MG_CORRECTED), v1, v2)


def test_1d_tolerances(mg):
    """V(1000,1000) reaches rtol 1e-6; V(2,2) does not converge in 1D (SURVEY App. B13) and runs to max_cycles."""
    for (v1, v2), rtol, cap in (((1000, 1000), 1e-6, 50), ((2, 2), 1e-6, 50)):
        a = mg.MultiGrid1D(1025, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        b = mg.MultiGrid1D(1025, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        a.solve(v1, v2, rtol=0.0, max_cycles=1)  # warm-up of the key
        a.init_problem()
        r = a.solve(v1, v2, rtol=rtol, max_cycles=cap)
        h = hand_loop(b, v1, v2, r.cycles)
        assert_bits_equal(r.history, h, "1D V(%d,%d) history" % (v1, v2))
        assert r.cycles == rule_cycles(h, rtol, 0.0, cap)
        assert_same_v(a, b, "1D V(%d,%d)" % (v1, v2))
        if (v1, v2) == (2, 2):
            assert r.cycles == cap and not r.converged
        else:
            assert r.converged


def _warm_reset(eng, v1=2, v2=2):
    eng.solve(v1, v2, rtol=0.0, max_cycles=1)
    eng.init_problem()


@pytest.mark.parametrize("n,rtol,cycles", [(33, 1e-6, 7), (129, 1e-5, 6)])
def test_known_cycle_counts(mg, n, rtol, cycles):
    """SURVEY.md 8c, fp64 CORRECTED V(2,2) from v = 0: 33^3 to rtol 1e-6 stops after 7 cycles (r_6 = 6.45e-3 above
    1.895e-3, r_7 = 7.46e-4 below), 129^3 to rtol 1e-5 after 6."""
    for warm in (False, True):  # host-driven (first call of the key), then the device loop
        eng = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        if warm:
            _warm_reset(eng)
        r = eng.solve(2, 2, rtol=rtol, max_cycles=100)
        assert r.converged and r.cycles == cycles, (warm, r.cycles, r.history)
        if n == 33:
            assert abs(r.history[6][0] - 6.45e-3) < 0.01e-3 and abs(r.history[7][0] - 7.46e-4) < 0.01e-4
            assert abs(rtol * r.history[0][0] - 1.895e-3) < 0.001e-3
        eng.close()


@pytest.mark.parametrize("n", [33, 65])
def test_oracle_answers(mg, n):
    """v bit-exact against the oracle(s) after `cycles` V-cycles; the history within 1e-12; the cycle count the rule gives on
    the oracle's own history, with tolerances at the geometric midpoints between successive oracle norms."""
    orc = oracles(3, np.float64, True, n)
    ohist = [np.array(o.residual_norms(0)) for o in orc[:1]]
    o0 = orc[0]
    for _ in range(8):
        o0.vcycle(0, 2, 2)
        ohist.append(np.array(o0.residual_norms(0)))
    ohist = np.array(ohist)
    for o in orc:
        o.close()
    eng = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    _warm_reset(eng)
    for j in range(1, 8):
        rtol = np.sqrt(ohist[j - 1][0] * ohist[j][0]) / ohist[0][0]
        eng.init_problem()
        r = eng.solve(2, 2, rtol=rtol, max_cycles=100)
        want = rule_cycles(ohist, rtol, 0.0, 100)
        assert r.cycles == want == j, (j, r.cycles, want)
        np.testing.assert_allclose(r.history, ohist[: r.cycles + 1], rtol=1e-12, atol=0)
        for o in oracles(3, np.float64, True, n):
            for _ in range(r.cycles):
                o.vcycle(0, 2, 2)
            for l in range(eng.numGrids):
                assert_bits_equal(eng.get_v(l), o.v(l), "n=%d rtol at midpoint %d: v level %d vs %s" % (n, j, l, type(o).__name__))
            o.close()
    eng.close()


def test_stopping_rules(mg):
    n = 33
    ref = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    h = hand_loop(ref, 2, 2, 6)
    ref.close()
    eng = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    _warm_reset(eng)
    # a start that meets the target: no cycle, r_0 reported
    r = eng.solve(2, 2, rtol=0.0, atol=1e30)
    assert (r.cycles, r.converged) == (0, True)
    assert_bits_equal(r.history, h[:1], "r_0")
    # the cycle limit
    r = eng.solve(2, 2, rtol=0.0, atol=0.0, max_cycles=3)
    assert (r.cycles, r.converged) == (3, False)
    assert_bits_equal(r.history, h[:4], "max_cycles")
    # max_cycles = 0 with a target not met
    eng.init_problem()
    r = eng.solve(2, 2, rtol=1e-3, max_cycles=0)
    assert (r.cycles, r.converged, r.history.shape) == (0, False, (1, 2))
    # atol only and rtol only, placed between r_2 and r_3
    mid = np.sqrt(h[2][0] * h[3][0])
    for rtol, atol in ((0.0, mid), (mid / h[0][0], 0.0)):
        eng.init_problem()
        r = eng.solve(2, 2, rtol=rtol, atol=atol, max_cycles=100)
        assert (r.cycles, r.converged) == (3, True), (rtol, atol, r)
        assert_bits_equal(r.history, h[:4], "rtol %g atol %g" % (rtol, atol))
    # the larger of the two targets wins
    eng.init_problem()
    r = eng.solve(2, 2, rtol=mid / h[0][0], atol=np.sqrt(h[0][0] * h[1][0]), max_cycles=100)
    assert (r.cycles, r.converged) == (1, True)
    # bad arguments: MG_ERR_ARG, nothing runs, the handle stays usable
    eng.init_problem()
    for kw in (dict(rtol=-1.0), dict(atol=-1e-3), dict(max_cycles=-1), dict(level=eng.numGrids), dict(level=-1),
               dict(v1=-1), dict(rtol=float("nan"))):
        with pytest.raises(mg.MGError) as ei:
            eng.solve(**kw)
        assert ei.value.code == mg._lib.MG_ERR_ARG
    assert eng.residual_norm(0) == tuple(h[0])
    r = eng.solve(2, 2, rtol=0.0, max_cycles=2)
    assert_bits_equal(r.history, h[:3], "after the refused calls")
    eng.close()


def test_nan_stops_at_once(mg):
    for warm in (False, True):
        eng = mg.MultiGrid3D(33, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        if warm:
            _warm_reset(eng)
        f = eng.get_f(0)
        f[16, 16, 16] = np.nan
        eng.set_f(0, f)
        v = eng.get_v(0)
        r = eng.solve(2, 2, rtol=1e-8, max_cycles=10)
        assert (r.cycles, r.converged) == (0, False) and np.isnan(r.history[0][0])
        assert_bits_equal(eng.get_v(0), v, "v untouched")
        eng.close()


def test_ref_compat_does_not_converge(mg):
    """REF_COMPAT keeps the reference's sign defect of the residual, and its V-cycle diverges like the reference's."""
    eng = mg.MultiGrid3D(33, dtype=np.float64, residual_mode=mg.MG_REF_COMPAT)
    r = eng.solve(2, 2, rtol=1e-6, max_cycles=20)
    assert not r.converged
    eng.close()


def test_reuse_and_fmg(mg):
    """Two device solves in a row with other tolerances and limits, a VCycle in between, and an FMG start: the bits of the
    hand-written loop."""
    n = 129
    a = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    b = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    for e in (a, b):
        e.FullMultiGridVCycle(0, 1, 2, 2)
    r0 = a.solve(2, 2, rtol=0.0, max_cycles=1)  # warm-up: host-driven
    r1 = a.solve(2, 2, rtol=0.3, max_cycles=50)
    a.VCycle(0, 2, 2)
    r2 = a.solve(2, 2, rtol=1e-3, max_cycles=4)
    assert r1.converged and r1.cycles >= 1 and r2.cycles >= 1
    h0 = hand_loop(b, 2, 2, r0.cycles + r1.cycles)
    b.VCycle(0, 2, 2)
    h2 = hand_loop(b, 2, 2, r2.cycles)
    assert_bits_equal(np.vstack([r0.history, r1.history[1:]]), h0, "FMG + solve + solve")
    assert_bits_equal(r2.history, h2, "after the VCycle")
    assert_same_v(a, b, "reuse")
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
if os.environ.get("SOLVE_PROFILE"):
    eng._call("profile", ctypes.c_int(1))
warm = eng.solve(2, 2, rtol=0.0, max_cycles=2)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    r = eng.solve(2, 2, rtol=0.0, atol=0.0, max_cycles=12)
prof.export_chrome_trace(out + ".trace.json")
ev = json.load(open(out + ".trace.json"))["traceEvents"]
def count(pred):
    return sum(1 for e in ev if e.get("ph") == "X" and pred(e.get("name", ""), e.get("cat", "")))
counts = dict(graph_launch=count(lambda n, c: "GraphLaunch" in n and c in ("cuda_runtime", "cuda_driver")),
              sync=count(lambda n, c: "StreamSynchronize" in n and c in ("cuda_runtime", "cuda_driver")),
              runtime=count(lambda n, c: c == "cuda_runtime"),
              dtoh=count(lambda n, c: c == "gpu_memcpy" and "DtoH" in n),
              kernels=count(lambda n, c: c == "kernel"))
np.savez(out, hist=r.history, cycles=r.cycles, warm=warm.history, **{"v%d" % l: eng.get_v(l) for l in range(eng.numGrids)})
print("COUNTS", json.dumps(counts))
'''


def _child(tmp_path, tag, **env):
    out = str(tmp_path / tag)
    e = dict(os.environ, **env)
    p = subprocess.run([sys.executable, "-c", CHILD, out], cwd=ROOT, env=e, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    counts = json.loads(p.stdout.split("COUNTS", 1)[1].strip().splitlines()[0])
    print(tag, counts)
    return np.load(out + ".npz"), counts


def test_device_loop_runs_on_the_device_and_fallbacks_agree(mg, tmp_path):
    dev, cd = _child(tmp_path, "device")
    host, ch = _child(tmp_path, "nograph", MG_B200_NO_GRAPH="1")
    prof, _ = _child(tmp_path, "profiled", SOLVE_PROFILE="1")
    assert int(dev["cycles"]) == 12
    for other, tag in ((host, "MG_B200_NO_GRAPH"), (prof, "profiling")):
        for k in dev.files:
            assert_bits_equal(dev[k], other[k], "%s: %s" % (tag, k))
    # what the GPU did: the device loop reads back twice per solve (the parameter block, the history), the host loop once
    # per cycle; this is recorded by CUPTI's activity API, whichever CUDA runtime issued the copies
    assert cd["kernels"] > 0 and ch["kernels"] > 0, (cd, ch)
    assert cd["dtoh"] <= 3, cd
    assert ch["dtoh"] >= 12, ch
    # the runtime calls: visible when CUPTI sees the library's own (statically linked) runtime
    if ch["runtime"] > 0:
        assert cd["graph_launch"] <= 2 and cd["sync"] <= 3, cd
        assert ch["sync"] >= 12, ch


def test_debug_bounds_build_runs_a_solve(mg):
    from pde_multigrid_b200.build import SO_DEBUG, build_debug_bounds
    syms = subprocess.run(["nm", "-D", "--defined-only", SO_DEBUG], capture_output=True, text=True).stdout if os.path.exists(SO_DEBUG) else ""
    if "mg3d_solve" not in syms:
        build_debug_bounds()
    code = ("import sys; sys.path.insert(0, '.'); import numpy as np, pde_multigrid_b200 as mg\n"
            "e = mg.MultiGrid3D(257, dtype=np.float64, residual_mode=mg.MG_CORRECTED)\n"
            "e.solve(2, 1, rtol=0.0, max_cycles=2); r = e.solve(2, 1, rtol=1e-6, max_cycles=30)\n"
            "print('SOLVE', r.cycles, r.converged)\n")
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, MG_B200_LIB=SO_DEBUG), capture_output=True,
                       text=True, timeout=600)
    assert p.returncode == 0 and "SOLVE" in p.stdout and "MG_DEBUG_BOUNDS" not in p.stdout + p.stderr, p.stdout[-2000:] + p.stderr[-2000:]


def test_multi_gpu_solve_matches_single_gpu(mg):
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs (found %d)" % ngpu)
    for world in (2, 4, 8):
        if world > ngpu:
            break
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
               "127.0.0.1", "--master-port", "29547", os.path.join(ROOT, "tests", "solve_dist_check.py")]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
        assert "SOLVE_DIST_CHECK OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]

"""GPU: the CUDA-graph cache of V-cycles and solves.

A call that captures or replays a graph must leave the handle where the same call leaves it with MG_B200_NO_GRAPH=1: the
same v on every level, the same solve history, and kernel_launches and halo_bytes advanced by the same amounts.  Changing
the Jacobi weight must drop every graph that carries the old weight, cycle and solve graphs alike."""
import os
import subprocess
import sys

import numpy as np
import pytest

from util import assert_bits_equal

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

# (dim, n, smoother, v1, v2); smoother None = the engine's default.  V(2,1) ends a 3D cycle on the other v buffers of
# the levels the temporally blocked smoother runs on (257^3 with the default smoother).
CASES = [(2, 65, None, 2, 2), (2, 1025, None, 2, 2)] + [
    (3, n, sm, v1, v2) for n in (33, 257) for sm in ("colour", None) for v1, v2 in ((2, 2), (2, 1))]


def case_id(case):
    dim, n, sm, v1, v2 = case
    return "%dd_%d_%s_V%d%d" % (dim, n, sm or "default", v1, v2)


def levels(e):
    return [e.get_v(l) for l in range(e.numGrids)]


def counter_sequence(mg, case):
    """Four VCycles (eager, captured, replayed, replayed) and two solves (host-driven, then on the device): the counter
    deltas of every call, v on every level and both histories.  The first solve runs an even number of cycles, so the
    second starts on the buffers the first did and finds its key warm."""
    dim, n, sm, v1, v2 = case
    if dim == 2:
        e = mg.MultiGrid2D(n, dtype=np.float64)
    else:
        e = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        if sm == "colour":
            e.set_smoother(mg.MG_SMOOTHER_COLOUR)

    def counters():
        return (e.kernel_launches, e.halo_bytes if dim == 3 else 0)

    deltas, out = [], {}
    for i, call in enumerate(["vcycle"] * 4 + ["solve"] * 2):
        c0 = counters()
        if call == "vcycle":
            e.VCycle(0, v1, v2)
        else:
            out["hist%d" % i] = e.solve(v1, v2, rtol=0.0, atol=0.0, max_cycles=2 if i == 4 else 3).history
        deltas.append(np.subtract(counters(), c0))
    out["deltas"] = np.array(deltas, dtype=np.int64)
    for l, v in enumerate(levels(e)):
        out["v%d" % l] = v
    e.close()
    return out


def jacobi_sequence(mg, weight_first):
    """65^3 Jacobi.  weight_first: weight 0.5, then two VCycles and a solve.  Otherwise three VCycles and two solves at the
    default weight (both caches then hold graphs), weight 0.5, the initial problem again, and the same calls."""
    e = mg.MultiGrid3D(65, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
    e.set_smoother(mg.MG_SMOOTHER_JACOBI)
    if not weight_first:
        for _ in range(3):
            e.VCycle(0, 2, 2)
        for _ in range(2):
            e.solve(2, 2, rtol=0.0, atol=0.0, max_cycles=2)
    e.set_jacobi_weight(0.5)
    if not weight_first:
        e.init_problem()
    for _ in range(2):
        e.VCycle(0, 2, 2)
    out = {"hist": e.solve(2, 2, rtol=0.0, atol=0.0, max_cycles=3).history}
    for l, v in enumerate(levels(e)):
        out["v%d" % l] = v
    e.close()
    return out


def record(path):
    """Runs every sequence in this process and saves the results (the child process of the eager_run fixture)."""
    import pde_multigrid_b200 as mg
    res = {}
    for case in CASES:
        res.update({case_id(case) + "." + k: a for k, a in counter_sequence(mg, case).items()})
    res.update({"jacobi." + k: a for k, a in jacobi_sequence(mg, weight_first=False).items()})
    np.savez(path, **res)


@pytest.fixture(scope="module")
def eager_run(mg, tmp_path_factory):
    path = str(tmp_path_factory.mktemp("graph_cache") / "eager.npz")
    code = "import sys; sys.path[:0] = [%r, %r]; import test_graph_cache_gpu as t; t.record(%r)" % (ROOT, HERE, path)
    p = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, MG_B200_NO_GRAPH="1"),
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    return np.load(path)


def assert_same(got, want, prefix):
    for k, a in got.items():
        assert_bits_equal(a, want[prefix + "." + k], "%s: %s" % (prefix, k))


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_counters_and_bits_match_eager_calls(mg, eager_run, case):
    assert_same(counter_sequence(mg, case), eager_run, case_id(case))


def test_jacobi_weight_change_drops_cycle_and_solve_graphs(mg, eager_run):
    changed = jacobi_sequence(mg, weight_first=False)
    assert_same(changed, eager_run, "jacobi")
    fresh = jacobi_sequence(mg, weight_first=True)
    for k, a in changed.items():
        assert_bits_equal(a, fresh[k], "weight changed after graphs were captured vs set first: %s" % k)

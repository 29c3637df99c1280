"""CPU: the numpy mirror of the multigrid-preconditioned CG schedule (tests/pcg_mirror.py) on the C oracle's V-cycle.

The mirror is what tests/test_pcg_gpu.py holds the engine to, so it is pinned here: its iteration counts to rtol 1e-9
in fp64 from init_problem, that its last true residual really meets the target, and that in fp32 it stops at the
attainable floor and says so instead of declaring convergence early."""
import numpy as np
import pytest

from oracle import port
from pcg_mirror import make_oracle, pcg

CASES = [  # (kind, shape, v1, v2, jacobi, iterations)
    ("cube", (65,), 2, 2, False, 6),
    ("cube", (129,), 2, 1, False, 8),
    ("cube", (65,), 2, 2, True, 9),
    ("box", (129, 65, 33), 2, 2, False, 16),
    ("box", (65, 65, 17), 2, 2, False, 17),
]


@pytest.mark.parametrize("kind,shape,v1,v2,jacobi,iters", CASES, ids=lambda c: str(c))
def test_mirror_iteration_counts(kind, shape, v1, v2, jacobi, iters):
    m = make_oracle(kind, shape, np.float64)
    k, conv, hist, x = pcg(m, v1, v2, rtol=1e-9, max_iters=100, jacobi=jacobi)
    assert conv and k == iters, (k, conv, hist[:, 0] / hist[0, 0])
    assert hist[-1, 0] <= 1e-9 * hist[0, 0]
    # the history is the true residual of the returned iterate
    m.v(0)[...] = x
    m.f(0)[...] = make_oracle(kind, shape, np.float64).f(0)
    assert port.norms(m.residual(0))[0] == hist[-1, 0]


def test_mirror_beats_the_stationary_cycle_on_a_box():
    """the point of the feature: on an anisotropic box the stationary V-cycle contracts slowly"""
    kind, shape = "box", (65, 65, 17)
    m = make_oracle(kind, shape, np.float64)
    r0 = m.residual_norms(0)[0]
    cycles = 0
    while m.residual_norms(0)[0] > 1e-9 * r0:
        m.vcycle(0, 2, 2)
        cycles += 1
    assert cycles >= 2 * 17, cycles


def test_fp32_stops_at_the_floor_and_says_so():
    m = make_oracle("cube", (65,), np.float32)
    k, conv, hist, _ = pcg(m, 2, 2, rtol=1e-6, max_iters=40)
    rel = hist[:, 0] / hist[0, 0]
    assert not conv and k == 40, (k, conv, rel)
    assert np.all(rel[1:] > 1e-6) and np.min(rel) < 1e-4, rel


def test_max_iters_zero_and_converged_start_leave_the_data():
    m = make_oracle("cube", (33,), np.float64)
    v0, f0 = m.v(0).copy(), m.f(0).copy()
    k, conv, hist, x = pcg(m, max_iters=0)
    assert k == 0 and not conv and hist.shape == (1, 2) and np.array_equal(x, v0)
    k, conv, hist, x = pcg(make_oracle("cube", (33,), np.float64), atol=1e30)
    assert k == 0 and conv and np.array_equal(x, v0)
    assert np.array_equal(f0, make_oracle("cube", (33,), np.float64).f(0))

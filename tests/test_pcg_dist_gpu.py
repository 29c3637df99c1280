"""GPU (>= 2 devices): pcg on a distributed 3D handle reproduces the single-GPU pcg (tests/pcg_dist_check.py under torchrun,
one rank per GPU, on 2, 4 and 8 GPUs as far as the box has them), and the bounds-checked build runs it without a report
(the p and x updates write one plane beyond the owned ones).  Skipped on a one-GPU box."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worlds():
    import torch
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip("needs >= 2 GPUs (found %d)" % ngpu)
    return [w for w in (2, 4, 8) if w <= ngpu]


def run_check(world, env=None):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", "29561", os.path.join(ROOT, "tests", "pcg_dist_check.py")]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=1800, env=env)


def test_multi_gpu_pcg_matches_single_gpu(mg):
    for world in worlds():
        out = run_check(world)
        assert "PCG_DIST_CHECK OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


def test_multi_gpu_pcg_debug_bounds_build(mg):
    from pde_multigrid_b200.build import SO, SO_DEBUG, build_debug_bounds
    world = worlds()[-1]
    if not os.path.exists(SO_DEBUG) or os.path.getmtime(SO_DEBUG) < os.path.getmtime(SO):  # older than the library under test
        build_debug_bounds()
    out = run_check(world, dict(os.environ, MG_B200_LIB=SO_DEBUG, PCG_DIST_CHECK_RUNS="129:65"))
    text = out.stdout + out.stderr
    assert "PCG_DIST_CHECK OK" in out.stdout and "MG_DEBUG_BOUNDS" not in text, out.stdout[-3000:] + out.stderr[-3000:]

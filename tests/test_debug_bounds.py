"""compute-sanitizer is closed on the GPU pool, so the library has a checking build of its own: -DMG_DEBUG_BOUNDS puts an
index assertion (report, then retire the thread before the access) in front of the global-memory accesses of the 3D kernels (csrc/mg3d_device.cuh).
CPU: the checking build compiles (libmg_b200_dbg.so, shipped to the GPU box).  GPU: scripts/sanitize_smoke.py -- every kernel
family at 257^3 / 513^3 incl. the guard fallback -- runs clean against it, and a deliberately out-of-range launch IS reported
(so a silent pass means something)."""
import os
import subprocess
import sys

import pytest

from pde_multigrid_b200.build import build_debug_bounds

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DBG = os.path.join(ROOT, "pde_multigrid_b200", "libmg_b200_dbg.so")

BAD = r'''
import ctypes, sys
sys.path.insert(0, ".")
import torch
import pde_multigrid_b200 as mg
class Geom(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int), ("hp", ctypes.c_int), ("plane", ctypes.c_longlong), ("cstride", ctypes.c_longlong),
                ("z0", ctypes.c_int), ("nzl", ctypes.c_int)]
L = mg.lib()
n, hp = 33, 32
g = Geom(n, hp, hp * n, hp * n * n, 0, n)
buf = torch.zeros(4 * hp * n * n, dtype=torch.float64, device="cuda")
L.mgk3d_set.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, Geom, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int]
print("launch", L.mgk3d_set(None, 1, buf.data_ptr(), g, 1.0, 1, 0, n + 3))  # three planes past the end of the field
torch.cuda.synchronize()
print("RETURNED", float(buf[: 2 * hp * n * n].sum()))
'''


@pytest.fixture(scope="module")
def dbg(mg):
    """The checking build, compiled afresh once per run: a library left over from older sources would be tested instead."""
    return build_debug_bounds()


def test_checking_build_compiles(dbg):
    so = dbg
    assert so == DBG and os.path.exists(DBG)
    syms = subprocess.run(["nm", "-D", "--defined-only", DBG], capture_output=True, text=True).stdout
    assert "mg3d_vcycle" in syms


@pytest.mark.gpu
def test_every_kernel_family_runs_clean_under_the_bounds_checks(dbg):
    env = dict(os.environ, MG_B200_LIB=DBG)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "sanitize_smoke.py")], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=900)
    assert out.returncode == 0 and "sanitize_smoke ok" in out.stdout and "MG_DEBUG_BOUNDS" not in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


@pytest.mark.gpu
def test_an_out_of_range_launch_is_reported(dbg):
    env = dict(os.environ, MG_B200_LIB=DBG)
    out = subprocess.run([sys.executable, "-c", BAD], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    # the three planes past the end are reported by every thread that would have written them, and nothing is written there
    assert "MG_DEBUG_BOUNDS" in out.stdout and "RETURNED" in out.stdout, out.stdout[-1500:] + out.stderr[-1500:]

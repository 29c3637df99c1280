"""Equivalence of the drop-in shim with the reference's own classes, at the level the reference itself offers for looking at
a result: the text dump PrintDiff() writes to log/diff.txt (N3/Grid3D.cpp:136-159, N2/Grid2D.cpp:82-103, N1/Grid1D.cpp:46-60).

tests/compat/drv{1,2,3}d.cpp hold the calls of the reference's main()s with PrintDiff() switched on.  In a container with the
reference (CPU part) they are built twice: with the reference's unmodified .cpp files -- that run produced the committed
tests/golden/compat_diff_?d.txt (tests/golden/make_compat_golden.py) and is repeated here -- and against include/compat/ +
libmg_b200.so (binaries in tests/_build/).  On the GPU the shim binaries must write the same bytes:
3D 17^3 FMG(2,3,3) (with the reference's own residual signs the iteration blows up, any deviation would be amplified), 2D 33^2
FMG(1,20,20), 1D 129 FMG(2,100,100); and a non-cubic 33 x 17 x 9 grid (FMG(2,3,3) plus a hand-made cycle through the free-array
operators) whose reference side is the same classes compiled with -DNDEBUG.

The CUDA_TESI faces (-DMG_COMPAT_CUDA_TESI: d_v / d_f / d_sizeXYZ members, device-pointer operands, Set, (size, pitch)
signatures) cannot be pinned to the twin's numbers (its smoother races, SURVEY.md 0.6); tests/compat/drv?d_cuda.cpp do the
V-cycle by hand through those operators, in the twin's own call sequence, and compare with the object's VCycle."""
import filecmp
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")
REF = os.environ.get("MG_REFERENCE_ROOT", "/root/reference")
CUDA_HOME = os.environ.get("CUDA_HOME", "/usr/local/cuda")
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_compat_golden as golden  # noqa: E402

ARGS = {dim: c[2] for dim, c in golden.CASES.items()}


def shim_cmd(src, out, cuda_face=False):
    cmd = ["g++", "-O2", "-w", "-I", os.path.join(ROOT, "include", "compat"), "-I", os.path.join(ROOT, "include"), src, "-o", out,
           "-L", os.path.join(ROOT, "pde_multigrid_b200"), "-lmg_b200", "-Wl,-rpath,$ORIGIN/../../pde_multigrid_b200", "-lm"]
    if cuda_face:
        cmd[3:3] = ["-DMG_COMPAT_CUDA_TESI", "-I", os.path.join(CUDA_HOME, "include")]
        cmd += ["-L", os.path.join(CUDA_HOME, "lib64"), "-lcudart"]
    return cmd


def build_driver(dim, cuda_face=False):
    """tests/compat/drv<dim>[_cuda].cpp against the shim -> tests/_build/eq_{shim,cuda}_<dim>; the CPU and the GPU tests both call it."""
    os.makedirs(BUILD, exist_ok=True)
    src = os.path.join(ROOT, "tests", "compat", "drv%s%s.cpp" % (dim, "_cuda" if cuda_face else ""))
    exe = os.path.join(BUILD, "eq_%s_%s" % ("cuda" if cuda_face else "shim", dim))
    subprocess.run(shim_cmd(src, exe, cuda_face), check=True)
    return exe


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference sources not mounted")
@pytest.mark.parametrize("dim", ["1d", "2d", "3d", "3d_box"])
def test_reference_classes_reproduce_the_committed_dump(dim, tmp_path):
    """the reference side of the comparison, re-run: the committed golden file IS what the reference's classes write"""
    exe = str(tmp_path / ("ref_drv" + dim))
    golden.build_reference_side(dim, exe)
    (tmp_path / "log").mkdir()
    subprocess.run([exe] + list(ARGS[dim]), cwd=str(tmp_path), check=True, capture_output=True)
    assert filecmp.cmp(str(tmp_path / "log" / "diff.txt"), os.path.join(ROOT, "tests", "golden", "compat_diff_%s.txt" % dim), shallow=False)


@pytest.mark.parametrize("dim", ["1d", "2d", "3d", "3d_box"])
def test_shim_side_builds(mg, dim):
    build_driver(dim)


@pytest.mark.parametrize("dim", ["1d", "2d", "3d"])
def test_cuda_tesi_faces_build(mg, dim):
    build_driver(dim, cuda_face=True)


@pytest.mark.gpu
@pytest.mark.parametrize("dim", ["1d", "2d", "3d", "3d_box"])
def test_shim_writes_the_reference_dump_byte_for_byte(mg, dim, tmp_path):
    exe = build_driver(dim)
    (tmp_path / "log").mkdir()
    out = subprocess.run([exe] + list(ARGS[dim]), cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr
    got, want = str(tmp_path / "log" / "diff.txt"), os.path.join(ROOT, "tests", "golden", "compat_diff_%s.txt" % dim)
    if not filecmp.cmp(got, want, shallow=False):
        a, b = open(got).read().splitlines(), open(want).read().splitlines()
        bad = [(i, x, y) for i, (x, y) in enumerate(zip(a, b)) if x != y]
        raise AssertionError("%d of %d lines differ (%d vs %d lines), first: %r" % (len(bad), len(b), len(a), len(b), bad[:3]))


@pytest.mark.gpu
@pytest.mark.parametrize("dim", ["1d", "2d", "3d"])
def test_cuda_tesi_faces_run(mg, dim, tmp_path):
    exe = build_driver(dim, cuda_face=True)
    out = subprocess.run([exe], cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "CUDA_FACE OK" in out.stdout, out.stdout + out.stderr

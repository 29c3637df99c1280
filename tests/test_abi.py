"""CPU tests of the drop-in boundary (no GPU needed): the C-ABI library builds, loads, exports every
symbol declared in include/mg_b200.h, reports errors through status codes, and refuses to run without
a CUDA device (there is no CPU fallback)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mg_b200.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"\b(mg(?:[123]d|3b)?_[a-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_header_declares_the_reference_interface():
    names = declared_functions()
    for dim in ("1d", "2d", "3d"):
        for op in ("create", "destroy", "num_levels", "level_size", "relax", "residual", "restrict", "interpolate",
                   "set_to_value", "vcycle", "fmg", "restrict_host", "interpolate_host", "apply_correction_host",
                   "set_to_value_host", "vcycle_host", "residual_norm", "set_field", "get_field"):
            assert "mg%s_%s" % (dim, op) in names
    for op in ("create", "destroy", "num_levels", "level_size", "relax", "residual", "restrict", "residual_restrict", "interpolate",
               "interpolate_correct", "set_to_value", "vcycle", "fmg", "restrict_host", "interpolate_host", "apply_correction_host",
               "set_to_value_host", "vcycle_host", "residual_norm", "set_field", "get_field"):
        assert "mg3b_" + op in names  # the same interface for non-cubic grids


def test_library_exports_every_declared_symbol(mg):
    L = mg.lib()
    missing = [n for n in declared_functions() if not hasattr(L, n)]
    assert not missing, missing


def test_header_compiles_as_c_and_cxx(tmp_path):
    for comp, ext in (("gcc", "c"), ("g++", "cpp")):
        src = tmp_path / ("t." + ext)
        src.write_text('#include "mg_b200.h"\nint main(void){return MG_OK;}\n')
        subprocess.run([comp, "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src), "-o",
                        str(tmp_path / ("t_%s.o" % ext))], check=True)


NO_DEVICE = r'''
import sys
sys.path.insert(0, sys.argv[1])
import pde_multigrid_b200 as mg
assert mg.lib().mg_device_count() == 0
for ctor in (lambda: mg.MultiGrid3D(17), lambda: mg.MultiGrid2D(17), lambda: mg.MultiGrid1D(17), lambda: mg.MultiGrid3DBox((33, 17, 9))):
    try:
        ctor()
    except mg.MGError as e:
        assert e.code == 2 and "no CPU fallback" in str(e), e
    else:
        raise AssertionError("created an engine without a CUDA device")
print("NO_FALLBACK_OK")
'''


def test_no_cpu_fallback(mg):
    """Without a CUDA device create() must fail with MG_ERR_CUDA.  Checked in a child process that sees no device, so a
    machine with a GPU checks it as well."""
    out = subprocess.run([sys.executable, "-c", NO_DEVICE, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True, timeout=300)
    assert out.returncode == 0 and "NO_FALLBACK_OK" in out.stdout, out.stdout + out.stderr


def test_argument_validation_precedes_device_probe(mg):
    with pytest.raises(mg.MGError) as ei:
        mg.MultiGrid3D([17, 17, 9])
    assert ei.value.code == 1
    with pytest.raises(mg.MGError) as ei:
        mg.MultiGrid1D(100)
    assert ei.value.code == 1
    with pytest.raises(mg.MGError) as ei:
        mg.MultiGrid3DBox((33, 18, 9))  # every size must be 2^k + 1
    assert ei.value.code == 1


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pde_multigrid_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".c", ".cu", ".h", ".cuh")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "oracle" not in text.replace("parity oracle", "").replace("is the oracle", "").lower() or f == "build.py", \
                    "%s mentions the oracle" % f


def test_compat_shim_headers_compile(tmp_path):
    """The reference's class interface (include/compat/) compiles with g++ against mg_b200.h."""
    compat = os.path.join(ROOT, "include", "compat")
    if not os.path.isdir(compat):
        pytest.skip("compat shim not built yet")
    src = tmp_path / "t.cpp"
    src.write_text('#include "Grid3D.h"\n#include "MultiGrid3D.h"\n#include "Grid2D.h"\n#include "MultiGrid2D.h"\n'
                   '#include "Grid1D.h"\n#include "MultiGrid1D.h"\nint main(){return 0;}\n')
    subprocess.run(["g++", "-Wall", "-I", compat, "-I", os.path.join(ROOT, "include"), "-c", str(src), "-o",
                    str(tmp_path / "t.o")], check=True)


EXAMPLE = os.path.join(ROOT, "tests", "_build", "example_poisson3d")


def build_example(src, exe):
    """Compile examples/<src> against libmg_b200.so into tests/_build/<exe>; the CPU and the GPU tests both call it."""
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.run(["gcc", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "examples", src), "-o", exe,
                    "-L", os.path.join(ROOT, "pde_multigrid_b200"), "-lmg_b200",
                    "-Wl,-rpath,$ORIGIN/../../pde_multigrid_b200", "-lm"], check=True)


def test_c_example_builds_and_fails_loudly_without_a_gpu(mg):
    """examples/poisson3d_vcycle.c: the ABI from plain C.  On a machine without a GPU it must stop at mg3d_create with
    the no-CPU-fallback message, not compute anything."""
    build_example("poisson3d_vcycle.c", EXAMPLE)
    import torch
    if not torch.cuda.is_available():
        out = subprocess.run([EXAMPLE, "33", "1"], capture_output=True, text=True)
        assert out.returncode == 1 and "no CPU fallback" in out.stderr, out.stderr


@pytest.mark.gpu
def test_c_example_runs_on_the_gpu(mg):
    build_example("poisson3d_vcycle.c", EXAMPLE)
    out = subprocess.run([EXAMPLE, "65", "3"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    norms = [float(l.split("||r||_2 =")[1].split()[0]) for l in out.stdout.splitlines() if "||r||_2 =" in l]
    assert len(norms) == 3 and norms[2] < 0.2 * norms[1] < 0.04 * norms[0] * 5, out.stdout
    centre = float(out.stdout.split("v(centre) =")[1].split()[0])
    assert abs(centre - 1.0) < 0.01, out.stdout


EXAMPLE_BOX = os.path.join(ROOT, "tests", "_build", "example_poisson3d_box")


def test_c_example_for_a_non_cubic_grid_builds(mg):
    build_example("poisson3d_box.c", EXAMPLE_BOX)
    import torch
    if not torch.cuda.is_available():
        out = subprocess.run([EXAMPLE_BOX], capture_output=True, text=True)
        assert out.returncode == 1 and "no CPU fallback" in out.stderr, out.stderr


@pytest.mark.gpu
def test_c_example_for_a_non_cubic_grid_runs_on_the_gpu(mg):
    build_example("poisson3d_box.c", EXAMPLE_BOX)
    out = subprocess.run([EXAMPLE_BOX, "129", "65", "33", "6"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert "5 levels down to 9 x 5 x 3" in out.stdout, out.stdout
    r0 = float(out.stdout.split("||r0||_2 =")[1].split()[0])
    r1 = float(out.stdout.split("||r||_2 =")[1].split()[0])
    assert r1 < 0.1 * r0, out.stdout
    centre = float(out.stdout.split("v(centre) =")[1].split()[0])
    assert abs(centre - 1.0) < 0.01, out.stdout

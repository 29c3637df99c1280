"""CPU test (no GPU needed): the built library really carries the Blackwell data path the design claims -- sm_100a cubins whose
hot kernels issue TMA tensor loads (UTMALDG) tracked by mbarriers (SYNCS), and no library kernels.  Reads the SASS of
pde_multigrid_b200/libmg_b200.so with cuobjdump (B200_PROFILING.md names these mnemonics as the proof of TMA use)."""
import os
import re
import shutil
import subprocess

import pytest


@pytest.fixture(scope="module")
def sass(mg):
    from pde_multigrid_b200 import build
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.path.dirname(build.NVCC), "cuobjdump")  # else the toolkit that built the library
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found")
    import pde_multigrid_b200._lib as L
    out = subprocess.run([cuobjdump, "-sass", L.SO_PATH], capture_output=True, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = {"UTMALDG": 0, "SYNCS": 0, "UTMAPF": 0, "n": 0}
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            kernels[cur]["n"] += 1
            for k in ("UTMALDG", "SYNCS", "UTMAPF"):
                if re.search(r"\b%s\b" % k, line):
                    kernels[cur][k] += 1
    return set(re.findall(r"arch = (sm_\w+)", out)), kernels


def test_cubins_are_sm_100a_only(sass):
    archs, kernels = sass
    assert archs == {"sm_100a"}, archs
    assert len(kernels) > 50


@pytest.mark.parametrize("name", ["k_relax_pipe2", "k_relax_colour_tma", "k_residual_restrict_tma", "k_relax_fused2"])
def test_hot_kernels_use_tma_and_mbarriers(sass, name):
    _, kernels = sass
    mine = {k: v for k, v in kernels.items() if name in k}
    assert mine, "no kernel named %s in the library" % name
    for k, v in mine.items():
        assert v["UTMALDG"] > 0 and v["SYNCS"] > 0, (k, v)


def test_residual_restrict_prefetches_f_through_tma(sass):
    _, kernels = sass
    assert any(v["UTMAPF"] > 0 for k, v in kernels.items() if "k_residual_restrict_tma" in k)

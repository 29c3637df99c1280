"""Every operator of a cubic 3D handle launches the kernels it launched when tests/golden/level_paths.json was written.

The kernel families that can relax a level (pipelined two-sweep, shared-memory fused, TMA colour, plain colour, Jacobi) and
the riders on them (fused prolongation+correction, coarse tail, colour-1-only correction) all produce the same bits, so a
level that takes another path fails no bit test: only its speed changes.  tests/golden/make_level_paths.py records, per case,
the ordered kernel names torch.profiler sees for Relax(0, 1..3), residual_norm(0), residual_restrict(0),
interpolate_correct(0) and V(1,1), V(2,2), V(3,3) on level 0, with the launch count of each call; this test records them
again and demands the stored ones.
"""
import json
import os
import subprocess
import sys

import pytest

from golden_util import GOLDEN_DIR

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAKER = os.path.join(GOLDEN_DIR, "make_level_paths.py")

with open(os.path.join(GOLDEN_DIR, "level_paths.json")) as _fh:
    WANT = json.load(_fh)


@pytest.fixture(scope="module")
def recorded(mg, tmp_path_factory):
    """one child process records every case (the profiler stays out of this process); graphs off before any handle exists"""
    out = tmp_path_factory.mktemp("level_paths") / "level_paths.json"
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("MG_B200_NO_GRAPH", "1")
        mp.delenv("MG_B200_FULL_CORRECTION", raising=False)
        p = subprocess.run([sys.executable, MAKER, "--out", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    with open(out) as fh:
        return json.load(fh)


def test_every_case_is_recorded(recorded):
    assert sorted(recorded) == sorted(WANT)


@pytest.mark.parametrize("case", sorted(WANT))
def test_level_path_is_unchanged(recorded, case):
    got = recorded[case]
    for call, want in WANT[case].items():
        assert got[call] == want, "%s %s:\n  got  %s\n  want %s" % (case, call, got[call], want)

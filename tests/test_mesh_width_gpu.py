"""GPU: the exact-arithmetic shortcuts across mesh widths and across the exponent range, against the oracle.

The 3D engine is bit-identical to the reference, and much of its speed comes from shortcuts that are exact only under
stated conditions, all of which depend on h:
  * the temporally blocked smoother (k_relax_pipe2) computes (s6 - f h^2)/6 instead of the reference's h^4-weighted sum,
    behind an exponent-range check whose window depends on h;
  * the colour, TMA, fused, Jacobi and tail kernels divide by den = 6 h^4 with a Markstein quotient (fast_den);
  * the residual kernels multiply by 1/h^2 (fast_h).
Every other 3D test runs them with h = 2^-k, k >= 2, on the unit cube, or turns them all off (h not a power of two).
Here the cubic grids have power-of-two h on both sides of 1, on offset domains [-a, a]:
  h = 16, 4, 1, 2^-7 ([-1,1]^3), 2^-20, and in float 2^-37 (den = 6 h^4 is subnormal there),
at 257^3 (the coarser levels bring h*2, h*4, ... on the plain kernels and the <= 17^3 tail kernel), plus one 513^3 case
with h = 4.  Fields: uniform random, and two "edge" fields whose values sit around the thresholds where, for that h, one
of the reference's own products (x h^4, f h^2, f h^4, f h^6), its six-term sum or its quotient overflows or underflows,
computed below from the reference's arithmetic, plus -0, subnormals and +-inf.  Every path is compared bit for bit with
the oracle (oracle.port.PortMG, and the compiled reference when it is present); two NaNs compare equal whatever their
payload and sign (x86 and the GPU produce different ones, and the reference's results do not promise one).
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import oracles

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

N = 257
# log2(h) per dtype; h = 2^-37 is float's last h whose h^4 is nonzero
LOG2H = {np.float64: [4, 2, 0, -7, -20], np.float32: [4, 2, 0, -7, -20, -37]}
FIELDS = ["random", "top", "bottom"]
PATHS = ["AUTO", "TMA", "FUSED", "COLOUR", "JACOBI"]


def domain(n, log2h):
    a = 2.0 ** log2h * (n - 1) / 2
    return (-a, a) * 3


# ---- the comparator -------------------------------------------------------------------------------------------------
def assert_same(got, want, what):
    """Bit equality, except that any two NaNs are equal."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.dtype == want.dtype and got.shape == want.shape, what
    u = np.uint32 if got.dtype == np.float32 else np.uint64
    same = (got.view(u) == want.view(u)) | (np.isnan(got) & np.isnan(want))
    if not same.all():
        bad = np.argwhere(~same)
        first = tuple(bad[0])
        raise AssertionError("%s: %d of %d values differ (first at %s: %r vs %r)" % (what, len(bad), got.size, first, got[first], want[first]))


def test_comparator_treats_nans_alike_and_nothing_else():
    a = np.array([np.nan, -np.nan, 0.0, 1.0], dtype=np.float64)
    b = np.array([-np.nan, np.nan, 0.0, 1.0], dtype=np.float64)
    b[0] = np.frombuffer(np.uint64(0x7ff0000000000123).tobytes(), dtype=np.float64)[0]  # another payload
    assert_same(a, b, "nan payloads")
    for x, y in ((0.0, -0.0), (1.0, np.nextafter(1.0, 2.0)), (np.nan, np.inf)):
        with pytest.raises(AssertionError):
            assert_same(np.array([x]), np.array([y]), "")


# ---- edge fields ------------------------------------------------------------------------------------------------------
def thresholds(dtype, log2h):
    """Exponents t (|x| ~ 2^t) at which, for this h, an intermediate of the reference's Relax
        (O*(hy2*hz2) + ... + U*(hx2*hy2) - f*hx2*hy2*hz2) / (2*(hy2*hz2 + hx2*hz2 + hx2*hy2))
    or of its CalculateResidual (x / h^2) leaves the normal range, from the format's emax, emin and precision p.
    Returns (top, bottom): overflow thresholds and underflow thresholds."""
    fi = np.finfo(dtype)
    emax, emin, p = fi.maxexp, fi.minexp, fi.nmant  # |x| < 2^emax, normal from 2^emin, p fraction bits
    L = log2h
    top = [emax - 4 * L,                      # x h^4 overflows
           emax - 4 * L - 3,                  # the sum of six x h^4 overflows (6 < 2^3)
           emax - 2 * L, emax - 4 * L, emax - 6 * L,  # f h^2, f h^4, f h^6 overflow
           emax + 2 * L,                      # x / h^2 overflows (residual)
           emax - 1]                          # the top of the format: the smoother's own sums
    bottom = [emin - 4 * L, emin - p - 4 * L,  # x h^4 becomes subnormal / zero
              emin - 6 * L, emin - p - 6 * L,  # f h^6 becomes subnormal / zero
              emin + 2 * p + 4 - 4 * L,        # the numerator where a quotient's residual r = a - b q could be subnormal
              emin + 2 * L,                    # x / h^2 becomes subnormal (residual)
              emin]
    return top, bottom


def pipe_window(dtype, log2h):
    """The range check of k_relax_pipe2 as documented in mg3d_smooth_pipe.cu (h = 2^-k): values are accepted with
    2^lo <= |x| < 2^(hi+1).  Only used to put values just inside and just outside it."""
    k = -log2h
    kl, kh = max(k, 0), min(k, 0)
    if dtype == np.float64:
        return max(-857 + 6 * kl, -697 + 2 * kl) + 8, 1010 + 6 * kh
    return -122 + 6 * kl, 115 + 6 * kh


def edge_field(rng, n, dtype, log2h, kind):
    """'top': values around the overflow thresholds and just inside the window's upper end, capped at the upper end for
    h <= 1 (so that there the pass itself computes them, where a single value outside would send the whole pass to the
    fallback); 'bottom': values around the underflow thresholds and just inside / outside the window's lower end, -0,
    subnormals, +-inf.  A few hundred sprinkled points in v and f, and 3x3x3 blocks in which all six neighbours of a point
    are extreme; the rest uniform in [-1, 1]."""
    fi = np.finfo(dtype)
    emax, emin, p = fi.maxexp, fi.minexp, fi.nmant
    top, bottom = thresholds(dtype, log2h)
    lo, hi = pipe_window(dtype, log2h)
    if kind == "top":
        cap = pipe_window(dtype, 0)[1]
        centres = [min(t, cap) for t in top] + [hi]
    else:
        centres = bottom + [lo, lo - 1]
    exps = sorted({int(np.clip(c + d, emin - p, emax - 1)) for c in centres for d in range(-3, 3)})
    if kind == "top":
        exps = [e for e in exps if e <= cap]

    def values(m):
        e = rng.choice(exps, size=m)
        mant = rng.uniform(1.0, 2.0, size=m)
        sign = rng.choice([-1.0, 1.0], size=m)
        return (sign * np.ldexp(mant, e)).astype(dtype)

    v = rng.uniform(-1.0, 1.0, size=(n,) * 3).astype(dtype)
    f = rng.uniform(-1.0, 1.0, size=(n,) * 3).astype(dtype)
    for a in (v, f):
        idx = rng.integers(1, n - 1, size=(300, 3))
        a[idx[:, 0], idx[:, 1], idx[:, 2]] = values(len(idx))
        for _ in range(12):
            z, y, x = rng.integers(2, n - 4, size=3)
            a[z:z + 3, y:y + 3, x:x + 3] = values(1)[0] * rng.choice([-1.0, 1.0], size=(3, 3, 3)).astype(dtype)
    if kind == "bottom":
        specials = np.array([-0.0, fi.smallest_subnormal, -fi.smallest_subnormal * 7, fi.tiny / 2, np.inf, -np.inf], dtype=dtype)
        for a in (v, f):
            idx = rng.integers(1, n - 1, size=(24, 3))
            a[idx[:, 0], idx[:, 1], idx[:, 2]] = specials[np.arange(24) % len(specials)]
        v[n // 2, n // 2, n // 2 - 1:n // 2 + 2] = -0.0
    return v, f


@functools.lru_cache(maxsize=1)
def fields(n, dtype, log2h, kind):
    rng = np.random.default_rng([n, np.dtype(dtype).itemsize, log2h + 64, FIELDS.index(kind)])
    if kind == "random":
        return rng.uniform(-1.0, 1.0, size=(n,) * 3).astype(dtype), rng.uniform(-1.0, 1.0, size=(n,) * 3).astype(dtype)
    with np.errstate(all="ignore"):
        return edge_field(rng, n, dtype, log2h, kind)


def test_edge_bands_are_where_the_reference_leaves_the_normal_range():
    """The thresholds are where they say: a value one binade below a top threshold keeps that product finite, one binade
    above makes it inf (checked in the dtype's own arithmetic, as the reference computes it)."""
    for dtype in (np.float32, np.float64):
        for L in LOG2H[dtype]:
            h = dtype(2.0 ** L)
            h2 = h * h
            top, bottom = thresholds(dtype, L)
            with np.errstate(all="ignore"):
                for t, prod in ((top[0], lambda x: x * (h2 * h2)), (top[4], lambda x: x * h2 * h2 * h2)):
                    if np.finfo(dtype).minexp < t - 1 < np.finfo(dtype).maxexp:
                        assert np.isfinite(prod(dtype(np.ldexp(1.5, t - 2))))
                    if np.finfo(dtype).minexp < t < np.finfo(dtype).maxexp:
                        assert np.isinf(prod(dtype(np.ldexp(1.0, t))))
                t = bottom[1]  # x h^4 is zero below it, nonzero above
                if np.finfo(dtype).minexp - np.finfo(dtype).nmant < t - 2 and t + 2 < np.finfo(dtype).maxexp and h2 * h2 != 0:
                    assert (dtype(np.ldexp(1.0, t - 2)) * (h2 * h2)) == 0
                    assert (dtype(np.ldexp(1.0, t + 2)) * (h2 * h2)) != 0


# ---- engine and oracle runs -------------------------------------------------------------------------------------------
def make_engine(mg, n, dtype, log2h, path, corrected, v0, f0):
    eng = mg.MultiGrid3D(n, domain(n, log2h), dtype=dtype, residual_mode=mg.MG_CORRECTED if corrected else mg.MG_REF_COMPAT)
    eng.set_smoother(getattr(mg, "MG_SMOOTHER_" + path))
    eng.set_arith(mg.MG_ARITH_EXACT)
    eng.set_v(0, v0)
    eng.set_f(0, f0)
    return eng


CYCLES = ((2, 2), (2, 2), (2, 2), (2, 1), (2, 1))  # V(2,2): eager, captured, replayed; V(2,1): eager, captured


@functools.lru_cache(maxsize=2)
def oracle_run(n, dtype, log2h, kind, what, jacobi, corrected, cycles=CYCLES):
    """Snapshots of every oracle (port, and the compiled reference when present) for one sequence of calls; V-cycles:
    v of level 0 after every cycle, v and f of every level after the last."""
    v0, f0 = fields(n, dtype, log2h, kind)
    out = []
    with np.errstate(all="ignore"):
        for o in oracles(3, dtype, corrected, n, range=domain(n, log2h)):
            o.v(0)[...] = v0
            o.f(0)[...] = f0
            snaps = []
            if what in ("relax2", "relax3"):
                (o.relax_jacobi if jacobi else o.relax)(0, int(what[-1]))
                snaps.append([o.v(0).copy()])
            elif what == "residual":
                r = o.residual(0)
                snaps.append([r, o.restrict(r), np.zeros(o.shape(1), dtype=dtype)])
            else:
                for c, (v1, v2) in enumerate(cycles):
                    (o.vcycle_jacobi if jacobi else o.vcycle)(0, v1, v2)
                    last = c == len(cycles) - 1
                    levels = range(o.num_levels) if last else [0]
                    snaps.append([o.v(l).copy() for l in levels] + ([o.f(l).copy() for l in levels] if last else []))
            out.append((type(o).__name__, snaps))
    return out


def cases(with_paths, kinds=FIELDS):
    out = []
    for dtype in (np.float64, np.float32):
        for L in LOG2H[dtype]:
            for kind in kinds:
                for path in with_paths:
                    out.append(pytest.param(dtype, L, kind, path, id="%s-h2^%d-%s-%s" % (np.dtype(dtype).name, L, kind, path)))
    return out


def relax_cases():
    out = []
    for p in cases(PATHS):
        for nu in (2, 3):
            if p.values[3] != "TMA" or nu == 3:  # the TMA colour kernel with an odd number of sweeps
                out.append(pytest.param(*p.values, nu, id="%s-nu%d" % (p.id, nu)))
    return sorted(out, key=lambda q: q.id.rsplit("-", 2)[0] + q.id[-1])


@pytest.mark.parametrize("dtype,log2h,kind,path,nu", relax_cases())
def test_relax(mg, dtype, log2h, kind, path, nu):
    v0, f0 = fields(N, dtype, log2h, kind)
    eng = make_engine(mg, N, dtype, log2h, path, True, v0, f0)
    eng.Relax(0, nu)
    got = eng.get_v(0)
    eng.close()
    for name, snaps in oracle_run(N, dtype, log2h, kind, "relax%d" % nu, path == "JACOBI", True):
        assert_same(got, snaps[0][0], "Relax(0, %d) vs %s" % (nu, name))


def residual_cases():
    out = []
    for p in cases(["AUTO", "COLOUR"]):
        for corrected in (True, False):
            if corrected or p.values[1] in (4, -7):  # the reference's own residual (REF_COMPAT) on both sides of h = 1
                out.append(pytest.param(*p.values, corrected, id="%s-%s" % (p.id, "corrected" if corrected else "ref_compat")))
    return sorted(out, key=lambda q: q.id.rsplit("-", 2)[0] + q.id.rsplit("-", 1)[1])


@pytest.mark.parametrize("dtype,log2h,kind,path,corrected", residual_cases())
def test_residual_and_residual_restrict(mg, dtype, log2h, kind, path, corrected):
    """CalculateResidual (plain kernel) and residual_restrict(0) (the TMA kernel on AUTO, the plain one on COLOUR)."""
    v0, f0 = fields(N, dtype, log2h, kind)
    eng = make_engine(mg, N, dtype, log2h, path, corrected, v0, f0)
    r = eng.CalculateResidual(0)
    eng.residual_restrict(0)
    got = [r, eng.get_f(1), eng.get_v(1)]
    eng.close()
    for name, snaps in oracle_run(N, dtype, log2h, kind, "residual", False, corrected):
        for what, a, b in zip(("residual", "restricted residual (f, level 1)", "v level 1"), got, snaps[0]):
            assert_same(a, b, "%s vs %s" % (what, name))


def run_cycles(mg, n, dtype, log2h, kind, path, corrected, cycles=CYCLES):
    v0, f0 = fields(n, dtype, log2h, kind)
    eng = make_engine(mg, n, dtype, log2h, path, corrected, v0, f0)
    got = []
    for c, (v1, v2) in enumerate(cycles):
        eng.VCycle(0, v1, v2)
        last = c == len(cycles) - 1
        levels = range(eng.numGrids) if last else [0]
        got.append([eng.get_v(l) for l in levels] + ([eng.get_f(l) for l in levels] if last else []))
    eng.close()
    for name, snaps in oracle_run(n, dtype, log2h, kind, "vcycle", path == "JACOBI", corrected, cycles):
        for c, (a, b) in enumerate(zip(got, snaps)):
            nl = len(a) // 2 if c == len(cycles) - 1 else 1
            for j, (x, y) in enumerate(zip(a, b)):
                what = "%s level %d" % ("v" if j < nl else "f", j % nl)
                assert_same(x, y, "cycle %d V%s, %s vs %s" % (c + 1, cycles[c], what, name))


@pytest.mark.parametrize("dtype,log2h,kind,path", cases(PATHS, kinds=["random", "top"]))
def test_vcycles(mg, dtype, log2h, kind, path):
    """V(2,2) x 3 then V(2,1) x 2: on AUTO the post-smoothing of V(2,2) folds the prolongation into the pipe (CORR), V(2,1)
    does not; the levels <= 17^3 run in the tail kernel."""
    run_cycles(mg, N, dtype, log2h, kind, path, True)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("kind", ["random", "top"])
def test_vcycles_ref_compat_residual(mg, dtype, kind):
    run_cycles(mg, N, dtype, 4, kind, "AUTO", False)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_513_with_h_above_one(mg, dtype):
    """513^3 on [-1024, 1024]^3 (h = 4): the pipe on a 513^3 level, then the same kernels on 257^3 .. 3^3 with h = 8 .. 512."""
    n = 513
    v0, f0 = fields(n, dtype, 2, "top")
    eng = make_engine(mg, n, dtype, 2, "AUTO", True, v0, f0)
    eng.Relax(0, 2)
    got = eng.get_v(0)
    eng.close()
    for name, snaps in oracle_run(n, dtype, 2, "top", "relax2", False, True):
        assert_same(got, snaps[0][0], "513^3 Relax(0, 2) vs %s" % name)
    oracle_run.cache_clear()
    run_cycles(mg, n, dtype, 2, "top", "AUTO", True, cycles=((2, 2), (2, 1)))
    oracle_run.cache_clear()


# ---- route check: the cases above run the kernels they are meant to test ----------------------------------------------
CHILD = r'''
import json, sys
sys.path.insert(0, "tests")
sys.path.insert(0, ".")
import numpy as np
import torch
import pde_multigrid_b200 as mg
from torch.profiler import profile, ProfilerActivity
from test_mesh_width_gpu import N, fields, make_engine
out = sys.argv[1]
torch.cuda.init()
CASES = {  # name: (log2h, field, path, call)
    "pipe": (4, "random", "AUTO", "relax2"),
    "pipe_guard": (4, "top", "AUTO", "relax2"),
    "tma": (4, "random", "TMA", "relax3"),
    "fused": (4, "random", "FUSED", "relax2"),
    "colour": (4, "random", "COLOUR", "relax2"),
    "jacobi": (4, "random", "JACOBI", "relax2"),
    "rr": (4, "random", "AUTO", "rr"),
    "vcycle": (4, "random", "AUTO", "vcycle"),
}
res = {}
for name, (L, kind, path, call) in CASES.items():
    v0, f0 = fields(N, np.float64, L, kind)
    eng = make_engine(mg, N, np.float64, L, path, True, v0, f0)
    eng.Relax(0, 2); eng.VCycle(0, 2, 2)  # first launches outside the trace
    eng.set_v(0, v0)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        if call.startswith("relax"):
            eng.Relax(0, int(call[-1]))
        elif call == "rr":
            eng.residual_restrict(0)
        else:
            eng.VCycle(0, 2, 2)
        eng.sync()
    fn = out + "." + name + ".json"
    prof.export_chrome_trace(fn)
    k = {}
    for e in json.load(open(fn))["traceEvents"]:
        if e.get("ph") == "X" and e.get("cat") == "kernel":
            k[e["name"]] = k.get(e["name"], 0.0) + float(e.get("dur", 0.0))
    res[name] = k
    eng.close()
print("KERNELS", json.dumps(res))
'''


def test_cases_take_the_kernels_they_test(mg, tmp_path):
    p = subprocess.run([sys.executable, "-c", CHILD, str(tmp_path / "trace")], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    res = json.loads(p.stdout.split("KERNELS", 1)[1].strip().splitlines()[0])

    def ran(case, name):
        return sum(d for k, d in res[case].items() if name in k)

    def has(case, name):
        return any(name in k for k in res[case])

    assert has("pipe", "k_relax_pipe2<double, 0, false>"), res["pipe"]
    assert has("pipe_guard", "k_relax_pipe2<double, 0, false>"), res["pipe_guard"]
    # the literal-arithmetic pass behind the pipe is always enqueued and returns at once unless the range check fired
    assert has("pipe", "k_relax_fused2") and has("pipe_guard", "k_relax_fused2")
    assert ran("pipe_guard", "k_relax_fused2") > 4 * ran("pipe", "k_relax_fused2"), (res["pipe"], res["pipe_guard"])
    assert has("tma", "k_relax_colour_tma"), res["tma"]
    assert has("fused", "k_relax_fused2") and not has("fused", "k_relax_pipe2"), res["fused"]
    assert has("colour", "k_relax_colour<") and not has("colour", "k_relax_colour_tma"), res["colour"]
    assert has("jacobi", "k_jacobi_colour"), res["jacobi"]
    assert has("rr", "k_residual_restrict_tma"), res["rr"]
    assert has("vcycle", "k_relax_pipe2<double, 0, true>") and has("vcycle", "k_vcycle_tail"), res["vcycle"]

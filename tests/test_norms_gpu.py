"""GPU: residual_norm and the abs-error reductions of every engine against a high-precision reference.

r = CalculateResidual(level), whose bits the parity tests pin to the oracle, is the input.  The reference l2 is the square
root of the exact sum of r^2: the squares are split exactly (Dekker) and summed with math.fsum up to 2^22 terms, with a
pairwise np.longdouble sum above that (its own error, about log2(terms) * 2^-64 relative, is far below the bound).

Tolerance.  Every kernel squares in double and adds in double; a partial sum goes through at most m - 1 roundings of
additions on its longest chain (the terms one thread adds in sequence, the warp and block trees, the final reduction of
the per-block partials), plus the rounding of its own square: the computed sum is within gamma_m = m u / (1 - m u) of the
exact one (u = 2^-53), so l2 is within gamma_m / 2 + u (its square root's rounding) of the exact l2, plus u for the
rounding of the reference's own sum to double.  m is derived below from each kernel's launch shape.  linf must equal
max |r| exactly.

fp32 residuals are also run near 1e-30 and 1e30, where r^2 underflows or overflows in fp32: a path that squared in T
instead of double would return 0 or inf there.  A NaN in the residual gives (nan, nan) -- like np.max(np.abs(r)) --, an
inf gives (inf, inf), both give (nan, nan), on every engine, in the solve's first history entry, and in abs_error.
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
DTYPES = [np.float32, np.float64]
GENERAL = (0.25, 1.75, -0.5, 0.7, 0.1, 3.3)  # h not a power of two: the plain kernel even on a large level


def cdiv(a, b):
    return -(-a // b)


# ---- the longest chain of additions of each reduction (constants of csrc/) ---------------------------------------
BLOCK_TREE = 10  # warp shuffle (5 levels) + shuffle over the per-warp partials (5 levels) of a 256/1024-thread block


def chain_3d_plain(n):
    """k_residual_norm: MGK_NORM_BLOCKS = 1184 blocks of 256 threads over rows (y, z), a thread adds x = 1+t, 1+t+256, ...;
    k_norm_final: 256 threads over the 1184 partials."""
    rows = (n - 2) * n
    return cdiv(rows, 1184) * cdiv(n - 2, 256) + BLOCK_TREE + cdiv(1184, 256) + BLOCK_TREE


def chain_3d_tma(n):
    """k_residual_restrict_tma<NORM>: a 256-thread CTA owns 32 x 8 coarse points and zchunk coarse planes (2 * zchunk fine
    planes, 4 points of each per thread); zchunk starts at 16 and halves while the grid has fewer than 4 * 148 CTAs
    (tile_grid); k_norm_final over the CTAs."""
    nc = (n - 1) // 2 + 1
    tiles = cdiv(nc, 32) * cdiv(nc, 8)
    zchunk = 16
    while zchunk > 8 and tiles * cdiv(nc, zchunk) < 148 * 4:
        zchunk //= 2
    parts = tiles * cdiv(nc, zchunk)
    return 4 * 2 * zchunk + BLOCK_TREE + cdiv(parts, 256) + BLOCK_TREE


def chain_box(shape):
    """k_bs_norm: MG3B_NPARTS = 1024 blocks of 256 threads over equal slices of all points; k_bs_norm_final: ONE thread adds
    the 1024 partials in sequence."""
    tot = shape[0] * shape[1] * shape[2]
    return cdiv(cdiv(tot, 1024), 256) + BLOCK_TREE + 1024


def chain_2d(n):
    """k_reduce: MG2D_REDUCE_BLOCKS = 592 blocks of 256 threads over rows; k_reduce_final: 256 threads over the partials."""
    return cdiv(n - 2, 592) * cdiv(n - 2, 256) + BLOCK_TREE + cdiv(592, 256) + BLOCK_TREE


def chain_1d(n):
    """k_ops1d OP_NORM: one block of the smallest power of two >= n threads (at most 1024)."""
    t = 32
    while t < 1024 and t < n:
        t *= 2
    return cdiv(n, t) + BLOCK_TREE


def l2_bound(chain):
    m = chain + 1  # + the square's rounding
    gamma = m * U / (1 - m * U)
    return gamma / 2 + U + U


# ---- the reference -------------------------------------------------------------------------------------------------
def exact_sum_of_squares(r):
    x = np.ascontiguousarray(r, dtype=np.float64).ravel()
    sq = x * x
    c = x * 134217729.0  # Dekker: x = hi + lo with 26-bit halves, x*x = sq + err exactly
    hi = c - (c - x)
    lo = x - hi
    err = ((hi * hi - sq) + 2.0 * hi * lo) + lo * lo
    if 2 * x.size <= 1 << 22:
        return math.fsum(np.concatenate([sq, err]).tolist())
    return float(np.sum(sq.astype(np.longdouble)) + np.sum(err.astype(np.longdouble)))


def check_norms(eng, what, chain):
    r = eng.CalculateResidual(0)
    l2, linf = eng.residual_norm(0)
    want_inf = float(np.max(np.abs(r.astype(np.float64))))
    assert linf == want_inf, "%s: linf %r, max|r| %r" % (what, linf, want_inf)
    want = math.sqrt(exact_sum_of_squares(r))
    bound = l2_bound(chain)
    assert abs(l2 - want) <= bound * want, "%s: l2 %r, exact %r, relative error %.3e > %.3e (chain %d)" % (
        what, l2, want, abs(l2 - want) / want, bound, chain)
    return r


# ---- engines ---------------------------------------------------------------------------------------------------------
def engine(mg, kind, size, dtype, rng_range=None):
    if kind == "3d":
        return mg.MultiGrid3D(size, rng_range or (0, 1) * 3, dtype=dtype, residual_mode=mg.MG_CORRECTED)
    if kind == "box":
        return mg.MultiGrid3DBox(size, dtype=dtype, residual_mode=mg.MG_CORRECTED)
    if kind == "2d":
        return mg.MultiGrid2D(size, dtype=dtype)
    return mg.MultiGrid1D(size, dtype=dtype, residual_mode=mg.MG_CORRECTED)


def fill(eng, rng, scale=1.0):
    dtype = eng.np_dtype
    shape = eng.shape(0)
    eng.set_v(0, (rng.uniform(-1.0, 1.0, size=shape) * scale).astype(dtype))
    eng.set_f(0, (rng.uniform(-1.0, 1.0, size=shape) * scale).astype(dtype))


def wide(n):  # h = 4
    return (-2.0 * (n - 1), 2.0 * (n - 1)) * 3


CASES = [  # (id, engine kind, size, range, chain)
    ("3d-33", "3d", 33, None, chain_3d_plain(33)),
    ("3d-129", "3d", 129, None, chain_3d_plain(129)),
    ("3d-257-unit", "3d", 257, None, chain_3d_tma(257)),
    ("3d-257-h2^-7", "3d", 257, (-1, 1) * 3, chain_3d_tma(257)),
    ("3d-257-h4", "3d", 257, wide(257), chain_3d_tma(257)),
    ("3d-257-general", "3d", 257, GENERAL, chain_3d_plain(257)),
    ("3d-513-unit", "3d", 513, None, chain_3d_tma(513)),
    ("3d-513-h2^-8", "3d", 513, (-1, 1) * 3, chain_3d_tma(513)),
    ("3d-513-h4", "3d", 513, wide(513), chain_3d_tma(513)),
    ("box-129x65x33", "box", (129, 65, 33), None, chain_box((129, 65, 33))),
    ("box-257x129x65", "box", (257, 129, 65), None, chain_box((257, 129, 65))),
    ("2d-65", "2d", 65, None, chain_2d(65)),
    ("2d-1025", "2d", 1025, None, chain_2d(1025)),
    ("1d-1025", "1d", 1025, None, chain_1d(1025)),
    ("1d-65537", "1d", 65537, None, chain_1d(65537)),
]
PARAMS = [pytest.param(k, s, rg, ch, id=i) for i, k, s, rg, ch in CASES]


def test_bounds_are_tight_enough_to_mean_something():
    """The derived bounds stay far below what a sum in fp32 (2^-24) or a dropped term would give."""
    for _, _, _, _, chain in CASES:
        assert chain >= BLOCK_TREE and l2_bound(chain) < 1e-12


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind,size,rng_range,chain", PARAMS)
def test_norms_match_the_exact_sum(mg, kind, size, rng_range, chain, dtype):
    eng = engine(mg, kind, size, dtype, rng_range)
    fill(eng, np.random.default_rng(77))
    check_norms(eng, "%s %s" % (kind, np.dtype(dtype).name), chain)
    eng.close()


@pytest.mark.parametrize("target", [-100, 100], ids=["r~1e-30", "r~1e30"])
@pytest.mark.parametrize("kind,size,rng_range,chain", [p for p in PARAMS if "513" not in p.id])
def test_fp32_norms_where_the_square_leaves_fp32(mg, kind, size, rng_range, chain, target):
    """Scale v and f by a power of two (the residual scales exactly) so that max|r| ~ 2^target: r^2 ~ 2^(2 target) is
    below fp32's smallest subnormal or above its largest value."""
    eng = engine(mg, kind, size, np.float32, rng_range)
    fill(eng, np.random.default_rng(78))
    r0 = np.max(np.abs(eng.CalculateResidual(0).astype(np.float64)))
    fill(eng, np.random.default_rng(78), 2.0 ** (target - math.ceil(math.log2(r0))))
    r = check_norms(eng, "%s float32 scaled to 2^%d" % (kind, target), chain)
    rmax = np.max(np.abs(r.astype(np.float64)))
    assert 2.0 ** (target - 2) <= rmax <= 2.0 ** (target + 1), rmax
    eng.close()


# ---- non-finite residuals --------------------------------------------------------------------------------------------
NONFINITE = [
    pytest.param("3d", 33, None, id="3d-33"),
    pytest.param("3d", 257, None, id="3d-257-tma"),
    pytest.param("3d", 257, GENERAL, id="3d-257-general"),
    pytest.param("box", (129, 65, 33), None, id="box"),
    pytest.param("2d", 65, None, id="2d"),
    pytest.param("1d", 1025, None, id="1d"),
]


def poisoned(mg, kind, size, dtype, rng_range, values):
    """An engine with random v, f and the given values written into f at interior points (each makes exactly one residual
    value non-finite)."""
    eng = engine(mg, kind, size, dtype, rng_range)
    rng = np.random.default_rng(5)
    fill(eng, rng)
    f = eng.get_f(0)
    for j, val in enumerate(values):
        idx = tuple(s // 2 + j for s in f.shape)
        f[idx] = val
    eng.set_f(0, f)
    return eng


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("poison,want", [((np.nan,), "nan"), ((np.inf,), "inf"), ((-np.inf,), "inf"), ((np.inf, np.nan), "nan"),
                                         ((np.nan, -np.inf), "nan")], ids=["nan", "inf", "-inf", "inf+nan", "nan+-inf"])
@pytest.mark.parametrize("kind,size,rng_range", NONFINITE)
def test_nonfinite_residual(mg, kind, size, rng_range, dtype, poison, want):
    eng = poisoned(mg, kind, size, dtype, rng_range, poison)
    r = eng.CalculateResidual(0)
    ref_linf = float(np.max(np.abs(r.astype(np.float64))))
    assert (np.isnan(ref_linf) if want == "nan" else ref_linf == np.inf), ref_linf  # the definition the suite uses
    got = eng.residual_norm(0)
    if want == "nan":
        assert np.isnan(got[0]) and np.isnan(got[1]), got
    else:
        assert got == (np.inf, np.inf), got
    res = eng.solve(2, 2, rtol=1e-6, max_cycles=3)
    assert res.cycles == 0 and not res.converged, res
    h0 = tuple(res.history[0])
    if want == "nan":
        assert np.isnan(h0[0]) and np.isnan(h0[1]), h0
    else:
        assert h0 == (np.inf, np.inf), h0
    eng.close()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind,n", [("3d", 33), ("3d", 257), ("1d", 1025), ("2d", 65)])
def test_abs_error_with_a_nan(mg, kind, n, dtype):
    eng = engine(mg, kind, n, dtype)
    eng.init_problem()
    v = eng.get_v(0)
    v[tuple(s // 2 for s in v.shape)] = np.nan
    eng.set_v(0, v)
    if kind == "2d":
        assert np.isnan(eng.mean_abs_error())
    else:
        mean, mx = eng.abs_error(0)
        assert np.isnan(mean) and np.isnan(mx), (mean, mx)
        v[tuple(s // 2 for s in v.shape)] = 0.0
        eng.set_v(0, v)
        mean, mx = eng.abs_error(0)
        assert np.isfinite(mean) and np.isfinite(mx), (mean, mx)
    eng.close()

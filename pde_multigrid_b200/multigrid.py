"""Python mirror of the reference's operator interface over the C ABI (include/mg_b200.h).

Class and method names follow the reference classes MultiGrid3D / MultiGrid2D / MultiGrid1D
(N3/MultiGrid3D.h:6-33, N2/MultiGrid2D.h:6-37, N1/MultiGrid1D.h:6-31) so that the parity tests read
like the reference's own driver code.  This layer is plumbing only (ctypes + numpy buffers): every
operator runs in libmg_b200.so on the GPU.
"""
import collections
import ctypes

import numpy as np

from . import _lib
from ._lib import (MG_CORRECTED, MG_F32, MG_F64, MG_FIELD_F, MG_FIELD_V, MG_REF_COMPAT, check)


SolveResult = collections.namedtuple("SolveResult", "cycles converged history")
SolveResult.__doc__ = """Outcome of solve(): cycles run, whether the target was met, and a (cycles + 1, 2) float64 array
of (l2, linf) of the residuals r_0 .. r_cycles."""


def _dtype_code(dtype):
    dt = np.dtype(dtype)
    if dt == np.dtype(np.float32):
        return MG_F32
    if dt == np.dtype(np.float64):
        return MG_F64
    raise ValueError("dtype must be float32 or float64")


class _MultiGridBase:
    dim = 0
    prefix = ""

    def _fn(self, name):
        return getattr(self._L, "%s_%s" % (self.prefix, name))

    def _call(self, name, *args):
        check(self._fn(name)(self._h, *args))

    # ---- lifetime ----
    def close(self):
        if getattr(self, "_h", None) is not None:
            self._fn("destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- introspection ----
    @property
    def numGrids(self):
        return self._fn("num_levels")(self._h)

    def level_size(self, level):
        return self._fn("level_size")(self._h, ctypes.c_int(level))

    def level_h(self, level):
        return self._fn("level_h")(self._h, ctypes.c_int(level))

    def shape(self, level):
        """Shape of the host array of a level as this rank sees it (multi-GPU 3D: the owned z-planes)."""
        return (self.level_size(level),) * self.dim

    @property
    def stream(self):
        return self._fn("stream")(self._h)

    @property
    def kernel_launches(self):
        return self._fn("kernel_launches")(self._h)

    def sync(self):
        self._call("sync")

    # ---- fields (host dense arrays, reference layout: x fastest) ----
    def _chk(self, arr, level=None, shape=None):
        a = np.ascontiguousarray(arr, dtype=self.np_dtype)
        want = shape if shape is not None else self.shape(level)
        if a.shape != tuple(want):
            raise ValueError("array shape %s, expected %s" % (a.shape, tuple(want)))
        return a

    def set_field(self, level, field, arr):
        a = self._chk(arr, level)
        self._call("set_field", ctypes.c_int(level), ctypes.c_int(field), a.ctypes.data_as(ctypes.c_void_p))

    def get_field(self, level, field):
        out = np.empty(self.shape(level), dtype=self.np_dtype)
        self._call("get_field", ctypes.c_int(level), ctypes.c_int(field), out.ctypes.data_as(ctypes.c_void_p))
        return out

    def set_v(self, level, arr):
        self.set_field(level, MG_FIELD_V, arr)

    def set_f(self, level, arr):
        self.set_field(level, MG_FIELD_F, arr)

    def get_v(self, level=0):
        return self.get_field(level, MG_FIELD_V)

    def get_f(self, level=0):
        return self.get_field(level, MG_FIELD_F)

    def init_problem(self):
        self._call("init_problem")

    # ---- operators on the engine's own level arrays ----
    def Relax(self, level, ncycles):
        self._call("relax", ctypes.c_int(level), ctypes.c_int(ncycles))

    def CalculateResidual(self, level=0):
        out = np.empty(self.shape(level), dtype=self.np_dtype)
        self._call("residual", ctypes.c_int(level), out.ctypes.data_as(ctypes.c_void_p))
        return out

    def residual_norm(self, level=0):
        l2, linf = ctypes.c_double(), ctypes.c_double()
        self._call("residual_norm", ctypes.c_int(level), ctypes.byref(l2), ctypes.byref(linf))
        return l2.value, linf.value

    def restrict_level(self, fine_level, field=MG_FIELD_F):
        self._call("restrict", ctypes.c_int(fine_level), ctypes.c_int(field))

    def residual_restrict(self, fine_level):
        self._call("residual_restrict", ctypes.c_int(fine_level))

    def interpolate_level(self, fine_level):
        self._call("interpolate", ctypes.c_int(fine_level))

    def interpolate_correct(self, fine_level):
        self._call("interpolate_correct", ctypes.c_int(fine_level))

    def set_level_to_value(self, level, field, value, modifyBoundaries):
        self._call("set_to_value", ctypes.c_int(level), ctypes.c_int(field), ctypes.c_double(value),
                   ctypes.c_int(1 if modifyBoundaries else 0))

    def VCycle(self, gridID, v1, v2):
        self._call("vcycle", ctypes.c_int(gridID), ctypes.c_int(v1), ctypes.c_int(v2))

    def FullMultiGridVCycle(self, gridID, v0, v1, v2):
        self._call("fmg", ctypes.c_int(gridID), ctypes.c_int(v0), ctypes.c_int(v1), ctypes.c_int(v2))

    def solve(self, v1=2, v2=2, rtol=1e-8, atol=0.0, max_cycles=100, level=0):
        """V-cycles VCycle(level, v1, v2) from the current v until ||r_k||_2 <= max(atol, rtol * ||r_0||_2) or
        max_cycles cycles have run (mg?d_solve).  On one GPU the loop runs on the device: one wait per solve."""
        hist = np.empty((max(int(max_cycles), 0) + 1, 2), dtype=np.float64)
        cycles, converged = ctypes.c_int(), ctypes.c_int()
        self._call("solve", ctypes.c_int(level), ctypes.c_int(v1), ctypes.c_int(v2), ctypes.c_double(rtol),
                   ctypes.c_double(atol), ctypes.c_int(max_cycles), ctypes.byref(cycles), ctypes.byref(converged),
                   hist.ctypes.data_as(ctypes.c_void_p))
        return SolveResult(cycles.value, bool(converged.value), hist[:cycles.value + 1].copy())

    # ---- reference-facing operators on caller-owned HOST arrays (NOCUDA signatures) ----
    def _sizes(self, n):
        if self.dim == 1:
            return ctypes.c_int(n)
        return (ctypes.c_int * self.dim)(*([n] * self.dim))

    def Restrict(self, fine):
        fine = np.ascontiguousarray(fine, dtype=self.np_dtype)
        fn = fine.shape[0]
        cn = (fn - 1) // 2 + 1
        coarse = np.zeros((cn,) * self.dim, dtype=self.np_dtype)
        self._call("restrict_host", fine.ctypes.data_as(ctypes.c_void_p), self._sizes(fn),
                   coarse.ctypes.data_as(ctypes.c_void_p), self._sizes(cn))
        return coarse

    def Interpolate(self, fine, coarse):
        """fine is modified in place (interior only), like the reference."""
        assert fine.dtype == self.np_dtype and fine.flags["C_CONTIGUOUS"]
        coarse = np.ascontiguousarray(coarse, dtype=self.np_dtype)
        self._call("interpolate_host", fine.ctypes.data_as(ctypes.c_void_p), self._sizes(fine.shape[0]),
                   coarse.ctypes.data_as(ctypes.c_void_p), self._sizes(coarse.shape[0]))
        return fine

    def ApplyCorrection(self, fine, error):
        assert fine.dtype == self.np_dtype and fine.flags["C_CONTIGUOUS"]
        error = np.ascontiguousarray(error, dtype=self.np_dtype)
        self._call("apply_correction_host", fine.ctypes.data_as(ctypes.c_void_p), self._sizes(fine.shape[0]),
                   error.ctypes.data_as(ctypes.c_void_p), self._sizes(error.shape[0]))
        return fine

    def setToValue(self, grid, value, modifyBoundaries):
        assert grid.dtype == self.np_dtype and grid.flags["C_CONTIGUOUS"]
        self._call("set_to_value_host", grid.ctypes.data_as(ctypes.c_void_p), self._sizes(grid.shape[0]),
                   ctypes.c_double(value), ctypes.c_int(1 if modifyBoundaries else 0))
        return grid

    def vcycle_host(self, v_host, f_host, v1, v2, cycles=1):
        """End-to-end call with HOST buffers: upload v,f -> cycles x VCycle(0,v1,v2) -> download v."""
        assert v_host.dtype == self.np_dtype and v_host.flags["C_CONTIGUOUS"]
        assert f_host.dtype == self.np_dtype and f_host.flags["C_CONTIGUOUS"]
        self._call("vcycle_host", v_host.ctypes.data_as(ctypes.c_void_p), f_host.ctypes.data_as(ctypes.c_void_p),
                   ctypes.c_int(v1), ctypes.c_int(v2), ctypes.c_int(cycles))
        return v_host


class _PCGMixin:
    """pcg() of the 3D engines.  CG needs a symmetric operator: the 2D Lyapunov operator and the first-order 1D
    equation are not, so the 2D and 1D classes do not have it."""

    def pcg(self, v1=2, v2=2, rtol=1e-8, atol=0.0, max_iters=100, level=0):
        """Conjugate gradients preconditioned by one VCycle(level, v1, v2) per iteration (mg3d_pcg / mg3b_pcg) on the
        MG_CORRECTED operator, from the current v, until the true residual meets ||r_k||_2 <= max(atol, rtol * ||r_0||_2)
        or max_iters iterations have run.  Returns a SolveResult whose `cycles` counts iterations (one V-cycle each).
        v of `level` holds the iterate afterwards, f of `level` is unchanged."""
        hist = np.empty((max(int(max_iters), 0) + 1, 2), dtype=np.float64)
        iters, converged = ctypes.c_int(), ctypes.c_int()
        self._call("pcg", ctypes.c_int(level), ctypes.c_int(v1), ctypes.c_int(v2), ctypes.c_double(rtol),
                   ctypes.c_double(atol), ctypes.c_int(max_iters), ctypes.byref(iters), ctypes.byref(converged),
                   hist.ctypes.data_as(ctypes.c_void_p))
        return SolveResult(iters.value, bool(converged.value), hist[:iters.value + 1].copy())


class MultiGrid3D(_PCGMixin, _MultiGridBase):
    """MultiGrid3D(finestGridSizeXYZ, range) -- N3/MultiGrid3D.h:12."""
    dim = 3
    prefix = "mg3d"

    def __init__(self, finestGridSizeXYZ, range=(0, 1, 0, 1, 0, 1), dtype=np.float32, residual_mode=MG_REF_COMPAT,
                 rank=0, nranks=1, nccl_unique_id=None):
        self._L = _lib.lib()
        self.np_dtype = np.dtype(dtype)
        if np.isscalar(finestGridSizeXYZ):
            finestGridSizeXYZ = [int(finestGridSizeXYZ)] * 3
        sz = (ctypes.c_int * 3)(*[int(s) for s in finestGridSizeXYZ])
        rg = (ctypes.c_double * 6)(*[float(r) for r in range])
        h = ctypes.c_void_p()
        self._h = None
        if nranks == 1:
            check(self._L.mg3d_create(ctypes.byref(h), sz, rg, _dtype_code(dtype), int(residual_mode)))
        else:
            check(self._L.mg3d_create_dist(ctypes.byref(h), sz, rg, _dtype_code(dtype), int(residual_mode),
                                           int(rank), int(nranks), nccl_unique_id))
        self._h = h

        self.rank, self.nranks = int(rank), int(nranks)

    def set_smoother(self, smoother, sweeps_per_pass=None):
        if sweeps_per_pass is None:
            sweeps_per_pass = 2 if smoother in (_lib.MG_SMOOTHER_FUSED, _lib.MG_SMOOTHER_PIPE) else 1
        self._call("set_smoother", ctypes.c_int(smoother), ctypes.c_int(sweeps_per_pass))

    def set_arith(self, arith):
        """MG_ARITH_EXACT (bit-identical to the reference, default) or MG_ARITH_FAST."""
        self._call("set_arith", ctypes.c_int(arith))

    def set_jacobi_weight(self, omega):
        """Relaxation weight of MG_SMOOTHER_JACOBI (default 6/7)."""
        self._call("set_jacobi_weight", ctypes.c_double(omega))

    def owned_range(self, level):
        """(z_begin, z_count) of the global planes this rank owns on `level`."""
        zb, zc = ctypes.c_int(), ctypes.c_int()
        self._call("owned_range", ctypes.c_int(level), ctypes.byref(zb), ctypes.byref(zc))
        return zb.value, zc.value

    def shape(self, level):
        n = self.level_size(level)
        return (self.owned_range(level)[1], n, n)

    @property
    def halo_bytes(self):
        return self._fn("halo_bytes")(self._h)

    def field_checksum(self, level=0, field=MG_FIELD_V):
        """Position-keyed additive checksum of a whole level field (all ranks return the global value)."""
        out = ctypes.c_ulonglong()
        self._call("field_checksum", ctypes.c_int(level), ctypes.c_int(field), ctypes.byref(out))
        return out.value

    def abs_error(self, level=0):
        """(mean, max) over all points of |sin(pi x)sin(pi y)sin(pi z) - v|: Grid3D::PrintDiff as a reduction."""
        mean, mx = ctypes.c_double(), ctypes.c_double()
        self._call("abs_error", ctypes.c_int(level), ctypes.byref(mean), ctypes.byref(mx))
        return mean.value, mx.value

    @staticmethod
    def plan_level(n, nranks, rank):
        """Slab plan (no GPU needed): dict(dist, z0, nzl, own_lo, own_hi)."""
        out = (ctypes.c_int * 5)()
        check(_lib.lib().mg3d_plan_level(ctypes.c_int(n), ctypes.c_int(nranks), ctypes.c_int(rank), out))
        return dict(zip(("dist", "z0", "nzl", "own_lo", "own_hi"), list(out)))


class MultiGrid3DBox(_PCGMixin, _MultiGridBase):
    """MultiGrid3D(finestGridSizeXYZ, range) with sizeX != sizeY != sizeZ (mg3b_* of the C ABI): the grids the reference
    asserts away at N3/Grid3D.cpp:10-11.  Host arrays have numpy shape (sizeZ, sizeY, sizeX) -- the dense x-fastest layout."""
    dim = 3
    prefix = "mg3b"

    def __init__(self, finestGridSizeXYZ, range=(0, 1, 0, 1, 0, 1), dtype=np.float32, residual_mode=MG_REF_COMPAT):
        self._L = _lib.lib()
        self._L.mg3b_stream.restype = ctypes.c_void_p
        self._L.mg3b_kernel_launches.restype = ctypes.c_longlong
        self.np_dtype = np.dtype(dtype)
        sz = (ctypes.c_int * 3)(*[int(s) for s in finestGridSizeXYZ])
        rg = (ctypes.c_double * 6)(*[float(r) for r in range])
        h = ctypes.c_void_p()
        self._h = None
        check(self._L.mg3b_create(ctypes.byref(h), sz, rg, _dtype_code(dtype), int(residual_mode)))
        self._h = h

    def level_size(self, level):
        """(sizeX, sizeY, sizeZ) of a level"""
        o = (ctypes.c_int * 3)()
        self._call("level_size", ctypes.c_int(level), o)
        return tuple(o)

    def level_h(self, level):
        o = (ctypes.c_double * 3)()
        self._call("level_h", ctypes.c_int(level), o)
        return tuple(o)

    def shape(self, level):
        nx, ny, nz = self.level_size(level)
        return (nz, ny, nx)


class MultiGrid2D(_MultiGridBase):
    """MultiGrid2D(finestGridSizeXY, range, A, A_size, alfa) -- N2/MultiGrid2D.h:16."""
    dim = 2
    prefix = "mg2d"

    def __init__(self, finestGridSizeXY, range=(0, 1, 0, 1), A=(-1.0, -2.0, 0.0, -3.0), alfa=2, dtype=np.float32):
        self._L = _lib.lib()
        self.np_dtype = np.dtype(dtype)
        if np.isscalar(finestGridSizeXY):
            finestGridSizeXY = [int(finestGridSizeXY)] * 2
        sz = (ctypes.c_int * 2)(*[int(s) for s in finestGridSizeXY])
        rg = (ctypes.c_double * 4)(*[float(r) for r in range])
        a4 = (ctypes.c_double * 4)(*[float(a) for a in A])
        h = ctypes.c_void_p()
        self._h = None
        check(self._L.mg2d_create(ctypes.byref(h), sz, rg, a4, int(alfa), _dtype_code(dtype)))
        self._h = h

    def mean_abs_error(self):
        out = ctypes.c_double()
        self._call("mean_abs_error", ctypes.byref(out))
        return out.value


class MultiGrid1D(_MultiGridBase):
    """MultiGrid1D(finestGridSize, range) -- N1/MultiGrid1D.h:12."""
    dim = 1
    prefix = "mg1d"

    def __init__(self, finestGridSize, range=(0, 1), dtype=np.float32, residual_mode=MG_REF_COMPAT):
        self._L = _lib.lib()
        self.np_dtype = np.dtype(dtype)
        rg = (ctypes.c_double * 2)(*[float(r) for r in range])
        h = ctypes.c_void_p()
        self._h = None
        check(self._L.mg1d_create(ctypes.byref(h), ctypes.c_int(int(finestGridSize)), rg, _dtype_code(dtype),
                                  int(residual_mode)))
        self._h = h

    def abs_error(self, level=0):
        """(mean, max) over all points of |approxsol - realsol|: Grid1D::PrintDiffApproxReal as a reduction."""
        mean, mx = ctypes.c_double(), ctypes.c_double()
        self._call("abs_error", ctypes.c_int(level), ctypes.byref(mean), ctypes.byref(mx))
        return mean.value, mx.value

"""oracle/port.py -- TEST INFRASTRUCTURE, not product code.

ctypes binding to oracle/libmg_oracle.so (mg_oracle.c, the plain-C restatement of the reference's
NOCUDA_TESI algorithm).  `PortMG` has the same interface as oracle.ref.RefMG so the tests can run
either one as the checker.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may
import this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libmg_oracle.so")
SRC = [os.path.join(_HERE, "mg_oracle.c"), os.path.join(_HERE, "mg_oracle_impl.h")]
_lib = None


def build(force=False):
    """gcc -O2, contraction off, never fast-math (the reference is built without FMA)."""
    if not force and os.path.exists(SO_PATH) and all(os.path.getmtime(SO_PATH) >= os.path.getmtime(s) for s in SRC):
        return SO_PATH
    cmd = [os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
           SRC[0], "-o", SO_PATH, "-lm"]
    subprocess.run(cmd, check=True)
    return SO_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            build()
        _lib = ctypes.CDLL(SO_PATH)
    return _lib


def level_sizes(n):
    """numGrids = (int)log2(n-1), n_l = (n_{l-1}-1)/2+1  (N3/MultiGrid3D.cpp:33-46)"""
    num = int(np.floor(np.log2(n - 1)))
    sizes = [n]
    for _ in range(1, num):
        sizes.append((sizes[-1] - 1) // 2 + 1)
    return sizes


def norms(r):
    r64 = np.asarray(r, dtype=np.float64).ravel()
    return float(np.sqrt(np.cumsum(r64 * r64)[-1])) if r64.size else 0.0, float(np.max(np.abs(r64)))


class PortMG:
    def __init__(self, dim, dtype, corrected=False, n=33, range=None, A=(-1.0, -2.0, 0.0, -3.0), alfa=2):
        self.dim = dim
        self.np_dtype = np.dtype(dtype)
        self.sfx = "_f32" if self.np_dtype == np.dtype(np.float32) else "_f64"
        self.corrected = 1 if (corrected and dim != 2) else 0
        self.L = lib()
        self.creal_p = ctypes.POINTER(ctypes.c_float if self.sfx == "_f32" else ctypes.c_double)
        if range is None:
            range = [0.0, 1.0] * dim
        self.range = (ctypes.c_double * (2 * dim))(*[float(x) for x in range])
        self.A = (ctypes.c_double * 4)(*[float(x) for x in A])
        self.alfa = int(alfa)
        self.sizes = level_sizes(n)
        self.num_levels = len(self.sizes)
        self._v = [np.zeros((s,) * dim, dtype=self.np_dtype) for s in self.sizes]
        self._f = [np.zeros((s,) * dim, dtype=self.np_dtype) for s in self.sizes]
        for l, s in enumerate(self.sizes):  # every level is initialised like the finest (Grid ctor)
            if dim == 3:
                self._call("init_v", self._p(self._v[l]), s)
                self._call("init_f", self._p(self._f[l]), s, self.range)
            elif dim == 2:
                self._call("init_v", self._p(self._v[l]), s, self.range)
                self._call("init_f", self._p(self._f[l]), s)
            else:
                self._call("init_v", self._p(self._v[l]), s, self.range)
                self._call("init_f", self._p(self._f[l]), s, self.range)

    def _call(self, name, *args):
        f = getattr(self.L, "orc%dd_%s%s" % (self.dim, name, self.sfx))
        f.restype = None
        conv = []
        for a in args:
            if isinstance(a, (int, np.integer)):
                conv.append(ctypes.c_int(int(a)))
            elif isinstance(a, float):
                conv.append(ctypes.c_double(a))
            else:
                conv.append(a)
        f(*conv)

    def close(self):
        pass

    def shape(self, l):
        return (self.sizes[l],) * self.dim

    def v(self, l=0):
        return self._v[l]

    def f(self, l=0):
        return self._f[l]

    def _p(self, arr):
        assert arr.dtype == self.np_dtype and arr.flags["C_CONTIGUOUS"]
        return arr.ctypes.data_as(self.creal_p)

    def _pp(self, arrs):
        return (self.creal_p * len(arrs))(*[self._p(a) for a in arrs])

    def _extra(self):
        return (self.range, self.A, self.alfa) if self.dim == 2 else (self.range,)

    def relax(self, l, ncycles):
        self._call("relax", self._p(self._v[l]), self._p(self._f[l]), self.sizes[l], *self._extra(), int(ncycles))

    def relax_jacobi(self, l, ncycles, omega=6.0 / 7.0):
        """Weighted Jacobi (3D only; not in the reference -- the port is its definition)."""
        assert self.dim == 3
        self._call("relax_jacobi", self._p(self._v[l]), self._p(self._f[l]), self.sizes[l], self.range, float(omega), int(ncycles))

    def vcycle_jacobi(self, l, v1, v2, omega=6.0 / 7.0):
        assert self.dim == 3
        self._call("vcycle_jacobi", self._pp(self._v), self._pp(self._f), self.sizes[0], self.num_levels, self.range, int(l),
                   int(v1), int(v2), self.corrected, float(omega))

    def residual(self, l=0):
        out = np.empty(self.shape(l), dtype=self.np_dtype)
        if self.dim == 2:
            self._call("residual", self._p(self._v[l]), self._p(self._f[l]), self._p(out), self.sizes[l],
                       *self._extra())
        else:
            self._call("residual", self._p(self._v[l]), self._p(self._f[l]), self._p(out), self.sizes[l],
                       self.range, self.corrected)
        return out

    def restrict(self, fine):
        cn = (fine.shape[0] - 1) // 2 + 1
        coarse = np.zeros((cn,) * self.dim, dtype=self.np_dtype)
        self._call("restrict", self._p(fine), fine.shape[0], self._p(coarse))
        return coarse

    def interpolate(self, fine, coarse):
        self._call("interpolate", self._p(fine), fine.shape[0], self._p(coarse))
        return fine

    def apply_correction(self, fine, err):
        self._call("apply_correction", self._p(fine), self._p(err), fine.shape[0])
        return fine

    def set_to_value(self, grid, value, modify_boundaries):
        self._call("set", self._p(grid), grid.shape[0], float(value), 1 if modify_boundaries else 0)
        return grid

    def vcycle(self, l, v1, v2):
        args = [self._pp(self._v), self._pp(self._f), self.sizes[0], self.num_levels, *self._extra(), int(l), int(v1),
                int(v2)]
        if self.dim != 2:
            args.append(self.corrected)
        self._call("vcycle", *args)

    def fmg(self, l, v0, v1, v2):
        args = [self._pp(self._v), self._pp(self._f), self.sizes[0], self.num_levels, *self._extra(), int(l), int(v0),
                int(v1), int(v2)]
        if self.dim != 2:
            args.append(self.corrected)
        self._call("fmg", *args)

    def residual_norms(self, l=0):
        return norms(self.residual(l))


def box_level_shapes(shape):
    """(nx, ny, nz) per level: numGrids from the smallest dimension, every dimension halved per level (N3/MultiGrid3D.cpp:19-47)"""
    nx, ny, nz = [int(s) for s in shape]
    num = int(np.floor(np.log2(min(nx, ny, nz) - 1)))
    out = [(nx, ny, nz)]
    for _ in range(1, num):
        nx, ny, nz = (nx - 1) // 2 + 1, (ny - 1) // 2 + 1, (nz - 1) // 2 + 1
        out.append((nx, ny, nz))
    return out


class PortBox3D:
    """The restatement on a NON-CUBIC 3D grid (orc3b_* in mg_oracle_impl.h); same interface as RefMG(3, ..., shape=...).
    Arrays have numpy shape (nz, ny, nx): the dense x-fastest layout of the reference."""

    def __init__(self, dtype, corrected=False, shape=(33, 17, 9), range=None):
        self.dim = 3
        self.np_dtype = np.dtype(dtype)
        self.sfx = "_f32" if self.np_dtype == np.dtype(np.float32) else "_f64"
        self.corrected = 1 if corrected else 0
        self.L = lib()
        self.creal_p = ctypes.POINTER(ctypes.c_float if self.sfx == "_f32" else ctypes.c_double)
        self.range = (ctypes.c_double * 6)(*[float(x) for x in (range if range is not None else [0.0, 1.0] * 3)])
        self.xyz = box_level_shapes(shape)
        self.n0 = (ctypes.c_int * 3)(*self.xyz[0])
        self.num_levels = len(self.xyz)
        self.shapes = [(nz, ny, nx) for nx, ny, nz in self.xyz]
        self._v = [np.zeros(s, dtype=self.np_dtype) for s in self.shapes]
        self._f = [np.zeros(s, dtype=self.np_dtype) for s in self.shapes]
        for l, (nx, ny, nz) in enumerate(self.xyz):
            self._call("init_v", self._p(self._v[l]), nx, ny, nz)
            self._call("init_f", self._p(self._f[l]), nx, ny, nz, self.range)

    def _call(self, name, *args):
        f = getattr(self.L, "orc3b_%s%s" % (name, self.sfx))
        f.restype = None
        f(*[ctypes.c_int(int(a)) if isinstance(a, (int, np.integer)) else (ctypes.c_double(a) if isinstance(a, float) else a) for a in args])

    def close(self):
        pass

    def shape(self, l):
        return self.shapes[l]

    def v(self, l=0):
        return self._v[l]

    def f(self, l=0):
        return self._f[l]

    def _p(self, arr):
        assert arr.dtype == self.np_dtype and arr.flags["C_CONTIGUOUS"]
        return arr.ctypes.data_as(self.creal_p)

    def _pp(self, arrs):
        return (self.creal_p * len(arrs))(*[self._p(a) for a in arrs])

    def relax(self, l, ncycles):
        self._call("relax", self._p(self._v[l]), self._p(self._f[l]), *self.xyz[l], self.range, int(ncycles))

    def residual(self, l=0):
        out = np.empty(self.shapes[l], dtype=self.np_dtype)
        self._call("residual", self._p(self._v[l]), self._p(self._f[l]), self._p(out), *self.xyz[l], self.range, self.corrected)
        return out

    def restrict(self, fine):
        nz, ny, nx = fine.shape
        coarse = np.zeros(((nz - 1) // 2 + 1, (ny - 1) // 2 + 1, (nx - 1) // 2 + 1), dtype=self.np_dtype)
        self._call("restrict", self._p(fine), nx, ny, nz, self._p(coarse))
        return coarse

    def interpolate(self, fine, coarse):
        nz, ny, nx = fine.shape
        self._call("interpolate", self._p(fine), nx, ny, nz, self._p(coarse))
        return fine

    def apply_correction(self, fine, err):
        nz, ny, nx = fine.shape
        self._call("apply_correction", self._p(fine), self._p(err), nx, ny, nz)
        return fine

    def set_to_value(self, grid, value, modify_boundaries):
        nz, ny, nx = grid.shape
        self._call("set", self._p(grid), nx, ny, nz, float(value), 1 if modify_boundaries else 0)
        return grid

    def vcycle(self, l, v1, v2):
        self._call("vcycle", self._pp(self._v), self._pp(self._f), self.n0, self.num_levels, self.range, int(l), int(v1), int(v2), self.corrected)

    def fmg(self, l, v0, v1, v2):
        self._call("fmg", self._pp(self._v), self._pp(self._f), self.n0, self.num_levels, self.range, int(l), int(v0), int(v1), int(v2),
                   self.corrected)

    def residual_norms(self, l=0):
        return norms(self.residual(l))

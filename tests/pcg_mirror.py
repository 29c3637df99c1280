"""A numpy mirror of the multigrid-preconditioned conjugate-gradient schedule of mg3d_pcg / mg3b_pcg (DESIGN.md §6b).

Vectors are in the level's dtype, scalars in fp64, the preconditioner is the C oracle's V-cycle (oracle.port:
PortMG.vcycle, PortMG.vcycle_jacobi, PortBox3D.vcycle) from v = 0 with f = r.  Every vector operation rounds like the
kernels of csrc/mg3d_cg.cu (a product, then a sum, each rounded to the dtype), the residual is the oracle's
CalculateResidual (sign-corrected), and the dot products are correctly rounded to fp64 like the engine's double-double
ones, so alpha, beta and the vectors are the engine's; only the order of the sum of squares in the norm differs.
Test infrastructure, not product code.
"""
import math

import numpy as np

from oracle import port


def make_oracle(kind, shape, dtype):
    """kind 'cube' (shape = (n,)) or 'box' (shape = (nx, ny, nz)), MG_CORRECTED, init_problem data"""
    if kind == "box":
        return port.PortBox3D(dtype, corrected=True, shape=shape)
    return port.PortMG(3, dtype, corrected=True, n=shape[0])


def _two_prod(a, b):
    """p = fl(a*b) and the exact error e = a*b - p (Dekker's product with Veltkamp splitting)"""
    p = a * b
    split = 134217729.0  # 2^27 + 1
    ca, cb = split * a, split * b
    ah, bh = ca - (ca - a), cb - (cb - b)
    al, bl = a - ah, b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def _dot(a, b):
    """the correctly rounded dot product in fp64 (the engine accumulates its dots in double-double, csrc/mg3d_cg.cu):
    exact products summed by math.fsum"""
    a64, b64 = a.ravel().astype(np.float64), b.ravel().astype(np.float64)
    p, e = _two_prod(a64, b64)
    nz = e != 0
    return math.fsum(np.concatenate([p, e[nz]]).tolist()) if nz.any() else math.fsum(p.tolist())


def pcg(m, v1=2, v2=2, rtol=1e-9, atol=0.0, max_iters=100, jacobi=False, omega=6.0 / 7.0):
    """PCG on level 0 of oracle `m` from its current v and f.  Returns (iterations, converged, history (k+1, 2), x):
    the history holds (l2, linf) of the true residuals r_0 .. r_k."""
    dt = m.np_dtype.type
    x = m.v(0).copy()
    b = m.f(0).copy()

    def resid(v, f):
        m.v(0)[...] = v
        m.f(0)[...] = f
        return m.residual(0)

    def precondition(r):
        m.v(0)[...] = 0
        m.f(0)[...] = r
        if jacobi:
            m.vcycle_jacobi(0, v1, v2, omega)
        else:
            m.vcycle(0, v1, v2)
        return m.v(0).copy()

    r = resid(x, b)
    hist = [port.norms(r)]
    thr = max(atol, rtol * hist[0][0])

    def stop(l2):
        finite = np.isfinite(l2)
        return (not finite) or l2 <= thr, bool(finite and l2 <= thr)

    done, conv = stop(hist[0][0])
    p = np.zeros_like(x)
    d = np.zeros_like(x)
    zeros = np.zeros_like(b)
    rho_prev = None
    k = 0
    while not done and k < max_iters:
        z = precondition(r)
        rho, sigma = _dot(z, r), _dot(z, d)
        beta = 0.0 if rho_prev is None else sigma / rho_prev
        rho_prev = rho
        p = z + dt(beta) * p
        q = -resid(p, zeros)
        alpha = rho / _dot(p, q)
        xn = x + dt(alpha) * p
        rn = resid(xn, b)
        d = rn - r
        x, r = xn, rn
        k += 1
        hist.append(port.norms(r))
        done, conv = stop(hist[-1][0])
    return k, conv, np.array(hist, dtype=np.float64), x

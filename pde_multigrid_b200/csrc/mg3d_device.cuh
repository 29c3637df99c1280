// mg3d_device.cuh -- device functions shared by the 3D kernel translation units: the per-point
// formulas of the reference (relax, residual, 27-point restriction, trilinear prolongation) and the
// colour-split addressing.  See mg3d_kernels.cu for the layout description.
#pragma once
#include <stdint.h>

#include "mg_exact.cuh"
#include "mg_launch.h"

// Raise a kernel's dynamic shared-memory limit once per DEVICE (the attribute is per device: a process may hold
// handles on several GPUs).  The static lives at the call site, i.e. once per kernel instantiation.
#define MG_SET_SMEM_LIMIT(kernel, bytes)                                                                        \
    do {                                                                                                        \
        static unsigned char done_[64];                                                                         \
        int dev_ = 0;                                                                                           \
        cudaGetDevice(&dev_);                                                                                   \
        if (dev_ < 0 || dev_ >= 64 || !done_[dev_]) {                                                           \
            cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));            \
            if (dev_ >= 0 && dev_ < 64) done_[dev_] = 1;                                                        \
        }                                                                                                       \
    } while (0)

// -DMG_DEBUG_BOUNDS (python -m pde_multigrid_b200.build --debug-bounds -> libmg_b200_dbg.so): every global-memory access of
// the 3D kernels asserts that its (half-index, row, plane) lies inside the field it addresses; otherwise it reports and retires the thread -- the
// stand-in for compute-sanitizer memcheck, which is closed on the GPU pool (tests/test_debug_bounds.py runs the suite's
// small cases against this build).  Compiled out of the product library.
#ifdef MG_DEBUG_BOUNDS
#include <stdio.h>
#define MG_CHK(cond)                                                                                              \
    do {                                                                                                          \
        if (!(cond)) {                                                                                            \
            printf("MG_DEBUG_BOUNDS: %s violated at %s:%d (block %d,%d,%d thread %d)\n", #cond, __FILE__, __LINE__, \
                   (int)blockIdx.x, (int)blockIdx.y, (int)blockIdx.z, (int)threadIdx.x);                          \
            asm volatile("exit;"); /* the thread ends here: the bad access never happens, the GPU takes no fault */  \
        }                                                                                                         \
    } while (0)
#else
#define MG_CHK(cond) ((void)0)
#endif
// site (half-index i, row y, local plane zl) inside the stored part of a colour array
#define MG_CHK_SITE(g, i, y, zl) MG_CHK((i) >= 0 && (i) < (g).hp && (y) >= 0 && (y) < (g).n && (zl) >= 0 && (zl) < (g).nzl)

namespace mg3 {
using namespace mgx;

template <typename T>
struct Coef3 {
    T hx2, hy2, hz2, cx, cy, cz, den, rden, ihx2, ihy2, ihz2;
};

template <typename T>
Coef3<T> narrow(const mg_coef3d& c)
{
    Coef3<T> r;
    r.hx2 = (T)c.hx2; r.hy2 = (T)c.hy2; r.hz2 = (T)c.hz2;
    r.cx = (T)c.cx; r.cy = (T)c.cy; r.cz = (T)c.cz;
    r.den = (T)c.den; r.rden = (T)c.rden;
    r.ihx2 = (T)c.ihx2; r.ihy2 = (T)c.ihy2; r.ihz2 = (T)c.ihz2;
    return r;
}

__device__ __forceinline__ long long off3(const mg_geom3d& g, int x, int y, int zl)
{
    MG_CHK(x >= 0 && x < g.n && y >= 0 && y < g.n && zl >= 0 && zl < g.nzl);
    const int c = (x + y + g.z0 + zl) & 1;
    return (long long)c * g.cstride + (long long)zl * g.plane + (long long)y * g.hp + (x >> 1);
}

// block-wide {sum, max} of one double pair per thread: warp shuffles, then one warp over the per-warp results
// (deterministic for a given block size); sh holds 64 doubles.  The result is valid in thread 0.
__device__ __forceinline__ void block_sum_max(double& s, double& m, double* sh)
{
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) { sh[w] = s; sh[32 + w] = m; }
    __syncthreads();
    if (w == 0) {
        s = (l < nw) ? sh[l] : 0.0;
        m = (l < nw) ? sh[32 + l] : 0.0;
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
        }
    }
}

// N3/MultiGrid3D.cpp:532 -- left-to-right sum of the six weighted neighbours, minus f*hx2*hy2*hz2,
// divided by 2*(hy2*hz2 + hx2*hz2 + hx2*hy2).  O/E = x-1/x+1, N/S = y-1/y+1, D/U = z-1/z+1.
// FAST: the divisor is 6*2^e (cubic grid, power-of-two h: the reference problem) -> correctly rounded
// quotient from the host reciprocal in 3 pipe ops (mg_exact.cuh); otherwise IEEE division.
template <typename T, bool FAST>
__device__ __forceinline__ T relax_point(T O, T E, T N, T S, T D, T U, T f, const Coef3<T>& c)
{
    T s = add(mul(O, c.cx), mul(E, c.cx));
    s = add(s, mul(N, c.cy));
    s = add(s, mul(S, c.cy));
    s = add(s, mul(D, c.cz));
    s = add(s, mul(U, c.cz));
    s = sub(s, mul(mul(mul(f, c.hx2), c.hy2), c.hz2));
    return FAST ? div_by_const(s, c.den, c.rden) : div(s, c.den);
}

// N3/MultiGrid3D.cpp:723 (REF_COMPAT, minus S / minus U) or the sign-corrected form.  FAST: every h^2
// is a power of two, so x/h^2 == x*(1/h^2) exactly.
template <typename T, bool FAST>
__device__ __forceinline__ T residual_point(T O, T E, T N, T S, T D, T U, T vc, T f, const Coef3<T>& c, int corrected)
{
    const T v2 = mul(T(2), vc);
    const T ax = add(sub(O, v2), E);
    const T ay = corrected ? add(sub(N, v2), S) : sub(sub(N, v2), S);
    const T az = corrected ? add(sub(D, v2), U) : sub(sub(D, v2), U);
    const T tx = FAST ? mul(ax, c.ihx2) : div(ax, c.hx2);
    const T ty = FAST ? mul(ay, c.ihy2) : div(ay, c.hy2);
    const T tz = FAST ? mul(az, c.ihz2) : div(az, c.hz2);
    return sub(sub(sub(f, tx), ty), tz);
}

// residual at interior fine point (x,y,zl) read from the colour-split arrays
template <typename T, bool FAST>
__device__ __forceinline__ T residual_at(const T* __restrict__ v, const T* __restrict__ f, const mg_geom3d& g, int x, int y,
                                         int zl, const Coef3<T>& c, int corrected)
{
    MG_CHK(x >= 1 && x <= g.n - 2 && y >= 1 && y <= g.n - 2 && zl >= 1 && zl <= g.nzl - 2);
    const int col = (x + y + g.z0 + zl) & 1, q = x & 1;
    const long long idx = (long long)zl * g.plane + (long long)y * g.hp + (x >> 1);
    const T* own = v + (long long)col * g.cstride + idx;
    const T* oth = v + (long long)(col ^ 1) * g.cstride + idx;
    return residual_point<T, FAST>(oth[q - 1], oth[q], oth[-g.hp], oth[g.hp], oth[-g.plane], oth[g.plane], own[0],
                                   f[(long long)col * g.cstride + idx], c, corrected);
}

// N3/MultiGrid3D.cpp:180 with the exact grouping.  R(dx,dy,dz) reads the fine value at offset
// (dx,dy,dz) from the fine centre; reference names: suffix _C dy=0, _N dy=-1, _S dy=+1;
// N dz=+1, S dz=-1, E dx=+1, O dx=-1.
template <typename T, typename Getter>
__device__ __forceinline__ T restrict_point(Getter R)
{
    T C_C = R(0, 0, 0), N_C = R(0, 0, 1), S_C = R(0, 0, -1), E_C = R(1, 0, 0), O_C = R(-1, 0, 0);
    T NE_C = R(1, 0, 1), NO_C = R(-1, 0, 1), SE_C = R(1, 0, -1), SO_C = R(-1, 0, -1);
    T C_N = R(0, -1, 0), N_N = R(0, -1, 1), S_N = R(0, -1, -1), E_N = R(1, -1, 0), O_N = R(-1, -1, 0);
    T NE_N = R(1, -1, 1), NO_N = R(-1, -1, 1), SE_N = R(1, -1, -1), SO_N = R(-1, -1, -1);
    T C_S = R(0, 1, 0), N_S = R(0, 1, 1), S_S = R(0, 1, -1), E_S = R(1, 1, 0), O_S = R(-1, 1, 0);
    T NE_S = R(1, 1, 1), NO_S = R(-1, 1, 1), SE_S = R(1, 1, -1), SO_S = R(-1, 1, -1);

    T t1 = mul(T(1 / 8.0f), C_C);
    T t2 = mul(T(1 / 16.0f), add(add(add(add(N_C, E_C), S_C), O_C), add(C_N, C_S)));
    T g1 = add(add(add(NE_C, SE_C), SO_C), NO_C);
    T g2 = add(add(add(N_N, E_N), S_N), O_N);
    T g3 = add(add(add(N_S, E_S), S_S), O_S);
    T t3 = mul(T(1 / 32.0f), add(add(g1, g2), g3));
    T h1 = add(add(add(NE_N, SE_N), SO_N), NO_N);
    T h2 = add(add(add(NE_S, SE_S), SO_S), NO_S);
    T t4 = mul(T(1 / 64.0f), add(h1, h2));
    return add(add(add(t1, t2), t3), t4);
}

// N3/MultiGrid3D.cpp:216-331: trilinear prolongation by parity of (y,x,z).  C(dx,dy,dz) reads the coarse
// value (fx/2+dx, fy/2+dy, fz/2+dz); summation orders as written in the reference.
template <typename T, typename Getter>
__device__ __forceinline__ T interp_point(Getter C, int ox, int oy, int oz)
{
    if (!oz) {
        if (!oy) {
            if (!ox) return C(0, 0, 0);                                                    // PPP :216
            return mul(T(0.5f), add(C(0, 0, 0), C(1, 0, 0)));                              // PDP :222  O + E
        }
        if (!ox) return mul(T(0.5f), add(C(0, 0, 0), C(0, 1, 0)));                         // DPP :233  N + S
        return mul(T(0.25f), add(add(add(C(0, 0, 0), C(1, 0, 0)), C(0, 1, 0)), C(1, 1, 0)));  // DDP :244
    }
    if (!oy) {
        if (!ox) return mul(T(0.5f), add(C(0, 0, 0), C(0, 0, 1)));                         // PPD :261  S + N
        return mul(T(0.25f), add(add(add(C(0, 0, 1), C(1, 0, 1)), C(0, 0, 0)), C(1, 0, 0)));  // PDD :272
    }
    if (!ox) return mul(T(0.25f), add(add(add(C(0, 0, 0), C(0, 0, 1)), C(0, 1, 0)), C(0, 1, 1)));  // DPD :287
    // DDD :302  USO + UNO + UNE + USE + DSO + DNO + DNE + DSE
    T s = add(C(0, 0, 0), C(0, 0, 1));
    s = add(s, C(1, 0, 1));
    s = add(s, C(1, 0, 0));
    s = add(s, C(0, 1, 0));
    s = add(s, C(0, 1, 1));
    s = add(s, C(1, 1, 1));
    s = add(s, C(1, 1, 0));
    return mul(T(0.125f), s);
}

}  // namespace mg3

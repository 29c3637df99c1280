// mg3d_box.cu -- the 3D Poisson operators on NON-CUBIC grids (sizeX != sizeY != sizeZ, each 2^k + 1).
//
// The reference asserts such grids away (N3/Grid3D.cpp:10-11; the author's own TODO, SURVEY.md 8f rank 4) although its
// hierarchy (N3/MultiGrid3D.cpp:19-47) and operators are written per dimension.  This file is the device side of that
// generalisation: the same per-point formulas as the cubic engine (mg3d_device.cuh: relax_point, residual_point,
// restrict_point, interp_point -- expression order of the reference, no FMA contraction, IEEE division because the three
// mesh widths differ) on the same colour-split layout (mg3d_box.h), so that a red or black half-sweep moves the algorithmic
// 12 B/point with unit stride.  One thread per point; the fine residual is evaluated on the fly inside the restriction and
// never written to memory, prolongation and correction are one kernel.  Not tuned beyond the layout: no TMA staging, no
// temporal blocking, no fused multi-level tail (those stay with the cubic path, where the headline configurations live).
#include "mg3d_box.h"
#include "mg3d_device.cuh"

using namespace mgx;
using namespace mg3;

namespace {

__device__ __forceinline__ long long soff(const mg_geom3b& g, int x, int y, int z)
{
    return (long long)((x + y + z) & 1) * g.cstride + (long long)z * g.plane + (long long)y * g.hp + (x >> 1);
}
__device__ __forceinline__ long long doff(int nx, int ny, int x, int y, int z) { return (long long)x + (long long)nx * ((long long)y + (long long)ny * z); }

// MultiGrid3D::Relax, one colour (N3/MultiGrid3D.cpp:515 / :544): thread = one point of the colour, unit stride in both arrays
template <typename T>
__global__ void __launch_bounds__(128) k_bs_relax(T* __restrict__ v, const T* __restrict__ f, mg_geom3b g, Coef3<T> c, int colour)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, y = 1 + blockIdx.y, z = 1 + blockIdx.z;
    const int q = (colour + y + z) & 1, x = 2 * i + q;
    if (x < 1 || x > g.nx - 2) return;
    const long long idx = (long long)z * g.plane + (long long)y * g.hp + i;
    const T* oth = v + (long long)(colour ^ 1) * g.cstride + idx;
    const long long own = (long long)colour * g.cstride + idx;
    v[own] = relax_point<T, false>(oth[q - 1], oth[q], oth[-g.hp], oth[g.hp], oth[-g.plane], oth[g.plane], f[own], c);
}

// FAST: every h^2 is a power of two (a power-of-two range on 2^k + 1 points per axis), so x / h^2 == x * (1 / h^2) exactly
template <typename T, bool FAST>
__device__ __forceinline__ T residual_s(const T* __restrict__ v, const T* __restrict__ f, const mg_geom3b& g, int x, int y, int z, const Coef3<T>& c,
                                        int corrected)
{
    if (x == 0 || x == g.nx - 1 || y == 0 || y == g.ny - 1 || z == 0 || z == g.nz - 1) return T(0);  // :704-705
    const int col = (x + y + z) & 1, q = x & 1;
    const long long idx = (long long)z * g.plane + (long long)y * g.hp + (x >> 1);
    const T* own = v + (long long)col * g.cstride + idx;
    const T* oth = v + (long long)(col ^ 1) * g.cstride + idx;
    return residual_point<T, FAST>(oth[q - 1], oth[q], oth[-g.hp], oth[g.hp], oth[-g.plane], oth[g.plane], own[0], f[(long long)col * g.cstride + idx], c,
                                    corrected);
}

// MultiGrid3D::CalculateResidual (N3/MultiGrid3D.cpp:678-730) into a caller-visible DENSE array
template <typename T, bool FAST>
__global__ void __launch_bounds__(128) k_bs_residual_dense(const T* __restrict__ v, const T* __restrict__ f, T* __restrict__ r, mg_geom3b g, Coef3<T> c,
                                                           int corrected)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
    if (x >= g.nx) return;
    r[doff(g.nx, g.ny, x, y, z)] = residual_s<T, FAST>(v, f, g, x, y, z, c, corrected);
}

// Restrict (N3/MultiGrid3D.cpp:50-184).  RESIDUAL: the fine operand is CalculateResidual(fine v, fine f), evaluated on the fly,
// and the coarse v is zeroed (setToValue(coarse v, 0, true), :634) -- the three steps of VCycle in one kernel.
template <typename T, bool RESIDUAL, bool FAST>
__global__ void __launch_bounds__(128) k_bs_restrict(const T* __restrict__ fv, const T* __restrict__ ff, mg_geom3b g, Coef3<T> c, int corrected,
                                                     T* __restrict__ cf, T* __restrict__ cv, mg_geom3b gc)
{
    const int cx = blockIdx.x * blockDim.x + threadIdx.x, cy = blockIdx.y, cz = blockIdx.z;
    if (cx >= gc.nx) return;
    const int fx = 2 * cx, fy = 2 * cy, fz = 2 * cz;
    auto R = [&](int dx, int dy, int dz) -> T {
        if (RESIDUAL) return residual_s<T, FAST>(fv, ff, g, fx + dx, fy + dy, fz + dz, c, corrected);
        return ff[soff(g, fx + dx, fy + dy, fz + dz)];
    };
    const bool bnd = cx == 0 || cx == gc.nx - 1 || cy == 0 || cy == gc.ny - 1 || cz == 0 || cz == gc.nz - 1;
    const long long ci = soff(gc, cx, cy, cz);
    cf[ci] = bnd ? R(0, 0, 0) : restrict_point<T>(R);  // :113-119 injection on the boundary
    if (RESIDUAL) cv[ci] = T(0);
}

// Interpolate (N3/MultiGrid3D.cpp:186-335), interior of the fine grid; ADD: + ApplyCorrection (:649-676)
template <typename T, bool ADD>
__global__ void __launch_bounds__(128) k_bs_interpolate(T* __restrict__ fv, mg_geom3b g, const T* __restrict__ cv, mg_geom3b gc)
{
    const int x = 1 + blockIdx.x * blockDim.x + threadIdx.x, y = 1 + blockIdx.y, z = 1 + blockIdx.z;
    if (x > g.nx - 2) return;
    const int cx = x >> 1, cy = y >> 1, cz = z >> 1;
    auto C = [&](int dx, int dy, int dz) -> T { return cv[soff(gc, cx + dx, cy + dy, cz + dz)]; };
    const T e = interp_point<T>(C, x & 1, y & 1, z & 1);
    const long long i = soff(g, x, y, z);
    fv[i] = ADD ? add(fv[i], e) : e;
}

// setToValue (N3/MultiGrid3D.cpp:587-621)
template <typename T>
__global__ void __launch_bounds__(128) k_bs_set(T* __restrict__ a, mg_geom3b g, T value, int modify_boundaries)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
    if (x >= g.nx) return;
    const bool bnd = x == 0 || x == g.nx - 1 || y == 0 || y == g.ny - 1 || z == 0 || z == g.nz - 1;
    if (modify_boundaries || !bnd) a[soff(g, x, y, z)] = value;
}

// Grid3D::InitF (N3/Grid3D.cpp:78-96): (real)(-3*PI*PI*sin(PI x)*sin(PI y)*sin(PI z)), the product in double, left to right;
// the sines are host-libm tables (the reference's own values)
template <typename T>
__global__ void __launch_bounds__(128) k_bs_init_f(T* __restrict__ f, mg_geom3b g, const double* __restrict__ sx, const double* __restrict__ sy,
                                                   const double* __restrict__ sz)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
    if (x >= g.nx) return;
    const double PI = 3.141592653589793;
    const double k = __dmul_rn(__dmul_rn(-3.0, PI), PI);
    f[soff(g, x, y, z)] = (T)__dmul_rn(__dmul_rn(__dmul_rn(k, sx[x]), sy[y]), sz[z]);
}

// dense (reference layout) <-> colour-split
template <typename T, bool TO_SPLIT>
__global__ void __launch_bounds__(128) k_bs_repack(T* __restrict__ split, mg_geom3b g, T* __restrict__ dense)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
    if (x >= g.nx) return;
    if (TO_SPLIT) split[soff(g, x, y, z)] = dense[doff(g.nx, g.ny, x, y, z)];
    else dense[doff(g.nx, g.ny, x, y, z)] = split[soff(g, x, y, z)];
}

// ||r||_2^2 and ||r||_inf of CalculateResidual, two deterministic stages: one partial pair per block, then one thread
template <typename T, bool FAST>
__global__ void __launch_bounds__(256) k_bs_norm(const T* __restrict__ v, const T* __restrict__ f, mg_geom3b g, Coef3<T> c, int corrected,
                                                 double* __restrict__ parts, int nparts)
{
    __shared__ double sh[64];
    const long long tot = (long long)g.nx * g.ny * g.nz, per = (tot + nparts - 1) / nparts;
    const long long lo = (long long)blockIdx.x * per, hi = lo + per < tot ? lo + per : tot;
    double s = 0.0, m = 0.0;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const int x = (int)(i % g.nx), y = (int)((i / g.nx) % g.ny), z = (int)(i / ((long long)g.nx * g.ny));
        const double r = (double)residual_s<T, FAST>(v, f, g, x, y, z, c, corrected);
        s += r * r;
        m = max_nan(m, fabs(r));
    }
    block_sum_max(s, m, sh);
    if (threadIdx.x == 0) { parts[blockIdx.x] = s; parts[nparts + blockIdx.x] = m; }
}

__global__ void k_bs_norm_final(const double* __restrict__ parts, int nparts, double* __restrict__ out2)
{
    if (threadIdx.x || blockIdx.x) return;
    double s = 0.0, m = 0.0;
    for (int i = 0; i < nparts; i++) { s += parts[i]; m = max_nan(m, parts[nparts + i]); }
    out2[0] = s;
    out2[1] = m;
}

// ---- the reference's operators on free DENSE arrays (the host-array entry points mg3b_*_host) ----
struct DGeom { int nx, ny, nz; };

template <typename T>
__global__ void __launch_bounds__(128) k_bd_restrict(const T* __restrict__ ff, DGeom g, T* __restrict__ cf, DGeom gc)
{
    const int cx = blockIdx.x * blockDim.x + threadIdx.x, cy = blockIdx.y, cz = blockIdx.z;
    if (cx >= gc.nx) return;
    const int fx = 2 * cx, fy = 2 * cy, fz = 2 * cz;
    auto R = [&](int dx, int dy, int dz) -> T { return ff[doff(g.nx, g.ny, fx + dx, fy + dy, fz + dz)]; };
    const bool bnd = cx == 0 || cx == gc.nx - 1 || cy == 0 || cy == gc.ny - 1 || cz == 0 || cz == gc.nz - 1;
    cf[doff(gc.nx, gc.ny, cx, cy, cz)] = bnd ? R(0, 0, 0) : restrict_point<T>(R);
}

template <typename T>
__global__ void __launch_bounds__(128) k_bd_interpolate(T* __restrict__ fv, DGeom g, const T* __restrict__ cv, DGeom gc)
{
    const int x = 1 + blockIdx.x * blockDim.x + threadIdx.x, y = 1 + blockIdx.y, z = 1 + blockIdx.z;
    if (x > g.nx - 2) return;
    const int cx = x >> 1, cy = y >> 1, cz = z >> 1;
    auto C = [&](int dx, int dy, int dz) -> T { return cv[doff(gc.nx, gc.ny, cx + dx, cy + dy, cz + dz)]; };
    fv[doff(g.nx, g.ny, x, y, z)] = interp_point<T>(C, x & 1, y & 1, z & 1);
}

template <typename T>
__global__ void __launch_bounds__(128) k_bd_apply_correction(T* __restrict__ fv, const T* __restrict__ err, DGeom g)
{
    const int x = 1 + blockIdx.x * blockDim.x + threadIdx.x, y = 1 + blockIdx.y, z = 1 + blockIdx.z;
    if (x > g.nx - 2) return;
    const long long i = doff(g.nx, g.ny, x, y, z);
    fv[i] = add(fv[i], err[i]);
}

template <typename T>
__global__ void __launch_bounds__(128) k_bd_set(T* __restrict__ a, DGeom g, T value, int modify_boundaries)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, z = blockIdx.z;
    if (x >= g.nx) return;
    const bool bnd = x == 0 || x == g.nx - 1 || y == 0 || y == g.ny - 1 || z == 0 || z == g.nz - 1;
    if (modify_boundaries || !bnd) a[doff(g.nx, g.ny, x, y, z)] = value;
}

inline dim3 grid_for(int w, int ny, int nz) { return dim3((unsigned)((w + 127) / 128), (unsigned)ny, (unsigned)nz); }
inline int ok() { return cudaPeekAtLastError() == cudaSuccess ? 1 : -1; }
inline DGeom dg(const int n[3]) { return DGeom{n[0], n[1], n[2]}; }

}  // namespace

#define BOX_DISPATCH(expr_f, expr_d) \
    do {                             \
        if (dtype == 0) { expr_f; }  \
        else { expr_d; }             \
    } while (0)

extern "C" {

int mgk3b_relax_colour(cudaStream_t s, int dtype, void* v, const void* f, mg_geom3b g, mg_coef3d c, int colour)
{
    if (g.nx < 3 || g.ny < 3 || g.nz < 3) return 0;
    const dim3 grid = grid_for(g.nx / 2 + 1, g.ny - 2, g.nz - 2);
    BOX_DISPATCH((k_bs_relax<float><<<grid, 128, 0, s>>>((float*)v, (const float*)f, g, narrow<float>(c), colour)),
                 (k_bs_relax<double><<<grid, 128, 0, s>>>((double*)v, (const double*)f, g, narrow<double>(c), colour)));
    return ok();
}

int mgk3b_residual_dense(cudaStream_t s, int dtype, const void* v, const void* f, void* r, mg_geom3b g, mg_coef3d c, int corrected)
{
    const dim3 grid = grid_for(g.nx, g.ny, g.nz);
    if (c.fast_h)
        BOX_DISPATCH((k_bs_residual_dense<float, true><<<grid, 128, 0, s>>>((const float*)v, (const float*)f, (float*)r, g, narrow<float>(c), corrected)),
                     (k_bs_residual_dense<double, true><<<grid, 128, 0, s>>>((const double*)v, (const double*)f, (double*)r, g, narrow<double>(c), corrected)));
    else
        BOX_DISPATCH((k_bs_residual_dense<float, false><<<grid, 128, 0, s>>>((const float*)v, (const float*)f, (float*)r, g, narrow<float>(c), corrected)),
                     (k_bs_residual_dense<double, false><<<grid, 128, 0, s>>>((const double*)v, (const double*)f, (double*)r, g, narrow<double>(c), corrected)));
    return ok();
}

int mgk3b_restrict(cudaStream_t s, int dtype, const void* fv, const void* ff, mg_geom3b g, mg_coef3d c, int corrected, void* cf, void* cv, mg_geom3b gc)
{
    const dim3 grid = grid_for(gc.nx, gc.ny, gc.nz);
    if (fv && c.fast_h)
        BOX_DISPATCH((k_bs_restrict<float, true, true><<<grid, 128, 0, s>>>((const float*)fv, (const float*)ff, g, narrow<float>(c), corrected, (float*)cf, (float*)cv, gc)),
                     (k_bs_restrict<double, true, true><<<grid, 128, 0, s>>>((const double*)fv, (const double*)ff, g, narrow<double>(c), corrected, (double*)cf, (double*)cv, gc)));
    else if (fv)
        BOX_DISPATCH((k_bs_restrict<float, true, false><<<grid, 128, 0, s>>>((const float*)fv, (const float*)ff, g, narrow<float>(c), corrected, (float*)cf, (float*)cv, gc)),
                     (k_bs_restrict<double, true, false><<<grid, 128, 0, s>>>((const double*)fv, (const double*)ff, g, narrow<double>(c), corrected, (double*)cf, (double*)cv, gc)));
    else
        BOX_DISPATCH((k_bs_restrict<float, false, false><<<grid, 128, 0, s>>>(nullptr, (const float*)ff, g, narrow<float>(c), corrected, (float*)cf, nullptr, gc)),
                     (k_bs_restrict<double, false, false><<<grid, 128, 0, s>>>(nullptr, (const double*)ff, g, narrow<double>(c), corrected, (double*)cf, nullptr, gc)));
    return ok();
}

int mgk3b_interpolate(cudaStream_t s, int dtype, void* fv, mg_geom3b g, const void* cv, mg_geom3b gc, int add)
{
    if (g.nx < 3 || g.ny < 3 || g.nz < 3) return 0;
    const dim3 grid = grid_for(g.nx - 2, g.ny - 2, g.nz - 2);
    if (add)
        BOX_DISPATCH((k_bs_interpolate<float, true><<<grid, 128, 0, s>>>((float*)fv, g, (const float*)cv, gc)),
                     (k_bs_interpolate<double, true><<<grid, 128, 0, s>>>((double*)fv, g, (const double*)cv, gc)));
    else
        BOX_DISPATCH((k_bs_interpolate<float, false><<<grid, 128, 0, s>>>((float*)fv, g, (const float*)cv, gc)),
                     (k_bs_interpolate<double, false><<<grid, 128, 0, s>>>((double*)fv, g, (const double*)cv, gc)));
    return ok();
}

int mgk3b_set(cudaStream_t s, int dtype, void* a, mg_geom3b g, double value, int modify_boundaries)
{
    const dim3 grid = grid_for(g.nx, g.ny, g.nz);
    BOX_DISPATCH((k_bs_set<float><<<grid, 128, 0, s>>>((float*)a, g, (float)value, modify_boundaries)),
                 (k_bs_set<double><<<grid, 128, 0, s>>>((double*)a, g, value, modify_boundaries)));
    return ok();
}

int mgk3b_init_f(cudaStream_t s, int dtype, void* f, mg_geom3b g, const double* sx, const double* sy, const double* sz)
{
    const dim3 grid = grid_for(g.nx, g.ny, g.nz);
    BOX_DISPATCH((k_bs_init_f<float><<<grid, 128, 0, s>>>((float*)f, g, sx, sy, sz)), (k_bs_init_f<double><<<grid, 128, 0, s>>>((double*)f, g, sx, sy, sz)));
    return ok();
}

int mgk3b_repack(cudaStream_t s, int dtype, void* split, mg_geom3b g, void* dense, int to_split)
{
    const dim3 grid = grid_for(g.nx, g.ny, g.nz);
    if (to_split)
        BOX_DISPATCH((k_bs_repack<float, true><<<grid, 128, 0, s>>>((float*)split, g, (float*)dense)),
                     (k_bs_repack<double, true><<<grid, 128, 0, s>>>((double*)split, g, (double*)dense)));
    else
        BOX_DISPATCH((k_bs_repack<float, false><<<grid, 128, 0, s>>>((float*)split, g, (float*)dense)),
                     (k_bs_repack<double, false><<<grid, 128, 0, s>>>((double*)split, g, (double*)dense)));
    return ok();
}

/* parts: 2 * nparts doubles of scratch; out2 = {sum r^2, max |r|} */
int mgk3b_residual_norm(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom3b g, mg_coef3d c, int corrected, double* parts, int nparts,
                        double* out2)
{
    if (c.fast_h)
        BOX_DISPATCH((k_bs_norm<float, true><<<nparts, 256, 0, s>>>((const float*)v, (const float*)f, g, narrow<float>(c), corrected, parts, nparts)),
                     (k_bs_norm<double, true><<<nparts, 256, 0, s>>>((const double*)v, (const double*)f, g, narrow<double>(c), corrected, parts, nparts)));
    else
        BOX_DISPATCH((k_bs_norm<float, false><<<nparts, 256, 0, s>>>((const float*)v, (const float*)f, g, narrow<float>(c), corrected, parts, nparts)),
                     (k_bs_norm<double, false><<<nparts, 256, 0, s>>>((const double*)v, (const double*)f, g, narrow<double>(c), corrected, parts, nparts)));
    if (ok() < 0) return -1;
    k_bs_norm_final<<<1, 32, 0, s>>>(parts, nparts, out2);
    return ok() < 0 ? -1 : 2;
}

int mgk3b_dense_restrict(cudaStream_t s, int dtype, const void* fine, const int n[3], void* coarse, const int cn[3])
{
    const dim3 grid = grid_for(cn[0], cn[1], cn[2]);
    BOX_DISPATCH((k_bd_restrict<float><<<grid, 128, 0, s>>>((const float*)fine, dg(n), (float*)coarse, dg(cn))),
                 (k_bd_restrict<double><<<grid, 128, 0, s>>>((const double*)fine, dg(n), (double*)coarse, dg(cn))));
    return ok();
}

int mgk3b_dense_interpolate(cudaStream_t s, int dtype, void* fine, const int n[3], const void* coarse, const int cn[3])
{
    const dim3 grid = grid_for(n[0] - 2, n[1] - 2, n[2] - 2);
    BOX_DISPATCH((k_bd_interpolate<float><<<grid, 128, 0, s>>>((float*)fine, dg(n), (const float*)coarse, dg(cn))),
                 (k_bd_interpolate<double><<<grid, 128, 0, s>>>((double*)fine, dg(n), (const double*)coarse, dg(cn))));
    return ok();
}

int mgk3b_dense_apply_correction(cudaStream_t s, int dtype, void* fine, const void* err, const int n[3])
{
    const dim3 grid = grid_for(n[0] - 2, n[1] - 2, n[2] - 2);
    BOX_DISPATCH((k_bd_apply_correction<float><<<grid, 128, 0, s>>>((float*)fine, (const float*)err, dg(n))),
                 (k_bd_apply_correction<double><<<grid, 128, 0, s>>>((double*)fine, (const double*)err, dg(n))));
    return ok();
}

int mgk3b_dense_set(cudaStream_t s, int dtype, void* a, const int n[3], double value, int modify_boundaries)
{
    const dim3 grid = grid_for(n[0], n[1], n[2]);
    BOX_DISPATCH((k_bd_set<float><<<grid, 128, 0, s>>>((float*)a, dg(n), (float)value, modify_boundaries)),
                 (k_bd_set<double><<<grid, 128, 0, s>>>((double*)a, dg(n), value, modify_boundaries)));
    return ok();
}

}  // extern "C"

// mg3d_kernels.cu -- sm_100a kernels of the 3D Poisson multigrid hot path.
//
// Replaces the operators of the reference class MultiGrid3D (CPU: NOCUDA_TESI/POISSON_3D(TESI)/
// MultiGrid3D.cpp; GPU twin: CUDA_TESI/CUDA Poisson 3D/MultiGrid3D.cu:362-793).  Arithmetic follows
// the reference expression by expression (SURVEY.md Appendix A) through the non-contracting helpers of
// mg_exact.cuh, so results are bit-identical to the CPU solver for float and double.
//
// DEVICE LAYOUT: colour-split.  Every field (v, f on every level) is stored as two arrays, one per
// red-black colour c = (x+y+z) & 1, each compacted along x:
//     element (x,y,zl) lives at  base[c*cstride + zl*plane + y*hp + (x>>1)]
// A red half-sweep then reads ONLY the black array of v, the red array of f and writes ONLY the red
// array of v, all with unit stride: 12 B/point per half-sweep in fp64, i.e. exactly the algorithmic
// 24 B/point per RB sweep of SURVEY.md 8(d).  With interleaved colours the same kernel pulls every
// 32-B sector of v and f and writes every sector of v (48 B/point per sweep; measured: profiles/
// r1_v1_relax_colour_ncu_full.txt).  Neighbours of a point of colour c at half-index i in row (y,z),
// q = x & 1:  O/E = other[i-1+q], other[i+q];  N/S = other[i -/+ hp];  D/U = other[i -/+ plane].
//
// All stages are HBM-bound stencils (<= 2 flop/B): no tensor cores.
#include <stdint.h>

#include "mg3d_device.cuh"

using namespace mgx;
using namespace mg3;

namespace {

// ---------------------------------------------------------------------------------------------
// Smoother: one colour per launch, in place.  Points of colour `colour` only read the other colour's
// array, so there is no race (unlike the reference's CUDARelax, which updates both colours in one launch
// behind a block-local barrier, C3/MultiGrid3D.cu:635-673).  Thread (i, y, zl) owns half-index i of row
// (y, zl): x = 2i + q with q = (colour + y + z) & 1.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FAST>
__global__ void __launch_bounds__(256)
k_relax_colour(T* __restrict__ v, const T* __restrict__ f, mg_geom3d g, Coef3<T> c, int colour, int zl_lo, int zl_step)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    const int zl = zl_lo + blockIdx.z * zl_step;
    if (y > g.n - 2) return;
    const int q = (colour + y + g.z0 + zl) & 1;
    const int x = 2 * i + q;
    if (x < 1 || x > g.n - 2) return;
    MG_CHK_SITE(g, i, y, zl);
    MG_CHK(zl >= 1 && zl <= g.nzl - 2 && i + q - 1 >= 0 && i + q < g.hp);
    const long long idx = (long long)zl * g.plane + (long long)y * g.hp + i;
    const T* oth = v + (long long)(colour ^ 1) * g.cstride + idx;
    const long long own = (long long)colour * g.cstride + idx;
    v[own] = relax_point<T, FAST>(oth[q - 1], oth[q], oth[-g.hp], oth[g.hp], oth[-g.plane], oth[g.plane], f[own], c);
}

// ---------------------------------------------------------------------------------------------
// Weighted-Jacobi half of a sweep on ONE colour array: every interior point of `colour` becomes
//     old + omega * (gs - old),   gs = the reference's Gauss-Seidel expression (N3/MultiGrid3D.cpp:532)
// evaluated on the OLD values of the six neighbours (all of the other colour).  The reference has no
// Jacobi smoother (SURVEY.md 8f rank 4): the tests check this against a CPU restatement of the same formula.
// dst/own/oth/f are colour-array base pointers.  dst may be `own` (in place: a point reads only its own
// old value of that array) or a scratch array, which then also receives the non-interior points so that
// it can stand in for the colour array in the next sweep.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FAST>
__global__ void __launch_bounds__(256)
k_jacobi_colour(T* __restrict__ dst, const T* own, const T* __restrict__ oth, const T* __restrict__ f, mg_geom3d g,
                Coef3<T> c, T omega, int colour, int zl_lo)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int zl = zl_lo + blockIdx.z, z = g.z0 + zl;
    if (y > g.n - 1) return;
    const int q = (colour + y + z) & 1;
    const int x = 2 * i + q;
    if (x > g.n - 1) return;
    MG_CHK_SITE(g, i, y, zl);
    const long long idx = (long long)zl * g.plane + (long long)y * g.hp + i;
    const T old = own[idx];
    const bool interior = x >= 1 && x <= g.n - 2 && y >= 1 && y <= g.n - 2 && z >= 1 && z <= g.n - 2;
    T out = old;
    if (interior) {
        const T* o = oth + idx;
        const T gs = relax_point<T, FAST>(o[q - 1], o[q], o[-g.hp], o[g.hp], o[-g.plane], o[g.plane], f[idx], c);
        out = add(old, mul(omega, sub(gs, old)));
    }
    if (interior || dst != own) dst[idx] = out;
}

// ---------------------------------------------------------------------------------------------
// CalculateResidual into a full (colour-split) array; only used when the caller asks for it.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FAST>
__global__ void k_residual(const T* __restrict__ v, const T* __restrict__ f, T* __restrict__ r, mg_geom3d g,
                           Coef3<T> c, int corrected, int zl_lo)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int zl = zl_lo + blockIdx.z;
    const int z = g.z0 + zl;
    if (x >= g.n || y >= g.n) return;
    T out = T(0);
    if (!(x == 0 || x == g.n - 1 || y == 0 || y == g.n - 1 || z == 0 || z == g.n - 1))
        out = residual_at<T, FAST>(v, f, g, x, y, zl, c, corrected);
    r[off3(g, x, y, zl)] = out;
}

// ---------------------------------------------------------------------------------------------
// Residual norms: sum r^2 (fp64) and max |r|, residual recomputed on the fly, warp-shuffle
// reduction, one partial per block (deterministic), finished by k_norm_final.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FAST>
__global__ void __launch_bounds__(256)
k_residual_norm(const T* __restrict__ v, const T* __restrict__ f, mg_geom3d g, Coef3<T> c, int corrected, int zl_lo,
                int zl_hi, double* __restrict__ part)
{
    __shared__ double sh[64];
    double s = 0.0, m = 0.0;
    const int ni = g.n - 2;
    const long long rows = (long long)ni * (zl_hi - zl_lo);
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const int zl = zl_lo + (int)(row / ni);
        const int y = 1 + (int)(row % ni);
        const int z = g.z0 + zl;
        if (z == 0 || z == g.n - 1) continue;
        for (int x = 1 + threadIdx.x; x <= g.n - 2; x += blockDim.x) {
            const double rd = (double)residual_at<T, FAST>(v, f, g, x, y, zl, c, corrected);
            s += rd * rd;
            m = max_nan(m, fabs(rd));
        }
    }
    block_sum_max(s, m, sh);
    if (threadIdx.x == 0) { part[blockIdx.x] = s; part[gridDim.x + blockIdx.x] = m; }
}

__global__ void k_norm_final(const double* __restrict__ part, int nparts, double* __restrict__ out2)
{
    __shared__ double sh[64];
    double s = 0.0, m = 0.0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        s += part[i];
        m = max_nan(m, part[nparts + i]);
    }
    block_sum_max(s, m, sh);
    if (threadIdx.x == 0) { out2[0] = s; out2[1] = m; }
}

// ---------------------------------------------------------------------------------------------
// Restrict (27-point full weighting, boundary injection), one thread per coarse point.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_restrict(const T* __restrict__ fine, mg_geom3d gf, T* __restrict__ coarse, mg_geom3d gc, int czl_lo)
{
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;
    const int cy = blockIdx.y * blockDim.y + threadIdx.y;
    const int czl = czl_lo + blockIdx.z;
    const int cz = gc.z0 + czl;
    if (cx >= gc.n || cy >= gc.n) return;
    const int fx = 2 * cx, fy = 2 * cy, fzl = 2 * cz - gf.z0;
    T out;
    if (cx == 0 || cx == gc.n - 1 || cy == 0 || cy == gc.n - 1 || cz == 0 || cz == gc.n - 1)
        out = fine[off3(gf, fx, fy, fzl)];  // N3/MultiGrid3D.cpp:113-119
    else
        out = restrict_point<T>([&](int dx, int dy, int dz) { return fine[off3(gf, fx + dx, fy + dy, fzl + dz)]; });
    coarse[off3(gc, cx, cy, czl)] = out;
}

// ---------------------------------------------------------------------------------------------
// Fused CalculateResidual -> Restrict -> coarse f, plus setToValue(coarse v, 0, true).
// A CTA owns a CX x CY x CZ tile of coarse points; it evaluates the fine residual on the
// (2CX+1)(2CY+1)(2CZ+1) fine points around the tile into shared memory (fine boundary = 0 as in
// CalculateResidual) and restricts from there.  The fine residual never goes to HBM.
// ---------------------------------------------------------------------------------------------
template <typename T, bool FAST, int CX, int CY, int CZ>
__global__ void __launch_bounds__(256)
k_residual_restrict(const T* __restrict__ v, const T* __restrict__ f, mg_geom3d gf, Coef3<T> c, int corrected,
                    T* __restrict__ cf, T* __restrict__ cv, mg_geom3d gc, int czl_lo, int czl_hi)
{
    constexpr int FX = 2 * CX + 1, FY = 2 * CY + 1, FZ = 2 * CZ + 1;
    __shared__ T r[FZ][FY][FX];

    const int cx0 = blockIdx.x * CX, cy0 = blockIdx.y * CY;
    const int czl0 = czl_lo + blockIdx.z * CZ;   // first coarse local plane of the tile
    const int cz0 = gc.z0 + czl0;                // global
    const int fx0 = 2 * cx0 - 1, fy0 = 2 * cy0 - 1, fz0 = 2 * cz0 - 1;  // global fine origin of the smem tile
    const int n = gf.n;

    for (int i = threadIdx.x; i < FX * FY * FZ; i += 256) {
        const int lx = i % FX, ly = (i / FX) % FY, lz = i / (FX * FY);
        const int fx = fx0 + lx, fy = fy0 + ly, fz = fz0 + lz;
        T val = T(0);
        if (fx >= 1 && fx <= n - 2 && fy >= 1 && fy <= n - 2 && fz >= 1 && fz <= n - 2) {
            const int fzl = fz - gf.z0;
            if (fzl >= 1 && fzl <= gf.nzl - 2) val = residual_at<T, FAST>(v, f, gf, fx, fy, fzl, c, corrected);
        }
        r[lz][ly][lx] = val;
    }
    __syncthreads();

    for (int i = threadIdx.x; i < CX * CY * CZ; i += 256) {
        const int tx = i % CX, ty = (i / CX) % CY, tz = i / (CX * CY);
        const int cx = cx0 + tx, cy = cy0 + ty, czl = czl0 + tz, cz = cz0 + tz;
        if (cx >= gc.n || cy >= gc.n || czl >= czl_hi) continue;
        T out = T(0);  // boundary: injection of the (zero) boundary residual, N3/MultiGrid3D.cpp:113-119 + :705
        if (!(cx == 0 || cx == gc.n - 1 || cy == 0 || cy == gc.n - 1 || cz == 0 || cz == gc.n - 1)) {
            const int lx = 2 * tx + 1, ly = 2 * ty + 1, lz = 2 * tz + 1;
            out = restrict_point<T>([&](int dx, int dy, int dz) { return r[lz + dz][ly + dy][lx + dx]; });
        }
        const long long ci = off3(gc, cx, cy, czl);
        cf[ci] = out;
        cv[ci] = T(0);  // setToValue(coarse->h_v, 0, true), N3/MultiGrid3D.cpp:634
    }
}

// ---------------------------------------------------------------------------------------------
// Interpolate (+ ApplyCorrection when add != 0), N3/MultiGrid3D.cpp:186-335 and :649-676, organised by coarse
// cell: a thread owns the coarse cell (cx, cy) and marches along z;
// per cell it holds the 8 corner values in registers (the 4 upper corners become the next cell's lower
// ones) and produces the 2x2x2 fine points (2cx+ox, 2cy+oy, 2cz+oz) with the reference's per-parity
// formulas.  One coarse load per fine point instead of up to eight, no per-point 64-bit index arithmetic;
// both colour arrays of the fine level are touched with unit stride (the pair x = 2cx, 2cx+1 shares the
// half-index cx).
// MASK selects the colours that are produced (bit c = colour c).  Inside a V-cycle with nu2 >= 1 the correction of
// the colour-0 points is dead: the first half-sweep of the post-smoothing overwrites every interior colour-0 point
// from its colour-1 neighbours alone (the Gauss-Seidel update never reads the point's own old value), so the cycle
// asks for MASK = 2 and this kernel moves half the fine-level bytes; results are bit-identical.
// The kernel is latency-bound on its global loads (ncu: long-scoreboard stalls 21 per issue at 4 blocks per SM), so the
// colour-1 variant is held to 40 registers for 6 blocks per SM: 2.04 -> 1.73 ms at 1025^3 fp64.
template <typename T, int MASK>
__global__ void __launch_bounds__(256, MASK == 2 ? 6 : 4)
k_interp_octet(T* __restrict__ fine, mg_geom3d gf, const T* __restrict__ coarse, mg_geom3d gc, int add_, int zl_lo,
               int zl_hi, int cz_first, int cz_last, int kchunk, const unsigned int* __restrict__ cond)
{
    if (cond && *cond == 0u) return;  // conditional launch: see mgk3d_interpolate
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;
    const int cy = blockIdx.y * blockDim.y + threadIdx.y;
    if (cx > gc.n - 2 || cy > gc.n - 2) return;
    const int k0 = cz_first + blockIdx.z * kchunk;
    const int k1 = min(k0 + kchunk - 1, cz_last);
    if (k0 > k1) return;
    // corner (dx,dy) of coarse plane cz: colour (cx+dx+cy+dy+cz)&1, half-index (cx+dx)>>1
    long long cbase[4];
    int cpar[4];
#pragma unroll
    for (int d = 0; d < 4; d++) {
        const int dx = d & 1, dy = d >> 1;
        cbase[d] = (long long)(cy + dy) * gc.hp + ((cx + dx) >> 1);
        cpar[d] = (cx + dx + cy + dy) & 1;
    }
    auto load_plane = [&](int cz, T (&dst)[4]) {
        MG_CHK(cz - gc.z0 >= 0 && cz - gc.z0 < gc.nzl && cy + 1 < gc.n && ((cx + 1) >> 1) < gc.hp);
        const long long pz = (long long)(cz - gc.z0) * gc.plane;
#pragma unroll
        for (int d = 0; d < 4; d++) dst[d] = coarse[(long long)((cpar[d] + cz) & 1) * gc.cstride + pz + cbase[d]];
    };
    T lo[4], hi[4];
    load_plane(k0, lo);
    const int n = gf.n;
    for (int k = k0; k <= k1; k++) {
        // all loads of the cell are issued before any arithmetic (12 independent requests per thread):
        // the first version loaded, added and stored point by point and was latency-bound (ncu:
        // long_scoreboard 46 of 50 stall cycles per issue, 43 % of DRAM bandwidth)
        load_plane(k + 1, hi);
        T* ptr[8];
        T old[8];
#pragma unroll
        for (int oz = 0; oz < 2; oz++) {
            const int z = 2 * k + oz, zl = z - gf.z0;
            const bool zok = z >= 1 && z <= n - 2 && zl >= zl_lo && zl < zl_hi;
#pragma unroll
            for (int oy = 0; oy < 2; oy++) {
                const int y = 2 * cy + oy;
                const int c0 = (oy + oz) & 1;  // colour of the even-x point of the pair: (2cx + y + z) & 1, a compile-time value
                const long long idx = (long long)zl * gf.plane + (long long)y * gf.hp + cx;
                const bool ok = zok && y >= 1;  // y <= n-2 holds for every cell row
                if (ok) MG_CHK_SITE(gf, cx, y, zl);
                ptr[oz * 4 + oy * 2 + 0] = (ok && cx >= 1 && ((MASK >> c0) & 1)) ? fine + (long long)c0 * gf.cstride + idx : nullptr;
                ptr[oz * 4 + oy * 2 + 1] = (ok && ((MASK >> (c0 ^ 1)) & 1)) ? fine + (long long)(c0 ^ 1) * gf.cstride + idx : nullptr;
            }
        }
        if (add_) {
#pragma unroll
            for (int m = 0; m < 8; m++) old[m] = ptr[m] ? *ptr[m] : T(0);
        }
        auto C = [&](int dx, int dy, int dz) { return dz ? hi[dy * 2 + dx] : lo[dy * 2 + dx]; };
#pragma unroll
        for (int m = 0; m < 8; m++) {
            const T e = interp_point<T>(C, m & 1, (m >> 1) & 1, m >> 2);
            if (ptr[m]) *ptr[m] = add_ ? add(old[m], e) : e;
        }
#pragma unroll
        for (int d = 0; d < 4; d++) lo[d] = hi[d];
    }
}

// zl_skip_lo < zl_skip_hi: the planes [zl_skip_lo, zl_skip_hi) are left out (a slab's own planes: only its ghost planes are set)
template <typename T>
__global__ void k_set(T* __restrict__ a, mg_geom3d g, T value, int modify_boundaries, int zl_lo, int zl_skip_lo, int zl_skip_hi)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    int zl = zl_lo + blockIdx.z;
    if (zl >= zl_skip_lo) zl += zl_skip_hi - zl_skip_lo;
    const int z = g.z0 + zl;
    if (x >= g.n || y >= g.n) return;
    if (!modify_boundaries && (x == 0 || x == g.n - 1 || y == 0 || y == g.n - 1 || z == 0 || z == g.n - 1)) return;
    a[off3(g, x, y, zl)] = value;
}

// N3/Grid3D.cpp:92: h_f = -3*PI*PI*sin(PI*x)*sin(PI*y)*sin(PI*z) evaluated left to right in double,
// narrowed to T.  The sines come from host libm tables so they are the reference's own values.
template <typename T>
__global__ void k_init_f(T* __restrict__ f, mg_geom3d g, const double* __restrict__ sx, const double* __restrict__ sy,
                         const double* __restrict__ sz, int zl_lo)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int zl = zl_lo + blockIdx.z;
    const int z = g.z0 + zl;
    if (x >= g.n || y >= g.n) return;
    const double PI = 3.141592653589793;
    const double k = __dmul_rn(__dmul_rn(-3.0, PI), PI);
    f[off3(g, x, y, zl)] = (T)__dmul_rn(__dmul_rn(__dmul_rn(k, sx[x]), sy[y]), sz[z]);
}

// dense (reference layout: x fastest, idx = x + y*n + zl*n*n) <-> colour-split device field
template <typename T, int TO_DEVICE>
__global__ void k_repack(T* __restrict__ split, mg_geom3d g, T* __restrict__ dense, int zl_lo)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int zl = zl_lo + blockIdx.z;
    if (x >= g.n || y >= g.n) return;
    const long long d = (long long)(zl - zl_lo) * g.n * g.n + (long long)y * g.n + x;
    if (TO_DEVICE) split[off3(g, x, y, zl)] = dense[d];
    else dense[d] = split[off3(g, x, y, zl)];
}

inline int launch_ok() { return cudaPeekAtLastError() == cudaSuccess ? 1 : -1; }

inline dim3 block2d(int nx) { int bx = nx >= 128 ? 128 : (nx >= 64 ? 64 : 32); return dim3(bx, 256 / bx, 1); }

// launch geometry of the row-of-half-indices kernels (relax, interpolate): `cols` threads per row
inline void half_row_launch(int cols, int n, int nz, dim3& block, dim3& grid)
{
    int bx = 32;
    while (bx < 128 && bx < cols) bx <<= 1;
    int by = 256 / bx;
    if (by > n - 2) by = n - 2;
    if (by < 1) by = 1;
    block = dim3(bx, by, 1);
    grid = dim3((cols + bx - 1) / bx, (n - 2 + by - 1) / by, nz);
}

template <typename T>
int relax_colour_t(cudaStream_t s, T* v, const T* f, mg_geom3d g, mg_coef3d c, int colour, int zl_lo, int nplanes, int zl_step)
{
    if (nplanes <= 0 || g.n < 3) return 0;
    dim3 block, grid;
    half_row_launch((g.n - 1) / 2, g.n, nplanes, block, grid);
    if (c.fast_den) k_relax_colour<T, true><<<grid, block, 0, s>>>(v, f, g, narrow<T>(c), colour, zl_lo, zl_step);
    else k_relax_colour<T, false><<<grid, block, 0, s>>>(v, f, g, narrow<T>(c), colour, zl_lo, zl_step);
    return launch_ok();
}

template <typename T>
int jacobi_colour_t(cudaStream_t s, T* dst, const T* own, const T* oth, const T* f, mg_geom3d g, mg_coef3d c, double omega, int colour,
                    int zl_lo, int zl_hi)
{
    if (zl_hi <= zl_lo || g.n < 3) return 0;
    const int cols = (g.n + 1) / 2;
    int bx = 32;
    while (bx < 128 && bx < cols) bx <<= 1;
    dim3 block(bx, 256 / bx, 1), grid((cols + bx - 1) / bx, (g.n + block.y - 1) / block.y, zl_hi - zl_lo);
    if (c.fast_den) k_jacobi_colour<T, true><<<grid, block, 0, s>>>(dst, own, oth, f, g, narrow<T>(c), (T)omega, colour, zl_lo);
    else k_jacobi_colour<T, false><<<grid, block, 0, s>>>(dst, own, oth, f, g, narrow<T>(c), (T)omega, colour, zl_lo);
    return launch_ok();
}

template <typename T>
int residual_t(cudaStream_t s, const T* v, const T* f, T* r, mg_geom3d g, mg_coef3d c, int corrected, int zl_lo, int zl_hi)
{
    if (zl_hi <= zl_lo) return 0;
    dim3 block = block2d(g.n), grid((g.n + block.x - 1) / block.x, (g.n + block.y - 1) / block.y, zl_hi - zl_lo);
    if (c.fast_h) k_residual<T, true><<<grid, block, 0, s>>>(v, f, r, g, narrow<T>(c), corrected, zl_lo);
    else k_residual<T, false><<<grid, block, 0, s>>>(v, f, r, g, narrow<T>(c), corrected, zl_lo);
    return launch_ok();
}

template <typename T>
int residual_norm_t(cudaStream_t s, const T* v, const T* f, mg_geom3d g, mg_coef3d c, int corrected, int zl_lo, int zl_hi,
                    double* scratch, double* out2)
{
    const int nb = MGK_NORM_BLOCKS;
    if (c.fast_h) k_residual_norm<T, true><<<nb, 256, 0, s>>>(v, f, g, narrow<T>(c), corrected, zl_lo, zl_hi, scratch);
    else k_residual_norm<T, false><<<nb, 256, 0, s>>>(v, f, g, narrow<T>(c), corrected, zl_lo, zl_hi, scratch);
    k_norm_final<<<1, 256, 0, s>>>(scratch, nb, out2);
    return launch_ok() < 0 ? -1 : 2;
}

template <typename T>
int residual_restrict_t(cudaStream_t s, const T* v, const T* f, mg_geom3d gf, mg_coef3d c, int corrected, T* cf, T* cv,
                        mg_geom3d gc, int czl_lo, int czl_hi)
{
    if (czl_hi <= czl_lo) return 0;
    constexpr int CX = 16, CY = 8, CZ = 4;
    dim3 grid((gc.n + CX - 1) / CX, (gc.n + CY - 1) / CY, (czl_hi - czl_lo + CZ - 1) / CZ);
    if (c.fast_h)
        k_residual_restrict<T, true, CX, CY, CZ><<<grid, 256, 0, s>>>(v, f, gf, narrow<T>(c), corrected, cf, cv, gc, czl_lo, czl_hi);
    else
        k_residual_restrict<T, false, CX, CY, CZ><<<grid, 256, 0, s>>>(v, f, gf, narrow<T>(c), corrected, cf, cv, gc, czl_lo, czl_hi);
    return launch_ok();
}

}  // namespace

#define DISPATCH(dtype, call_f32, call_f64) ((dtype) == 0 ? (call_f32) : (call_f64))

extern "C" {

int mgk3d_relax_colour(cudaStream_t s, int dtype, void* v, const void* f, mg_geom3d g, mg_coef3d c, int colour,
                       int zl_lo, int zl_hi)
{
    return DISPATCH(dtype, relax_colour_t<float>(s, (float*)v, (const float*)f, g, c, colour, zl_lo, zl_hi - zl_lo, 1),
                    relax_colour_t<double>(s, (double*)v, (const double*)f, g, c, colour, zl_lo, zl_hi - zl_lo, 1));
}

/* {sum, max} of nparts partial pairs (part[0..nparts) sums, part[nparts..2 nparts) maxima) into out2 */
int mgk_norm_final(cudaStream_t s, const double* part, int nparts, double* out2)
{
    k_norm_final<<<1, 256, 0, s>>>(part, nparts, out2);
    return launch_ok();
}

/* weighted-Jacobi update of one colour array on local planes [zl_lo, zl_hi): see k_jacobi_colour */
int mgk3d_jacobi_colour(cudaStream_t s, int dtype, void* dst, const void* own, const void* oth, const void* f, mg_geom3d g,
                        mg_coef3d c, double omega, int colour, int zl_lo, int zl_hi)
{
    return DISPATCH(dtype,
                    jacobi_colour_t<float>(s, (float*)dst, (const float*)own, (const float*)oth, (const float*)f, g, c, omega, colour, zl_lo, zl_hi),
                    jacobi_colour_t<double>(s, (double*)dst, (const double*)own, (const double*)oth, (const double*)f, g, c, omega, colour, zl_lo, zl_hi));
}

/* the same half-sweep on the two planes zl_a and zl_b only (the boundary planes of a slab), one launch */
int mgk3d_relax_colour_pair(cudaStream_t s, int dtype, void* v, const void* f, mg_geom3d g, mg_coef3d c, int colour,
                            int zl_a, int zl_b)
{
    if (zl_b <= zl_a) return -1;
    return DISPATCH(dtype, relax_colour_t<float>(s, (float*)v, (const float*)f, g, c, colour, zl_a, 2, zl_b - zl_a),
                    relax_colour_t<double>(s, (double*)v, (const double*)f, g, c, colour, zl_a, 2, zl_b - zl_a));
}

int mgk3d_residual(cudaStream_t s, int dtype, const void* v, const void* f, void* r, mg_geom3d g, mg_coef3d c,
                   int corrected, int zl_lo, int zl_hi)
{
    return DISPATCH(dtype, residual_t<float>(s, (const float*)v, (const float*)f, (float*)r, g, c, corrected, zl_lo, zl_hi),
                    residual_t<double>(s, (const double*)v, (const double*)f, (double*)r, g, c, corrected, zl_lo, zl_hi));
}

int mgk3d_residual_norm(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom3d g, mg_coef3d c,
                        int corrected, int zl_lo, int zl_hi, double* scratch, double* out2)
{
    return DISPATCH(dtype, residual_norm_t<float>(s, (const float*)v, (const float*)f, g, c, corrected, zl_lo, zl_hi, scratch, out2),
                    residual_norm_t<double>(s, (const double*)v, (const double*)f, g, c, corrected, zl_lo, zl_hi, scratch, out2));
}

int mgk3d_restrict(cudaStream_t s, int dtype, const void* fine, mg_geom3d gf, void* coarse, mg_geom3d gc, int czl_lo,
                   int czl_hi)
{
    if (czl_hi <= czl_lo) return 0;
    dim3 block = block2d(gc.n), grid((gc.n + block.x - 1) / block.x, (gc.n + block.y - 1) / block.y, czl_hi - czl_lo);
    if (dtype == 0)
        k_restrict<float><<<grid, block, 0, s>>>((const float*)fine, gf, (float*)coarse, gc, czl_lo);
    else
        k_restrict<double><<<grid, block, 0, s>>>((const double*)fine, gf, (double*)coarse, gc, czl_lo);
    return launch_ok();
}

int mgk3d_residual_restrict(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom3d gf, mg_coef3d c,
                            int corrected, void* coarse_f, void* coarse_v, mg_geom3d gc, int czl_lo, int czl_hi)
{
    return DISPATCH(dtype,
                    residual_restrict_t<float>(s, (const float*)v, (const float*)f, gf, c, corrected, (float*)coarse_f, (float*)coarse_v, gc, czl_lo, czl_hi),
                    residual_restrict_t<double>(s, (const double*)v, (const double*)f, gf, c, corrected, (double*)coarse_f, (double*)coarse_v, gc, czl_lo, czl_hi));
}

int mgk3d_interpolate(cudaStream_t s, int dtype, void* fine, mg_geom3d gf, const void* coarse, mg_geom3d gc, int add,
                      int colour_mask, int zl_lo, int zl_hi, const unsigned int* cond)
{
    if (zl_hi <= zl_lo || gf.n < 3) return 0;
    const int cells = gc.n - 1;  // coarse cells per axis: cell c covers fine 2c, 2c+1
    // coarse cells (global z) touching the fine local planes [zl_lo, zl_hi)
    const int cz_first = (gf.z0 + zl_lo) >> 1, cz_last_raw = (gf.z0 + zl_hi - 1) >> 1;
    const int cz_last = cz_last_raw > gc.n - 2 ? gc.n - 2 : cz_last_raw;
    if (cz_last < cz_first) return 0;
    int bx = 32;
    while (bx < 128 && bx < cells) bx <<= 1;
    int by = 256 / bx;
    if (by > cells) by = cells;
    const int ncz = cz_last - cz_first + 1;
    int kchunk = cond ? 64 : 8;  // a conditional launch almost always exits at once: few, long CTAs
    while (kchunk > 1 && (long long)((cells + bx - 1) / bx) * ((cells + by - 1) / by) * ((ncz + kchunk - 1) / kchunk) < 148 * 8) kchunk /= 2;
    dim3 block(bx, by, 1), grid((cells + bx - 1) / bx, (cells + by - 1) / by, (ncz + kchunk - 1) / kchunk);
    if (dtype == 0)
        if (colour_mask == 2) k_interp_octet<float, 2><<<grid, block, 0, s>>>((float*)fine, gf, (const float*)coarse, gc, add, zl_lo, zl_hi, cz_first, cz_last, kchunk, cond);
        else k_interp_octet<float, 3><<<grid, block, 0, s>>>((float*)fine, gf, (const float*)coarse, gc, add, zl_lo, zl_hi, cz_first, cz_last, kchunk, cond);
    else
        if (colour_mask == 2) k_interp_octet<double, 2><<<grid, block, 0, s>>>((double*)fine, gf, (const double*)coarse, gc, add, zl_lo, zl_hi, cz_first, cz_last, kchunk, cond);
        else k_interp_octet<double, 3><<<grid, block, 0, s>>>((double*)fine, gf, (const double*)coarse, gc, add, zl_lo, zl_hi, cz_first, cz_last, kchunk, cond);
    return launch_ok();
}

int mgk3d_set(cudaStream_t s, int dtype, void* a, mg_geom3d g, double value, int modify_boundaries, int zl_lo,
              int zl_hi)
{
    if (zl_hi <= zl_lo) return 0;
    dim3 block = block2d(g.n), grid((g.n + block.x - 1) / block.x, (g.n + block.y - 1) / block.y, zl_hi - zl_lo);
    if (dtype == 0)
        k_set<float><<<grid, block, 0, s>>>((float*)a, g, (float)value, modify_boundaries, zl_lo, 0, 0);
    else
        k_set<double><<<grid, block, 0, s>>>((double*)a, g, value, modify_boundaries, zl_lo, 0, 0);
    return launch_ok();
}

/* every stored plane EXCEPT [own_lo, own_hi): the ghost planes of a slab */
int mgk3d_set_ghosts(cudaStream_t s, int dtype, void* a, mg_geom3d g, double value, int own_lo, int own_hi)
{
    const int nz = g.nzl - (own_hi - own_lo);
    if (nz <= 0) return 0;
    dim3 block = block2d(g.n), grid((g.n + block.x - 1) / block.x, (g.n + block.y - 1) / block.y, nz);
    if (dtype == 0)
        k_set<float><<<grid, block, 0, s>>>((float*)a, g, (float)value, 1, 0, own_lo, own_hi);
    else
        k_set<double><<<grid, block, 0, s>>>((double*)a, g, value, 1, 0, own_lo, own_hi);
    return launch_ok();
}

int mgk3d_init_f(cudaStream_t s, int dtype, void* f, mg_geom3d g, const double* sx, const double* sy,
                 const double* sz, int zl_lo, int zl_hi)
{
    if (zl_hi <= zl_lo) return 0;
    dim3 block = block2d(g.n), grid((g.n + block.x - 1) / block.x, (g.n + block.y - 1) / block.y, zl_hi - zl_lo);
    if (dtype == 0)
        k_init_f<float><<<grid, block, 0, s>>>((float*)f, g, sx, sy, sz, zl_lo);
    else
        k_init_f<double><<<grid, block, 0, s>>>((double*)f, g, sx, sy, sz, zl_lo);
    return launch_ok();
}

int mgk3d_repack(cudaStream_t s, int dtype, void* split, mg_geom3d g, void* dense, int to_device, int zl_lo, int zl_hi)
{
    if (zl_hi <= zl_lo) return 0;
    dim3 block = block2d(g.n), grid((g.n + block.x - 1) / block.x, (g.n + block.y - 1) / block.y, zl_hi - zl_lo);
    if (dtype == 0) {
        if (to_device) k_repack<float, 1><<<grid, block, 0, s>>>((float*)split, g, (float*)dense, zl_lo);
        else k_repack<float, 0><<<grid, block, 0, s>>>((float*)split, g, (float*)dense, zl_lo);
    } else {
        if (to_device) k_repack<double, 1><<<grid, block, 0, s>>>((double*)split, g, (double*)dense, zl_lo);
        else k_repack<double, 0><<<grid, block, 0, s>>>((double*)split, g, (double*)dense, zl_lo);
    }
    return launch_ok();
}

}  // extern "C"

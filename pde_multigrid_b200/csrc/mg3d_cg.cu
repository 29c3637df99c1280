// mg3d_cg.cu -- the vector kernels of the multigrid-preconditioned conjugate-gradient solve (mg3d_pcg / mg3b_pcg,
// DESIGN.md §6b), written once for the colour-split layout the cubic and the box engine share (mg_launch.h, mg3d_box.h).
//
// One PCG iteration outside its V-cycle is three passes over the level:
//   dots:  rho = z.r, sigma = z.d                                          (reads z, r, d)
//   dir:   p' = z + beta*p, pi = p'.(Laplacian p'), p' at the six
//          neighbours recomputed on the fly                                (reads z, p; writes p')
//   upd:   x' = x + alpha*p', r' = b - Laplacian x' (x' at the neighbours
//          recomputed on the fly), d = r' - r, f = r', sum r'^2, max|r'|  (reads x, p', b, r; writes x', d, r')
// The stencil passes read their input at the neighbours while other blocks write their output, so both work out of
// place (p and x ping-pong between two buffers).  Every field value goes through the non-contracting helpers of
// mg_exact.cuh: r' is CalculateResidual(x') of the reference bit for bit (sign-corrected form, N3/MultiGrid3D.cpp:723).
// The three dot products that steer the iteration (rho, sigma, pi) are accumulated in double-double: every product is
// split exactly into two doubles (TwoProd through an FMA), and every sum carries its rounding error (TwoSum).  Their
// value is then the correctly rounded dot product of the stored vectors, whatever the order of the terms (the error of
// the double-double sum is ~n*2^-106 of the sum of |terms|, far below half an ulp of the result), so alpha and beta do not
// depend on the grid of blocks and equal those of any correctly rounded restatement (tests/pcg_mirror.py).  The norm
// partials are plain fp64 like the families' norm passes.  Every block writes one partial, and one block adds the partials
// in a fixed order: no atomics, so every launch of the same shapes gives the same bits.  alpha and beta are read from
// device memory.
//
// Thread layout: one warp per half-row (colour, plane, row), lanes over the half-index i (x = 2i + q); a fixed grid of
// MGK_PCG_BLOCKS blocks (two per SM) strides over the rows.  The rows in flight then span about one plane, and with the
// planes on either side the stencil inputs stay in L2 until every point that needs them has read them (at 1025^3 fp64,
// about 3 planes of 8.6 MB per field); each lane keeps four points in flight to cover the latency.
#include <stdint.h>

#include "mg3d_device.cuh"

using namespace mgx;
using namespace mg3;

#ifdef MG_DEBUG_BOUNDS
#define CG_CHK_SITE(g, i, y, zl) MG_CHK((i) >= 0 && (i) < (g).hp && (y) >= 0 && (y) < (g).ny && (zl) >= 0 && (zl) < (g).nzl)
#else
#define CG_CHK_SITE(g, i, y, zl) ((void)0)
#endif

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

// the half-row a warp works on: colour array `col`, local plane zl, row y; q = x & 1 of its points
struct Row {
    int col, zl, y, z, q;
    long long base;  // element offset of (i = 0, y, zl) inside one colour array
    bool bnd;        // the row lies on a face of the box (y or z on the boundary): every point is a Dirichlet point
};

// rows in the order (plane, row, colour): both colours of a row are worked on together, so the values a half-row reads as
// stencil neighbours are the other colour's half-row of the same and the adjacent rows and planes, which the blocks
// read at about the same time
__device__ __forceinline__ Row row_of(const mg_geom3cg& g, long long row, int zl_lo)
{
    Row r;
    r.col = (int)(row & 1);
    const long long yz = row >> 1;
    const int dz = (int)(yz / g.ny);
    r.zl = zl_lo + dz;
    r.y = (int)(yz - (long long)dz * g.ny);
    r.z = g.z0 + r.zl;
    r.q = (r.col + r.y + r.z) & 1;
    r.base = (long long)r.zl * g.plane + (long long)r.y * g.hp;
    r.bnd = r.y == 0 || r.y == g.ny - 1 || r.z == 0 || r.z == g.nz - 1;
    return r;
}

// the six neighbours of interior point (i, row) of colour r.col read from the OTHER colour array `o` (already offset
// to the row): O/E = x-1/x+1, N/S = y-1/y+1, D/U = z-1/z+1 (mg3d_kernels.cu)
#define CG_NB(o, i, q, g)                                                                                               \
    MG_CHK((i) + (q) - 1 >= 0 && (i) + (q) < (g).hp);                                                                   \
    const long long o_O = (i) + (q) - 1, o_E = (i) + (q), o_N = (i) - (g).hp, o_S = (i) + (g).hp, o_D = (i) - (g).plane, \
                    o_U = (i) + (g).plane

// ---- double-double accumulation (Dekker 1971, Knuth TwoSum), written with the non-contracting intrinsics ----
// (h, l) += a*b, the product split exactly into p + e
__device__ __forceinline__ void dd_fma(double& h, double& l, double a, double b)
{
    const double p = __dmul_rn(a, b), e = __fma_rn(a, b, -p);
    const double s = __dadd_rn(h, p), v = __dsub_rn(s, h);
    const double t = __dadd_rn(__dsub_rn(h, __dsub_rn(s, v)), __dsub_rn(p, v));
    h = s;
    l = __dadd_rn(l, __dadd_rn(t, e));
}

// (h, l) += (bh, bl), renormalised so that h = RN(h + l)
__device__ __forceinline__ void dd_add(double& h, double& l, double bh, double bl)
{
    const double s = __dadd_rn(h, bh), v = __dsub_rn(s, h);
    const double t = __dadd_rn(__dsub_rn(h, __dsub_rn(s, v)), __dsub_rn(bh, v));
    const double e = __dadd_rn(t, __dadd_rn(l, bl));
    h = __dadd_rn(s, e);
    l = __dsub_rn(e, __dsub_rn(h, s));
}

// two double-double values per thread summed over the block in a fixed order; valid in thread 0.  sh: 128 doubles
__device__ __forceinline__ void block_sum_dd2(double& ah, double& al, double& bh, double& bl, double* sh)
{
    for (int o = 16; o > 0; o >>= 1) {
        const double xh = __shfl_xor_sync(0xffffffffu, ah, o), xl = __shfl_xor_sync(0xffffffffu, al, o);
        const double yh = __shfl_xor_sync(0xffffffffu, bh, o), yl = __shfl_xor_sync(0xffffffffu, bl, o);
        dd_add(ah, al, xh, xl);
        dd_add(bh, bl, yh, yl);
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    if (l == 0) { sh[w] = ah; sh[32 + w] = al; sh[64 + w] = bh; sh[96 + w] = bl; }
    __syncthreads();
    if (w == 0) {
        ah = (l < nw) ? sh[l] : 0.0;
        al = (l < nw) ? sh[32 + l] : 0.0;
        bh = (l < nw) ? sh[64 + l] : 0.0;
        bl = (l < nw) ? sh[96 + l] : 0.0;
        for (int o = 16; o > 0; o >>= 1) {
            const double xh = __shfl_xor_sync(0xffffffffu, ah, o), xl = __shfl_xor_sync(0xffffffffu, al, o);
            const double yh = __shfl_xor_sync(0xffffffffu, bh, o), yl = __shfl_xor_sync(0xffffffffu, bl, o);
            dd_add(ah, al, xh, xl);
            dd_add(bh, bl, yh, yl);
        }
    }
}

// the partials of the dot passes: {a hi, a lo, b hi, b lo} of every block, MGK_PCG_BLOCKS each
__device__ __forceinline__ void store_dd2(double* part, double ah, double al, double bh, double bl)
{
    if (threadIdx.x == 0) {
        part[blockIdx.x] = ah;
        part[gridDim.x + blockIdx.x] = al;
        part[2 * gridDim.x + blockIdx.x] = bh;
        part[3 * gridDim.x + blockIdx.x] = bl;
    }
}

// rho = z.r and sigma = z.d over the stored points of local planes [zl_lo, zl_hi) (boundary values of z and r are 0)
template <typename T>
__global__ void __launch_bounds__(kThreads)
k_pcg_dots(const T* __restrict__ zv, const T* __restrict__ r, const T* __restrict__ d, mg_geom3cg g, int zl_lo, int zl_hi,
           double* __restrict__ part)
{
    __shared__ double sh[128];
    double rho = 0.0, rho_l = 0.0, sig = 0.0, sig_l = 0.0;
    const int nzr = zl_hi - zl_lo;
    const long long rows = 2LL * nzr * g.ny;
    const int lane = threadIdx.x & 31;
    for (long long row = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5); row < rows; row += (long long)gridDim.x * kWarps) {
        const Row R = row_of(g, row, zl_lo);
        const long long own = (long long)R.col * g.cstride + R.base;
#pragma unroll 4
        for (int i = lane; 2 * i + R.q < g.nx; i += 32) {
            CG_CHK_SITE(g, i, R.y, R.zl);
            const double zz = (double)zv[own + i];
            dd_fma(rho, rho_l, zz, (double)r[own + i]);
            dd_fma(sig, sig_l, zz, (double)d[own + i]);
        }
    }
    block_sum_dd2(rho, rho_l, sig, sig_l, sh);
    store_dd2(part, rho, rho_l, sig, sig_l);
}

// p_out = z + beta*p_in everywhere; pi = sum over the interior of p_out * (Laplacian p_out), the Laplacian taken as
// -(CalculateResidual of p_out with f = 0), i.e. the residual expression's own grouping
template <typename T, bool FAST>
__global__ void __launch_bounds__(kThreads)
k_pcg_dir(const T* __restrict__ zv, const T* __restrict__ p_in, T* __restrict__ p_out, mg_geom3cg g, Coef3<T> c,
          const double* __restrict__ sc, int zl_lo, int zl_hi, double* __restrict__ part)
{
    __shared__ double sh[128];
    const T beta = (T)sc[MGK_PCG_BETA];
    double pi = 0.0, pi_l = 0.0, zero = 0.0, zero_l = 0.0;
    const int nzr = zl_hi - zl_lo;
    const long long rows = 2LL * nzr * g.ny;
    const int lane = threadIdx.x & 31;
    for (long long row = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5); row < rows; row += (long long)gridDim.x * kWarps) {
        const Row R = row_of(g, row, zl_lo);
        const long long own = (long long)R.col * g.cstride + R.base, oth = (long long)(R.col ^ 1) * g.cstride + R.base;
#pragma unroll 4
        for (int i = lane; 2 * i + R.q < g.nx; i += 32) {
            CG_CHK_SITE(g, i, R.y, R.zl);
            const int x = 2 * i + R.q;
            const T pc = add(zv[own + i], mul(beta, p_in[own + i]));
            p_out[own + i] = pc;
            if (R.bnd || x == 0 || x == g.nx - 1) continue;
            CG_NB(oth, i, R.q, g);
            const T* zo = zv + oth;
            const T* po = p_in + oth;
            const T pO = add(zo[o_O], mul(beta, po[o_O])), pE = add(zo[o_E], mul(beta, po[o_E]));
            const T pN = add(zo[o_N], mul(beta, po[o_N])), pS = add(zo[o_S], mul(beta, po[o_S]));
            const T pD = add(zo[o_D], mul(beta, po[o_D])), pU = add(zo[o_U], mul(beta, po[o_U]));
            const T q = -residual_point<T, FAST>(pO, pE, pN, pS, pD, pU, pc, T(0), c, 1);
            dd_fma(pi, pi_l, (double)pc, (double)q);
        }
    }
    block_sum_dd2(pi, pi_l, zero, zero_l, sh);
    store_dd2(part, pi, pi_l, zero, zero_l);
}

// UPDATE: x_out = x_in + alpha*p, r' = b - Laplacian x_out into r (in place: a point reads only its own r), d = r' - r,
//         {sum r'^2, max |r'|} partials in the layout of mgk_norm_final.  Dirichlet points keep x, get r' = d = 0.
// !UPDATE (prologue): r = b - Laplacian x_in only, and the scalar block is marked "first iteration".
template <typename T, bool FAST, bool UPDATE>
__global__ void __launch_bounds__(kThreads)
k_pcg_upd(const T* __restrict__ x_in, const T* __restrict__ p, const T* __restrict__ b, T* __restrict__ r, T* __restrict__ x_out,
          T* __restrict__ d, mg_geom3cg g, Coef3<T> c, double* __restrict__ sc, int zl_lo, int zl_hi, double* __restrict__ part)
{
    __shared__ double sh[64];
    const T alpha = UPDATE ? (T)sc[MGK_PCG_ALPHA] : T(0);
    double s = 0.0, m = 0.0;
    const int nzr = zl_hi - zl_lo;
    const long long rows = 2LL * nzr * g.ny;
    const int lane = threadIdx.x & 31;
    for (long long row = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5); row < rows; row += (long long)gridDim.x * kWarps) {
        const Row R = row_of(g, row, zl_lo);
        const long long own = (long long)R.col * g.cstride + R.base, oth = (long long)(R.col ^ 1) * g.cstride + R.base;
#pragma unroll 4
        for (int i = lane; 2 * i + R.q < g.nx; i += 32) {
            CG_CHK_SITE(g, i, R.y, R.zl);
            const int x = 2 * i + R.q;
            const T xo = x_in[own + i];
            T xc = xo, rn = T(0);
            if (!(R.bnd || x == 0 || x == g.nx - 1)) {
                CG_NB(oth, i, R.q, g);
                const T* xq = x_in + oth;
                if (UPDATE) {
                    const T* pq = p + oth;
                    xc = add(xo, mul(alpha, p[own + i]));
                    rn = residual_point<T, FAST>(add(xq[o_O], mul(alpha, pq[o_O])), add(xq[o_E], mul(alpha, pq[o_E])),
                                                 add(xq[o_N], mul(alpha, pq[o_N])), add(xq[o_S], mul(alpha, pq[o_S])),
                                                 add(xq[o_D], mul(alpha, pq[o_D])), add(xq[o_U], mul(alpha, pq[o_U])), xc,
                                                 b[own + i], c, 1);
                } else {
                    rn = residual_point<T, FAST>(xq[o_O], xq[o_E], xq[o_N], xq[o_S], xq[o_D], xq[o_U], xo, b[own + i], c, 1);
                }
            }
            if (UPDATE) {
                x_out[own + i] = xc;
                d[own + i] = sub(rn, r[own + i]);
                const double rd = (double)rn;
                s += rd * rd;
                m = max_nan(m, fabs(rd));
            }
            r[own + i] = rn;
        }
    }
    if (!UPDATE) {
        if (blockIdx.x == 0 && threadIdx.x == 0) sc[MGK_PCG_FIRST] = 1.0;
        return;
    }
    block_sum_max(s, m, sh);
    if (threadIdx.x == 0) { part[blockIdx.x] = s; part[gridDim.x + blockIdx.x] = m; }
}

// which 0 (after k_pcg_dots): rho, sigma -> beta = sigma / rho_prev (0 on the first iteration), rho_prev = rho;
// which 1 (after k_pcg_dir): pi -> alpha = rho / pi.  The partials are double-double (store_dd2); each sum is rounded once.
__global__ void __launch_bounds__(kThreads) k_pcg_scalars(const double* __restrict__ part, int nparts, double* __restrict__ sc, int which)
{
    __shared__ double sh[128];
    double ah = 0.0, al = 0.0, bh = 0.0, bl = 0.0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        dd_add(ah, al, part[i], part[nparts + i]);
        dd_add(bh, bl, part[2 * nparts + i], part[3 * nparts + i]);
    }
    block_sum_dd2(ah, al, bh, bl, sh);
    if (threadIdx.x != 0) return;
    const double a = __dadd_rn(ah, al), b = __dadd_rn(bh, bl);
    if (which == 0) {
        const int first = sc[MGK_PCG_FIRST] != 0.0;
        sc[MGK_PCG_BETA] = first ? 0.0 : b / sc[MGK_PCG_RHO];
        sc[MGK_PCG_RHO] = a;
        sc[MGK_PCG_FIRST] = 0.0;
    } else {
        sc[MGK_PCG_PI] = a;
        sc[MGK_PCG_ALPHA] = sc[MGK_PCG_RHO] / a;
    }
}

template <typename T>
int launch_dots(cudaStream_t s, const void* z, const void* r, const void* d, mg_geom3cg g, int zl_lo, int zl_hi, double* part, double* sc)
{
    k_pcg_dots<T><<<MGK_PCG_BLOCKS, kThreads, 0, s>>>((const T*)z, (const T*)r, (const T*)d, g, zl_lo, zl_hi, part);
    k_pcg_scalars<<<1, kThreads, 0, s>>>(part, MGK_PCG_BLOCKS, sc, 0);
    return cudaPeekAtLastError() == cudaSuccess ? 2 : -1;
}

template <typename T>
int launch_dir(cudaStream_t s, const void* z, const void* p_in, void* p_out, mg_geom3cg g, mg_coef3d c, int zl_lo, int zl_hi, double* part,
               double* sc)
{
    if (c.fast_h)
        k_pcg_dir<T, true><<<MGK_PCG_BLOCKS, kThreads, 0, s>>>((const T*)z, (const T*)p_in, (T*)p_out, g, narrow<T>(c), sc, zl_lo, zl_hi, part);
    else
        k_pcg_dir<T, false><<<MGK_PCG_BLOCKS, kThreads, 0, s>>>((const T*)z, (const T*)p_in, (T*)p_out, g, narrow<T>(c), sc, zl_lo, zl_hi, part);
    k_pcg_scalars<<<1, kThreads, 0, s>>>(part, MGK_PCG_BLOCKS, sc, 1);
    return cudaPeekAtLastError() == cudaSuccess ? 2 : -1;
}

template <typename T, bool UPDATE>
int launch_upd(cudaStream_t s, const void* x_in, const void* p, const void* b, void* r, void* x_out, void* d, mg_geom3cg g, mg_coef3d c,
               double* sc, int zl_lo, int zl_hi, double* part)
{
    if (c.fast_h)
        k_pcg_upd<T, true, UPDATE><<<MGK_PCG_BLOCKS, kThreads, 0, s>>>((const T*)x_in, (const T*)p, (const T*)b, (T*)r, (T*)x_out, (T*)d,
                                                                        g, narrow<T>(c), sc, zl_lo, zl_hi, part);
    else
        k_pcg_upd<T, false, UPDATE><<<MGK_PCG_BLOCKS, kThreads, 0, s>>>((const T*)x_in, (const T*)p, (const T*)b, (T*)r, (T*)x_out, (T*)d,
                                                                         g, narrow<T>(c), sc, zl_lo, zl_hi, part);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace

extern "C" int mgk3cg_dots(cudaStream_t s, int dtype, const void* z, const void* r, const void* d, mg_geom3cg g, int zl_lo, int zl_hi,
                           double* part, double* sc)
{
    return dtype == 0 ? launch_dots<float>(s, z, r, d, g, zl_lo, zl_hi, part, sc) : launch_dots<double>(s, z, r, d, g, zl_lo, zl_hi, part, sc);
}

extern "C" int mgk3cg_dir(cudaStream_t s, int dtype, const void* z, const void* p_in, void* p_out, mg_geom3cg g, mg_coef3d c, int zl_lo,
                          int zl_hi, double* part, double* sc)
{
    return dtype == 0 ? launch_dir<float>(s, z, p_in, p_out, g, c, zl_lo, zl_hi, part, sc)
                      : launch_dir<double>(s, z, p_in, p_out, g, c, zl_lo, zl_hi, part, sc);
}

extern "C" int mgk3cg_update(cudaStream_t s, int dtype, const void* x_in, const void* p, const void* b, void* r, void* x_out, void* d,
                             mg_geom3cg g, mg_coef3d c, const double* sc, int zl_lo, int zl_hi, double* part)
{
    double* scw = const_cast<double*>(sc);
    return dtype == 0 ? launch_upd<float, true>(s, x_in, p, b, r, x_out, d, g, c, scw, zl_lo, zl_hi, part)
                      : launch_upd<double, true>(s, x_in, p, b, r, x_out, d, g, c, scw, zl_lo, zl_hi, part);
}

extern "C" int mgk3cg_residual(cudaStream_t s, int dtype, const void* x, const void* b, void* r, mg_geom3cg g, mg_coef3d c, double* sc,
                               int zl_lo, int zl_hi)
{
    return dtype == 0 ? launch_upd<float, false>(s, x, nullptr, b, r, nullptr, nullptr, g, c, sc, zl_lo, zl_hi, nullptr)
                      : launch_upd<double, false>(s, x, nullptr, b, r, nullptr, nullptr, g, c, sc, zl_lo, zl_hi, nullptr);
}

// mg2d_kernels.cu -- sm_100a kernels of the 2D Lyapunov multigrid path.
//
// Replaces the operators of the reference class MultiGrid2D (CPU: NOCUDA_TESI/PDE Lyapunov 2D/
// MultiGrid2D.cpp; GPU twin CUDA_TESI/CUDA Lyapunov 2D/MultiGrid2D.cu:243-462 -- whose smoother drops
// f, SURVEY.md App. B4; the CPU solver is the oracle).  K1, K2 and den vary per point, so this path IS
// FMA-sensitive: everything goes through the non-contracting helpers of mg_exact.cuh and true IEEE
// division.  At the benchmark size (1025^2 fp32 = 4.2 MB per field) the whole hierarchy is L2-resident;
// the kernels are latency/launch bound, not HBM bound.
#include "mg_exact.cuh"
#include "mg_launch.h"

using namespace mgx;

namespace {

template <typename T>
struct Coef2 {
    T hx, hy, xa, ya, A0, A1, A2, A3, alfa;
};

template <typename T>
Coef2<T> narrow(const mg_coef2d& c)
{
    Coef2<T> r;
    r.hx = (T)c.hx; r.hy = (T)c.hy; r.xa = (T)c.xa; r.ya = (T)c.ya;
    r.A0 = (T)c.A[0]; r.A1 = (T)c.A[1]; r.A2 = (T)c.A[2]; r.A3 = (T)c.A[3];
    r.alfa = (T)c.alfa;  // int -> real, as in `alfa*h_x*h_y`
    return r;
}

// K1 = A[0]*xj + A[1]*yi, K2 = A[2]*xj + A[3]*yi with xj = x_a + posX*h_x, yi = y_a + posY*h_y
// (N2/MultiGrid2D.cpp:230-234)
template <typename T>
__device__ __forceinline__ void k1k2(int x, int y, const Coef2<T>& c, T& K1, T& K2)
{
    const T xj = add(c.xa, mul((T)x, c.hx));
    const T yi = add(c.ya, mul((T)y, c.hy));
    K1 = add(mul(c.A0, xj), mul(c.A1, yi));
    K2 = add(mul(c.A2, xj), mul(c.A3, yi));
}

// N2/MultiGrid2D.cpp:236-241
template <typename T>
__device__ __forceinline__ T relax_point(int x, int y, T vE, T vS, T f, const Coef2<T>& c)
{
    T K1, K2;
    k1k2(x, y, c, K1, K2);
    const T den = sub(add(mul(K1, c.hy), mul(K2, c.hx)), mul(mul(c.alfa, c.hx), c.hy));
    const T num = sub(add(mul(mul(c.hy, K1), vE), mul(mul(c.hx, K2), vS)), mul(mul(f, c.hx), c.hy));
    return div(num, den);
}

// N2/MultiGrid2D.cpp:395-403
template <typename T>
__device__ __forceinline__ T residual_point(int x, int y, T vC, T vE, T vS, T f, const Coef2<T>& c)
{
    T K1, K2;
    k1k2(x, y, c, K1, K2);
    const T inner = sub(add(mul(c.hy, K1), mul(c.hx, K2)), mul(mul(c.alfa, c.hx), c.hy));
    const T num = sub(add(mul(mul(c.hy, K1), vE), mul(mul(c.hx, K2), vS)), mul(vC, inner));
    return sub(f, div(num, mul(c.hx, c.hy)));
}

// residual at fine point (x,y), zero on the boundary (N2/MultiGrid2D.cpp:389-392)
template <typename T>
__device__ __forceinline__ T residual_at(const T* __restrict__ v, const T* __restrict__ f, int x, int y, int n, int p,
                                         const Coef2<T>& c)
{
    if (x == 0 || x == n - 1 || y == 0 || y == n - 1) return T(0);
    const long long i = (long long)y * p + x;
    return residual_point<T>(x, y, v[i], v[i + 1], v[i + p], f[i], c);
}

// N2/MultiGrid2D.cpp:123: (1/16)*(NO+NE+SO+SE + 2*(O+E+N+S) + 4*C); N = y-1, S = y+1, E = x+1, O = x-1
template <typename T, typename Getter>
__device__ __forceinline__ T restrict_point(Getter R)
{
    const T C = R(0, 0), N = R(0, -1), S = R(0, 1), E = R(1, 0), O = R(-1, 0);
    const T NE = R(1, -1), NO = R(-1, -1), SE = R(1, 1), SO = R(-1, 1);
    const T corners = add(add(add(NO, NE), SO), SE);
    const T edges = mul(T(2), add(add(add(O, E), N), S));
    return mul(T(1 / 16.0f), add(add(corners, edges), mul(T(4), C)));
}

template <typename T>
__global__ void k_relax_colour(T* __restrict__ v, const T* __restrict__ f, mg_geom2d g, Coef2<T> c, int colour)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    if (y > g.n - 2) return;
    const int x = 2 * t + 2 - ((y + colour) & 1);
    if (x > g.n - 2) return;
    const long long i = (long long)y * g.pitch + x;
    v[i] = relax_point<T>(x, y, v[i + 1], v[i + g.pitch], f[i], c);
}

// Small levels (n <= 65: the whole grid fits in one CTA's shared memory): ALL ncycles sweeps in one launch.
// v lives in shared memory, colours are separated by __syncthreads(), and the per-point quantities that do not
// change between sweeps (hy*K1, hx*K2, f*hx*hy, den -- the same operations in the same order as
// N2/MultiGrid2D.cpp:230-241) stay in registers.  With the thesis parameters (nu = 500) this replaces 1000 launches
// per Relax call on 7 of the 10 levels of a 1025^2 hierarchy.
constexpr int SMALL_NT = 1024, SMALL_PPT = 4;  // (65-2)^2 = 3969 interior points <= 4 * 1024

template <typename T>
__global__ void __launch_bounds__(SMALL_NT) k_relax_small(T* __restrict__ v, const T* __restrict__ f, mg_geom2d g, Coef2<T> c, int ncycles)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T* sv = reinterpret_cast<T*>(smem_raw);
    const int n = g.n, ni = n - 2, tid = threadIdx.x;
    for (int i = tid; i < n * n; i += SMALL_NT) sv[i] = v[(long long)(i / n) * g.pitch + (i % n)];
    int pos[SMALL_PPT];
    T a[SMALL_PPT], b[SMALL_PPT], fh[SMALL_PPT], den[SMALL_PPT];
#pragma unroll
    for (int k = 0; k < SMALL_PPT; k++) {
        const int idx = tid + k * SMALL_NT;
        pos[k] = -1;
        a[k] = b[k] = fh[k] = T(0);
        den[k] = T(1);
        if (idx < ni * ni) {
            const int y = 1 + idx / ni, x = 1 + idx % ni;
            T K1, K2;
            k1k2(x, y, c, K1, K2);
            den[k] = sub(add(mul(K1, c.hy), mul(K2, c.hx)), mul(mul(c.alfa, c.hx), c.hy));
            a[k] = mul(c.hy, K1);
            b[k] = mul(c.hx, K2);
            fh[k] = mul(mul(f[(long long)y * g.pitch + x], c.hx), c.hy);
            pos[k] = (y * n + x) | (((x + y) & 1) << 30);
        }
    }
    __syncthreads();
    for (int it = 0; it < ncycles; it++)
        for (int colour = 0; colour < 2; colour++) {
#pragma unroll
            for (int k = 0; k < SMALL_PPT; k++)
                if (pos[k] >= 0 && (pos[k] >> 30) == colour) {
                    const int i = pos[k] & 0x3fffffff;
                    sv[i] = div(sub(add(mul(a[k], sv[i + 1]), mul(b[k], sv[i + n])), fh[k]), den[k]);
                }
            __syncthreads();
        }
#pragma unroll
    for (int k = 0; k < SMALL_PPT; k++)
        if (pos[k] >= 0) {
            const int i = pos[k] & 0x3fffffff;
            v[(long long)(i / n) * g.pitch + (i % n)] = sv[i];
        }
}

template <typename T>
__global__ void k_residual(const T* __restrict__ v, const T* __restrict__ f, T* __restrict__ r, mg_geom2d g, Coef2<T> c)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= g.n || y >= g.n) return;
    r[(long long)y * g.pitch + x] = residual_at<T>(v, f, x, y, g.n, g.pitch, c);
}

__device__ __forceinline__ void block_reduce_sum_max(double& s, double& m, double* sh)
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

// mode 0: sum r^2 / max|r| of the residual; mode 1: sum / max of |v - exact| over interior points
// (PrintMeanAbsoluteError, C2/Grid2D.cu:123-154: diff in T, accumulation in double)
template <typename T>
__global__ void k_reduce(const T* __restrict__ v, const T* __restrict__ f, mg_geom2d g, Coef2<T> c, int mode,
                         double* __restrict__ part)
{
    __shared__ double sh[64];
    double s = 0.0, m = 0.0;
    for (int y = 1 + blockIdx.x; y <= g.n - 2; y += gridDim.x)
        for (int x = 1 + threadIdx.x; x <= g.n - 2; x += blockDim.x) {
            const long long i = (long long)y * g.pitch + x;
            double d;
            if (mode == 0) {
                d = (double)residual_point<T>(x, y, v[i], v[i + 1], v[i + g.pitch], f[i], c);
                s += d * d;
            } else {
                const T xj = add(c.xa, mul((T)x, c.hx));
                const T yi = add(c.ya, mul((T)y, c.hy));
                const T real = add(sub(mul(mul(T(2), xj), xj), mul(mul(T(4), xj), yi)), mul(mul(T(2), yi), yi));
                d = fabs((double)sub(v[i], real));
                s += d;
            }
            m = max_nan(m, fabs(d));
        }
    block_reduce_sum_max(s, m, sh);
    if (threadIdx.x == 0) { part[blockIdx.x] = s; part[gridDim.x + blockIdx.x] = m; }
}

__global__ void k_reduce_final(const double* __restrict__ part, int nparts, double* __restrict__ out2)
{
    __shared__ double sh[64];
    double s = 0.0, m = 0.0;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) {
        s += part[i];
        m = max_nan(m, part[nparts + i]);
    }
    block_reduce_sum_max(s, m, sh);
    if (threadIdx.x == 0) { out2[0] = s; out2[1] = m; }
}

// Restrict; FUSED != 0: the fine values are residuals evaluated on the fly (never stored) and the
// coarse v is zeroed, boundary included (N2/MultiGrid2D.cpp:320-326)
template <typename T, int FUSED>
__global__ void k_restrict(const T* __restrict__ fine, const T* __restrict__ f, mg_geom2d gf, Coef2<T> c,
                           T* __restrict__ coarse, T* __restrict__ coarse_v, mg_geom2d gc)
{
    const int cx = blockIdx.x * blockDim.x + threadIdx.x;
    const int cy = blockIdx.y * blockDim.y + threadIdx.y;
    if (cx >= gc.n || cy >= gc.n) return;
    const long long ci = (long long)cy * gc.pitch + cx;
    const int fx = 2 * cx, fy = 2 * cy;
    auto R = [&](int dx, int dy) -> T {
        if (FUSED) return residual_at<T>(fine, f, fx + dx, fy + dy, gf.n, gf.pitch, c);
        return fine[(long long)(fy + dy) * gf.pitch + fx + dx];
    };
    T out;
    if (cx == 0 || cx == gc.n - 1 || cy == 0 || cy == gc.n - 1) out = R(0, 0);  // N2/MultiGrid2D.cpp:95-101
    else out = restrict_point<T>(R);
    coarse[ci] = out;
    if (FUSED) coarse_v[ci] = T(0);
}

// N2/MultiGrid2D.cpp:128-196; thread owns the fine pair (2i, 2i+1)
template <typename T>
__global__ void k_interpolate(T* __restrict__ fine, mg_geom2d gf, const T* __restrict__ coarse, mg_geom2d gc, int add_)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    if (y > gf.n - 2 || 2 * i > gf.n - 2) return;
    const int oy = y & 1;
    const T* c = coarse + (long long)(y >> 1) * gc.pitch + i;
    const int cp = gc.pitch;
    T* p = fine + (long long)y * gf.pitch + 2 * i;
    if (i >= 1) {
        const T e = oy ? mul(T(0.5f), add(c[0], c[cp])) : c[0];
        p[0] = add_ ? add(p[0], e) : e;
    }
    if (2 * i + 1 <= gf.n - 2) {
        const T e = oy ? mul(T(0.25f), add(add(add(c[0], c[1]), c[cp]), c[cp + 1])) : mul(T(0.5f), add(c[0], c[1]));
        p[1] = add_ ? add(p[1], e) : e;
    }
}

template <typename T>
__global__ void k_apply_correction(T* __restrict__ fine, const T* __restrict__ err, mg_geom2d g)
{
    const int x = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    const int y = 1 + blockIdx.y * blockDim.y + threadIdx.y;
    if (x > g.n - 2 || y > g.n - 2) return;
    const long long i = (long long)y * g.pitch + x;
    fine[i] = add(fine[i], err[i]);
}

template <typename T>
__global__ void k_set(T* __restrict__ a, mg_geom2d g, T value, int modify_boundaries)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= g.n || y >= g.n) return;
    if (!modify_boundaries && (x == 0 || x == g.n - 1 || y == 0 || y == g.n - 1)) return;
    a[(long long)y * g.pitch + x] = value;
}

// Grid2D::InitV, N2/Grid2D.cpp:50-68: boundary = 2x^2 - 4xy + 2y^2, interior 0
template <typename T>
__global__ void k_init_v(T* __restrict__ v, mg_geom2d g, Coef2<T> c)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= g.n || y >= g.n) return;
    T val = T(0);
    if (x == 0 || x == g.n - 1 || y == 0 || y == g.n - 1) {
        const T yi = add(c.ya, mul((T)y, c.hy));
        const T xj = add(c.xa, mul((T)x, c.hx));
        val = add(sub(mul(mul(T(2), xj), xj), mul(mul(T(4), xj), yi)), mul(mul(T(2), yi), yi));
    }
    v[(long long)y * g.pitch + x] = val;
}

inline int launch_ok() { return cudaPeekAtLastError() == cudaSuccess ? 1 : -1; }
inline dim3 blk(int nx) { int bx = nx >= 128 ? 128 : (nx >= 64 ? 64 : 32); return dim3(bx, 256 / bx, 1); }
inline dim3 grd(int nx, int ny, dim3 b) { return dim3((nx + b.x - 1) / b.x, (ny + b.y - 1) / b.y, 1); }
#define MG2D_REDUCE_BLOCKS 592

}  // namespace

extern "C" {

int mgk2d_relax_colour(cudaStream_t s, int dtype, void* v, const void* f, mg_geom2d g, mg_coef2d c, int colour)
{
    if (g.n < 3) return 0;
    const int halfw = (g.n - 1) / 2;
    int bx = halfw < 128 ? halfw : 128;
    int by = 256 / bx;
    if (by > g.n - 2) by = g.n - 2;
    dim3 b(bx, by, 1), gr((halfw + bx - 1) / bx, (g.n - 2 + by - 1) / by, 1);
    if (dtype == 0) k_relax_colour<float><<<gr, b, 0, s>>>((float*)v, (const float*)f, g, narrow<float>(c), colour);
    else k_relax_colour<double><<<gr, b, 0, s>>>((double*)v, (const double*)f, g, narrow<double>(c), colour);
    return launch_ok();
}

int mgk2d_relax_small(cudaStream_t s, int dtype, void* v, const void* f, mg_geom2d g, mg_coef2d c, int ncycles)
{
    if (g.n < 3 || ncycles <= 0) return 0;
    if (g.n > MGK2D_SMALL_N) return -1;
    const size_t smem = (size_t)g.n * g.n * (dtype == 0 ? 4 : 8);
    if (dtype == 0) k_relax_small<float><<<1, SMALL_NT, smem, s>>>((float*)v, (const float*)f, g, narrow<float>(c), ncycles);
    else k_relax_small<double><<<1, SMALL_NT, smem, s>>>((double*)v, (const double*)f, g, narrow<double>(c), ncycles);
    return launch_ok();
}

int mgk2d_residual(cudaStream_t s, int dtype, const void* v, const void* f, void* r, mg_geom2d g, mg_coef2d c)
{
    dim3 b = blk(g.n), gr = grd(g.n, g.n, b);
    if (dtype == 0) k_residual<float><<<gr, b, 0, s>>>((const float*)v, (const float*)f, (float*)r, g, narrow<float>(c));
    else k_residual<double><<<gr, b, 0, s>>>((const double*)v, (const double*)f, (double*)r, g, narrow<double>(c));
    return launch_ok();
}

static int reduce2d(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom2d g, mg_coef2d c, int mode,
                    double* scratch, double* out2)
{
    const int nb = MG2D_REDUCE_BLOCKS;
    if (dtype == 0) k_reduce<float><<<nb, 256, 0, s>>>((const float*)v, (const float*)f, g, narrow<float>(c), mode, scratch);
    else k_reduce<double><<<nb, 256, 0, s>>>((const double*)v, (const double*)f, g, narrow<double>(c), mode, scratch);
    k_reduce_final<<<1, 256, 0, s>>>(scratch, nb, out2);
    return launch_ok() < 0 ? -1 : 2;
}

int mgk2d_residual_norm(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom2d g, mg_coef2d c,
                        double* scratch, double* out2)
{
    return reduce2d(s, dtype, v, f, g, c, 0, scratch, out2);
}

int mgk2d_abs_error_sum(cudaStream_t s, int dtype, const void* v, mg_geom2d g, mg_coef2d c, double* scratch,
                        double* out2)
{
    return reduce2d(s, dtype, v, v, g, c, 1, scratch, out2);
}

int mgk2d_restrict(cudaStream_t s, int dtype, const void* fine, mg_geom2d gf, void* coarse, mg_geom2d gc)
{
    dim3 b = blk(gc.n), gr = grd(gc.n, gc.n, b);
    mg_coef2d c0 = {};
    if (dtype == 0) k_restrict<float, 0><<<gr, b, 0, s>>>((const float*)fine, nullptr, gf, narrow<float>(c0), (float*)coarse, nullptr, gc);
    else k_restrict<double, 0><<<gr, b, 0, s>>>((const double*)fine, nullptr, gf, narrow<double>(c0), (double*)coarse, nullptr, gc);
    return launch_ok();
}

int mgk2d_residual_restrict(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom2d gf, mg_coef2d c,
                            void* coarse_f, void* coarse_v, mg_geom2d gc)
{
    dim3 b = blk(gc.n), gr = grd(gc.n, gc.n, b);
    if (dtype == 0) k_restrict<float, 1><<<gr, b, 0, s>>>((const float*)v, (const float*)f, gf, narrow<float>(c), (float*)coarse_f, (float*)coarse_v, gc);
    else k_restrict<double, 1><<<gr, b, 0, s>>>((const double*)v, (const double*)f, gf, narrow<double>(c), (double*)coarse_f, (double*)coarse_v, gc);
    return launch_ok();
}

int mgk2d_interpolate(cudaStream_t s, int dtype, void* fine, mg_geom2d gf, const void* coarse, mg_geom2d gc, int add)
{
    if (gf.n < 3) return 0;
    const int pairs = (gf.n - 1) / 2;
    int bx = pairs < 128 ? pairs : 128;
    int by = 256 / bx;
    if (by > gf.n - 2) by = gf.n - 2;
    dim3 b(bx, by, 1), gr((pairs + bx - 1) / bx, (gf.n - 2 + by - 1) / by, 1);
    if (dtype == 0) k_interpolate<float><<<gr, b, 0, s>>>((float*)fine, gf, (const float*)coarse, gc, add);
    else k_interpolate<double><<<gr, b, 0, s>>>((double*)fine, gf, (const double*)coarse, gc, add);
    return launch_ok();
}

int mgk2d_apply_correction(cudaStream_t s, int dtype, void* fine, const void* err, mg_geom2d g)
{
    if (g.n < 3) return 0;
    dim3 b = blk(g.n), gr = grd(g.n - 2, g.n - 2, b);
    if (dtype == 0) k_apply_correction<float><<<gr, b, 0, s>>>((float*)fine, (const float*)err, g);
    else k_apply_correction<double><<<gr, b, 0, s>>>((double*)fine, (const double*)err, g);
    return launch_ok();
}

int mgk2d_set(cudaStream_t s, int dtype, void* a, mg_geom2d g, double value, int modify_boundaries)
{
    dim3 b = blk(g.n), gr = grd(g.n, g.n, b);
    if (dtype == 0) k_set<float><<<gr, b, 0, s>>>((float*)a, g, (float)value, modify_boundaries);
    else k_set<double><<<gr, b, 0, s>>>((double*)a, g, value, modify_boundaries);
    return launch_ok();
}

int mgk2d_init_v(cudaStream_t s, int dtype, void* v, mg_geom2d g, mg_coef2d c)
{
    dim3 b = blk(g.n), gr = grd(g.n, g.n, b);
    if (dtype == 0) k_init_v<float><<<gr, b, 0, s>>>((float*)v, g, narrow<float>(c));
    else k_init_v<double><<<gr, b, 0, s>>>((double*)v, g, narrow<double>(c));
    return launch_ok();
}

}  // extern "C"

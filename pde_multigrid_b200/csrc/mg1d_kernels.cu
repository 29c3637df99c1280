// mg1d_kernels.cu -- sm_100a kernels of the 1D two-point BVP multigrid path (u' - u/(e^x+1) = e^x).
//
// Replaces the operators of the reference class MultiGrid1D (CPU: NOCUDA_TESI/EQUAZIONE 1D/
// MultiGrid1D.cpp; GPU twin CUDA_TESI/CUDA 1D/MultiGrid1D.cu:206-319, whose one-launch red/black sweep
// races across blocks, SURVEY.md App. B3).
//
// The whole hierarchy is tiny (2 055 points at n = 1025), so the design is the opposite of the 3D
// path: ONE persistent CTA walks whole V-cycles / FMG solves in a single launch; colours are
// separated by __syncthreads(), levels never leave L1.  The thesis parameters (nu = 1000 sweeps per
// Relax) would otherwise cost two launches per sweep.  The transcendental exp(x_j) is not evaluated
// on the device: the host driver tabulates e1[j] = exp(x_j)+1 and d[j] = exp(x_j)+1+h with the same
// libm the reference calls (N1/MultiGrid1D.cpp:101), which keeps the path bit-exact.
#include "mg_exact.cuh"
#include "mg_launch.h"

using namespace mgx;

namespace {

template <typename T>
struct Lvl {
    T* v;
    T* f;
    const T* e1;
    const T* d;
    T h;
    int n;
};

template <typename T>
__device__ __forceinline__ Lvl<T> level_of(T* arena, const mg_hier1d& H, int l)
{
    Lvl<T> L;
    L.v = arena + H.off_v[l];
    L.f = arena + H.off_f[l];
    L.e1 = arena + H.off_e[l];
    L.d = arena + H.off_d[l];
    L.h = (T)H.h[l];
    L.n = H.n[l];
    return L;
}

// Relax: ncycles x (even points, then odd points), N1/MultiGrid1D.cpp:79-118
//   v[j] = (v[j+1]*(exp(xj)+1) - f[j]*h*(exp(xj)+1)) / (exp(xj)+1+h)
template <typename T>
__device__ void relax1d(const Lvl<T>& L, int ncycles)
{
    for (int k = 0; k < ncycles; k++)
        for (int colour = 0; colour < 2; colour++) {
            for (int j = 2 - colour + 2 * threadIdx.x; j <= L.n - 2; j += 2 * blockDim.x) {  // colour 0: even j >= 2
                const T e1 = L.e1[j];
                L.v[j] = div(sub(mul(L.v[j + 1], e1), mul(mul(L.f[j], L.h), e1)), L.d[j]);
            }
            __syncthreads();
        }
}

// CalculateResidual, N1/MultiGrid1D.cpp:190-214 (REF_COMPAT: minus v/(e^x+1); CORRECTED: plus)
template <typename T>
__device__ __forceinline__ T residual1d_at(const Lvl<T>& L, int j, int corrected)
{
    if (j == 0 || j == L.n - 1) return T(0);
    const T a = sub(L.f[j], div(sub(L.v[j + 1], L.v[j]), L.h));
    const T b = div(L.v[j], L.e1[j]);
    return corrected ? add(a, b) : sub(a, b);
}

// Restrict(CalculateResidual(fine)) -> coarse f; coarse v = 0 incl. boundary (N1/MultiGrid1D.cpp:156-162);
// restriction (1/4)*(O + 2*C + E), end points by injection (N1/MultiGrid1D.cpp:34-58)
template <typename T>
__device__ void residual_restrict1d(const Lvl<T>& F, const Lvl<T>& C, int corrected)
{
    for (int c = threadIdx.x; c < C.n; c += blockDim.x) {
        T out;
        if (c == 0 || c == C.n - 1) out = residual1d_at(F, 2 * c, corrected);
        else {
            const T O = residual1d_at(F, 2 * c - 1, corrected), Cc = residual1d_at(F, 2 * c, corrected),
                    E = residual1d_at(F, 2 * c + 1, corrected);
            out = mul(T(0.25f), add(add(O, mul(T(2), Cc)), E));
        }
        C.f[c] = out;
        C.v[c] = T(0);
    }
    __syncthreads();
}

template <typename T>
__device__ void restrict_f1d(const Lvl<T>& F, const Lvl<T>& C)
{
    for (int c = threadIdx.x; c < C.n; c += blockDim.x) {
        if (c == 0 || c == C.n - 1) C.f[c] = F.f[2 * c];
        else C.f[c] = mul(T(0.25f), add(add(F.f[2 * c - 1], mul(T(2), F.f[2 * c])), F.f[2 * c + 1]));
    }
    __syncthreads();
}

// Interpolate (N1/MultiGrid1D.cpp:60-77) into v (add == 0) or Interpolate + ApplyCorrection (add != 0)
template <typename T>
__device__ void interpolate1d(const Lvl<T>& F, const Lvl<T>& C, int add_)
{
    for (int j = 1 + threadIdx.x; j <= F.n - 2; j += blockDim.x) {
        const int c = j >> 1;
        const T e = (j & 1) ? mul(T(0.5f), add(C.v[c], C.v[c + 1])) : C.v[c];
        F.v[j] = add_ ? add(F.v[j], e) : e;
    }
    __syncthreads();
}

template <typename T>
__device__ void vcycle1d(T* arena, const mg_hier1d& H, int level, int v1, int v2, int corrected)
{
    const int last = H.nlevels - 1;
    for (int k = level; k < last; k++) {  // N1/MultiGrid1D.cpp:150-175, recursion unrolled
        relax1d(level_of(arena, H, k), v1);
        residual_restrict1d(level_of(arena, H, k), level_of(arena, H, k + 1), corrected);
    }
    relax1d(level_of(arena, H, last), v1);
    relax1d(level_of(arena, H, last), v2);
    for (int k = last - 1; k >= level; k--) {
        interpolate1d(level_of(arena, H, k), level_of(arena, H, k + 1), 1);
        relax1d(level_of(arena, H, k), v2);
    }
}

enum { OP_RELAX = 0, OP_RESIDUAL = 1, OP_NORM = 2, OP_RESIDUAL_RESTRICT = 3, OP_VCYCLE = 4, OP_FMG = 5, OP_RESTRICT_F = 6,
       OP_INTERP = 7, OP_INTERP_ADD = 8 };

// One persistent CTA executes a whole operator / V-cycle / FMG solve.
template <typename T>
__global__ void __launch_bounds__(1024) k_ops1d(T* arena, mg_hier1d H, int op, int level, int a0, int a1, int a2,
                                                int corrected, T* r_out, double* out2)
{
    __shared__ double sh[64];
    const int last = H.nlevels - 1;
    switch (op) {
        case OP_RELAX:
            relax1d(level_of(arena, H, level), a0);
            break;
        case OP_RESIDUAL: {
            const Lvl<T> L = level_of(arena, H, level);
            for (int j = threadIdx.x; j < L.n; j += blockDim.x) r_out[j] = residual1d_at(L, j, corrected);
            break;
        }
        case OP_NORM: {
            const Lvl<T> L = level_of(arena, H, level);
            double s = 0.0, m = 0.0;
            for (int j = threadIdx.x; j < L.n; j += blockDim.x) {
                const double r = (double)residual1d_at(L, j, corrected);
                s += r * r;
                m = max_nan(m, fabs(r));
            }
            for (int o = 16; o > 0; o >>= 1) {
                s += __shfl_xor_sync(0xffffffffu, s, o);
                m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
            }
            const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
            if (l == 0) { sh[w] = s; sh[32 + w] = m; }
            __syncthreads();
            if (w == 0) {
                s = l < nw ? sh[l] : 0.0;
                m = l < nw ? sh[32 + l] : 0.0;
                for (int o = 16; o > 0; o >>= 1) {
                    s += __shfl_xor_sync(0xffffffffu, s, o);
                    m = max_nan(m, __shfl_xor_sync(0xffffffffu, m, o));
                }
                if (l == 0) { out2[0] = s; out2[1] = m; }
            }
            break;
        }
        case OP_RESIDUAL_RESTRICT:
            residual_restrict1d(level_of(arena, H, level), level_of(arena, H, level + 1), corrected);
            break;
        case OP_RESTRICT_F:
            restrict_f1d(level_of(arena, H, level), level_of(arena, H, level + 1));
            break;
        case OP_INTERP:
        case OP_INTERP_ADD:
            interpolate1d(level_of(arena, H, level), level_of(arena, H, level + 1), op == OP_INTERP_ADD);
            break;
        case OP_VCYCLE:
            for (int i = 0; i < a0; i++) vcycle1d(arena, H, level, a1, a2, corrected);
            break;
        case OP_FMG: {  // N1/MultiGrid1D.cpp:132-148, recursion unrolled: restrict f down, then climb
            for (int k = level; k < last; k++) restrict_f1d(level_of(arena, H, k), level_of(arena, H, k + 1));
            {
                const Lvl<T> L = level_of(arena, H, last);
                for (int j = 1 + threadIdx.x; j <= L.n - 2; j += blockDim.x) L.v[j] = T(0);  // setToValue(.., 0, false)
                __syncthreads();
            }
            for (int k = last; k >= level; k--) {
                if (k < last) interpolate1d(level_of(arena, H, k), level_of(arena, H, k + 1), 0);
                for (int i = 0; i < a0; i++) vcycle1d(arena, H, k, a1, a2, corrected);
            }
            break;
        }
    }
}

template <typename T>
__global__ void k_restrict1(const T* __restrict__ fine, int fn, T* __restrict__ coarse, int cn)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cn) return;
    if (c == 0 || c == cn - 1) coarse[c] = fine[2 * c];
    else coarse[c] = mul(T(0.25f), add(add(fine[2 * c - 1], mul(T(2), fine[2 * c])), fine[2 * c + 1]));
}

template <typename T>
__global__ void k_interp1(T* __restrict__ fine, int fn, const T* __restrict__ coarse, int add_)
{
    const int j = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    if (j > fn - 2) return;
    const int c = j >> 1;
    const T e = (j & 1) ? mul(T(0.5f), add(coarse[c], coarse[c + 1])) : coarse[c];
    fine[j] = add_ ? add(fine[j], e) : e;
}

template <typename T>
__global__ void k_correct1(T* __restrict__ fine, const T* __restrict__ err, int n)
{
    const int j = 1 + blockIdx.x * blockDim.x + threadIdx.x;
    if (j > n - 2) return;
    fine[j] = add(fine[j], err[j]);
}

template <typename T>
__global__ void k_set1(T* __restrict__ a, int n, T value, int modify_boundaries)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (!modify_boundaries && (j == 0 || j == n - 1)) return;
    a[j] = value;
}

inline int launch_ok() { return cudaPeekAtLastError() == cudaSuccess ? 1 : -1; }

inline int threads_for(const mg_hier1d& H, int level)
{
    int n = H.n[level];
    int t = 32;
    while (t < 1024 && t < n) t <<= 1;
    return t;
}

int ops(cudaStream_t s, int dtype, void* arena, const mg_hier1d& H, int op, int level, int a0, int a1, int a2,
        int corrected, void* r_out, double* out2)
{
    const int t = threads_for(H, level);
    if (dtype == 0) k_ops1d<float><<<1, t, 0, s>>>((float*)arena, H, op, level, a0, a1, a2, corrected, (float*)r_out, out2);
    else k_ops1d<double><<<1, t, 0, s>>>((double*)arena, H, op, level, a0, a1, a2, corrected, (double*)r_out, out2);
    return launch_ok();
}

}  // namespace

// |v - table| reduced to {sum, max} by one block (N1/Grid1D.cpp:46-60 as a reduction; `table` holds the analytic solution
// computed with the host libm, in the grid's own precision; the difference is taken in that precision too)
template <typename T>
__global__ void __launch_bounds__(256) k_abs_error1(const T* __restrict__ v, const T* __restrict__ table, int n, double* __restrict__ out2)
{
    __shared__ double ss[256], sm[256];
    double s = 0.0, m = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double d = fabs((double)mgx::sub(v[i], table[i]));
        s += d;
        m = max_nan(m, d);
    }
    ss[threadIdx.x] = s;
    sm[threadIdx.x] = m;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            ss[threadIdx.x] += ss[threadIdx.x + o];
            sm[threadIdx.x] = max_nan(sm[threadIdx.x], sm[threadIdx.x + o]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out2[0] = ss[0]; out2[1] = sm[0]; }
}

extern "C" {

int mgk1d_relax(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int ncycles)
{
    return ops(s, dtype, arena, H, OP_RELAX, level, ncycles, 0, 0, 0, nullptr, nullptr);
}

int mgk1d_residual(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected, void* r_out)
{
    return ops(s, dtype, arena, H, OP_RESIDUAL, level, 0, 0, 0, corrected, r_out, nullptr);
}

int mgk1d_residual_norm(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected, double* out2)
{
    return ops(s, dtype, arena, H, OP_NORM, level, 0, 0, 0, corrected, nullptr, out2);
}

int mgk1d_residual_restrict(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected)
{
    return ops(s, dtype, arena, H, OP_RESIDUAL_RESTRICT, level, 0, 0, 0, corrected, nullptr, nullptr);
}

int mgk1d_cycle(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int v0, int v1, int v2, int corrected,
                int fmg)
{
    return ops(s, dtype, arena, H, fmg ? OP_FMG : OP_VCYCLE, level, v0, v1, v2, corrected, nullptr, nullptr);
}

int mgk1d_level_op(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int which)
{
    /* which: 0 Restrict(f) fine->coarse, 1 Interpolate into v, 2 Interpolate + ApplyCorrection */
    return ops(s, dtype, arena, H, which == 0 ? OP_RESTRICT_F : (which == 1 ? OP_INTERP : OP_INTERP_ADD), level, 0, 0, 0, 0,
               nullptr, nullptr);
}

int mgk1d_abs_error(cudaStream_t s, int dtype, const void* v, const void* table, int n, double* out2)
{
    if (dtype == 0) k_abs_error1<float><<<1, 256, 0, s>>>((const float*)v, (const float*)table, n, out2);
    else k_abs_error1<double><<<1, 256, 0, s>>>((const double*)v, (const double*)table, n, out2);
    return launch_ok();
}

int mgk1d_restrict(cudaStream_t s, int dtype, const void* fine, int fn, void* coarse, int cn)
{
    const int b = 256, g = (cn + b - 1) / b;
    if (dtype == 0) k_restrict1<float><<<g, b, 0, s>>>((const float*)fine, fn, (float*)coarse, cn);
    else k_restrict1<double><<<g, b, 0, s>>>((const double*)fine, fn, (double*)coarse, cn);
    return launch_ok();
}

int mgk1d_interpolate(cudaStream_t s, int dtype, void* fine, int fn, const void* coarse, int cn, int add)
{
    (void)cn;
    if (fn < 3) return 0;
    const int b = 256, g = (fn - 2 + b - 1) / b;
    if (dtype == 0) k_interp1<float><<<g, b, 0, s>>>((float*)fine, fn, (const float*)coarse, add);
    else k_interp1<double><<<g, b, 0, s>>>((double*)fine, fn, (const double*)coarse, add);
    return launch_ok();
}

int mgk1d_apply_correction(cudaStream_t s, int dtype, void* fine, const void* err, int n)
{
    if (n < 3) return 0;
    const int b = 256, g = (n - 2 + b - 1) / b;
    if (dtype == 0) k_correct1<float><<<g, b, 0, s>>>((float*)fine, (const float*)err, n);
    else k_correct1<double><<<g, b, 0, s>>>((double*)fine, (const double*)err, n);
    return launch_ok();
}

int mgk1d_set(cudaStream_t s, int dtype, void* a, int n, double value, int modify_boundaries)
{
    const int b = 256, g = (n + b - 1) / b;
    if (dtype == 0) k_set1<float><<<g, b, 0, s>>>((float*)a, n, (float)value, modify_boundaries);
    else k_set1<double><<<g, b, 0, s>>>((double*)a, n, value, modify_boundaries);
    return launch_ok();
}

}  // extern "C"

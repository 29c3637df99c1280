// mg3d_diag.cu -- device-side diagnostics of the 3D engine (no reference counterpart on the device; the reference
// prints text dumps from the host):
//   * k_field_checksum: position-keyed additive checksum of a field -- the quantity bench.py prints to prove that a
//     run on N GPUs produced the bits the reference CPU solver produces (tests/golden/hashes3d.json holds the
//     reference's numbers, tests/golden_util.py:field_checksum is the same sum in numpy);
//   * k_abs_error: |analytic - v| reduced to {sum, max}: what Grid3D::PrintDiff (N3/Grid3D.cpp:136-159) writes point
//     by point into log/diff.txt, as a reduction (SURVEY.md 8f rank 3).
#include <stdint.h>

#include "mg3d_device.cuh"

using namespace mgx;
using namespace mg3;

namespace {

__device__ __forceinline__ unsigned long long mix64(unsigned long long z)
{
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return z;
}
__device__ __forceinline__ unsigned long long bits_of(double x) { return (unsigned long long)__double_as_longlong(x); }
__device__ __forceinline__ unsigned long long bits_of(float x) { return (unsigned long long)__float_as_uint(x); }

// sum over the points (x, y, z0+zl), zl in [zl_lo, zl_hi), of mix64(bits(a) + (idx+1)*GOLD), idx = x + n*(y + n*z):
// integer addition is associative and commutative, so the atomics make the result order-independent and slabs add up.
template <typename T>
__global__ void __launch_bounds__(256)
k_field_checksum(const T* __restrict__ a, mg_geom3d g, int zl_lo, int zl_hi, unsigned long long* __restrict__ out)
{
    const int hw = (g.n + 1) / 2;  // half-indices that exist in a row
    const long long rows = (long long)g.n * (zl_hi - zl_lo);
    unsigned long long acc = 0;
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const int zl = zl_lo + (int)(row / g.n), y = (int)(row % g.n), z = g.z0 + zl;
        const long long rbase = (long long)zl * g.plane + (long long)y * g.hp;
        const unsigned long long ibase = ((unsigned long long)z * g.n + y) * g.n;
        for (int k = threadIdx.x; k < 2 * hw; k += blockDim.x) {
            const int col = k >= hw, i = col ? k - hw : k;
            const int x = 2 * i + ((col + y + z) & 1);
            if (x >= g.n) continue;
            const T val = a[(long long)col * g.cstride + rbase + i];
            acc += mix64(bits_of(val) + (ibase + x + 1) * 0x9E3779B97F4A7C15ull);
        }
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

// N3/Grid3D.cpp:146-152: realSol = (real)(sin(PI*x)*sin(PI*y)*sin(PI*z)) (double product, narrowed),
// diff = realSol - approxSol in the grid's own precision.  sx/sy/sz: host-libm tables of sin(PI*coord).
template <typename T>
__global__ void __launch_bounds__(256)
k_abs_error(const T* __restrict__ v, mg_geom3d g, const double* __restrict__ sx, const double* __restrict__ sy,
            const double* __restrict__ sz, int zl_lo, int zl_hi, double* __restrict__ part)
{
    __shared__ double sh[64];
    double s = 0.0, m = 0.0;
    const long long rows = (long long)g.n * (zl_hi - zl_lo);
    for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
        const int zl = zl_lo + (int)(row / g.n), y = (int)(row % g.n), z = g.z0 + zl;
        const double syz = sy[y], szz = sz[z];
        for (int x = threadIdx.x; x < g.n; x += blockDim.x) {
            const T real_sol = (T)__dmul_rn(__dmul_rn(sx[x], syz), szz);
            const double d = fabs((double)sub(real_sol, v[off3(g, x, y, zl)]));
            s += d;
            m = max_nan(m, d);
        }
    }
    block_sum_max(s, m, sh);
    if (threadIdx.x == 0) { part[blockIdx.x] = s; part[gridDim.x + blockIdx.x] = m; }
}

}  // namespace

extern "C" {

/* *out += checksum of local planes [zl_lo, zl_hi) of the colour-split field a (the caller zeroes *out) */
int mgk3d_field_checksum(cudaStream_t s, int dtype, const void* a, mg_geom3d g, int zl_lo, int zl_hi, unsigned long long* out)
{
    if (zl_hi <= zl_lo) return 0;
    const long long rows = (long long)g.n * (zl_hi - zl_lo);
    const int nb = (int)(rows < 148 * 16 ? rows : 148 * 16);
    if (dtype == 0) k_field_checksum<float><<<nb, 256, 0, s>>>((const float*)a, g, zl_lo, zl_hi, out);
    else k_field_checksum<double><<<nb, 256, 0, s>>>((const double*)a, g, zl_lo, zl_hi, out);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

/* {sum, max} of |analytic - v| over local planes [zl_lo, zl_hi): partials into scratch (2*MGK_NORM_BLOCKS doubles),
   finished by mgk_norm_final into out2 */
int mgk3d_abs_error(cudaStream_t s, int dtype, const void* v, mg_geom3d g, const double* sx, const double* sy, const double* sz,
                    int zl_lo, int zl_hi, double* scratch, double* out2)
{
    const int nb = MGK_NORM_BLOCKS;
    if (dtype == 0) k_abs_error<float><<<nb, 256, 0, s>>>((const float*)v, g, sx, sy, sz, zl_lo, zl_hi, scratch);
    else k_abs_error<double><<<nb, 256, 0, s>>>((const double*)v, g, sx, sy, sz, zl_lo, zl_hi, scratch);
    if (cudaPeekAtLastError() != cudaSuccess) return -1;
    return mgk_norm_final(s, scratch, nb, out2) < 0 ? -1 : 2;
}

}  // extern "C"

// mg_exact.cuh -- rounding-exact arithmetic helpers shared by all kernels.
//
// The parity contract is bit-equality with the reference CPU solver, which is compiled for
// baseline x86-64: every +,-,*,/ is a separately rounded IEEE operation (no FMA contraction,
// SURVEY.md 7.2).  nvcc contracts a*b+c into FMA by default, so the kernels never write infix
// arithmetic on field values: they go through these intrinsics, which ptxas may not contract.
#pragma once
#include <cuda_runtime.h>

namespace mgx {

__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }

__device__ __forceinline__ double fma_(double a, double b, double c) { return __fma_rn(a, b, c); }
__device__ __forceinline__ float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }

// max that keeps a NaN (fmax drops it): the linf of a field with a NaN is NaN, like np.max(np.abs(r)).  For the
// linf and abs-error reductions; every finite result is fmax's.
__device__ __forceinline__ double max_nan(double a, double b) { return (a > b || a != a) ? a : b; }

// Correctly rounded a/b from a correctly rounded reciprocal y = RN(1/b) computed once on the host
// (Markstein 1990: q = RN(a*y); r = a - b*q exactly with one FMA; q' = RN(q + r*y) is the correctly
// rounded quotient).  Three pipe operations instead of the ~20-instruction IEEE division sequence.
// Bit-identical to a/b in every case:
//   * r == 0: q is already the exact quotient (this also keeps the sign of a zero: the FMA chain would turn -0 into +0);
//   * |a| below 2^(emin + 2p + 4) (p = significand bits): the residual r could be subnormal and lose bits, so the
//     IEEE division is used there -- never reached by values of an actual solve, see tests/test_smoother_pipe_gpu.py;
//   * non-finite q (inf/NaN input): passed through, so that overflowed REF_COMPAT runs still match the reference.
__device__ __forceinline__ bool div_small(double a) { return fabs(a) < 0x1p-914; }
__device__ __forceinline__ bool div_small(float a) { return fabsf(a) < 0x1p-76f; }

template <typename T>
__device__ __forceinline__ T div_by_const(T a, T b, T y)
{
    if (div_small(a)) return div(a, b);
    T q = mul(a, y);
    T r = fma_(-b, q, a);
    T q2 = fma_(r, y, q);
    return (q - q == T(0) && r != T(0)) ? q2 : q;  // q - q is NaN for inf/NaN
}

}  // namespace mgx

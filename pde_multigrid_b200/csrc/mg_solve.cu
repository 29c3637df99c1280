// mg_solve.cu -- the device side of the tolerance-driven solve (mg?d_solve in include/mg_b200.h): one thread that reads the
// (sum of squares, max) pair a family's norm finaliser has just written, applies the stopping rule and steers the
// CUDA-graph WHILE (and IF) node of the solve.  The same kernel decides in the host-driven loop, where it sets no handle,
// so both paths stop on exactly the same comparison.
#include "mg_launch.h"

namespace {

__global__ void k_solve_check(const double* __restrict__ out2, mg_solve_par* __restrict__ p, int nhandles,
                              cudaGraphConditionalHandle h0, cudaGraphConditionalHandle h1)
{
    // IEEE double sqrt is correctly rounded: the same bits as the host's sqrt in mg?d_residual_norm
    const double l2 = sqrt(out2[0]), linf = out2[1];
    const int k = p->k;
    if (k == 0) {
        const double t = p->rtol * l2;
        p->thr = p->atol > t ? p->atol : t;
    }
    if (k < p->hist_cap) {
        p->hist[2 * k] = l2;
        p->hist[2 * k + 1] = linf;
    }
    const int finite = isfinite(l2);
    const int conv = finite && l2 <= p->thr;
    const int done = !finite || conv || k >= p->max_cycles;
    p->k = k + 1;
    p->done = done;
    p->converged = conv;
    if (nhandles > 0) cudaGraphSetConditional(h0, done ? 0u : 1u);
    if (nhandles > 1) cudaGraphSetConditional(h1, done ? 0u : 1u);
}

}  // namespace

extern "C" int mgk_solve_check(cudaStream_t s, const double* out2, mg_solve_par* par, int nhandles, cudaGraphConditionalHandle h0,
                               cudaGraphConditionalHandle h1)
{
    k_solve_check<<<1, 1, 0, s>>>(out2, par, nhandles, h0, h1);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

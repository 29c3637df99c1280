/*
 * mg1d_host.c -- C host driver of the 1D multigrid (first-order ODE BVP u' - u/(e^x+1) = e^x).
 *
 * Mirrors the reference class MultiGrid1D (NOCUDA_TESI/EQUAZIONE 1D/MultiGrid1D.cpp: InitGrids :19-31,
 * VCycle :150-175, FullMultiGridVCycle :132-148).  The hierarchy (v, f and the two coefficient tables
 * e1 = exp(x)+1, d = exp(x)+1+h per level) lives in one device arena; a whole V-cycle or FMG solve is
 * ONE kernel launch (mg1d_kernels.cu).  The host evaluates exp() with libm, exactly as the reference
 * does (exp(float) -> expf in the float build, exp(double) in the double build, SURVEY.md 8a), so the
 * device never needs a transcendental and stays bit-exact.  No CPU solve path exists here.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mg_host_common.h"

struct mg1d_s {
    mg_core core; /* core.nlevels == H.nlevels, which the kernels take by value */
    int mode;
    double range[2];
    mg_hier1d H;
    size_t arena_elems;
    void* arena;
    double* d_out2;
};

static void* elem_ptr(mg1d_t* mg, long long off) { return (char*)mg->arena + (size_t)off * mg_esize(mg->core.dtype); }
static void* field_ptr(mg1d_t* mg, int level, int field) { return elem_ptr(mg, field == MG_FIELD_V ? mg->H.off_v[level] : mg->H.off_f[level]); }

int mg1d_create(mg1d_t** out, int n, const double range[2], int dtype, int residual_mode)
{
    if (!out || !range) return mg_fail(MG_ERR_ARG, "null argument");
    *out = NULL;
    if (n < 3 || ((n - 1) & (n - 2)) != 0) return mg_fail(MG_ERR_ARG, "size must be 2^k+1 with k >= 1 (got %d)", n); /* N1/Grid1D.cpp:6-7 */
    if (!(range[1] > range[0])) return mg_fail(MG_ERR_ARG, "range must satisfy b > a");                               /* N1/Grid1D.cpp:10 */
    if (dtype != MG_F32 && dtype != MG_F64) return mg_fail(MG_ERR_ARG, "dtype must be MG_F32 or MG_F64");
    if (residual_mode != MG_REF_COMPAT && residual_mode != MG_CORRECTED) return mg_fail(MG_ERR_ARG, "bad residual_mode");
    int st = mg_require_device();
    if (st) return st;
    mg1d_t* mg = (mg1d_t*)calloc(1, sizeof *mg);
    if (!mg) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    mg->core.dtype = dtype;
    mg->mode = residual_mode;
    mg->range[0] = range[0];
    mg->range[1] = range[1];
    mg->H.nlevels = mg->core.nlevels = mg_num_levels_for(n);
    if (mg->H.nlevels > MG1D_MAX_LEVELS) { free(mg); return mg_fail(MG_ERR_ARG, "too many levels"); }
    long long off = 0;
    int nl = n;
    for (int l = 0; l < mg->H.nlevels; l++) {
        long long padded = (nl + 31) / 32 * 32;
        mg->H.n[l] = nl;
        mg->H.off_v[l] = off; off += padded;
        mg->H.off_f[l] = off; off += padded;
        mg->H.off_e[l] = off; off += padded;
        mg->H.off_d[l] = off; off += padded;
        nl = (nl - 1) / 2 + 1; /* N1/MultiGrid1D.cpp:28 */
    }
    mg->arena_elems = (size_t)off;
    if ((st = mg_core_init(&mg->core))) { mg1d_destroy(mg); return st; }
    if (cudaMalloc(&mg->arena, mg->arena_elems * mg_esize(dtype)) != cudaSuccess ||
        cudaMalloc((void**)&mg->d_out2, 2 * sizeof(double)) != cudaSuccess) {
        int code = mg_fail(MG_ERR_CUDA, "device setup failed: %s", cudaGetErrorString(cudaGetLastError()));
        mg1d_destroy(mg);
        return code;
    }
    st = mg1d_init_problem(mg);
    if (st) { mg1d_destroy(mg); return st; }
    *out = mg;
    return MG_OK;
}

int mg1d_destroy(mg1d_t* mg)
{
    if (!mg) return MG_OK;
    mg_core_free(&mg->core);
    if (mg->arena) cudaFree(mg->arena);
    if (mg->d_out2) cudaFree(mg->d_out2);
    free(mg);
    return MG_OK;
}

int mg1d_num_levels(const mg1d_t* mg) { return mg ? mg->H.nlevels : 0; }
int mg1d_level_size(const mg1d_t* mg, int level) { return (mg && level >= 0 && level < mg->H.nlevels) ? mg->H.n[level] : 0; }
double mg1d_level_h(const mg1d_t* mg, int level) { return (mg && level >= 0 && level < mg->H.nlevels) ? mg->H.h[level] : 0.0; }
void* mg1d_stream(mg1d_t* mg) { return mg ? (void*)mg->core.stream : NULL; }
long long mg1d_kernel_launches(const mg1d_t* mg) { return mg ? mg->core.launches : 0; }

int mg1d_sync(mg1d_t* mg) { return mg_sync(MG_CORE(mg)); }
int mg1d_profile(mg1d_t* mg, int enable) { return mg_profile_enable(MG_CORE(mg), enable); }
int mg1d_profile_read(mg1d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls)
{
    return mg_profile_read(MG_CORE(mg), level, op, ms_total, kernel_launches, calls);
}

/* Grid1D ctor on every level (N1/Grid1D.cpp:4-43): h, InitV (analytic end points; interior zeroed,
   SURVEY.md App. B8), InitF (f = exp(x)), plus the smoother's coefficient tables. */
int mg1d_init_problem(mg1d_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    const size_t es = mg_esize(mg->core.dtype);
    void* host = calloc(mg->arena_elems, es);
    if (!host) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    for (int l = 0; l < mg->H.nlevels; l++) {
        const int n = mg->H.n[l];
        if (mg->core.dtype == MG_F32) {
            float* a = (float*)host;
            float x_a = (float)mg->range[0], x_b = (float)mg->range[1];
            float x_range = x_b - x_a;
            float h_x = x_range / (float)(n - 1);
            mg->H.h[l] = h_x;
            float *v = a + mg->H.off_v[l], *f = a + mg->H.off_f[l], *e1 = a + mg->H.off_e[l], *d = a + mg->H.off_d[l];
            v[0] = (expf(x_a) + x_a - 3) / (1 + expf(-x_a));
            v[n - 1] = (expf(x_b) + x_b - 3) / (1 + expf(-x_b));
            for (int j = 0; j < n; j++) {
                float xj = x_a + j * h_x;
                f[j] = expf(xj);
                e1[j] = expf(xj) + 1;
                d[j] = expf(xj) + 1 + h_x;
            }
        } else {
            double* a = (double*)host;
            double x_a = mg->range[0], x_b = mg->range[1];
            double x_range = x_b - x_a;
            double h_x = x_range / (double)(n - 1);
            mg->H.h[l] = h_x;
            double *v = a + mg->H.off_v[l], *f = a + mg->H.off_f[l], *e1 = a + mg->H.off_e[l], *d = a + mg->H.off_d[l];
            v[0] = (exp(x_a) + x_a - 3) / (1 + exp(-x_a));
            v[n - 1] = (exp(x_b) + x_b - 3) / (1 + exp(-x_b));
            for (int j = 0; j < n; j++) {
                double xj = x_a + j * h_x;
                f[j] = exp(xj);
                e1[j] = exp(xj) + 1;
                d[j] = exp(xj) + 1 + h_x;
            }
        }
    }
    cudaError_t e = cudaMemcpyAsync(mg->arena, host, mg->arena_elems * es, cudaMemcpyHostToDevice, mg->core.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
    free(host);
    if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "arena upload failed: %s", cudaGetErrorString(e));
    return MG_OK;
}

int mg1d_set_field(mg1d_t* mg, int level, int field, const void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, level, field), host_dense, (size_t)mg->H.n[level] * mg_esize(mg->core.dtype), cudaMemcpyHostToDevice, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg1d_get_field(mg1d_t* mg, int level, int field, void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaMemcpyAsync(host_dense, field_ptr(mg, level, field), (size_t)mg->H.n[level] * mg_esize(mg->core.dtype), cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg1d_relax(mg1d_t* mg, int level, int ncycles)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (ncycles < 0) return mg_fail(MG_ERR_ARG, "ncycles < 0");
    PROF_BEGIN(mg, level, MG_OP_RELAX);
    MG_LAUNCH(mg->core.launches, mgk1d_relax(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, ncycles));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_residual(mg1d_t* mg, int level, void* host_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_out) return mg_fail(MG_ERR_ARG, "null output");
    const size_t bytes = (size_t)mg->H.n[level] * mg_esize(mg->core.dtype);
    void* r = NULL;
    MG_CUDA(cudaMalloc(&r, bytes));
    int k = mgk1d_residual(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, r);
    cudaError_t e = cudaSuccess;
    if (k >= 0) {
        mg->core.launches += k;
        e = cudaMemcpyAsync(host_out, r, bytes, cudaMemcpyDeviceToHost, mg->core.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
    }
    cudaFree(r);
    if (k < 0 || e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "residual failed: %s", cudaGetErrorString(e));
    return MG_OK;
}

/* Grid1D::PrintDiffApproxReal (N1/Grid1D.cpp:46-60) as a reduction: mean and max over all points of |approxsol - realsol|,
   realsol = (exp(xj) + xj - 3)/(1 + exp(-xj)) with the host libm in the grid's precision (float: expf, like the reference) */
int mg1d_abs_error(mg1d_t* mg, int level, double* mean_abs, double* max_abs)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    const int n = mg->H.n[level];
    const size_t es = mg_esize(mg->core.dtype);
    void* host = malloc((size_t)n * es);
    if (!host) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    if (mg->core.dtype == MG_F32) {
        float x_a = (float)mg->range[0], h_x = ((float)mg->range[1] - x_a) / (float)(n - 1);
        for (int j = 0; j < n; j++) {
            float xj = x_a + j * h_x;
            ((float*)host)[j] = (expf(xj) + xj - 3) / (1 + expf(-xj));
        }
    } else {
        double x_a = mg->range[0], h_x = (mg->range[1] - x_a) / (double)(n - 1);
        for (int j = 0; j < n; j++) {
            double xj = x_a + j * h_x;
            ((double*)host)[j] = (exp(xj) + xj - 3) / (1 + exp(-xj));
        }
    }
    void* d = NULL;
    cudaError_t e = cudaMalloc(&d, (size_t)n * es);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d, host, (size_t)n * es, cudaMemcpyHostToDevice, mg->core.stream);
    if (e != cudaSuccess) { free(host); if (d) cudaFree(d); return mg_fail(MG_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e)); }
    const char* v = (const char*)mg->arena + (size_t)mg->H.off_v[level] * es;
    int k = mgk1d_abs_error(mg->core.stream, mg->core.dtype, v, d, n, mg->d_out2);
    if (k >= 0) e = cudaMemcpyAsync(mg->core.h_out2, mg->d_out2, 2 * sizeof(double), cudaMemcpyDeviceToHost, mg->core.stream);
    if (k >= 0 && e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
    free(host);
    cudaFree(d);
    if (k < 0 || e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "abs error reduction failed: %s", cudaGetErrorString(cudaGetLastError()));
    mg->core.launches += k;
    if (mean_abs) *mean_abs = mg->core.h_out2[0] / n;
    if (max_abs) *max_abs = mg->core.h_out2[1];
    return MG_OK;
}

/* the norm pass of mg1d_residual_norm: {sum of r^2, max |r|} into d_out2, nothing read back */
static int residual_norm_enqueue(mg1d_t* mg, int level)
{
    MG_LAUNCH(mg->core.launches, mgk1d_residual_norm(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, mg->d_out2));
    return MG_OK;
}

int mg1d_residual_norm(mg1d_t* mg, int level, double* l2, double* linf)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if ((st = residual_norm_enqueue(mg, level))) return st;
    return mg_read_norm(&mg->core, mg->d_out2, l2, linf);
}

int mg1d_restrict(mg1d_t* mg, int fine_level, int field)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    MG_LAUNCH(mg->core.launches, mgk1d_restrict(mg->core.stream, mg->core.dtype, field_ptr(mg, fine_level, field), mg->H.n[fine_level],
                                           field_ptr(mg, fine_level + 1, field), mg->H.n[fine_level + 1]));
    return MG_OK;
}

int mg1d_residual_restrict(mg1d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    PROF_BEGIN(mg, fine_level, MG_OP_RESIDUAL_RESTRICT);
    MG_LAUNCH(mg->core.launches, mgk1d_residual_restrict(mg->core.stream, mg->core.dtype, mg->arena, mg->H, fine_level, mg->mode == MG_CORRECTED));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_interpolate(mg1d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    MG_LAUNCH(mg->core.launches, mgk1d_level_op(mg->core.stream, mg->core.dtype, mg->arena, mg->H, fine_level, 1));
    return MG_OK;
}

int mg1d_interpolate_correct(mg1d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    PROF_BEGIN(mg, fine_level, MG_OP_INTERPOLATE);
    MG_LAUNCH(mg->core.launches, mgk1d_level_op(mg->core.stream, mg->core.dtype, mg->arena, mg->H, fine_level, 2));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_set_to_value(mg1d_t* mg, int level, int field, double value, int modify_boundaries)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    MG_LAUNCH(mg->core.launches, mgk1d_set(mg->core.stream, mg->core.dtype, field_ptr(mg, level, field), mg->H.n[level], value, modify_boundaries));
    return MG_OK;
}

/* VCycle (N1/MultiGrid1D.cpp:150-175): the whole cycle is one launch of the persistent CTA */
int mg1d_vcycle(mg1d_t* mg, int level, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    PROF_BEGIN(mg, level, MG_OP_OTHER);
    MG_LAUNCH(mg->core.launches, mgk1d_cycle(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, 1, v1, v2, mg->mode == MG_CORRECTED, 0));
    PROF_END(mg);
    return MG_OK;
}

/* tolerance-driven solve (mg_host_common.c builds and runs it): the body is the one-launch cycle, the norm and the check */
static int s1_norm(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return residual_norm_enqueue(x->h, x->level); }
static int s1_cycle(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return mg1d_vcycle(x->h, x->level, x->v1, x->v2); }

int mg1d_solve(mg1d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles, int* cycles_out, int* converged_out,
               double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_cycles, v1, v2);
    if (st) return st;
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = {&x, mg->core.stream, &mg->core.launches, NULL, s1_cycle, s1_cycle, s1_norm, mg->d_out2, NULL, NULL};
    const int key[MG_GRAPH_KEY] = {level, v1, v2};
    /* one launch per cycle: no bound on the sweep counts */
    return mg_solve_run(&mg->core.graphs, mg_graphs_on(&mg->core.graphs, mg->core.prof.enabled, 1) ? key : NULL, &ops, rtol, atol, max_cycles,
                        cycles_out, converged_out, history);
}

/* FullMultiGridVCycle (N1/MultiGrid1D.cpp:132-148): one launch */
int mg1d_fmg(mg1d_t* mg, int level, int v0, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v0 < 0 || v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative cycle/sweep count");
    PROF_BEGIN(mg, level, MG_OP_OTHER);
    MG_LAUNCH(mg->core.launches, mgk1d_cycle(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, v0, v1, v2, mg->mode == MG_CORRECTED, 1));
    PROF_END(mg);
    return MG_OK;
}

/* ---- reference-facing operators on HOST arrays (N1/MultiGrid1D.h:16-22) ---------------------- */

int mg1d_restrict_host(mg1d_t* mg, const void* fine, int fn, void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N1/MultiGrid1D.cpp:36 */
    void *df, *dc;
    int st = mg_tmp_begin(&mg->core, &df, fn, fine, &dc, cn, NULL);
    if (st) return st;
    return mg_tmp_finish(&mg->core, mgk1d_restrict(mg->core.stream, mg->core.dtype, df, fn, dc, cn), coarse, dc, cn, df, dc);
}

int mg1d_interpolate_host(mg1d_t* mg, void* fine, int fn, const void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N1/MultiGrid1D.cpp:62 */
    void *df, *dc;
    int st = mg_tmp_begin(&mg->core, &df, fn, fine, &dc, cn, coarse);
    if (st) return st;
    return mg_tmp_finish(&mg->core, mgk1d_interpolate(mg->core.stream, mg->core.dtype, df, fn, dc, cn, 0), fine, df, fn, df, dc);
}

int mg1d_apply_correction_host(mg1d_t* mg, void* fine, int fn, const void* error, int en)
{
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn != en || fn < 3) return mg_fail(MG_ERR_ARG, "fsize != esize"); /* N1/MultiGrid1D.cpp:179 */
    void *df, *de;
    int st = mg_tmp_begin(&mg->core, &df, fn, fine, &de, en, error);
    if (st) return st;
    return mg_tmp_finish(&mg->core, mgk1d_apply_correction(mg->core.stream, mg->core.dtype, df, de, fn), fine, df, fn, df, de);
}

int mg1d_set_to_value_host(mg1d_t* mg, void* grid, int n, double value, int modify_boundaries)
{
    if (!mg || !grid || n < 1) return mg_fail(MG_ERR_ARG, "bad argument");
    void *d, *unused;
    int st = mg_tmp_begin(&mg->core, &d, n, grid, &unused, 0, NULL);
    if (st) return st;
    return mg_tmp_finish(&mg->core, mgk1d_set(mg->core.stream, mg->core.dtype, d, n, value, modify_boundaries), grid, d, n, d, NULL);
}

/* ---- the CUDA_TESI faces (C1/MultiGrid1D.h:16-23, C1/Grid1D.h:15-18): operators on DEVICE arrays.  The engine's 1D fields
        are dense device arrays already, so a level's d_v / d_f are the engine's own storage. ------------------------- */
int mg1d_level_device_ptr(mg1d_t* mg, int level, int field, void** ptr)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!ptr || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    const long long off = field == MG_FIELD_V ? mg->H.off_v[level] : mg->H.off_f[level];
    *ptr = (char*)mg->arena + (size_t)off * mg_esize(mg->core.dtype);
    return MG_OK;
}

int mg1d_restrict_device(mg1d_t* mg, const void* fine, int fn, void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk1d_restrict(mg->core.stream, mg->core.dtype, fine, fn, coarse, cn));
}

int mg1d_interpolate_device(mg1d_t* mg, void* fine, int fn, const void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk1d_interpolate(mg->core.stream, mg->core.dtype, fine, fn, coarse, cn, 0));
}

int mg1d_apply_correction_device(mg1d_t* mg, void* fine, int fn, const void* error, int en)
{
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn != en || fn < 1) return mg_fail(MG_ERR_ARG, "fsize != esize");
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk1d_apply_correction(mg->core.stream, mg->core.dtype, fine, error, fn));
}

int mg1d_set_device(mg1d_t* mg, void* d_v, int n, double value, int modify_boundaries)
{
    if (!mg || !d_v || n < 1) return mg_fail(MG_ERR_ARG, "bad argument");
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk1d_set(mg->core.stream, mg->core.dtype, d_v, n, value, modify_boundaries));
}

/* CalculateResidual(grid) into a caller-owned DEVICE array (C1/MultiGrid1D.cu:86-104) */
int mg1d_residual_device(mg1d_t* mg, int level, void* dev_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!dev_out) return mg_fail(MG_ERR_ARG, "null output");
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk1d_residual(mg->core.stream, mg->core.dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, dev_out));
}

int mg1d_vcycle_host(mg1d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles)
{
    if (!mg || !v_host || !f_host) return mg_fail(MG_ERR_ARG, "null argument");
    if (v1 < 0 || v2 < 0 || cycles < 0) return mg_fail(MG_ERR_ARG, "negative count");
    const size_t bytes = (size_t)mg->H.n[0] * mg_esize(mg->core.dtype);
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, 0, MG_FIELD_V), v_host, bytes, cudaMemcpyHostToDevice, mg->core.stream));
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, 0, MG_FIELD_F), f_host, bytes, cudaMemcpyHostToDevice, mg->core.stream));
    MG_LAUNCH(mg->core.launches, mgk1d_cycle(mg->core.stream, mg->core.dtype, mg->arena, mg->H, 0, cycles, v1, v2, mg->mode == MG_CORRECTED, 0));
    MG_CUDA(cudaMemcpyAsync(v_host, field_ptr(mg, 0, MG_FIELD_V), bytes, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

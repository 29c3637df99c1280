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
#include "mg_profile.h"

struct mg1d_s {
    int dtype, mode;
    double range[2];
    mg_hier1d H;
    size_t arena_elems;
    void* arena;
    cudaStream_t stream;
    double* d_out2;
    double* h_out2;
    long long launches;
    mg_prof prof;
    mg_graphs graphs; /* mg1d_solve graphs */
};

#define PROF_BEGIN(mg, level, op) mg_prof_begin(&(mg)->prof, (mg)->stream, (level), (op), (mg)->launches)
#define PROF_END(mg) mg_prof_end(&(mg)->prof, (mg)->stream, (mg)->launches)

static int check_level(const mg1d_t* mg, int level)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    if (level < 0 || level >= mg->H.nlevels) return mg_fail(MG_ERR_ARG, "level %d out of range [0,%d)", level, mg->H.nlevels);
    return MG_OK;
}

static void* elem_ptr(mg1d_t* mg, long long off) { return (char*)mg->arena + (size_t)off * mg_esize(mg->dtype); }
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
    mg->dtype = dtype;
    mg->mode = residual_mode;
    mg_graphs_init(&mg->graphs);
    mg->range[0] = range[0];
    mg->range[1] = range[1];
    mg->H.nlevels = mg_num_levels_for(n);
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
    if (cudaMalloc(&mg->arena, mg->arena_elems * mg_esize(dtype)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&mg->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaMalloc((void**)&mg->d_out2, 2 * sizeof(double)) != cudaSuccess ||
        cudaMallocHost((void**)&mg->h_out2, 2 * sizeof(double)) != cudaSuccess) {
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
    if (mg->stream) cudaStreamSynchronize(mg->stream);
    mg_graphs_free(&mg->graphs);
    if (mg->stream) cudaStreamDestroy(mg->stream);
    if (mg->arena) cudaFree(mg->arena);
    if (mg->d_out2) cudaFree(mg->d_out2);
    if (mg->h_out2) cudaFreeHost(mg->h_out2);
    mg_prof_free(&mg->prof);
    free(mg);
    return MG_OK;
}

int mg1d_num_levels(const mg1d_t* mg) { return mg ? mg->H.nlevels : 0; }
int mg1d_level_size(const mg1d_t* mg, int level) { return (mg && level >= 0 && level < mg->H.nlevels) ? mg->H.n[level] : 0; }
double mg1d_level_h(const mg1d_t* mg, int level) { return (mg && level >= 0 && level < mg->H.nlevels) ? mg->H.h[level] : 0.0; }
void* mg1d_stream(mg1d_t* mg) { return mg ? (void*)mg->stream : NULL; }
long long mg1d_kernel_launches(const mg1d_t* mg) { return mg ? mg->launches : 0; }

int mg1d_sync(mg1d_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    return MG_OK;
}

int mg1d_profile(mg1d_t* mg, int enable)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    return mg_prof_enable(&mg->prof, mg->stream, enable);
}

int mg1d_profile_read(mg1d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (op < 0 || op >= MG_OP_COUNT) return mg_fail(MG_ERR_ARG, "bad op %d", op);
    st = mg_prof_collect(&mg->prof, mg->stream);
    if (st) return st;
    if (ms_total) *ms_total = mg->prof.ms[level][op];
    if (kernel_launches) *kernel_launches = mg->prof.kl[level][op];
    if (calls) *calls = mg->prof.calls[level][op];
    return MG_OK;
}

/* Grid1D ctor on every level (N1/Grid1D.cpp:4-43): h, InitV (analytic end points; interior zeroed,
   SURVEY.md App. B8), InitF (f = exp(x)), plus the smoother's coefficient tables. */
int mg1d_init_problem(mg1d_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    const size_t es = mg_esize(mg->dtype);
    void* host = calloc(mg->arena_elems, es);
    if (!host) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    for (int l = 0; l < mg->H.nlevels; l++) {
        const int n = mg->H.n[l];
        if (mg->dtype == MG_F32) {
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
    cudaError_t e = cudaMemcpyAsync(mg->arena, host, mg->arena_elems * es, cudaMemcpyHostToDevice, mg->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(mg->stream);
    free(host);
    if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "arena upload failed: %s", cudaGetErrorString(e));
    return MG_OK;
}

int mg1d_set_field(mg1d_t* mg, int level, int field, const void* host_dense)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, level, field), host_dense, (size_t)mg->H.n[level] * mg_esize(mg->dtype), cudaMemcpyHostToDevice, mg->stream));
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    return MG_OK;
}

int mg1d_get_field(mg1d_t* mg, int level, int field, void* host_dense)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaMemcpyAsync(host_dense, field_ptr(mg, level, field), (size_t)mg->H.n[level] * mg_esize(mg->dtype), cudaMemcpyDeviceToHost, mg->stream));
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    return MG_OK;
}

int mg1d_relax(mg1d_t* mg, int level, int ncycles)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (ncycles < 0) return mg_fail(MG_ERR_ARG, "ncycles < 0");
    PROF_BEGIN(mg, level, MG_OP_RELAX);
    MG_LAUNCH(mg->launches, mgk1d_relax(mg->stream, mg->dtype, mg->arena, mg->H, level, ncycles));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_residual(mg1d_t* mg, int level, void* host_out)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (!host_out) return mg_fail(MG_ERR_ARG, "null output");
    const size_t bytes = (size_t)mg->H.n[level] * mg_esize(mg->dtype);
    void* r = NULL;
    MG_CUDA(cudaMalloc(&r, bytes));
    int k = mgk1d_residual(mg->stream, mg->dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, r);
    cudaError_t e = cudaSuccess;
    if (k >= 0) {
        mg->launches += k;
        e = cudaMemcpyAsync(host_out, r, bytes, cudaMemcpyDeviceToHost, mg->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(mg->stream);
    }
    cudaFree(r);
    if (k < 0 || e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "residual failed: %s", cudaGetErrorString(e));
    return MG_OK;
}

/* Grid1D::PrintDiffApproxReal (N1/Grid1D.cpp:46-60) as a reduction: mean and max over all points of |approxsol - realsol|,
   realsol = (exp(xj) + xj - 3)/(1 + exp(-xj)) with the host libm in the grid's precision (float: expf, like the reference) */
int mg1d_abs_error(mg1d_t* mg, int level, double* mean_abs, double* max_abs)
{
    int st = check_level(mg, level);
    if (st) return st;
    const int n = mg->H.n[level];
    const size_t es = mg_esize(mg->dtype);
    void* host = malloc((size_t)n * es);
    if (!host) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    if (mg->dtype == MG_F32) {
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
    if (e == cudaSuccess) e = cudaMemcpyAsync(d, host, (size_t)n * es, cudaMemcpyHostToDevice, mg->stream);
    if (e != cudaSuccess) { free(host); if (d) cudaFree(d); return mg_fail(MG_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e)); }
    const char* v = (const char*)mg->arena + (size_t)mg->H.off_v[level] * es;
    int k = mgk1d_abs_error(mg->stream, mg->dtype, v, d, n, mg->d_out2);
    if (k >= 0) e = cudaMemcpyAsync(mg->h_out2, mg->d_out2, 2 * sizeof(double), cudaMemcpyDeviceToHost, mg->stream);
    if (k >= 0 && e == cudaSuccess) e = cudaStreamSynchronize(mg->stream);
    free(host);
    cudaFree(d);
    if (k < 0 || e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "abs error reduction failed: %s", cudaGetErrorString(cudaGetLastError()));
    mg->launches += k;
    if (mean_abs) *mean_abs = mg->h_out2[0] / n;
    if (max_abs) *max_abs = mg->h_out2[1];
    return MG_OK;
}

/* the norm pass of mg1d_residual_norm: {sum of r^2, max |r|} into d_out2, nothing read back */
static int residual_norm_enqueue(mg1d_t* mg, int level)
{
    MG_LAUNCH(mg->launches, mgk1d_residual_norm(mg->stream, mg->dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, mg->d_out2));
    return MG_OK;
}

int mg1d_residual_norm(mg1d_t* mg, int level, double* l2, double* linf)
{
    int st = check_level(mg, level);
    if (st) return st;
    if ((st = residual_norm_enqueue(mg, level))) return st;
    MG_CUDA(cudaMemcpyAsync(mg->h_out2, mg->d_out2, 2 * sizeof(double), cudaMemcpyDeviceToHost, mg->stream));
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    if (l2) *l2 = sqrt(mg->h_out2[0]);
    if (linf) *linf = mg->h_out2[1];
    return MG_OK;
}

static int not_coarsest(mg1d_t* mg, int level)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (level == mg->H.nlevels - 1) return mg_fail(MG_ERR_ARG, "level %d is the coarsest", level);
    return MG_OK;
}

int mg1d_restrict(mg1d_t* mg, int fine_level, int field)
{
    int st = not_coarsest(mg, fine_level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    MG_LAUNCH(mg->launches, mgk1d_restrict(mg->stream, mg->dtype, field_ptr(mg, fine_level, field), mg->H.n[fine_level],
                                           field_ptr(mg, fine_level + 1, field), mg->H.n[fine_level + 1]));
    return MG_OK;
}

int mg1d_residual_restrict(mg1d_t* mg, int fine_level)
{
    int st = not_coarsest(mg, fine_level);
    if (st) return st;
    PROF_BEGIN(mg, fine_level, MG_OP_RESIDUAL_RESTRICT);
    MG_LAUNCH(mg->launches, mgk1d_residual_restrict(mg->stream, mg->dtype, mg->arena, mg->H, fine_level, mg->mode == MG_CORRECTED));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_interpolate(mg1d_t* mg, int fine_level)
{
    int st = not_coarsest(mg, fine_level);
    if (st) return st;
    MG_LAUNCH(mg->launches, mgk1d_level_op(mg->stream, mg->dtype, mg->arena, mg->H, fine_level, 1));
    return MG_OK;
}

int mg1d_interpolate_correct(mg1d_t* mg, int fine_level)
{
    int st = not_coarsest(mg, fine_level);
    if (st) return st;
    PROF_BEGIN(mg, fine_level, MG_OP_INTERPOLATE);
    MG_LAUNCH(mg->launches, mgk1d_level_op(mg->stream, mg->dtype, mg->arena, mg->H, fine_level, 2));
    PROF_END(mg);
    return MG_OK;
}

int mg1d_set_to_value(mg1d_t* mg, int level, int field, double value, int modify_boundaries)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    MG_LAUNCH(mg->launches, mgk1d_set(mg->stream, mg->dtype, field_ptr(mg, level, field), mg->H.n[level], value, modify_boundaries));
    return MG_OK;
}

/* VCycle (N1/MultiGrid1D.cpp:150-175): the whole cycle is one launch of the persistent CTA */
int mg1d_vcycle(mg1d_t* mg, int level, int v1, int v2)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    PROF_BEGIN(mg, level, MG_OP_OTHER);
    MG_LAUNCH(mg->launches, mgk1d_cycle(mg->stream, mg->dtype, mg->arena, mg->H, level, 1, v1, v2, mg->mode == MG_CORRECTED, 0));
    PROF_END(mg);
    return MG_OK;
}

/* tolerance-driven solve (mg_host_common.c builds and runs it): the body is the one-launch cycle, the norm and the check */
typedef struct {
    mg1d_t* mg;
    int level, v1, v2;
} solve1d_ctx;

static int s1_norm(void* c) { solve1d_ctx* x = (solve1d_ctx*)c; return residual_norm_enqueue(x->mg, x->level); }
static int s1_cycle(void* c) { solve1d_ctx* x = (solve1d_ctx*)c; return mg1d_vcycle(x->mg, x->level, x->v1, x->v2); }

int mg1d_solve(mg1d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles, int* cycles_out, int* converged_out,
               double* history)
{
    int st = check_level(mg, level);
    if (st) return st;
    if ((st = mg_solve_check_args(rtol, atol, max_cycles, v1, v2))) return st;
    solve1d_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = {&x, mg->stream, &mg->launches, NULL, s1_cycle, s1_cycle, s1_norm, mg->d_out2, NULL, NULL};
    const int key[MG_GRAPH_KEY] = {level, v1, v2};
    /* one launch per cycle: no bound on the sweep counts */
    return mg_solve_run(&mg->graphs, mg_graphs_on(&mg->graphs, mg->prof.enabled, 1) ? key : NULL, &ops, rtol, atol, max_cycles,
                        cycles_out, converged_out, history);
}

/* FullMultiGridVCycle (N1/MultiGrid1D.cpp:132-148): one launch */
int mg1d_fmg(mg1d_t* mg, int level, int v0, int v1, int v2)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (v0 < 0 || v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative cycle/sweep count");
    PROF_BEGIN(mg, level, MG_OP_OTHER);
    MG_LAUNCH(mg->launches, mgk1d_cycle(mg->stream, mg->dtype, mg->arena, mg->H, level, v0, v1, v2, mg->mode == MG_CORRECTED, 1));
    PROF_END(mg);
    return MG_OK;
}

/* ---- reference-facing operators on HOST arrays (N1/MultiGrid1D.h:16-22) ---------------------- */

static int up(mg1d_t* mg, void** d, const void* h, int n)
{
    MG_CUDA(cudaMalloc(d, (size_t)n * mg_esize(mg->dtype)));
    if (h) MG_CUDA(cudaMemcpyAsync(*d, h, (size_t)n * mg_esize(mg->dtype), cudaMemcpyHostToDevice, mg->stream));
    return MG_OK;
}

static int down(mg1d_t* mg, void* h, const void* d, int n)
{
    MG_CUDA(cudaMemcpyAsync(h, d, (size_t)n * mg_esize(mg->dtype), cudaMemcpyDeviceToHost, mg->stream));
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    return MG_OK;
}

int mg1d_restrict_host(mg1d_t* mg, const void* fine, int fn, void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N1/MultiGrid1D.cpp:36 */
    void *df = NULL, *dc = NULL;
    int st = up(mg, &df, fine, fn);
    if (!st) st = up(mg, &dc, NULL, cn);
    if (!st) {
        int k = mgk1d_restrict(mg->stream, mg->dtype, df, fn, dc, cn);
        if (k < 0) st = mg_fail(MG_ERR_CUDA, "restrict launch failed"); else mg->launches += k;
    }
    if (!st) st = down(mg, coarse, dc, cn);
    cudaFree(df); cudaFree(dc);
    return st;
}

int mg1d_interpolate_host(mg1d_t* mg, void* fine, int fn, const void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N1/MultiGrid1D.cpp:62 */
    void *df = NULL, *dc = NULL;
    int st = up(mg, &df, fine, fn);
    if (!st) st = up(mg, &dc, coarse, cn);
    if (!st) {
        int k = mgk1d_interpolate(mg->stream, mg->dtype, df, fn, dc, cn, 0);
        if (k < 0) st = mg_fail(MG_ERR_CUDA, "interpolate launch failed"); else mg->launches += k;
    }
    if (!st) st = down(mg, fine, df, fn);
    cudaFree(df); cudaFree(dc);
    return st;
}

int mg1d_apply_correction_host(mg1d_t* mg, void* fine, int fn, const void* error, int en)
{
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn != en || fn < 3) return mg_fail(MG_ERR_ARG, "fsize != esize"); /* N1/MultiGrid1D.cpp:179 */
    void *df = NULL, *de = NULL;
    int st = up(mg, &df, fine, fn);
    if (!st) st = up(mg, &de, error, en);
    if (!st) {
        int k = mgk1d_apply_correction(mg->stream, mg->dtype, df, de, fn);
        if (k < 0) st = mg_fail(MG_ERR_CUDA, "apply_correction launch failed"); else mg->launches += k;
    }
    if (!st) st = down(mg, fine, df, fn);
    cudaFree(df); cudaFree(de);
    return st;
}

int mg1d_set_to_value_host(mg1d_t* mg, void* grid, int n, double value, int modify_boundaries)
{
    if (!mg || !grid || n < 1) return mg_fail(MG_ERR_ARG, "bad argument");
    void* d = NULL;
    int st = up(mg, &d, grid, n);
    if (!st) {
        int k = mgk1d_set(mg->stream, mg->dtype, d, n, value, modify_boundaries);
        if (k < 0) st = mg_fail(MG_ERR_CUDA, "set launch failed"); else mg->launches += k;
    }
    if (!st) st = down(mg, grid, d, n);
    cudaFree(d);
    return st;
}

/* ---- the CUDA_TESI faces (C1/MultiGrid1D.h:16-23, C1/Grid1D.h:15-18): operators on DEVICE arrays.  The engine's 1D fields
        are dense device arrays already, so a level's d_v / d_f are the engine's own storage. ------------------------- */
int mg1d_level_device_ptr(mg1d_t* mg, int level, int field, void** ptr)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (!ptr || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    const long long off = field == MG_FIELD_V ? mg->H.off_v[level] : mg->H.off_f[level];
    *ptr = (char*)mg->arena + (size_t)off * mg_esize(mg->dtype);
    return MG_OK;
}

static int dev1_done(mg1d_t* mg, int k)
{
    if (k < 0) return mg_fail(MG_ERR_CUDA, "operator launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    mg->launches += k;
    MG_CUDA(cudaStreamSynchronize(mg->stream));
    return MG_OK;
}

int mg1d_restrict_device(mg1d_t* mg, const void* fine, int fn, void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize());
    return dev1_done(mg, mgk1d_restrict(mg->stream, mg->dtype, fine, fn, coarse, cn));
}

int mg1d_interpolate_device(mg1d_t* mg, void* fine, int fn, const void* coarse, int cn)
{
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn < 3 || cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize());
    return dev1_done(mg, mgk1d_interpolate(mg->stream, mg->dtype, fine, fn, coarse, cn, 0));
}

int mg1d_apply_correction_device(mg1d_t* mg, void* fine, int fn, const void* error, int en)
{
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if (fn != en || fn < 1) return mg_fail(MG_ERR_ARG, "fsize != esize");
    MG_CUDA(cudaDeviceSynchronize());
    return dev1_done(mg, mgk1d_apply_correction(mg->stream, mg->dtype, fine, error, fn));
}

int mg1d_set_device(mg1d_t* mg, void* d_v, int n, double value, int modify_boundaries)
{
    if (!mg || !d_v || n < 1) return mg_fail(MG_ERR_ARG, "bad argument");
    MG_CUDA(cudaDeviceSynchronize());
    return dev1_done(mg, mgk1d_set(mg->stream, mg->dtype, d_v, n, value, modify_boundaries));
}

/* CalculateResidual(grid) into a caller-owned DEVICE array (C1/MultiGrid1D.cu:86-104) */
int mg1d_residual_device(mg1d_t* mg, int level, void* dev_out)
{
    int st = check_level(mg, level);
    if (st) return st;
    if (!dev_out) return mg_fail(MG_ERR_ARG, "null output");
    MG_CUDA(cudaDeviceSynchronize());
    return dev1_done(mg, mgk1d_residual(mg->stream, mg->dtype, mg->arena, mg->H, level, mg->mode == MG_CORRECTED, dev_out));
}

int mg1d_vcycle_host(mg1d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles)
{
    if (!mg || !v_host || !f_host) return mg_fail(MG_ERR_ARG, "null argument");
    if (v1 < 0 || v2 < 0 || cycles < 0) return mg_fail(MG_ERR_ARG, "negative count");
    const size_t bytes = (size_t)mg->H.n[0] * mg_esize(mg->dtype);
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, 0, MG_FIELD_V), v_host, bytes, cudaMemcpyHostToDevice, mg->stream));
    MG_CUDA(cudaMemcpyAsync(field_ptr(mg, 0, MG_FIELD_F), f_host, bytes, cudaMemcpyHostToDevice, mg->stream));
    MG_LAUNCH(mg->launches, mgk1d_cycle(mg->stream, mg->dtype, mg->arena, mg->H, 0, cycles, v1, v2, mg->mode == MG_CORRECTED, 0));
    return down(mg, v_host, field_ptr(mg, 0, MG_FIELD_V), mg->H.n[0]);
}

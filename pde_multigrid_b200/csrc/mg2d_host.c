/*
 * mg2d_host.c -- C host driver of the 2D Lyapunov multigrid (first-order upwind PDE
 * K1 V_x + K2 V_y + alfa V = f, K = A x): hierarchy, V-cycle, FMG, field I/O.
 *
 * Mirrors the reference class MultiGrid2D (NOCUDA_TESI/PDE Lyapunov 2D/MultiGrid2D.cpp: InitGrids
 * :20-42, InitA :45-60, VCycle :314-340, FullMultiGridVCycle :296-312) over the kernels of
 * mg2d_kernels.cu.  No CPU compute path: the host only derives h per level.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mg_host_common.h"

typedef struct {
    mg_geom2d g;
    mg_coef2d c;
    void* v;
    void* f;
} mg_level2d;

/* core.graphs holds the V-cycle graphs keyed (level, v1, v2): at 1025^2 a V(2,2) is ~60 dependent launches on L2-resident
   fields, i.e. pure launch latency */
struct mg2d_s {
    mg_core core;
    mg_level2d* lv;
    void* arena;
    double* d_scratch; /* 2*1184 partials + 2 outputs */
};

#define SCRATCH_PARTS 1184

static size_t field_bytes2(const mg_geom2d* g, int dtype) { return mg_align256((size_t)g->pitch * g->n * mg_esize(dtype)); }

static void* field_ptr(mg_level2d* L, int field) { return field == MG_FIELD_V ? L->v : L->f; }

/* h = range/(real)(n-1) in the level's precision, N2/Grid2D.cpp:24-35 */
static void level_coefs(int dtype, int n, const double* range, const double* A4, int alfa, mg_coef2d* c)
{
    if (dtype == MG_F32) {
        float xr = (float)range[1] - (float)range[0], yr = (float)range[3] - (float)range[2];
        c->hx = xr / (float)(n - 1);
        c->hy = yr / (float)(n - 1);
        c->xa = (float)range[0];
        c->ya = (float)range[2];
        for (int i = 0; i < 4; i++) c->A[i] = (float)A4[i];
    } else {
        double xr = range[1] - range[0], yr = range[3] - range[2];
        c->hx = xr / (double)(n - 1);
        c->hy = yr / (double)(n - 1);
        c->xa = range[0];
        c->ya = range[2];
        for (int i = 0; i < 4; i++) c->A[i] = A4[i];
    }
    c->alfa = alfa;
}

int mg2d_create(mg2d_t** out, const int sz[2], const double range[4], const double A4[4], int alfa, int dtype)
{
    if (!out || !sz || !range || !A4) return mg_fail(MG_ERR_ARG, "null argument");
    *out = NULL;
    if (sz[0] != sz[1]) return mg_fail(MG_ERR_ARG, "sizeX == sizeY required (got %d,%d)", sz[0], sz[1]); /* N2/Grid2D.cpp:9 */
    const int n = sz[0];
    if (n < 3 || ((n - 1) & (n - 2)) != 0) return mg_fail(MG_ERR_ARG, "size must be 2^k+1 with k >= 1 (got %d)", n);
    if (!(range[1] > range[0]) || !(range[3] > range[2])) return mg_fail(MG_ERR_ARG, "range must satisfy b > a on every axis");
    if (dtype != MG_F32 && dtype != MG_F64) return mg_fail(MG_ERR_ARG, "dtype must be MG_F32 or MG_F64");
    int st = mg_require_device();
    if (st) return st;
    mg2d_t* mg = (mg2d_t*)calloc(1, sizeof *mg);
    if (!mg) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    mg->core.dtype = dtype;
    mg->core.nlevels = mg_num_levels_for(n);
    mg->lv = (mg_level2d*)calloc((size_t)mg->core.nlevels, sizeof(mg_level2d));
    if (!mg->lv) { free(mg); return mg_fail(MG_ERR_NOMEM, "host allocation failed"); }
    size_t total = 0;
    int nl = n;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level2d* L = &mg->lv[l];
        L->g.n = nl;
        L->g.pitch = mg_pitch(nl, dtype);
        level_coefs(dtype, nl, range, A4, alfa, &L->c);
        total += 2 * field_bytes2(&L->g, dtype);
        nl = (nl - 1) / 2 + 1;
    }
    if ((st = mg_core_init(&mg->core))) { mg2d_destroy(mg); return st; }
    cudaError_t e = cudaMalloc(&mg->arena, total);
    if (e != cudaSuccess) {
        mg2d_destroy(mg);
        return mg_fail(e == cudaErrorMemoryAllocation ? MG_ERR_NOMEM : MG_ERR_CUDA, "cudaMalloc of %zu bytes failed: %s", total, cudaGetErrorString(e));
    }
    char* p = (char*)mg->arena;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level2d* L = &mg->lv[l];
        L->v = p; p += field_bytes2(&L->g, dtype);
        L->f = p; p += field_bytes2(&L->g, dtype);
    }
    if (cudaMalloc((void**)&mg->d_scratch, (2 * SCRATCH_PARTS + 2) * sizeof(double)) != cudaSuccess ||
        cudaMemsetAsync(mg->arena, 0, total, mg->core.stream) != cudaSuccess) {
        int code = mg_fail(MG_ERR_CUDA, "stream/scratch setup failed: %s", cudaGetErrorString(cudaGetLastError()));
        mg2d_destroy(mg);
        return code;
    }
    st = mg2d_init_problem(mg);
    if (st) { mg2d_destroy(mg); return st; }
    *out = mg;
    return MG_OK;
}

int mg2d_destroy(mg2d_t* mg)
{
    if (!mg) return MG_OK;
    mg_core_free(&mg->core);
    if (mg->arena) cudaFree(mg->arena);
    if (mg->d_scratch) cudaFree(mg->d_scratch);
    free(mg->lv);
    free(mg);
    return MG_OK;
}

int mg2d_num_levels(const mg2d_t* mg) { return mg ? mg->core.nlevels : 0; }
int mg2d_level_size(const mg2d_t* mg, int level) { return (mg && level >= 0 && level < mg->core.nlevels) ? mg->lv[level].g.n : 0; }
double mg2d_level_h(const mg2d_t* mg, int level) { return (mg && level >= 0 && level < mg->core.nlevels) ? mg->lv[level].c.hx : 0.0; }
void* mg2d_stream(mg2d_t* mg) { return mg ? (void*)mg->core.stream : NULL; }
long long mg2d_kernel_launches(const mg2d_t* mg) { return mg ? mg->core.launches : 0; }

int mg2d_sync(mg2d_t* mg) { return mg_sync(MG_CORE(mg)); }
int mg2d_profile(mg2d_t* mg, int enable) { return mg_profile_enable(MG_CORE(mg), enable); }
int mg2d_profile_read(mg2d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls)
{
    return mg_profile_read(MG_CORE(mg), level, op, ms_total, kernel_launches, calls);
}

static int copy_in(mg2d_t* mg, void* dev, const mg_geom2d* g, const void* host)
{
    size_t es = mg_esize(mg->core.dtype);
    MG_CUDA(cudaMemcpy2DAsync(dev, (size_t)g->pitch * es, host, (size_t)g->n * es, (size_t)g->n * es, (size_t)g->n,
                              cudaMemcpyHostToDevice, mg->core.stream));
    return MG_OK;
}

static int copy_out(mg2d_t* mg, void* host, const void* dev, const mg_geom2d* g)
{
    size_t es = mg_esize(mg->core.dtype);
    MG_CUDA(cudaMemcpy2DAsync(host, (size_t)g->n * es, dev, (size_t)g->pitch * es, (size_t)g->n * es, (size_t)g->n,
                              cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg2d_set_field(mg2d_t* mg, int level, int field, const void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    st = copy_in(mg, field_ptr(&mg->lv[level], field), &mg->lv[level].g, host_dense);
    if (st) return st;
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg2d_get_field(mg2d_t* mg, int level, int field, void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    return copy_out(mg, host_dense, field_ptr(&mg->lv[level], field), &mg->lv[level].g);
}

/* Grid2D::InitV / InitF on every level, N2/Grid2D.cpp:50-80 */
int mg2d_init_problem(mg2d_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level2d* L = &mg->lv[l];
        MG_LAUNCH(mg->core.launches, mgk2d_init_v(mg->core.stream, mg->core.dtype, L->v, L->g, L->c));
        MG_LAUNCH(mg->core.launches, mgk2d_set(mg->core.stream, mg->core.dtype, L->f, L->g, 0.0, 1));
    }
    return MG_OK;
}

/* Relax, N2/MultiGrid2D.cpp:199-273 */
static int relax_level(mg2d_t* mg, int level, int ncycles)
{
    mg_level2d* L = &mg->lv[level];
    if (ncycles <= 0) return MG_OK;
    PROF_BEGIN(mg, level, MG_OP_RELAX);
    if (L->g.n <= MGK2D_SMALL_N) { /* the whole level fits in one CTA: every sweep in a single launch */
        MG_LAUNCH(mg->core.launches, mgk2d_relax_small(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, ncycles));
    } else {
        for (int k = 0; k < ncycles; k++)
            for (int colour = 0; colour < 2; colour++)
                MG_LAUNCH(mg->core.launches, mgk2d_relax_colour(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, colour));
    }
    PROF_END(mg);
    return MG_OK;
}

int mg2d_relax(mg2d_t* mg, int level, int ncycles)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (ncycles < 0) return mg_fail(MG_ERR_ARG, "ncycles < 0");
    return relax_level(mg, level, ncycles);
}

int mg2d_residual(mg2d_t* mg, int level, void* host_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_out) return mg_fail(MG_ERR_ARG, "null output");
    mg_level2d* L = &mg->lv[level];
    void* r = NULL;
    MG_CUDA(cudaMalloc(&r, field_bytes2(&L->g, mg->core.dtype)));
    int k = mgk2d_residual(mg->core.stream, mg->core.dtype, L->v, L->f, r, L->g, L->c);
    if (k < 0) { cudaFree(r); return mg_fail(MG_ERR_CUDA, "residual launch failed"); }
    mg->core.launches += k;
    st = copy_out(mg, host_out, r, &L->g);
    cudaFree(r);
    return st;
}

/* the norm pass of mg2d_residual_norm: {sum of r^2, max |r|} into d_scratch + 2*SCRATCH_PARTS, nothing read back */
static int residual_norm_enqueue(mg2d_t* mg, int level)
{
    mg_level2d* L = &mg->lv[level];
    MG_LAUNCH(mg->core.launches, mgk2d_residual_norm(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, mg->d_scratch, mg->d_scratch + 2 * SCRATCH_PARTS));
    return MG_OK;
}

int mg2d_residual_norm(mg2d_t* mg, int level, double* l2, double* linf)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if ((st = residual_norm_enqueue(mg, level))) return st;
    return mg_read_norm(&mg->core, mg->d_scratch + 2 * SCRATCH_PARTS, l2, linf);
}

int mg2d_mean_abs_error(mg2d_t* mg, double* mae)
{
    if (!mg || !mae) return mg_fail(MG_ERR_ARG, "null argument");
    mg_level2d* L = &mg->lv[0];
    MG_LAUNCH(mg->core.launches, mgk2d_abs_error_sum(mg->core.stream, mg->core.dtype, L->v, L->g, L->c, mg->d_scratch, mg->d_scratch + 2 * SCRATCH_PARTS));
    int st = mg_read_out2(&mg->core, mg->d_scratch + 2 * SCRATCH_PARTS);
    if (st) return st;
    long long ni = (long long)(L->g.n - 2) * (L->g.n - 2); /* interior points only, C2/Grid2D.cu:130-148 */
    *mae = ni > 0 ? mg->core.h_out2[0] / (double)ni : 0.0;
    return MG_OK;
}

int mg2d_restrict(mg2d_t* mg, int fine_level, int field)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level2d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    MG_LAUNCH(mg->core.launches, mgk2d_restrict(mg->core.stream, mg->core.dtype, field_ptr(F, field), F->g, field_ptr(C, field), C->g));
    return MG_OK;
}

static int residual_restrict_level(mg2d_t* mg, int level)
{
    mg_level2d *F = &mg->lv[level], *C = &mg->lv[level + 1];
    PROF_BEGIN(mg, level, MG_OP_RESIDUAL_RESTRICT);
    MG_LAUNCH(mg->core.launches, mgk2d_residual_restrict(mg->core.stream, mg->core.dtype, F->v, F->f, F->g, F->c, C->f, C->v, C->g));
    PROF_END(mg);
    return MG_OK;
}

int mg2d_residual_restrict(mg2d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return residual_restrict_level(mg, fine_level);
}

static int interpolate_level(mg2d_t* mg, int fine_level, int add)
{
    mg_level2d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    PROF_BEGIN(mg, fine_level, MG_OP_INTERPOLATE);
    MG_LAUNCH(mg->core.launches, mgk2d_interpolate(mg->core.stream, mg->core.dtype, F->v, F->g, C->v, C->g, add));
    PROF_END(mg);
    return MG_OK;
}

int mg2d_interpolate(mg2d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 0);
}

int mg2d_interpolate_correct(mg2d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 1);
}

int mg2d_set_to_value(mg2d_t* mg, int level, int field, double value, int modify_boundaries)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level2d* L = &mg->lv[level];
    MG_LAUNCH(mg->core.launches, mgk2d_set(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, value, modify_boundaries));
    return MG_OK;
}

/* VCycle, N2/MultiGrid2D.cpp:314-340 */
static int vcycle_rec(mg2d_t* mg, int level, int v1, int v2)
{
    int st = relax_level(mg, level, v1);
    if (st) return st;
    if (level != mg->core.nlevels - 1) {
        if ((st = residual_restrict_level(mg, level))) return st;
        if ((st = vcycle_rec(mg, level + 1, v1, v2))) return st;
        if ((st = interpolate_level(mg, level, 1))) return st;
    }
    return relax_level(mg, level, v2);
}

/* one cycle on `level` with fixed sweep counts, as the graph cache (mg_host_common.c) runs, captures and replays it */
static int c2_cycle(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return vcycle_rec(x->h, x->level, x->v1, x->v2); }
static int c2_public(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return mg2d_vcycle(x->h, x->level, x->v1, x->v2); }
static int c2_norm(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return residual_norm_enqueue(x->h, x->level); }

static mg_cycle_ops cycle_ops(mg_cycle_ctx* x)
{
    mg2d_t* mg = x->h;
    const mg_cycle_ops ops = {x, mg->core.stream, &mg->core.launches, NULL, c2_cycle, c2_public, c2_norm, mg->d_scratch + 2 * SCRATCH_PARTS, NULL, NULL};
    return ops;
}

/* graphs for cycles of up to MG_GRAPH_MAX_LAUNCHES launches */
static int graphs_on(const mg2d_t* mg, int level, int v1, int v2)
{
    return mg_graphs_on(&mg->core.graphs, mg->core.prof.enabled, 2LL * (v1 + v2) * (mg->core.nlevels - level));
}

int mg2d_vcycle(mg2d_t* mg, int level, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = cycle_ops(&x);
    const int key[MG_GRAPH_KEY] = {level, v1, v2};
    return mg_graph_cycle(&mg->core.graphs, graphs_on(mg, level, v1, v2) ? key : NULL, &ops);
}

int mg2d_solve(mg2d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles, int* cycles_out, int* converged_out,
               double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_cycles, v1, v2);
    if (st) return st;
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = cycle_ops(&x);
    const int key[MG_GRAPH_KEY] = {level, v1, v2};
    return mg_solve_run(&mg->core.graphs, graphs_on(mg, level, v1, v2) ? key : NULL, &ops, rtol, atol, max_cycles, cycles_out,
                        converged_out, history);
}

/* FullMultiGridVCycle, N2/MultiGrid2D.cpp:296-312 */
static int fmg_rec(mg2d_t* mg, int level, int v0, int v1, int v2)
{
    int st;
    if (level != mg->core.nlevels - 1) {
        mg_level2d *F = &mg->lv[level], *C = &mg->lv[level + 1];
        MG_LAUNCH(mg->core.launches, mgk2d_restrict(mg->core.stream, mg->core.dtype, F->f, F->g, C->f, C->g));
        if ((st = fmg_rec(mg, level + 1, v0, v1, v2))) return st;
        if ((st = interpolate_level(mg, level, 0))) return st;
    } else {
        mg_level2d* L = &mg->lv[level];
        MG_LAUNCH(mg->core.launches, mgk2d_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 0));
    }
    for (int i = 0; i < v0; i++)
        if ((st = vcycle_rec(mg, level, v1, v2))) return st;
    return MG_OK;
}

int mg2d_fmg(mg2d_t* mg, int level, int v0, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v0 < 0 || v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative cycle/sweep count");
    return fmg_rec(mg, level, v0, v1, v2);
}

/* ---- reference-facing operators on HOST arrays (N2/MultiGrid2D.h:21-27) ---------------------- */

static int square(const int s[2], int* n)
{
    if (!s || s[0] != s[1] || s[0] < 3) return mg_fail(MG_ERR_ARG, "square size >= 3 required");
    *n = s[0];
    return MG_OK;
}

/* dense temporaries: the 2D kernels take any pitch >= size */
int mg2d_restrict_host(mg2d_t* mg, const void* fine, const int fs[2], void* coarse, const int cs[2])
{
    int fn = 0, cn = 0, st;
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = square(fs, &fn)) || (st = square(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N2/MultiGrid2D.cpp:71-72 */
    const mg_geom2d gf = {fn, fn}, gc = {cn, cn};
    void *df, *dc;
    if ((st = mg_tmp_begin(&mg->core, &df, (size_t)fn * fn, fine, &dc, (size_t)cn * cn, NULL))) return st;
    return mg_tmp_finish(&mg->core, mgk2d_restrict(mg->core.stream, mg->core.dtype, df, gf, dc, gc), coarse, dc, (size_t)cn * cn, df, dc);
}

int mg2d_interpolate_host(mg2d_t* mg, void* fine, const int fs[2], const void* coarse, const int cs[2])
{
    int fn = 0, cn = 0, st;
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = square(fs, &fn)) || (st = square(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N2/MultiGrid2D.cpp:136-137 */
    const mg_geom2d gf = {fn, fn}, gc = {cn, cn};
    void *df, *dc;
    if ((st = mg_tmp_begin(&mg->core, &df, (size_t)fn * fn, fine, &dc, (size_t)cn * cn, coarse))) return st;
    return mg_tmp_finish(&mg->core, mgk2d_interpolate(mg->core.stream, mg->core.dtype, df, gf, dc, gc, 0), fine, df, (size_t)fn * fn, df, dc);
}

int mg2d_apply_correction_host(mg2d_t* mg, void* fine, const int fs[2], const void* error, const int es[2])
{
    int fn = 0, en = 0, st;
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = square(fs, &fn)) || (st = square(es, &en))) return st;
    if (fn != en) return mg_fail(MG_ERR_ARG, "fsize != esize"); /* N2/MultiGrid2D.cpp:351-352 */
    const mg_geom2d g = {fn, fn};
    void *df, *de;
    if ((st = mg_tmp_begin(&mg->core, &df, (size_t)fn * fn, fine, &de, (size_t)fn * fn, error))) return st;
    return mg_tmp_finish(&mg->core, mgk2d_apply_correction(mg->core.stream, mg->core.dtype, df, de, g), fine, df, (size_t)fn * fn, df, de);
}

int mg2d_set_to_value_host(mg2d_t* mg, void* grid, const int s[2], double value, int modify_boundaries)
{
    int n = 0, st;
    if (!mg || !grid) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = square(s, &n))) return st;
    const mg_geom2d g = {n, n};
    void *d, *unused;
    if ((st = mg_tmp_begin(&mg->core, &d, (size_t)n * n, grid, &unused, 0, NULL))) return st;
    return mg_tmp_finish(&mg->core, mgk2d_set(mg->core.stream, mg->core.dtype, d, g, value, modify_boundaries), grid, d, (size_t)n * n, d, NULL);
}

/* ---- the CUDA_TESI faces (C2/MultiGrid2D.h:20-25, C2/Grid2D.h:19-22): operators on pitched DEVICE arrays given as
        (pointer, size, pitch in elements).  The engine's own 2D layout is pitched as well, so the kernels run on the
        caller's arrays in place, and a level's fields can be handed out without a copy. ---------------------------------- */
int mg2d_level_device_ptr(mg2d_t* mg, int level, int field, void** ptr, int* pitch_elems)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!ptr || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    *ptr = field == MG_FIELD_V ? mg->lv[level].v : mg->lv[level].f;
    if (pitch_elems) *pitch_elems = mg->lv[level].g.pitch;
    return MG_OK;
}

static int dev2_args(mg2d_t* mg, const void* a, int an, int ap, const void* b, int bn, int bp, int need_b)
{
    if (!mg || !a || (need_b && !b)) return mg_fail(MG_ERR_ARG, "null argument");
    if (an < 3 || ap < an || (need_b && (bn < 3 || bp < bn))) return mg_fail(MG_ERR_ARG, "size >= 3 and pitch >= size required");
    MG_CUDA(cudaDeviceSynchronize()); /* the caller's arrays may have been produced on any stream */
    return MG_OK;
}

int mg2d_restrict_device(mg2d_t* mg, const void* fine, int fsize, int f_pitch, void* coarse, int csize, int c_pitch)
{
    int st = dev2_args(mg, fine, fsize, f_pitch, coarse, csize, c_pitch, 1);
    if (st) return st;
    if (csize != (fsize - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    mg_geom2d gf = {fsize, f_pitch}, gc = {csize, c_pitch};
    return mg_launch_done(&mg->core, mgk2d_restrict(mg->core.stream, mg->core.dtype, fine, gf, coarse, gc));
}

int mg2d_interpolate_device(mg2d_t* mg, void* fine, int fsize, int f_pitch, const void* coarse, int csize, int c_pitch)
{
    int st = dev2_args(mg, fine, fsize, f_pitch, coarse, csize, c_pitch, 1);
    if (st) return st;
    if (csize != (fsize - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    mg_geom2d gf = {fsize, f_pitch}, gc = {csize, c_pitch};
    return mg_launch_done(&mg->core, mgk2d_interpolate(mg->core.stream, mg->core.dtype, fine, gf, coarse, gc, 0));
}

int mg2d_apply_correction_device(mg2d_t* mg, void* fine, int fsize, int f_pitch, const void* error, int esize, int e_pitch)
{
    int st = dev2_args(mg, fine, fsize, f_pitch, error, esize, e_pitch, 1);
    if (st) return st;
    if (fsize != esize || f_pitch != e_pitch) return mg_fail(MG_ERR_ARG, "fine and error must have the same size and pitch");
    mg_geom2d g = {fsize, f_pitch};
    return mg_launch_done(&mg->core, mgk2d_apply_correction(mg->core.stream, mg->core.dtype, fine, error, g));
}

int mg2d_set_device(mg2d_t* mg, void* v, int size, int pitch, double value, int modify_border)
{
    int st = dev2_args(mg, v, size, pitch, NULL, 0, 0, 0);
    if (st) return st;
    mg_geom2d g = {size, pitch};
    return mg_launch_done(&mg->core, mgk2d_set(mg->core.stream, mg->core.dtype, v, g, value, modify_border));
}

/* CalculateResidual(grid) into a caller-owned pitched DEVICE array with the level's own pitch (C2/MultiGrid2D.cu:105-127) */
int mg2d_residual_device(mg2d_t* mg, int level, void* dev_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!dev_out) return mg_fail(MG_ERR_ARG, "null output");
    mg_level2d* L = &mg->lv[level];
    MG_CUDA(cudaDeviceSynchronize());
    return mg_launch_done(&mg->core, mgk2d_residual(mg->core.stream, mg->core.dtype, L->v, L->f, dev_out, L->g, L->c));
}

int mg2d_vcycle_host(mg2d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles)
{
    if (!mg || !v_host || !f_host) return mg_fail(MG_ERR_ARG, "null argument");
    if (v1 < 0 || v2 < 0 || cycles < 0) return mg_fail(MG_ERR_ARG, "negative count");
    mg_level2d* L = &mg->lv[0];
    int st = copy_in(mg, L->v, &L->g, v_host);
    if (!st) st = copy_in(mg, L->f, &L->g, f_host);
    for (int i = 0; i < cycles && !st; i++) st = vcycle_rec(mg, 0, v1, v2);
    if (!st) st = copy_out(mg, v_host, L->v, &L->g);
    return st;
}

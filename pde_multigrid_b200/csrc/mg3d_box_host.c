/*
 * mg3d_box_host.c -- C host driver of the 3D Poisson multigrid on NON-CUBIC grids (mg3b_* in include/mg_b200.h).
 *
 * The reference's constructor takes three sizes (MultiGrid3D(int finestGridSizeXYZ[], float range[]),
 * N3/MultiGrid3D.cpp:5-8) and its hierarchy is already written per dimension -- numGrids = (int)log2(minSize - 1),
 * every dimension halved per level (InitGrids, :19-47) -- but Grid3D asserts sizeX == sizeY == sizeZ
 * (N3/Grid3D.cpp:10-11; lifting that is the author's own TODO, SURVEY.md 8f rank 4).  This driver mirrors the same
 * control flow (VCycle :623-647, FullMultiGridVCycle :569-585) over the kernels of mg3d_box.cu.  The coarsest level of
 * an anisotropic hierarchy has more than one unknown (e.g. 9 x 5 x 3): like the reference it gets v1 + v2 sweeps.
 * Fields live on the device colour-split like the cubic engine's (mg3d_box.h); set/get repack through a dense staging field.
 * No CPU compute path.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mg_host_common.h"

#include "mg3d_box.h"

#define MG3B_NPARTS 1024

typedef struct {
    int n[3];
    mg_geom3b g;   /* colour-split device layout of the level's fields */
    mg_coef3d c;
    double h[3];
    void* v;
    void* f;
} mg_level3b;

struct mg3b_s {
    mg_core core;      /* core.graphs holds the mg3b_solve graphs */
    int mode;
    double range[6];
    mg_level3b* lv;
    void* arena;
    void* staging;     /* one dense field of the finest level: host <-> device copies pass through it (repack) */
    double* d_scratch; /* 2 * MG3B_NPARTS partials + 2 outputs */
    double* d_tables;  /* sin tables of InitF: nx + ny + nz doubles of the finest level */
    mg_pcg_vecs* pcg;  /* per level, allocated by the first mg3b_pcg of the level */
};

static size_t level_count(const mg_level3b* L) { return (size_t)L->n[0] * (size_t)L->n[1] * (size_t)L->n[2]; }
static size_t field_bytes(const mg_level3b* L, int dtype) { return mg_align256(2 * (size_t)L->g.cstride * mg_esize(dtype)); }
static void set_geom3b(mg_geom3b* g, const int n[3], int dtype)
{
    g->nx = n[0]; g->ny = n[1]; g->nz = n[2];
    g->hp = mg_pitch((n[0] + 1) / 2, dtype);
    g->plane = (long long)g->hp * n[1];
    g->cstride = g->plane * n[2];
}

/* h = range/(real)(size-1) per axis (N3/Grid3D.cpp:31-45) and the products of N3/MultiGrid3D.cpp:498-500, :532, in the level's
   own precision exactly like the reference computes them on the host */
static void box_coefs(int dtype, const int n[3], const double* range, double h[3], mg_coef3d* c)
{
    memset(c, 0, sizeof *c);
    if (dtype == MG_F32) {
        float xr = (float)range[1] - (float)range[0], yr = (float)range[3] - (float)range[2], zr = (float)range[5] - (float)range[4];
        float hx = xr / (float)(n[0] - 1), hy = yr / (float)(n[1] - 1), hz = zr / (float)(n[2] - 1);
        float hx2 = hx * hx, hy2 = hy * hy, hz2 = hz * hz;
        float cx = hy2 * hz2, cy = hx2 * hz2, cz = hx2 * hy2;
        float den = 2 * (cx + cy + cz);
        h[0] = hx; h[1] = hy; h[2] = hz;
        c->hx2 = hx2; c->hy2 = hy2; c->hz2 = hz2;
        c->cx = cx; c->cy = cy; c->cz = cz;
        c->den = den; c->rden = 1.0f / den;
        c->ihx2 = 1.0f / hx2; c->ihy2 = 1.0f / hy2; c->ihz2 = 1.0f / hz2;
    } else {
        double xr = range[1] - range[0], yr = range[3] - range[2], zr = range[5] - range[4];
        double hx = xr / (double)(n[0] - 1), hy = yr / (double)(n[1] - 1), hz = zr / (double)(n[2] - 1);
        double hx2 = hx * hx, hy2 = hy * hy, hz2 = hz * hz;
        double cx = hy2 * hz2, cy = hx2 * hz2, cz = hx2 * hy2;
        double den = 2 * (cx + cy + cz);
        h[0] = hx; h[1] = hy; h[2] = hz;
        c->hx2 = hx2; c->hy2 = hy2; c->hz2 = hz2;
        c->cx = cx; c->cy = cy; c->cz = cz;
        c->den = den; c->rden = 1.0 / den;
        c->ihx2 = 1.0 / hx2; c->ihy2 = 1.0 / hy2; c->ihz2 = 1.0 / hz2;
    }
    /* three different mesh widths: the smoother's divisor is not of the 6*2^e form, IEEE division there; the residual's x / h^2
       becomes the exact x * (1/h^2) when every h^2 is a power of two (mg_exact.cuh) */
    int e;
    c->fast_den = 0;
    c->fast_h = frexp(c->hx2, &e) == 0.5 && frexp(c->hy2, &e) == 0.5 && frexp(c->hz2, &e) == 0.5;
}

static int pow2_plus_1(int n)
{
    if (n < 3) return 0;
    int m = n - 1;
    return (m & (m - 1)) == 0;
}

int mg3b_destroy(mg3b_t* mg)
{
    if (!mg) return MG_OK;
    mg_core_free(&mg->core);
    if (mg->arena) cudaFree(mg->arena);
    if (mg->staging) cudaFree(mg->staging);
    if (mg->d_scratch) cudaFree(mg->d_scratch);
    if (mg->d_tables) cudaFree(mg->d_tables);
    for (int l = 0; mg->pcg && l < mg->core.nlevels; l++) mg_pcg_vecs_free(&mg->pcg[l]);
    free(mg->pcg);
    free(mg->lv);
    free(mg);
    return MG_OK;
}

int mg3b_create(mg3b_t** out, const int finest_size_xyz[3], const double range[6], int dtype, int residual_mode)
{
    if (!out || !finest_size_xyz) return mg_fail(MG_ERR_ARG, "null argument");
    *out = NULL;
    for (int a = 0; a < 3; a++)
        if (!pow2_plus_1(finest_size_xyz[a]))
            return mg_fail(MG_ERR_ARG, "size %d on axis %d is not 2^k + 1 (N3/Grid3D.cpp:13-20)", finest_size_xyz[a], a);
    if (dtype != MG_F32 && dtype != MG_F64) return mg_fail(MG_ERR_ARG, "bad dtype");
    if (residual_mode != MG_REF_COMPAT && residual_mode != MG_CORRECTED) return mg_fail(MG_ERR_ARG, "bad residual mode");
    static const double unit[6] = {0, 1, 0, 1, 0, 1};
    if (!range) range = unit;
    if (!(range[1] > range[0]) || !(range[3] > range[2]) || !(range[5] > range[4]))
        return mg_fail(MG_ERR_ARG, "empty range (N3/Grid3D.cpp:27-29)");
    int st = mg_require_device();
    if (st) return st;
    mg3b_t* mg = (mg3b_t*)calloc(1, sizeof *mg);
    if (!mg) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    mg->core.dtype = dtype;
    mg->mode = residual_mode;
    memcpy(mg->range, range, sizeof mg->range);
    int mn = finest_size_xyz[0];
    if (finest_size_xyz[1] < mn) mn = finest_size_xyz[1];
    if (finest_size_xyz[2] < mn) mn = finest_size_xyz[2];
    mg->core.nlevels = mg_num_levels_for(mn); /* numGrids = (int)log2(minSize - 1), N3/MultiGrid3D.cpp:24-34 */
    mg->lv = (mg_level3b*)calloc((size_t)mg->core.nlevels, sizeof *mg->lv);
    if (!mg->lv) { free(mg); return mg_fail(MG_ERR_NOMEM, "host allocation failed"); }
    size_t bytes = 0;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3b* L = &mg->lv[l];
        for (int a = 0; a < 3; a++) L->n[a] = l == 0 ? finest_size_xyz[a] : (mg->lv[l - 1].n[a] - 1) / 2 + 1;
        box_coefs(dtype, L->n, range, L->h, &L->c);
        set_geom3b(&L->g, L->n, dtype);
        bytes += 2 * field_bytes(L, dtype);
    }
#define MG3B_TRY(call)                                                                                                        \
    do {                                                                                                                      \
        cudaError_t e_ = (call);                                                                                              \
        if (e_ != cudaSuccess) {                                                                                              \
            mg3b_destroy(mg);                                                                                                 \
            return mg_fail(MG_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));                                      \
        }                                                                                                                     \
    } while (0)
    if ((st = mg_core_init(&mg->core))) { mg3b_destroy(mg); return st; }
    MG3B_TRY(cudaMalloc(&mg->arena, bytes));
    MG3B_TRY(cudaMemsetAsync(mg->arena, 0, bytes, mg->core.stream)); /* the row padding is never read for a result, but keep it defined */
    MG3B_TRY(cudaMalloc(&mg->staging, level_count(&mg->lv[0]) * mg_esize(dtype)));
    MG3B_TRY(cudaMalloc((void**)&mg->d_scratch, (2 * MG3B_NPARTS + 2) * sizeof(double)));
    MG3B_TRY(cudaMalloc((void**)&mg->d_tables, (size_t)(finest_size_xyz[0] + finest_size_xyz[1] + finest_size_xyz[2]) * sizeof(double)));
    char* p = (char*)mg->arena;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3b* L = &mg->lv[l];
        const size_t fb = field_bytes(L, dtype);
        L->v = p; p += fb;
        L->f = p; p += fb;
    }
    st = mg3b_init_problem(mg);
    if (st) { mg3b_destroy(mg); return st; }
    *out = mg;
    return MG_OK;
}

int mg3b_num_levels(const mg3b_t* mg) { return mg ? mg->core.nlevels : 0; }

int mg3b_level_size(const mg3b_t* mg, int level, int out_xyz[3])
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!out_xyz) return mg_fail(MG_ERR_ARG, "null output");
    memcpy(out_xyz, mg->lv[level].n, 3 * sizeof(int));
    return MG_OK;
}

int mg3b_level_h(const mg3b_t* mg, int level, double out_xyz[3])
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!out_xyz) return mg_fail(MG_ERR_ARG, "null output");
    memcpy(out_xyz, mg->lv[level].h, 3 * sizeof(double));
    return MG_OK;
}

int mg3b_sync(mg3b_t* mg) { return mg_sync(MG_CORE(mg)); }

void* mg3b_stream(mg3b_t* mg) { return mg ? (void*)mg->core.stream : NULL; }
long long mg3b_kernel_launches(const mg3b_t* mg) { return mg ? mg->core.launches : 0; }

/* Grid3D::InitV / InitF on every level (N3/Grid3D.cpp:61-96); the interior of v is zeroed as well (SURVEY.md App. B8).
   sin(PI x) with x = x_a + pos*h in the level's precision, evaluated by the host libm the reference calls. */
int mg3b_init_problem(mg3b_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    const double PI = 3.141592653589793;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3b* L = &mg->lv[l];
        const int tot = L->n[0] + L->n[1] + L->n[2];
        double* tab = (double*)malloc((size_t)tot * sizeof(double));
        if (!tab) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
        int o = 0;
        for (int a = 0; a < 3; a++)
            for (int i = 0; i < L->n[a]; i++) {
                double x;
                if (mg->core.dtype == MG_F32) {
                    float xf = (float)mg->range[2 * a] + i * (float)L->h[a];
                    x = xf;
                } else {
                    x = mg->range[2 * a] + i * L->h[a];
                }
                tab[o++] = sin(PI * x);
            }
        cudaError_t e = cudaMemcpyAsync(mg->d_tables, tab, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, mg->core.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
        free(tab);
        if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e));
        MG_LAUNCH(mg->core.launches, mgk3b_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 1));
        MG_LAUNCH(mg->core.launches, mgk3b_init_f(mg->core.stream, mg->core.dtype, L->f, L->g, mg->d_tables, mg->d_tables + L->n[0], mg->d_tables + L->n[0] + L->n[1]));
        MG_CUDA(cudaStreamSynchronize(mg->core.stream)); /* d_tables is reused by the next level */
    }
    return MG_OK;
}

static void* field_ptr(mg_level3b* L, int field) { return field == MG_FIELD_V ? L->v : L->f; }

int mg3b_set_field(mg3b_t* mg, int level, int field, const void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3b* L = &mg->lv[level];
    MG_CUDA(cudaMemcpyAsync(mg->staging, host_dense, level_count(L) * mg_esize(mg->core.dtype), cudaMemcpyHostToDevice, mg->core.stream));
    MG_LAUNCH(mg->core.launches, mgk3b_repack(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, mg->staging, 1));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg3b_get_field(mg3b_t* mg, int level, int field, void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3b* L = &mg->lv[level];
    MG_LAUNCH(mg->core.launches, mgk3b_repack(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, mg->staging, 0));
    MG_CUDA(cudaMemcpyAsync(host_dense, mg->staging, level_count(L) * mg_esize(mg->core.dtype), cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

/* Relax: ncycles x (red half-sweep, black half-sweep), N3/MultiGrid3D.cpp:489-567 */
static int relax_level(mg3b_t* mg, int level, int ncycles)
{
    mg_level3b* L = &mg->lv[level];
    for (int k = 0; k < ncycles; k++)
        for (int colour = 0; colour < 2; colour++)
            MG_LAUNCH(mg->core.launches, mgk3b_relax_colour(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, colour));
    return MG_OK;
}

int mg3b_relax(mg3b_t* mg, int level, int ncycles)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (ncycles < 0) return mg_fail(MG_ERR_ARG, "ncycles < 0");
    return relax_level(mg, level, ncycles);
}

int mg3b_residual(mg3b_t* mg, int level, void* host_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_out) return mg_fail(MG_ERR_ARG, "null output");
    mg_level3b* L = &mg->lv[level];
    const size_t bytes = level_count(L) * mg_esize(mg->core.dtype);
    MG_LAUNCH(mg->core.launches, mgk3b_residual_dense(mg->core.stream, mg->core.dtype, L->v, L->f, mg->staging, L->g, L->c, mg->mode == MG_CORRECTED));
    MG_CUDA(cudaMemcpyAsync(host_out, mg->staging, bytes, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

/* the norm pass of mg3b_residual_norm: {sum of r^2, max |r|} into d_scratch + 2*MG3B_NPARTS, nothing read back */
static int residual_norm_enqueue(mg3b_t* mg, int level)
{
    mg_level3b* L = &mg->lv[level];
    MG_LAUNCH(mg->core.launches, mgk3b_residual_norm(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, mg->mode == MG_CORRECTED, mg->d_scratch, MG3B_NPARTS,
                                                mg->d_scratch + 2 * MG3B_NPARTS));
    return MG_OK;
}

int mg3b_residual_norm(mg3b_t* mg, int level, double* l2, double* linf)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if ((st = residual_norm_enqueue(mg, level))) return st;
    return mg_read_norm(&mg->core, mg->d_scratch + 2 * MG3B_NPARTS, l2, linf);
}

int mg3b_restrict(mg3b_t* mg, int fine_level, int field)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level3b *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    MG_LAUNCH(mg->core.launches, mgk3b_restrict(mg->core.stream, mg->core.dtype, NULL, field_ptr(F, field), F->g, F->c, 0, field_ptr(C, field), NULL, C->g));
    return MG_OK;
}

static int residual_restrict_level(mg3b_t* mg, int fine_level)
{
    mg_level3b *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    MG_LAUNCH(mg->core.launches, mgk3b_restrict(mg->core.stream, mg->core.dtype, F->v, F->f, F->g, F->c, mg->mode == MG_CORRECTED, C->f, C->v, C->g));
    return MG_OK;
}

int mg3b_residual_restrict(mg3b_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return residual_restrict_level(mg, fine_level);
}

static int interpolate_level(mg3b_t* mg, int fine_level, int add)
{
    mg_level3b *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    MG_LAUNCH(mg->core.launches, mgk3b_interpolate(mg->core.stream, mg->core.dtype, F->v, F->g, C->v, C->g, add));
    return MG_OK;
}

int mg3b_interpolate(mg3b_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 0);
}

int mg3b_interpolate_correct(mg3b_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 1);
}

int mg3b_set_to_value(mg3b_t* mg, int level, int field, double value, int modify_boundaries)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level3b* L = &mg->lv[level];
    MG_LAUNCH(mg->core.launches, mgk3b_set(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, value, modify_boundaries));
    return MG_OK;
}

/* VCycle, N3/MultiGrid3D.cpp:623-647: CalculateResidual + Restrict + setToValue(coarse v, 0, true) are one kernel,
   Interpolate + ApplyCorrection are one kernel */
static int vcycle_rec(mg3b_t* mg, int level, int v1, int v2)
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

int mg3b_vcycle(mg3b_t* mg, int level, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    return vcycle_rec(mg, level, v1, v2);
}

/* tolerance-driven solve (mg_host_common.c builds and runs it) */
static int s3b_norm(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return residual_norm_enqueue(x->h, x->level); }
static int s3b_cycle(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return vcycle_rec(x->h, x->level, x->v1, x->v2); }

int mg3b_solve(mg3b_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles, int* cycles_out, int* converged_out,
               double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_cycles, v1, v2);
    if (st) return st;
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = {&x, mg->core.stream, &mg->core.launches, NULL, s3b_cycle, s3b_cycle, s3b_norm, mg->d_scratch + 2 * MG3B_NPARTS, NULL, NULL};
    const int key[MG_GRAPH_KEY] = {level, v1, v2};
    return mg_solve_run(&mg->core.graphs, mg_graphs_on(&mg->core.graphs, 0, 2LL * (v1 + v2) * (mg->core.nlevels - level)) ? key : NULL, &ops,
                        rtol, atol, max_cycles, cycles_out, converged_out, history);
}

/* multigrid-preconditioned conjugate gradients (mg_host_common.c runs the loop, mg3d_cg.cu has the vector passes) */
static void* p3b_v(mg_cycle_ctx* x) { return ((mg3b_t*)x->h)->lv[x->level].v; }
static int p3b_vcycle(mg_cycle_ctx* x) { return vcycle_rec(x->h, x->level, x->v1, x->v2); }
static int p3b_norm0(mg_cycle_ctx* x) { return residual_norm_enqueue(x->h, x->level); }
static int p3b_zero_v(mg_cycle_ctx* x)
{
    mg3b_t* mg = x->h;
    mg_level3b* L = &mg->lv[x->level];
    MG_LAUNCH(mg->core.launches, mgk3b_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 1));
    return MG_OK;
}

int mg3b_pcg(mg3b_t* mg, int level, int v1, int v2, double rtol, double atol, int max_iters, int* iters_out, int* converged_out,
             double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_iters, v1, v2);
    if (st) return st;
    if (mg->mode != MG_CORRECTED) return mg_fail(MG_ERR_STATE, "pcg needs MG_CORRECTED: the MG_REF_COMPAT residual is not a symmetric operator");
    if (!mg->pcg && !(mg->pcg = (mg_pcg_vecs*)calloc((size_t)mg->core.nlevels, sizeof *mg->pcg)))
        return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    mg_level3b* L = &mg->lv[level];
    if ((st = mg_pcg_vecs_alloc(&mg->pcg[level], field_bytes(L, mg->core.dtype), mg->core.stream))) return st;
    mg_pcg_ctx pc;
    memset(&pc, 0, sizeof pc);
    pc.cx.h = mg; pc.cx.level = level; pc.cx.v1 = v1; pc.cx.v2 = v2;
    pc.P = &mg->pcg[level];
    pc.dtype = mg->core.dtype;
    pc.stream = mg->core.stream;
    pc.launches = &mg->core.launches;
    pc.g.nx = L->g.nx; pc.g.ny = L->g.ny; pc.g.nz = L->g.nz;
    pc.g.hp = L->g.hp; pc.g.plane = L->g.plane; pc.g.cstride = L->g.cstride;
    pc.g.z0 = 0; pc.g.nzl = L->g.nz;
    pc.c = L->c;
    pc.f = L->f;
    pc.out2 = mg->d_scratch + 2 * MG3B_NPARTS;
    pc.v = p3b_v; pc.zero_v = p3b_zero_v; pc.vcycle = p3b_vcycle; pc.norm0 = p3b_norm0;
    const int key[MG_GRAPH_KEY] = {level, v1, v2, 0, 0, 0, 0, MG_GRAPH_PCG};
    return mg_pcg_run(&pc, &mg->core.graphs, mg_graphs_on(&mg->core.graphs, 0, 2LL * (v1 + v2) * (mg->core.nlevels - level)) ? key : NULL, rtol,
                      atol, max_iters, iters_out, converged_out, history);
}

/* FullMultiGridVCycle, N3/MultiGrid3D.cpp:569-585 */
static int fmg_rec(mg3b_t* mg, int level, int v0, int v1, int v2)
{
    int st;
    if (level != mg->core.nlevels - 1) {
        mg_level3b *F = &mg->lv[level], *C = &mg->lv[level + 1];
        MG_LAUNCH(mg->core.launches, mgk3b_restrict(mg->core.stream, mg->core.dtype, NULL, F->f, F->g, F->c, 0, C->f, NULL, C->g));
        if ((st = fmg_rec(mg, level + 1, v0, v1, v2))) return st;
        if ((st = interpolate_level(mg, level, 0))) return st;
    } else {
        mg_level3b* L = &mg->lv[level];
        MG_LAUNCH(mg->core.launches, mgk3b_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 0));
    }
    for (int i = 0; i < v0; i++)
        if ((st = vcycle_rec(mg, level, v1, v2))) return st;
    return MG_OK;
}

int mg3b_fmg(mg3b_t* mg, int level, int v0, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v0 < 0 || v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative count");
    return fmg_rec(mg, level, v0, v1, v2);
}

/* end to end on HOST arrays of the finest level: upload v, f -> cycles x VCycle(0, v1, v2) -> download v */
int mg3b_vcycle_host(mg3b_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles)
{
    if (!mg || !v_host || !f_host) return mg_fail(MG_ERR_ARG, "null argument");
    if (v1 < 0 || v2 < 0 || cycles < 0) return mg_fail(MG_ERR_ARG, "negative count");
    mg_level3b* L = &mg->lv[0];
    const size_t bytes = level_count(L) * mg_esize(mg->core.dtype);
    MG_CUDA(cudaMemcpyAsync(mg->staging, v_host, bytes, cudaMemcpyHostToDevice, mg->core.stream));
    MG_LAUNCH(mg->core.launches, mgk3b_repack(mg->core.stream, mg->core.dtype, L->v, L->g, mg->staging, 1));
    MG_CUDA(cudaMemcpyAsync(mg->staging, f_host, bytes, cudaMemcpyHostToDevice, mg->core.stream));
    MG_LAUNCH(mg->core.launches, mgk3b_repack(mg->core.stream, mg->core.dtype, L->f, L->g, mg->staging, 1));
    for (int i = 0; i < cycles; i++) {
        int st = vcycle_rec(mg, 0, v1, v2);
        if (st) return st;
    }
    MG_LAUNCH(mg->core.launches, mgk3b_repack(mg->core.stream, mg->core.dtype, L->v, L->g, mg->staging, 0));
    MG_CUDA(cudaMemcpyAsync(v_host, mg->staging, bytes, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

/* ---- reference-facing calls on caller-owned HOST arrays (N3/MultiGrid3D.h:16-27 with three different sizes): upload, run, download ---- */
static int box_sizes_ok(const int s[3]) { return s && s[0] >= 3 && s[1] >= 3 && s[2] >= 3; }
static int coarse_of(const int f[3], const int c[3])
{
    for (int a = 0; a < 3; a++)
        if (c[a] != (f[a] - 1) / 2 + 1) return 0; /* the reference's own check, N3/MultiGrid3D.cpp:60-62 */
    return 1;
}
static size_t count3(const int s[3]) { return (size_t)s[0] * (size_t)s[1] * (size_t)s[2]; }

int mg3b_restrict_host(mg3b_t* mg, const void* fine, const int fsize_xyz[3], void* coarse, const int csize_xyz[3])
{
    if (!mg || !fine || !coarse || !box_sizes_ok(fsize_xyz) || !box_sizes_ok(csize_xyz) || !coarse_of(fsize_xyz, csize_xyz))
        return mg_fail(MG_ERR_ARG, "bad arrays or sizes (coarse = (fine-1)/2+1 per axis)");
    void *df, *dc;
    int st = mg_tmp_begin(&mg->core, &df, count3(fsize_xyz), fine, &dc, count3(csize_xyz), NULL);
    if (st) return st;
    int k = mgk3b_dense_restrict(mg->core.stream, mg->core.dtype, df, fsize_xyz, dc, csize_xyz);
    return mg_tmp_finish(&mg->core, k, coarse, dc, count3(csize_xyz), df, dc);
}

int mg3b_interpolate_host(mg3b_t* mg, void* fine, const int fsize_xyz[3], const void* coarse, const int csize_xyz[3])
{
    if (!mg || !fine || !coarse || !box_sizes_ok(fsize_xyz) || !box_sizes_ok(csize_xyz) || !coarse_of(fsize_xyz, csize_xyz))
        return mg_fail(MG_ERR_ARG, "bad arrays or sizes (coarse = (fine-1)/2+1 per axis)");
    void *df, *dc;
    int st = mg_tmp_begin(&mg->core, &df, count3(fsize_xyz), fine, &dc, count3(csize_xyz), coarse); /* the boundary of fine is kept */
    if (st) return st;
    int k = mgk3b_dense_interpolate(mg->core.stream, mg->core.dtype, df, fsize_xyz, dc, csize_xyz);
    return mg_tmp_finish(&mg->core, k, fine, df, count3(fsize_xyz), df, dc);
}

int mg3b_apply_correction_host(mg3b_t* mg, void* fine, const int fsize_xyz[3], const void* error, const int esize_xyz[3])
{
    if (!mg || !fine || !error || !box_sizes_ok(fsize_xyz) || !esize_xyz || memcmp(fsize_xyz, esize_xyz, 3 * sizeof(int)))
        return mg_fail(MG_ERR_ARG, "bad arrays or sizes (N3/MultiGrid3D.cpp:659-661)");
    void *df, *de;
    int st = mg_tmp_begin(&mg->core, &df, count3(fsize_xyz), fine, &de, count3(fsize_xyz), error);
    if (st) return st;
    int k = mgk3b_dense_apply_correction(mg->core.stream, mg->core.dtype, df, de, fsize_xyz);
    return mg_tmp_finish(&mg->core, k, fine, df, count3(fsize_xyz), df, de);
}

int mg3b_set_to_value_host(mg3b_t* mg, void* grid, const int size_xyz[3], double value, int modify_boundaries)
{
    if (!mg || !grid || !box_sizes_ok(size_xyz)) return mg_fail(MG_ERR_ARG, "bad array or sizes");
    void *dg, *unused;
    int st = mg_tmp_begin(&mg->core, &dg, count3(size_xyz), grid, &unused, 0, NULL);
    if (st) return st;
    int k = mgk3b_dense_set(mg->core.stream, mg->core.dtype, dg, size_xyz, value, modify_boundaries);
    return mg_tmp_finish(&mg->core, k, grid, dg, count3(size_xyz), dg, NULL);
}

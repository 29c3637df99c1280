/* mg_host_common.c -- error state, device probing and the CUDA-graph cache shared by the host drivers. */
#include "mg_host_common.h"

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static __thread char g_err[512] = "";

int mg_fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

const char* mg_last_error(void) { return g_err; }

const char* mg_version(void) { return "pde_multigrid_b200 0.1 (sm_100a)"; }

int mg_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

/* ---- CUDA-graph cache ------------------------------------------------------------------------- */

void mg_graphs_init(mg_graphs* gr) { gr->enabled = getenv("MG_B200_NO_GRAPH") ? 0 : 1; }

static void drop_slot(mg_graph_slot* g)
{
    if (g->exec) cudaGraphExecDestroy(g->exec);
    memset(g, 0, sizeof *g);
}

void mg_graphs_free(mg_graphs* gr)
{
    for (int i = 0; i < MG_CYCLE_SLOTS; i++) drop_slot(&gr->cycles[i]);
    for (int i = 0; i < MG_SOLVE_SLOTS; i++) drop_slot(&gr->solves[i]);
    if (gr->h_par) cudaFreeHost(gr->h_par);
    if (gr->d_par) cudaFree(gr->d_par);
    if (gr->d_hist) cudaFree(gr->d_hist);
    memset(gr, 0, sizeof *gr);
}

int mg_graphs_on(const mg_graphs* gr, int profiling, long long launches_per_cycle)
{
    return gr->enabled && !profiling && launches_per_cycle <= MG_GRAPH_MAX_LAUNCHES;
}

void mg_graphs_drop(mg_graphs* gr, int pos, int value)
{
    for (int i = 0; i < MG_CYCLE_SLOTS; i++)
        if (gr->cycles[i].used && gr->cycles[i].key[pos] == value) drop_slot(&gr->cycles[i]);
    for (int i = 0; i < MG_SOLVE_SLOTS; i++)
        if (gr->solves[i].used && gr->solves[i].key[pos] == value) drop_slot(&gr->solves[i]);
}

/* the slot with this key, or a free one claimed for it (NULL: the cache is full) */
static mg_graph_slot* slot_for(mg_graph_slot* slots, int n, const int key[MG_GRAPH_KEY])
{
    for (int i = 0; i < n; i++)
        if (slots[i].used && !memcmp(slots[i].key, key, sizeof slots[i].key)) return &slots[i];
    for (int i = 0; i < n; i++)
        if (!slots[i].used) {
            memset(&slots[i], 0, sizeof slots[i]);
            slots[i].used = 1;
            memcpy(slots[i].key, key, sizeof slots[i].key);
            return &slots[i];
        }
    return NULL;
}

int mg_graph_cycle(mg_graphs* gr, const int key[MG_GRAPH_KEY], const mg_cycle_ops* ops)
{
    mg_graph_slot* g = key ? slot_for(gr->cycles, MG_CYCLE_SLOTS, key) : NULL;
    if (!g || !g->warm) { /* no graphs, the cache is full, or the first call of the key */
        if (g) g->warm = 1;
        return ops->cycle(ops->ctx);
    }
    if (!g->exec) {
        const long long l0 = *ops->launches, h0 = ops->halo_bytes ? *ops->halo_bytes : 0;
        cudaGraph_t graph = NULL;
        if (ops->save) ops->save(ops->ctx, g->snap[0]);
        MG_CUDA(cudaStreamBeginCapture(ops->stream, cudaStreamCaptureModeThreadLocal));
        int st = ops->cycle(ops->ctx);
        cudaError_t e = cudaStreamEndCapture(ops->stream, &graph);
        if (ops->save) { /* nothing ran during the capture: undo the host-side state changes, keep the end state */
            ops->save(ops->ctx, g->snap[1]);
            ops->load(ops->ctx, g->snap[0]);
        }
        g->launches[0] = *ops->launches - l0;
        *ops->launches = l0;
        if (ops->halo_bytes) {
            g->halo_bytes = *ops->halo_bytes - h0;
            *ops->halo_bytes = h0;
        }
        if (!st && e == cudaSuccess && graph) e = cudaGraphInstantiate(&g->exec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (st || e != cudaSuccess || !g->exec) {
            g->exec = NULL;
            cudaGetLastError();
            gr->enabled = 0; /* capture is not possible here: stay eager, and keep solves host-driven */
            return st ? st : ops->cycle(ops->ctx);
        }
    }
    MG_CUDA(cudaGraphLaunch(g->exec, ops->stream));
    if (ops->load) ops->load(ops->ctx, g->snap[1]); /* the replay leaves the host-side state the capture ended in */
    *ops->launches += g->launches[0];
    if (ops->halo_bytes) *ops->halo_bytes += g->halo_bytes;
    return MG_OK;
}

/* ---- the handle core -------------------------------------------------------------------------- */

int mg_core_init(mg_core* c)
{
    mg_graphs_init(&c->graphs);
    MG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    MG_CUDA(cudaMallocHost((void**)&c->h_out2, 2 * sizeof(double)));
    return MG_OK;
}

void mg_core_free(mg_core* c)
{
    if (c->stream) cudaStreamSynchronize(c->stream);
    mg_graphs_free(&c->graphs);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->h_out2) cudaFreeHost(c->h_out2);
    mg_prof_free(&c->prof);
}

int mg_check_level(const mg_core* c, int level)
{
    if (!c) return mg_fail(MG_ERR_ARG, "null handle");
    if (level < 0 || level >= c->nlevels) return mg_fail(MG_ERR_ARG, "level %d out of range [0,%d)", level, c->nlevels);
    return MG_OK;
}

int mg_check_fine_level(const mg_core* c, int level)
{
    int st = mg_check_level(c, level);
    if (st) return st;
    if (level == c->nlevels - 1) return mg_fail(MG_ERR_ARG, "level %d is the coarsest", level);
    return MG_OK;
}

int mg_sync(mg_core* c)
{
    if (!c) return mg_fail(MG_ERR_ARG, "null handle");
    MG_CUDA(cudaStreamSynchronize(c->stream));
    return MG_OK;
}

int mg_profile_enable(mg_core* c, int enable)
{
    if (!c) return mg_fail(MG_ERR_ARG, "null handle");
    return mg_prof_enable(&c->prof, c->stream, enable);
}

int mg_profile_read(mg_core* c, int level, int op, double* ms_total, long long* kernel_launches, long long* calls)
{
    int st = mg_check_level(c, level);
    if (st) return st;
    if (op < 0 || op >= MG_OP_COUNT) return mg_fail(MG_ERR_ARG, "bad op %d", op);
    if ((st = mg_prof_collect(&c->prof, c->stream))) return st;
    if (ms_total) *ms_total = c->prof.ms[level][op];
    if (kernel_launches) *kernel_launches = c->prof.kl[level][op];
    if (calls) *calls = c->prof.calls[level][op];
    return MG_OK;
}

int mg_read_out2(mg_core* c, const double* d_out2)
{
    MG_CUDA(cudaMemcpyAsync(c->h_out2, d_out2, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    MG_CUDA(cudaStreamSynchronize(c->stream));
    return MG_OK;
}

int mg_read_norm(mg_core* c, const double* d_out2, double* l2, double* linf)
{
    int st = mg_read_out2(c, d_out2);
    if (st) return st;
    if (l2) *l2 = sqrt(c->h_out2[0]);
    if (linf) *linf = c->h_out2[1];
    return MG_OK;
}

/* ---- the reference's operators on caller arrays ----------------------------------------------- */

int mg_tmp_begin(mg_core* c, void** da, size_t na, const void* ha, void** db, size_t nb, const void* hb)
{
    const size_t es = mg_esize(c->dtype);
    *da = *db = NULL;
    cudaError_t e = cudaMalloc(da, na * es);
    if (e == cudaSuccess && nb) e = cudaMalloc(db, nb * es);
    if (e == cudaSuccess && ha) e = cudaMemcpyAsync(*da, ha, na * es, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess && hb && nb) e = cudaMemcpyAsync(*db, hb, nb * es, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) return MG_OK;
    cudaFree(*da);
    cudaFree(*db);
    *da = *db = NULL;
    return mg_fail(MG_ERR_CUDA, "temporary device arrays: %s", cudaGetErrorString(e));
}

int mg_tmp_finish(mg_core* c, int k, void* host_out, const void* dev_out, size_t n, void* da, void* db)
{
    cudaError_t e = cudaSuccess;
    if (k >= 0 && host_out) e = cudaMemcpyAsync(host_out, dev_out, n * mg_esize(c->dtype), cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(da);
    if (db) cudaFree(db);
    if (k < 0) return mg_fail(MG_ERR_CUDA, "launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "copy failed: %s", cudaGetErrorString(e));
    c->launches += k;
    return MG_OK;
}

int mg_launch_done(mg_core* c, int k)
{
    if (k < 0) return mg_fail(MG_ERR_CUDA, "operator launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    c->launches += k;
    MG_CUDA(cudaStreamSynchronize(c->stream));
    return MG_OK;
}

/* ---- tolerance-driven solve ------------------------------------------------------------------- */

int mg_solve_check_args(const mg_core* c, int level, double rtol, double atol, int max_cycles, int v1, int v2)
{
    int st = mg_check_level(c, level);
    if (st) return st;
    if (!(rtol >= 0.0) || !(atol >= 0.0)) return mg_fail(MG_ERR_ARG, "rtol and atol must be >= 0 (got %g, %g)", rtol, atol);
    if (max_cycles < 0) return mg_fail(MG_ERR_ARG, "max_cycles %d < 0", max_cycles);
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    return MG_OK;
}

/* writes the parameter block of the next solve (the graph reads everything it needs from it: one graph serves every
   tolerance, cycle limit and history size) */
static int solver_begin(mg_graphs* gr, cudaStream_t s, double rtol, double atol, int max_cycles, int want_history)
{
    if (!gr->h_par) {
        MG_CUDA(cudaMallocHost((void**)&gr->h_par, sizeof *gr->h_par));
        MG_CUDA(cudaMalloc((void**)&gr->d_par, sizeof *gr->d_par));
    }
    const int need = want_history ? max_cycles + 1 : 0;
    if (need > gr->hist_cap) {
        MG_CUDA(cudaStreamSynchronize(s)); /* a previous solve may still write the old buffer */
        if (gr->d_hist) cudaFree(gr->d_hist);
        gr->d_hist = NULL;
        gr->hist_cap = 0;
        MG_CUDA(cudaMalloc((void**)&gr->d_hist, 2 * (size_t)need * sizeof(double)));
        gr->hist_cap = need;
    }
    mg_solve_par* p = gr->h_par;
    memset(p, 0, sizeof *p);
    p->rtol = rtol;
    p->atol = atol;
    p->hist = gr->d_hist;
    p->max_cycles = max_cycles;
    p->hist_cap = need;
    MG_CUDA(cudaMemcpyAsync(gr->d_par, p, sizeof *p, cudaMemcpyHostToDevice, s));
    return MG_OK;
}

static int read_par(mg_graphs* gr, cudaStream_t s)
{
    MG_CUDA(cudaMemcpyAsync(gr->h_par, gr->d_par, sizeof *gr->h_par, cudaMemcpyDeviceToHost, s));
    MG_CUDA(cudaStreamSynchronize(s));
    return MG_OK;
}

static int solver_finish(mg_graphs* gr, cudaStream_t s, int* cycles_out, int* converged_out, double* history)
{
    const int k = gr->h_par->k;
    if (history && k > 0) {
        MG_CUDA(cudaMemcpyAsync(history, gr->d_hist, 2 * (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, s));
        MG_CUDA(cudaStreamSynchronize(s));
    }
    if (cycles_out) *cycles_out = k - 1;
    if (converged_out) *converged_out = gr->h_par->converged;
    return MG_OK;
}

static int launch_check(const mg_cycle_ops* ops, mg_graphs* gr, int nhandles, cudaGraphConditionalHandle h0,
                        cudaGraphConditionalHandle h1)
{
    MG_LAUNCH(*ops->launches, mgk_solve_check(ops->stream, ops->out2, gr->d_par, nhandles, h0, h1));
    return MG_OK;
}

/* host-driven: the family's own cycle call, the norm pass and the check kernel, one read-back per cycle */
static int first_norm(const mg_cycle_ops* ops) { return ops->first ? ops->first(ops->ctx) : ops->norm(ops->ctx); }

static int solve_host(const mg_cycle_ops* ops, mg_graphs* gr)
{
    int st;
    if ((st = first_norm(ops))) return st;
    if ((st = launch_check(ops, gr, 0, 0, 0))) return st;
    for (;;) {
        if ((st = read_par(gr, ops->stream))) return st;
        if (gr->h_par->done) return MG_OK;
        if ((st = ops->public_cycle(ops->ctx))) return st;
        if ((st = ops->norm(ops->ctx))) return st;
        if ((st = launch_check(ops, gr, 0, 0, 0))) return st;
    }
}

#define SOLVE_TRY(call)                                                                                   \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) {                                                                          \
            st = mg_fail(MG_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_));                    \
            goto out;                                                                                     \
        }                                                                                                 \
    } while (0)
#define SOLVE_STEP(expr)                                                                                  \
    do {                                                                                                  \
        if ((st = (expr))) goto out;                                                                      \
    } while (0)

/* a conditional node behind everything captured so far on `s`; *body = the graph it runs */
static int add_conditional(cudaStream_t s, cudaGraphConditionalHandle h, enum cudaGraphConditionalNodeType type, cudaGraph_t* body)
{
    enum cudaStreamCaptureStatus cs;
    cudaGraph_t g = NULL;
    const cudaGraphNode_t* deps = NULL;
    size_t nd = 0;
    MG_CUDA(cudaStreamGetCaptureInfo(s, &cs, NULL, &g, &deps, &nd));
    struct cudaGraphNodeParams p;
    memset(&p, 0, sizeof p);
    p.type = cudaGraphNodeTypeConditional;
    p.conditional.handle = h;
    p.conditional.type = type;
    p.conditional.size = 1;
    cudaGraphNode_t node;
    MG_CUDA(cudaGraphAddNode(&node, g, deps, nd, &p));
    *body = p.conditional.phGraph_out[0];
    MG_CUDA(cudaStreamUpdateCaptureDependencies(s, &node, 1, cudaStreamSetCaptureDependencies));
    return MG_OK;
}

static int capture_segment_end(cudaStream_t s)
{
    cudaGraph_t g = NULL;
    MG_CUDA(cudaStreamEndCapture(s, &g)); /* capture to an existing graph hands back that graph: nothing to free */
    return MG_OK;
}

/* norm(r_0) -> check -> WHILE { cycle -> norm -> check [-> IF { cycle -> norm -> check }] }, instantiated into slot->exec.
   Nothing runs; the host-side state the captured cycles changed is put back, and the launch counter too. */
static int solve_build(const mg_cycle_ops* ops, mg_graph_slot* slot, mg_graphs* gr)
{
    cudaStream_t s = ops->stream;
    const long long l0 = *ops->launches;
    long long mark = l0;
    cudaGraph_t g = NULL, body = NULL, ibody = NULL;
    cudaGraphConditionalHandle hw = 0, hi = 0;
    int st = MG_OK;
    if (ops->save) ops->save(ops->ctx, slot->snap[0]);
    SOLVE_TRY(cudaGraphCreate(&g, 0));
    SOLVE_TRY(cudaGraphConditionalHandleCreate(&hw, g, 0, cudaGraphCondAssignDefault));

    SOLVE_TRY(cudaStreamBeginCaptureToGraph(s, g, NULL, NULL, 0, cudaStreamCaptureModeThreadLocal));
    SOLVE_STEP(first_norm(ops));
    SOLVE_STEP(launch_check(ops, gr, 1, hw, 0));
    SOLVE_STEP(add_conditional(s, hw, cudaGraphCondTypeWhile, &body));
    SOLVE_STEP(capture_segment_end(s));
    slot->launches[0] = *ops->launches - mark;
    mark = *ops->launches;

    SOLVE_TRY(cudaStreamBeginCaptureToGraph(s, body, NULL, NULL, 0, cudaStreamCaptureModeThreadLocal));
    SOLVE_STEP(ops->cycle(ops->ctx));
    if (ops->save) {
        ops->save(ops->ctx, slot->snap[1]);
        slot->two = slot->snap[1][0] != slot->snap[0][0];
    } else {
        memcpy(slot->snap[1], slot->snap[0], sizeof slot->snap[0]);
    }
    if (slot->two) SOLVE_TRY(cudaGraphConditionalHandleCreate(&hi, body, 0, cudaGraphCondAssignDefault));
    SOLVE_STEP(ops->norm(ops->ctx));
    SOLVE_STEP(launch_check(ops, gr, slot->two ? 2 : 1, hw, hi));
    if (slot->two) SOLVE_STEP(add_conditional(s, hi, cudaGraphCondTypeIf, &ibody));
    SOLVE_STEP(capture_segment_end(s));
    slot->launches[1] = *ops->launches - mark;
    mark = *ops->launches;

    if (slot->two) {
        SOLVE_TRY(cudaStreamBeginCaptureToGraph(s, ibody, NULL, NULL, 0, cudaStreamCaptureModeThreadLocal));
        SOLVE_STEP(ops->cycle(ops->ctx));
        ops->save(ops->ctx, slot->snap[2]);
        SOLVE_STEP(ops->norm(ops->ctx));
        SOLVE_STEP(launch_check(ops, gr, 1, hw, 0));
        SOLVE_STEP(capture_segment_end(s));
        slot->launches[2] = *ops->launches - mark;
        if (slot->snap[2][0] != slot->snap[0][0]) {
            st = mg_fail(MG_ERR_STATE, "two cycles do not return to the starting buffers");
            goto out;
        }
    }
    SOLVE_TRY(cudaGraphInstantiate(&slot->exec, g, 0));
out:
    if (st) {
        enum cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
            cudaGraph_t tmp = NULL;
            cudaStreamEndCapture(s, &tmp);
        }
        slot->exec = NULL;
        cudaGetLastError();
    }
    if (g) cudaGraphDestroy(g);
    *ops->launches = l0;
    if (ops->load) ops->load(ops->ctx, slot->snap[0]);
    return st;
}

int mg_solve_run(mg_graphs* gr, const int key[MG_GRAPH_KEY], const mg_cycle_ops* ops, double rtol, double atol,
                 int max_cycles, int* cycles_out, int* converged_out, double* history)
{
    cudaStream_t s = ops->stream;
    mg_graph_slot* slot = key ? slot_for(gr->solves, MG_SOLVE_SLOTS, key) : NULL; /* NULL: the solve runs host-driven */
    int st = solver_begin(gr, s, rtol, atol, max_cycles, history != NULL);
    if (st) return st;
    /* like the cycle graphs: a capture only after an eager run of the same cycle (kernel attributes, lazily loaded
       modules and lazily allocated buffers must exist before it) */
    if (slot && slot->warm && !slot->exec && !slot->failed && solve_build(ops, slot, gr) != MG_OK) slot->failed = 1;
    if (!slot || !slot->exec) {
        if ((st = solve_host(ops, gr))) return st;
        if (slot && gr->h_par->k > 1) slot->warm = 1;
        return solver_finish(gr, s, cycles_out, converged_out, history);
    }
    MG_CUDA(cudaGraphLaunch(slot->exec, s));
    if ((st = read_par(gr, s))) return st;
    const int cycles = gr->h_par->k - 1;
    *ops->launches += slot->launches[0];
    for (int c = 1; c <= cycles; c++) *ops->launches += slot->launches[slot->two && c % 2 == 0 ? 2 : 1];
    if (ops->load) ops->load(ops->ctx, cycles == 0 ? slot->snap[0] : (slot->two && cycles % 2 == 0) ? slot->snap[2] : slot->snap[1]);
    return solver_finish(gr, s, cycles_out, converged_out, history);
}

/* ---- multigrid-preconditioned conjugate gradients ------------------------------------------------ */

int mg_pcg_vecs_alloc(mg_pcg_vecs* P, size_t field_bytes, cudaStream_t s)
{
    if (P->b) return MG_OK;
    void** f[6] = {&P->b, &P->x[0], &P->x[1], &P->p[0], &P->p[1], &P->d};
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 6 && e == cudaSuccess; i++) e = cudaMalloc(f[i], field_bytes);
    if (e == cudaSuccess) e = cudaMalloc((void**)&P->parts, (MGK_PCG_PARTS + MGK_PCG_SCALARS) * sizeof(double));
    /* the row padding is never read for a result, but it is copied into v at the end: keep it defined */
    for (int i = 0; i < 6 && e == cudaSuccess; i++) e = cudaMemsetAsync(*f[i], 0, field_bytes, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(P->parts, 0, (MGK_PCG_PARTS + MGK_PCG_SCALARS) * sizeof(double), s);
    if (e == cudaSuccess) {
        P->bytes = field_bytes;
        return MG_OK;
    }
    cudaGetLastError();
    mg_pcg_vecs_free(P);
    return mg_fail(MG_ERR_NOMEM, "PCG vectors (6 x %zu bytes): %s", field_bytes, cudaGetErrorString(e));
}

void mg_pcg_vecs_free(mg_pcg_vecs* P)
{
    void* f[7] = {P->b, P->x[0], P->x[1], P->p[0], P->p[1], P->d, P->parts};
    for (int i = 0; i < 7; i++)
        if (f[i]) cudaFree(f[i]);
    memset(P, 0, sizeof *P);
}

static double* pcg_sc(const mg_pcg_ctx* pc) { return pc->P->parts + MGK_PCG_PARTS; }

/* norm(r_0) with the family's own pass (the same bits as mg?d_residual_norm), then b <- f, x <- v, r_0 = b - Laplacian x into f */
static int pcg_first(void* c)
{
    mg_pcg_ctx* pc = (mg_pcg_ctx*)c;
    mg_pcg_vecs* P = pc->P;
    int st = pc->norm0(&pc->cx);
    if (st) return st;
    pc->par = 0;
    MG_CUDA(cudaMemcpyAsync(P->b, pc->f, P->bytes, cudaMemcpyDeviceToDevice, pc->stream));
    MG_CUDA(cudaMemcpyAsync(P->x[0], pc->v(&pc->cx), P->bytes, cudaMemcpyDeviceToDevice, pc->stream));
    MG_CUDA(cudaMemsetAsync(P->p[0], 0, P->bytes, pc->stream)); /* beta = 0 multiplies it on the first iteration */
    MG_CUDA(cudaMemsetAsync(P->d, 0, P->bytes, pc->stream));
    MG_LAUNCH(*pc->launches, mgk3cg_residual(pc->stream, pc->dtype, P->x[0], P->b, pc->f, pc->g, pc->c, pcg_sc(pc), 0, pc->g.nzl));
    return MG_OK;
}

/* one iteration: z = VCycle(0; r) in v, beta, p, alpha, x, r, the norm partials of the new r */
static int pcg_step(void* c)
{
    mg_pcg_ctx* pc = (mg_pcg_ctx*)c;
    mg_pcg_vecs* P = pc->P;
    const int a = pc->par, n = a ^ 1;
    double *part = P->parts, *sc = pcg_sc(pc);
    int st;
    if ((st = pc->zero_v(&pc->cx)) || (st = pc->vcycle(&pc->cx))) return st;
    const void* z = pc->v(&pc->cx);
    MG_LAUNCH(*pc->launches, mgk3cg_dots(pc->stream, pc->dtype, z, pc->f, P->d, pc->g, 0, pc->g.nzl, part, sc));
    MG_LAUNCH(*pc->launches, mgk3cg_dir(pc->stream, pc->dtype, z, P->p[a], P->p[n], pc->g, pc->c, 0, pc->g.nzl, part + MGK_PCG_DIR_PARTS, sc));
    MG_LAUNCH(*pc->launches, mgk3cg_update(pc->stream, pc->dtype, P->x[a], P->p[n], P->b, pc->f, P->x[n], P->d, pc->g, pc->c, sc, 0, pc->g.nzl,
                                           part + MGK_PCG_UPD_PARTS));
    pc->par = n;
    return MG_OK;
}

static int pcg_norm(void* c)
{
    mg_pcg_ctx* pc = (mg_pcg_ctx*)c;
    MG_LAUNCH(*pc->launches, mgk_norm_final(pc->stream, pc->P->parts + MGK_PCG_UPD_PARTS, MGK_PCG_BLOCKS, pc->out2));
    return MG_OK;
}

static void pcg_save(void* c, unsigned out[2])
{
    mg_pcg_ctx* pc = (mg_pcg_ctx*)c;
    out[0] = out[1] = 0;
    if (pc->save) pc->save(&pc->cx, out);
    out[0] = (out[0] & 0x7fffffffu) | ((unsigned)pc->par << 31);
}

static void pcg_load(void* c, const unsigned in[2])
{
    mg_pcg_ctx* pc = (mg_pcg_ctx*)c;
    if (pc->load) {
        const unsigned fam[2] = {in[0] & 0x7fffffffu, in[1]};
        pc->load(&pc->cx, fam);
    }
    pc->par = (int)(in[0] >> 31);
}

int mg_pcg_run(mg_pcg_ctx* pc, mg_graphs* gr, const int key[MG_GRAPH_KEY], double rtol, double atol, int max_iters, int* iters_out,
               int* converged_out, double* history)
{
    const mg_cycle_ops ops = {pc, pc->stream, pc->launches, NULL, pcg_step, pcg_step, pcg_norm, pc->out2, pcg_save, pcg_load, pcg_first};
    int st = mg_solve_run(gr, key, &ops, rtol, atol, max_iters, iters_out, converged_out, history);
    if (st) return st;
    /* v of the level (the buffer the last V-cycle ended on) <- x, f <- b: the caller's f bit for bit */
    MG_CUDA(cudaMemcpyAsync(pc->v(&pc->cx), pc->P->x[pc->par], pc->P->bytes, cudaMemcpyDeviceToDevice, pc->stream));
    MG_CUDA(cudaMemcpyAsync(pc->f, pc->P->b, pc->P->bytes, cudaMemcpyDeviceToDevice, pc->stream));
    MG_CUDA(cudaStreamSynchronize(pc->stream));
    return MG_OK;
}

int mg_require_device(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n < 1) {
        cudaGetLastError();
        return mg_fail(MG_ERR_CUDA, "no CUDA device available (%s): this engine has no CPU fallback",
                       e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    return MG_OK;
}

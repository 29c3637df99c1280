/* mg_host_common.c -- error state and device probing shared by the host drivers. */
#include "mg_host_common.h"

#include <stdarg.h>
#include <stdio.h>
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

/* ---- tolerance-driven solve ------------------------------------------------------------------- */

int mg_solve_check_args(double rtol, double atol, int max_cycles, int v1, int v2)
{
    if (!(rtol >= 0.0) || !(atol >= 0.0)) return mg_fail(MG_ERR_ARG, "rtol and atol must be >= 0 (got %g, %g)", rtol, atol);
    if (max_cycles < 0) return mg_fail(MG_ERR_ARG, "max_cycles %d < 0", max_cycles);
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    return MG_OK;
}

mg_solve_slot* mg_solve_slot_for(mg_solve_slot slots[MG_SOLVE_SLOTS], const int key[MG_SOLVE_KEY])
{
    for (int i = 0; i < MG_SOLVE_SLOTS; i++)
        if (slots[i].used && !memcmp(slots[i].key, key, sizeof slots[i].key)) return &slots[i];
    for (int i = 0; i < MG_SOLVE_SLOTS; i++)
        if (!slots[i].used) {
            memset(&slots[i], 0, sizeof slots[i]);
            slots[i].used = 1;
            memcpy(slots[i].key, key, sizeof slots[i].key);
            return &slots[i];
        }
    return NULL;
}

void mg_solve_free(mg_solver* sv, mg_solve_slot slots[MG_SOLVE_SLOTS])
{
    for (int i = 0; i < MG_SOLVE_SLOTS; i++)
        if (slots[i].used && slots[i].exec) cudaGraphExecDestroy(slots[i].exec);
    if (sv->h_par) cudaFreeHost(sv->h_par);
    if (sv->d_par) cudaFree(sv->d_par);
    if (sv->d_hist) cudaFree(sv->d_hist);
    memset(sv, 0, sizeof *sv);
}

/* writes the parameter block of the next solve (the graph reads everything it needs from it: one graph serves every
   tolerance, cycle limit and history size) */
static int solver_begin(mg_solver* sv, cudaStream_t s, double rtol, double atol, int max_cycles, int want_history)
{
    if (!sv->h_par) {
        MG_CUDA(cudaMallocHost((void**)&sv->h_par, sizeof *sv->h_par));
        MG_CUDA(cudaMalloc((void**)&sv->d_par, sizeof *sv->d_par));
    }
    const int need = want_history ? max_cycles + 1 : 0;
    if (need > sv->hist_cap) {
        MG_CUDA(cudaStreamSynchronize(s)); /* a previous solve may still write the old buffer */
        if (sv->d_hist) cudaFree(sv->d_hist);
        sv->d_hist = NULL;
        sv->hist_cap = 0;
        MG_CUDA(cudaMalloc((void**)&sv->d_hist, 2 * (size_t)need * sizeof(double)));
        sv->hist_cap = need;
    }
    mg_solve_par* p = sv->h_par;
    memset(p, 0, sizeof *p);
    p->rtol = rtol;
    p->atol = atol;
    p->hist = sv->d_hist;
    p->max_cycles = max_cycles;
    p->hist_cap = need;
    MG_CUDA(cudaMemcpyAsync(sv->d_par, p, sizeof *p, cudaMemcpyHostToDevice, s));
    return MG_OK;
}

static int read_par(mg_solver* sv, cudaStream_t s)
{
    MG_CUDA(cudaMemcpyAsync(sv->h_par, sv->d_par, sizeof *sv->h_par, cudaMemcpyDeviceToHost, s));
    MG_CUDA(cudaStreamSynchronize(s));
    return MG_OK;
}

static int solver_finish(mg_solver* sv, cudaStream_t s, int* cycles_out, int* converged_out, double* history)
{
    const int k = sv->h_par->k;
    if (history && k > 0) {
        MG_CUDA(cudaMemcpyAsync(history, sv->d_hist, 2 * (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, s));
        MG_CUDA(cudaStreamSynchronize(s));
    }
    if (cycles_out) *cycles_out = k - 1;
    if (converged_out) *converged_out = sv->h_par->converged;
    return MG_OK;
}

static int launch_check(const mg_solve_ops* ops, mg_solver* sv, int nhandles, cudaGraphConditionalHandle h0,
                        cudaGraphConditionalHandle h1)
{
    MG_LAUNCH(*ops->launches, mgk_solve_check(ops->stream, ops->out2, sv->d_par, nhandles, h0, h1));
    return MG_OK;
}

/* host-driven: the family's own cycle call, the norm pass and the check kernel, one read-back per cycle */
static int solve_host(const mg_solve_ops* ops, mg_solver* sv)
{
    int st;
    if ((st = ops->norm(ops->ctx))) return st;
    if ((st = launch_check(ops, sv, 0, 0, 0))) return st;
    for (;;) {
        if ((st = read_par(sv, ops->stream))) return st;
        if (sv->h_par->done) return MG_OK;
        if ((st = ops->cycle(ops->ctx))) return st;
        if ((st = ops->norm(ops->ctx))) return st;
        if ((st = launch_check(ops, sv, 0, 0, 0))) return st;
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
static int solve_build(const mg_solve_ops* ops, mg_solve_slot* slot, mg_solver* sv)
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
    SOLVE_STEP(ops->norm(ops->ctx));
    SOLVE_STEP(launch_check(ops, sv, 1, hw, 0));
    SOLVE_STEP(add_conditional(s, hw, cudaGraphCondTypeWhile, &body));
    SOLVE_STEP(capture_segment_end(s));
    slot->launches[0] = *ops->launches - mark;
    mark = *ops->launches;

    SOLVE_TRY(cudaStreamBeginCaptureToGraph(s, body, NULL, NULL, 0, cudaStreamCaptureModeThreadLocal));
    SOLVE_STEP(ops->capture_cycle(ops->ctx));
    if (ops->save) {
        ops->save(ops->ctx, slot->snap[1]);
        slot->two = slot->snap[1][0] != slot->snap[0][0];
    } else {
        memcpy(slot->snap[1], slot->snap[0], sizeof slot->snap[0]);
    }
    if (slot->two) SOLVE_TRY(cudaGraphConditionalHandleCreate(&hi, body, 0, cudaGraphCondAssignDefault));
    SOLVE_STEP(ops->norm(ops->ctx));
    SOLVE_STEP(launch_check(ops, sv, slot->two ? 2 : 1, hw, hi));
    if (slot->two) SOLVE_STEP(add_conditional(s, hi, cudaGraphCondTypeIf, &ibody));
    SOLVE_STEP(capture_segment_end(s));
    slot->launches[1] = *ops->launches - mark;
    mark = *ops->launches;

    if (slot->two) {
        SOLVE_TRY(cudaStreamBeginCaptureToGraph(s, ibody, NULL, NULL, 0, cudaStreamCaptureModeThreadLocal));
        SOLVE_STEP(ops->capture_cycle(ops->ctx));
        ops->save(ops->ctx, slot->snap[2]);
        SOLVE_STEP(ops->norm(ops->ctx));
        SOLVE_STEP(launch_check(ops, sv, 1, hw, 0));
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

int mg_solve_run(const mg_solve_ops* ops, mg_solver* sv, mg_solve_slot* slot, double rtol, double atol, int max_cycles,
                 int* cycles_out, int* converged_out, double* history)
{
    cudaStream_t s = ops->stream;
    int st = solver_begin(sv, s, rtol, atol, max_cycles, history != NULL);
    if (st) return st;
    /* like the cycle graphs: a capture only after an eager run of the same cycle (kernel attributes, lazily loaded
       modules and lazily allocated buffers must exist before it) */
    if (slot && slot->warm && !slot->exec && !slot->failed && solve_build(ops, slot, sv) != MG_OK) slot->failed = 1;
    if (!slot || !slot->exec) {
        if ((st = solve_host(ops, sv))) return st;
        if (slot && sv->h_par->k > 1) slot->warm = 1;
        return solver_finish(sv, s, cycles_out, converged_out, history);
    }
    MG_CUDA(cudaGraphLaunch(slot->exec, s));
    if ((st = read_par(sv, s))) return st;
    const int cycles = sv->h_par->k - 1;
    *ops->launches += slot->launches[0];
    for (int c = 1; c <= cycles; c++) *ops->launches += slot->launches[slot->two && c % 2 == 0 ? 2 : 1];
    if (ops->load) ops->load(ops->ctx, cycles == 0 ? slot->snap[0] : (slot->two && cycles % 2 == 0) ? slot->snap[2] : slot->snap[1]);
    return solver_finish(sv, s, cycles_out, converged_out, history);
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

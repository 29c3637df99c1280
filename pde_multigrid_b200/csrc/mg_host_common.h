/*
 * mg_host_common.h -- shared helpers of the C host drivers: error reporting, CUDA call checking,
 * pitched-layout arithmetic, the handle core every family embeds, operators on caller arrays, the CUDA-graph cache of
 * cycles and solves.  Internal; the public ABI is include/mg_b200.h.
 */
#ifndef MG_HOST_COMMON_H
#define MG_HOST_COMMON_H

#include <cuda_runtime_api.h>
#include <stddef.h>

#include "../../include/mg_b200.h"
#include "mg_launch.h"
#include "mg_profile.h"

#ifdef __cplusplus
extern "C" {
#endif

int mg_fail(int code, const char* fmt, ...); /* records the message for mg_last_error(), returns code */

#define MG_CUDA(call)                                                                                         \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess)                                                                                \
            return mg_fail(MG_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

/* launcher return value -> status; adds to the handle's launch counter */
#define MG_LAUNCH(counter, call)                                                                     \
    do {                                                                                             \
        int k_ = (call);                                                                             \
        if (k_ < 0)                                                                                  \
            return mg_fail(MG_ERR_CUDA, "%s: launch failed: %s", #call, cudaGetErrorString(cudaGetLastError())); \
        (counter) += k_;                                                                             \
    } while (0)

static inline size_t mg_esize(int dtype) { return dtype == MG_F32 ? 4 : 8; }
/* row pitch in elements: n rounded up to 128 bytes */
static inline int mg_pitch(int n, int dtype)
{
    int per = (int)(128 / mg_esize(dtype));
    return (n + per - 1) / per * per;
}
static inline size_t mg_align256(size_t b) { return (b + 255) & ~(size_t)255; }
/* numGrids = (int)log2(minSize-1), N3/MultiGrid3D.cpp:33-34 */
static inline int mg_num_levels_for(int n)
{
    int k = 0, m = n - 1;
    while (m > 1) { m >>= 1; k++; }
    return k;
}
/* 128-byte CUtensorMap over one colour array of a colour-split 3D field (mg_tma_host.c) */
int mg_tma_make_colour_map(void* out128, int dtype, void* base, const mg_geom3d* g, int box_i, int box_y);
int mg_require_device(void); /* MG_OK, or MG_ERR_CUDA with a message: there is no CPU fallback */

/* ---- CUDA-graph cache of a handle, shared by the four families ----
   Cycle graphs (mg_graph_cycle, the public *_vcycle of 2D and 3D): a whole V-cycle is dozens to hundreds of dependent
   launches, most of them tiny, so replaying it from a graph removes the per-launch gaps.  The first call with a key runs
   eagerly (kernel attributes, lazily loaded modules and lazily allocated buffers must exist before a capture), the second
   captures and launches the graph, later calls replay it.
   Solve graphs (mg_solve_run, every *_solve): one graph  norm(r_0) -> check -> WHILE { cycle -> norm -> check }.  When a
   cycle does not end on the buffers it started on (the 3D temporally blocked smoother ping-pongs), the body holds two
   cycles: cycle(s0 -> s1) -> norm -> check -> IF { cycle(s1 -> s0) -> norm -> check }.  The first solve of a key runs
   host-driven: the same kernels and the same check kernel, one read-back of the parameter block per cycle.
   Either way nothing runs while a graph is captured, so the host-side state and the counters the captured cycle changed
   are put back; a replay applies the end state and adds the counts an eager run would have added. */

/* a cycle estimated to make more launches than this runs eagerly: it is not dominated by launch gaps, and its graph
   would be large to capture and keep */
#define MG_GRAPH_MAX_LAUNCHES 4096
#define MG_GRAPH_KEY 8     /* (level, v1, v2, smoother, arith, buffer bits, ghost bits, kind); the families use a prefix */
#define MG_GRAPH_KEY_SMOOTHER 3
#define MG_GRAPH_KEY_KIND 7 /* 0: cycles and solves, MG_GRAPH_PCG: *_pcg graphs */
#define MG_GRAPH_PCG 1
#define MG_CYCLE_SLOTS 16
#define MG_SOLVE_SLOTS 8

typedef struct {
    int used, key[MG_GRAPH_KEY];
    int warm;              /* a call with this key has run eagerly (a solve: host-driven, at least one cycle) */
    int failed;            /* solve graphs: the build failed, the key stays host-driven */
    int two;               /* solve graphs: the body holds two cycles */
    unsigned snap[3][2];   /* family state (ops.save) at the start, after the first and after the second captured cycle */
    cudaGraphExec_t exec;
    long long launches[3]; /* cycle: [0] the cycle; solve: norm(r_0) + check; first body cycle + norm + check; second */
    long long halo_bytes;  /* cycle graphs: what the captured cycle added to *ops.halo_bytes */
} mg_graph_slot;

typedef struct {
    int enabled;           /* 0: MG_B200_NO_GRAPH, or a cycle could not be captured: everything runs eagerly */
    mg_graph_slot cycles[MG_CYCLE_SLOTS];
    mg_graph_slot solves[MG_SOLVE_SLOTS];
    /* the solve's parameter block and history on the device */
    mg_solve_par* h_par;   /* pinned */
    mg_solve_par* d_par;
    double* d_hist;
    int hist_cap;          /* pairs d_hist has room for */
} mg_graphs;

/* what the cache needs of a family to run, capture and replay one cycle on one level with fixed sweep counts */
typedef struct {
    void* ctx;
    cudaStream_t stream;
    long long* launches;            /* the handle's kernel counter */
    long long* halo_bytes;          /* NULL, or a second counter the cycle advances (3D; solve graphs exist only where it
                                       stays put, on one GPU) */
    int (*cycle)(void* ctx);        /* one cycle as plain launches: what is captured, and what an eager call runs */
    int (*public_cycle)(void* ctx); /* one cycle the way the family's public *_vcycle runs it (host-driven solve) */
    int (*norm)(void* ctx);         /* enqueue the norm pass of the cycle's level into out2 */
    const double* out2;             /* where norm() leaves {sum of squares, max} */
    /* NULL for families whose cycle always ends on the buffers it started on; otherwise the host-side state:
       [0] = which buffer every level works on, [1] = further bookkeeping */
    void (*save)(void* ctx, unsigned out[2]);
    void (*load)(void* ctx, const unsigned in[2]);
    /* NULL, or what runs instead of norm() for r_0: its norm into out2, then whatever the loop needs set up (the PCG prologue) */
    int (*first)(void* ctx);
} mg_cycle_ops;

void mg_graphs_init(mg_graphs* gr); /* reads MG_B200_NO_GRAPH */
void mg_graphs_free(mg_graphs* gr);
/* graphs may be used: the cache is enabled, per-operator timers are off (they need eager launches) and the cycle's
   launch estimate is at most MG_GRAPH_MAX_LAUNCHES */
int mg_graphs_on(const mg_graphs* gr, int profiling, long long launches_per_cycle);
/* drops every cycle and solve graph whose key[pos] == value */
void mg_graphs_drop(mg_graphs* gr, int pos, int value);
/* one cycle: eager when key is NULL, the cache is full or the key is new; otherwise captured on first need, then replayed */
int mg_graph_cycle(mg_graphs* gr, const int key[MG_GRAPH_KEY], const mg_cycle_ops* ops);

/* what a family's mg_cycle_ops callbacks get as ctx: one cycle of handle h on `level` with fixed sweep counts */
typedef struct {
    void* h;
    int level, v1, v2;
} mg_cycle_ctx;

/* the whole solve: device-driven when key != NULL, the key is warm and its graph builds; host-driven otherwise */
int mg_solve_run(mg_graphs* gr, const int key[MG_GRAPH_KEY], const mg_cycle_ops* ops, double rtol, double atol,
                 int max_cycles, int* cycles_out, int* converged_out, double* history);

/* ---- multigrid-preconditioned conjugate gradients (mg3d_pcg, mg3b_pcg; DESIGN.md §6b) ----
   The loop is mg_solve_run's: ops.first = norm(r_0) + prologue, ops.cycle = one PCG iteration (its V-cycle included),
   ops.norm = the norm finaliser of the iteration's update pass.  x and p ping-pong between two buffers, so the iteration's
   parity is part of the state ops.save / ops.load carry (bit 31 of [0]) and a device loop always has the two-iteration body.
   A slab of a distributed level (DESIGN.md section 6b) adds the hooks and plane ranges of mg_pcg_ctx; its loop is host-driven. */
typedef struct {
    void* b;          /* the caller's f of the level, put back at the end */
    void* x[2];       /* the iterate */
    void* p[2];       /* the search direction */
    void* d;          /* r_k - r_{k-1} */
    double* parts;    /* MGK_PCG_PARTS partials of the three passes (mg_launch.h), MGK_PCG_SCALARS scalars, then (slabs) the
                         all-gathered double-double dot sums, 4 per rank */
    size_t bytes;     /* of one field */
} mg_pcg_vecs;

typedef struct {
    mg_cycle_ctx cx;              /* the family's cycle context: handle, level, sweeps */
    mg_pcg_vecs* P;
    int par;                      /* which of x[], p[] holds the current iterate and direction */
    int dtype;
    cudaStream_t stream;
    long long* launches;
    mg_geom3cg g;
    mg_coef3d c;
    void* f;                      /* the level's f */
    double* out2;                 /* where the family's norm pass leaves {sum of squares, max} */
    void* (*v)(mg_cycle_ctx* cx); /* the level's current v buffer */
    int (*zero_v)(mg_cycle_ctx* cx);
    int (*vcycle)(mg_cycle_ctx* cx);
    int (*norm0)(mg_cycle_ctx* cx); /* the family's residual-norm pass (mg?d_residual_norm without the read-back) */
    void (*save)(void* cx, unsigned out[2]); /* NULL, or the family's host-side buffer state */
    void (*load)(void* cx, const unsigned in[2]);
    /* local planes: the dots, residual and norm cover [own_lo, own_hi), the pointwise updates of p and x [wr_lo, wr_hi).
       One GPU (and a level every rank holds whole): both are all planes and the hooks below are NULL. */
    int own_lo, own_hi, wr_lo, wr_hi;
    int rank, nranks;
    int (*r_written)(mg_cycle_ctx* cx);    /* f (= r) holds new owned planes: bring its ghost planes up to date */
    int (*z_ready)(mg_cycle_ctx* cx);      /* the preconditioner has left z in v: at least one ghost plane of v each way */
    int (*allgather)(mg_cycle_ctx* cx, double* dd); /* dd[4*rank .. 4*rank+3] of every rank into every rank's dd, in place */
    int (*allreduce)(mg_cycle_ctx* cx, double* out2); /* {sum, max} over the ranks, in place */
    int (*v_restored)(mg_cycle_ctx* cx);   /* v holds the iterate on the owned planes: refresh its ghost planes as after set_field */
} mg_pcg_ctx;

/* allocates the vectors of one level on first use (MG_ERR_NOMEM, nothing allocated, when that fails); nranks: room for the
   dot sums of that many ranks (0 where the level is not distributed) */
int mg_pcg_vecs_alloc(mg_pcg_vecs* P, size_t field_bytes, int nranks, cudaStream_t s);
void mg_pcg_vecs_free(mg_pcg_vecs* P);
/* the whole PCG: the loop through mg_solve_run (device-driven when key != NULL), then v <- x, f <- b */
int mg_pcg_run(mg_pcg_ctx* pc, mg_graphs* gr, const int key[MG_GRAPH_KEY], double rtol, double atol, int max_iters, int* iters_out,
               int* converged_out, double* history);

/* ---- the handle core ----
   Every family's handle (mg1d_s, mg2d_s, mg3b_s, mg3d_s) has an mg_core named `core`.  A public call passes
   MG_CORE(handle) to the checking helpers below: NULL for a NULL handle, which they report as "null handle". */
typedef struct {
    int dtype, nlevels;
    cudaStream_t stream;  /* non-blocking: every operator of the handle runs on it */
    long long launches;   /* kernel launches, *_kernel_launches */
    double* h_out2;       /* pinned {sum of squares, max} read-back */
    mg_prof prof;         /* per-operator timers; the box engine never enables them */
    mg_graphs graphs;
} mg_core;

/* the stream, h_out2 and the graph cache; dtype and nlevels are the family's to set.  On failure the family frees the
   handle as usual: mg_core_free takes a partly initialised core, once. */
int mg_core_init(mg_core* c);
void mg_core_free(mg_core* c); /* synchronises the stream first */

#define MG_CORE(h) ((h) ? &(h)->core : NULL)

int mg_check_level(const mg_core* c, int level);
int mg_check_fine_level(const mg_core* c, int level); /* ... and level is not the coarsest */
int mg_sync(mg_core* c);
int mg_profile_enable(mg_core* c, int enable);
int mg_profile_read(mg_core* c, int level, int op, double* ms_total, long long* kernel_launches, long long* calls);
/* the arguments of a *_solve: mg_check_level, then the tolerances and counts */
int mg_solve_check_args(const mg_core* c, int level, double rtol, double atol, int max_cycles, int v1, int v2);
int mg_read_out2(mg_core* c, const double* d_out2); /* d_out2[0..1] -> c->h_out2, synchronised */
int mg_read_norm(mg_core* c, const double* d_out2, double* l2, double* linf); /* l2 = sqrt(sum of squares), linf = max */

/* per-operator timers around a family operator; h is a family handle */
#define PROF_BEGIN(h, level, op) mg_prof_begin(&(h)->core.prof, (h)->core.stream, (level), (op), (h)->core.launches)
#define PROF_END(h) mg_prof_end(&(h)->core.prof, (h)->core.stream, (h)->core.launches)

/* ---- the reference's operators on caller arrays ----
   Host arrays: up to two dense device temporaries (*da of na elements, *db of nb, none when nb == 0), uploaded from ha /
   hb when given; then the family launches one kernel on them and mg_tmp_finish downloads n elements of dev_out into
   host_out, frees both temporaries and counts the launch (k: the launcher's return value).  Nothing leaks on any error
   path.  Device arrays: the kernel runs in place and mg_launch_done counts it and synchronises the stream (the caller's
   next access may be on any stream). */
int mg_tmp_begin(mg_core* c, void** da, size_t na, const void* ha, void** db, size_t nb, const void* hb);
int mg_tmp_finish(mg_core* c, int k, void* host_out, const void* dev_out, size_t n, void* da, void* db);
int mg_launch_done(mg_core* c, int k);

#ifdef __cplusplus
}
#endif
#endif

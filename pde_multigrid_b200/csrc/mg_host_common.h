/*
 * mg_host_common.h -- shared helpers of the C host drivers: error reporting, CUDA call checking,
 * pitched-layout arithmetic.  Internal; the public ABI is include/mg_b200.h.
 */
#ifndef MG_HOST_COMMON_H
#define MG_HOST_COMMON_H

#include <cuda_runtime_api.h>
#include <stddef.h>

#include "../../include/mg_b200.h"
#include "mg_launch.h"

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

/* ---- tolerance-driven solve, shared by the four families (mg?d_solve) ----
   Device loop: one graph  norm(r_0) -> check -> WHILE { cycle -> norm -> check }.  When a cycle does not end on the
   buffers it started on (the 3D temporally blocked smoother ping-pongs), the body holds two cycles:
   cycle(s0 -> s1) -> norm -> check -> IF { cycle(s1 -> s0) -> norm -> check }.
   Host loop: the same kernels and the same check kernel, one read-back of the parameter block per cycle. */
typedef struct {
    mg_solve_par* h_par; /* pinned */
    mg_solve_par* d_par;
    double* d_hist;
    int hist_cap;        /* pairs d_hist has room for */
} mg_solver;

#define MG_SOLVE_SLOTS 8
#define MG_SOLVE_KEY 6
typedef struct {
    int used, failed;
    int warm;            /* a host-driven solve with this key has run a cycle: everything a capture needs exists */
    int key[MG_SOLVE_KEY];
    int two;             /* the body holds two cycles */
    unsigned snap[3][2]; /* family state (ops.save) at the start, after the first and after the second body cycle */
    cudaGraphExec_t exec;
    long long launches[3]; /* norm(r_0) + check; first body cycle + norm + check; second */
} mg_solve_slot;

typedef struct {
    void* ctx;
    cudaStream_t stream;
    const double* out2;       /* where norm() leaves {sum of squares, max} */
    long long* launches;      /* the handle's kernel counter */
    int (*norm)(void* ctx);   /* enqueue the norm pass of the solve's level into out2 */
    int (*cycle)(void* ctx);  /* one cycle the way the family's public *_vcycle runs it (host loop) */
    int (*capture_cycle)(void* ctx); /* one cycle as plain launches (device loop) */
    /* NULL for families whose cycle always ends on the buffers it started on; otherwise the host-side state:
       [0] = which buffer every level works on (must return to its start value), [1] = further bookkeeping */
    void (*save)(void* ctx, unsigned out[2]);
    void (*load)(void* ctx, const unsigned in[2]);
} mg_solve_ops;

int mg_solve_check_args(double rtol, double atol, int max_cycles, int v1, int v2);
/* slot with this key, or a free one (NULL: the cache is full, the solve runs host-driven) */
mg_solve_slot* mg_solve_slot_for(mg_solve_slot slots[MG_SOLVE_SLOTS], const int key[MG_SOLVE_KEY]);
/* the whole solve: device-driven when slot != NULL, it is warm and its graph builds; host-driven otherwise */
int mg_solve_run(const mg_solve_ops* ops, mg_solver* sv, mg_solve_slot* slot, double rtol, double atol, int max_cycles,
                 int* cycles_out, int* converged_out, double* history);
void mg_solve_free(mg_solver* sv, mg_solve_slot slots[MG_SOLVE_SLOTS]);

#ifdef __cplusplus
}
#endif
#endif

/*
 * mg3d_host.c -- C host driver of the 3D Poisson multigrid: hierarchy, V-cycle, FMG, field I/O, and the
 * multi-GPU z-slab decomposition.
 *
 * Mirrors the control flow of the reference class MultiGrid3D
 * (NOCUDA_TESI/POISSON_3D(TESI)/MultiGrid3D.cpp: InitGrids :19-47, VCycle :623-647,
 * FullMultiGridVCycle :569-585) over the sm_100a kernels of mg3d_*.cu.  Host code is C; all device work
 * goes through the launchers declared in mg_launch.h.  No CPU compute path exists here: the host only
 * computes per-level scalars (h, h^2 products, sin tables for InitF).
 *
 * Multi-GPU (the reference has none; thesis p.75 names it as future work): one process per GPU, the
 * grid is cut into z-slabs.  Rank g of P owns the global planes [g*m, (g+1)*m), m = (n-1)/P, the last
 * rank also the Dirichlet plane n-1.  A slab stores 4 ghost planes below and above (two RB sweeps per pass of the
 * temporally blocked smoother reach four planes; the fused residual+restrict needs v two planes under its first
 * coarse plane).  A level is slab-distributed while
 * m >= 8 and n >= 257; coarser levels are agglomerated: every rank holds them whole (one all-gather of the
 * restricted right-hand side on the way down, nothing on the way up) and smooths them redundantly.
 * RB Gauss-Seidel only couples opposite colours, so exchanging the just-updated colour's boundary
 * plane after every half-sweep reproduces the sequential red-then-black order exactly: the P-GPU result
 * is bit-identical to the 1-GPU result.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "mg3d_box.h"
#include "mg_comm.h"
#include "mg_host_common.h"

/* ghost planes a slab stores below / above its own planes: the temporally blocked smoother consumes four planes of
   colour 1 (and of f) on each side per pass; the fused residual+restrict reads v two planes below its first coarse plane */
#define MG_GHOST_LO 4
#define MG_GHOST_HI 4
/* bytes of addressable slack in front of and behind the fields of the arena: the pipelined smoother (mg3d_smooth_pipe.cu)
   issues unclamped, masked loads for halo sites up to 4 rows outside a field */
#define MG_ARENA_SLACK ((size_t)1 << 20)

typedef struct {
    mg_geom3d g;
    mg_coef3d c;
    void* v;
    void* f;
    double h[3];    /* h_x, h_y, h_z (values of the level's dtype) */
    int dist;       /* 1: slab-distributed over the ranks; 0: the whole level lives on this rank */
    int own_lo;     /* local plane range [own_lo, own_hi) owned by this rank */
    int own_hi;
    /* temporally blocked smoother: it works out of place, v ping-pongs between two buffers */
    void* vbuf[2];  /* vbuf[cur] == v; vbuf[1] is NULL when the level has no second buffer */
    int cur;
    void* jscratch; /* weighted Jacobi: one colour array of scratch, allocated on first use */
    unsigned char tmap_v[2][2][128] __attribute__((aligned(64)));  /* [buffer][colour] smoother boxes */
    unsigned char tmap_rr[2][2][128] __attribute__((aligned(64))); /* residual+restrict boxes */
    unsigned char tmap_fu[2][2][128] __attribute__((aligned(64))); /* fused-smoother boxes of v */
    unsigned char tmap_ff[2][128] __attribute__((aligned(64)));    /* fused-smoother boxes of f: [colour] */
    unsigned char tmap_pp[2][128] __attribute__((aligned(64)));    /* pipelined smoother: colour-1 array of v, [buffer] */
    unsigned char tmap_pf[2][128] __attribute__((aligned(64)));    /* pipelined smoother: f, [colour] */
    unsigned char tmap_pc[2][2][128] __attribute__((aligned(64))); /* this level's v as the COARSE operand of the finer level's pass: [buffer][colour] */
    /* distributed levels: 1 = the ghost planes of v (both colours, 2 below / 1 above) hold the neighbours' current values.
       Every operator leaves it 1 except the temporally blocked smoother, whose pass only writes the planes a rank owns;
       whoever reads ghost planes of v calls ensure_v_ghosts() first. */
    int vg_valid;
    /* 1 = the colour-1 ghost planes of v are valid to the full depth (InitV, set_field, setToValue, and the coarse v that
       residual+restrict has just zeroed everywhere): the pass that comes next needs no exchange in front of it */
    int vg_deep;
} mg_level3d;

/* direct NVLink halo path (mg_halo_p2p.cu): the neighbours' arenas and flag words mapped with CUDA IPC */
typedef struct {
    int enabled;
    char* peer_arena[2];          /* [0] rank-1, [1] rank+1 */
    unsigned int* flags;          /* local words, one per 128-B line: [0] raised by rank-1, [32] by rank+1, [64] push counter, [96] wait error */
    unsigned int* peer_flags[2];
    size_t* nb_off[2];            /* neighbour's byte offset of field fi (0: v buffer 0, 1: f, 2: v buffer 1) of level l inside its arena: [3*l + fi] */
    mg_geom3d* nb_geom[2];        /* neighbour's slab geometry per level */
    int* nb_own[2];               /* neighbour's own_lo, own_hi per level: [2*l], [2*l+1] */
    /* every rank of the job (the agglomeration gather stores into all of them): [rank]; the own entries are the local pointers */
    char** all_arena;
    unsigned int** all_flags;
    size_t* all_off;              /* byte offset of field fi of level l inside rank p's arena: [(p*nlevels + l)*3 + fi] */
    int gather_p2p;               /* 1: gather_level stores directly into the peers (at most MG_GATHER_MAX_PEERS of them) */
} mg_p2p;

/* core.graphs holds the V-cycle graphs: the cycle is ~100 dependent launches, most of them tiny (coarse levels, halo
   kernels); replaying them removes the per-launch gaps that dominate at 257^3 and on the 8-GPU slabs */
struct mg3d_s {
    mg_core core;
    int mode;
    int rank, nranks;
    int smoother;
    double range[6];
    cudaStream_t cstream;       /* side stream: halo exchange of the boundary planes overlapping the interior sweep */
    cudaEvent_t ev_fork, ev_join;
    mg_comm* comm;
    mg_p2p p2p;
    mg_level3d* lv;
    void* arena;     /* first field */
    void* arena_raw; /* the allocation: arena - MG_ARENA_SLACK */
    double* d_scratch; /* 2*MGK_NORM_MAX_PARTS partials + 2 outputs */
    double* d_tables;  /* 3*n0 doubles: sin tables of InitF */
    void* staging;     /* two dense device staging slots for host<->device field copies */
    size_t staging_bytes;
    cudaStream_t xstream; /* copy stream of copy_in / copy_out */
    cudaEvent_t ev_copied[2], ev_packed[2];
    long long halo_bytes; /* bytes sent by this rank in halo exchanges / gathers */
    double omega;   /* weight of MG_SMOOTHER_JACOBI */
    int arith;           /* MG_ARITH_EXACT / MG_ARITH_FAST */
    unsigned int* d_flag; /* {exactness flag of the pipelined smoother, completion counter of its fallback} */
    int full_correction; /* MG_B200_FULL_CORRECTION: correct both colours after prolongation inside a cycle */
    mg_pcg_vecs* pcg;    /* per level, allocated by the first mg3d_pcg of the level */
};

/* h = range/(real)(n-1) (N3/Grid3D.cpp:31-45) and the products of N3/MultiGrid3D.cpp:498-500,532,
   computed in the level's own precision exactly like the reference does on the host */
static void level_coefs(int dtype, int n, const double* range, double h[3], mg_coef3d* c)
{
    if (dtype == MG_F32) {
        float xr = (float)range[1] - (float)range[0];
        float yr = (float)range[3] - (float)range[2];
        float zr = (float)range[5] - (float)range[4];
        float hx = xr / (float)(n - 1), hy = yr / (float)(n - 1), hz = zr / (float)(n - 1);
        float hx2 = hx * hx, hy2 = hy * hy, hz2 = hz * hz;
        float cx = hy2 * hz2, cy = hx2 * hz2, cz = hx2 * hy2;
        float den = 2 * (cx + cy + cz);
        float rden = 1.0f / den;
        h[0] = hx; h[1] = hy; h[2] = hz;
        c->hx2 = hx2; c->hy2 = hy2; c->hz2 = hz2;
        c->cx = cx; c->cy = cy; c->cz = cz;
        c->den = den; c->rden = rden;
        c->ihx2 = 1.0f / hx2; c->ihy2 = 1.0f / hy2; c->ihz2 = 1.0f / hz2;
    } else {
        double xr = range[1] - range[0], yr = range[3] - range[2], zr = range[5] - range[4];
        double hx = xr / (double)(n - 1), hy = yr / (double)(n - 1), hz = zr / (double)(n - 1);
        double hx2 = hx * hx, hy2 = hy * hy, hz2 = hz * hz;
        double cx = hy2 * hz2, cy = hx2 * hz2, cz = hx2 * hy2;
        double den = 2 * (cx + cy + cz);
        h[0] = hx; h[1] = hy; h[2] = hz;
        c->hx2 = hx2; c->hy2 = hy2; c->hz2 = hz2;
        c->cx = cx; c->cy = cy; c->cz = cz;
        c->den = den; c->rden = 1.0 / den;
        c->ihx2 = 1.0 / hx2; c->ihy2 = 1.0 / hy2; c->ihz2 = 1.0 / hz2;
    }
    /* exact-arithmetic shortcuts (mg_exact.cuh): a power of two has frexp mantissa 0.5; den = 6*2^e has 0.75 */
    int e;
    c->fast_h = frexp(c->hx2, &e) == 0.5 && frexp(c->hy2, &e) == 0.5 && frexp(c->hz2, &e) == 0.5;
    /* ... and its reciprocal must be finite: a subnormal den (float h <= 2^-33, double h <= 2^-257) has 1/den = inf */
    c->fast_den = c->fast_h && frexp(c->den, &e) == 0.75 && isfinite(c->rden);
}

static void set_geom(mg_geom3d* g, int n, int dtype, int z0, int nzl)
{
    g->n = n;
    g->hp = mg_pitch((n + 1) / 2, dtype);
    g->plane = (long long)g->hp * n;
    g->cstride = g->plane * nzl;
    g->z0 = z0;
    g->nzl = nzl;
}

/* Slab plan of one level (pure arithmetic, also exported for tests): is the level distributed, and which
   global planes does `rank` store and own?  out = {dist, z0, nzl, own_lo, own_hi} in local indices. */
int mg3d_plan_level(int n, int nranks, int rank, int out5[5])
{
    if (!out5 || n < 3 || nranks < 1 || rank < 0 || rank >= nranks) return mg_fail(MG_ERR_ARG, "bad plan arguments");
    const int m = (n - 1) / nranks;
    /* distribute while a slab keeps >= 8 planes and the level is big enough for the halo latency to pay off:
       at 8 GPUs the 129^3 and 65^3 levels cost 0.3 ms per cycle each when distributed (11 latency-bound
       exchanges) against 0.1 ms when every GPU smooths them whole (profiles/r1_scaling.md) */
    const char* env = getenv("MG_B200_DIST_MIN_N");
    const int min_n = env ? atoi(env) : 257;
    const int dist = nranks > 1 && (n - 1) % nranks == 0 && m >= 8 && n >= min_n;
    if (!dist) {
        out5[0] = 0; out5[1] = 0; out5[2] = n; out5[3] = 0; out5[4] = n;
        return MG_OK;
    }
    const int a = rank * m, b = (rank + 1) * m + (rank == nranks - 1 ? 1 : 0);
    const int glo = rank > 0 ? MG_GHOST_LO : 0, ghi = rank < nranks - 1 ? MG_GHOST_HI : 0;
    out5[0] = 1;
    out5[1] = a - glo;
    out5[2] = (b - a) + glo + ghi;
    out5[3] = glo;
    out5[4] = glo + (b - a);
    return MG_OK;
}

static size_t field_bytes(const mg_level3d* L, int dtype)
{
    return mg_align256(2 * (size_t)L->g.cstride * mg_esize(dtype));
}

/* the levels with tensor maps (create_common makes them or fails).  The temporally blocked smoothers run there only, so
   these are the levels that keep a second v in the arena behind v and f. */
static int level_uses_tma(int n) { return (n - 1) / 2 >= MGK3D_TMA_IT; }

static void* field_ptr(mg_level3d* L, int field) { return field == MG_FIELD_V ? L->v : L->f; }

/* device address of local plane zl of colour `col` of a field */
static char* plane_ptr(const mg3d_t* mg, const mg_level3d* L, void* field, int col, int zl)
{
    return (char*)field + ((size_t)col * (size_t)L->g.cstride + (size_t)zl * (size_t)L->g.plane) * mg_esize(mg->core.dtype);
}

/* ------------------------------------------------------------------------------------------------
 * Halo exchange of a distributed level (grouped ncclSend/ncclRecv on the handle's stream).
 *   up:   my top `depth_up` owned planes        -> the lower ghosts of rank+1
 *   down: my bottom owned plane (if `down` != 0) -> the upper ghost of rank-1
 * colour_mask: bit 0 = colour-0 array, bit 1 = colour-1 array.
 * ---------------------------------------------------------------------------------------------- */
static int exchange_p2p2(mg3d_t* mg, int level, void* field, const int up2[2], const int down2[2], cudaStream_t xs);

static int exchange_p2p(mg3d_t* mg, int level, void* field, int colour_mask, int depth_up, int depth_down, cudaStream_t xs)
{
    const int up2[2] = {(colour_mask & 1) ? depth_up : 0, (colour_mask & 2) ? depth_up : 0};
    const int down2[2] = {(colour_mask & 1) ? depth_down : 0, (colour_mask & 2) ? depth_down : 0};
    return exchange_p2p2(mg, level, field, up2, down2, xs);
}

/* per-colour depths: up2[c] top owned planes of colour c go to the lower ghosts of rank+1, down2[c] bottom owned planes to the
   upper ghosts of rank-1 (0 = that colour does not travel in that direction); still ONE launch and one flag per direction */
static int exchange_p2p2(mg3d_t* mg, int level, void* field, const int up2[2], const int down2[2], cudaStream_t xs)
{
    mg_level3d* L = &mg->lv[level];
    mg_p2p* q = &mg->p2p;
    const size_t es = mg_esize(mg->core.dtype), pb = (size_t)L->g.plane * es; /* bytes per colour plane */
    const int r = mg->rank, P = mg->nranks;
    /* the neighbours run the same program: their current v buffer is the one with my index */
    const int fi = field == L->f ? 1 : (field == L->vbuf[1] && L->vbuf[1] ? 2 : 0);
    const void* src[4] = {0, 0, 0, 0};
    void* dst[4] = {0, 0, 0, 0};
    unsigned long long bytes[4] = {0, 0, 0, 0};
    unsigned int* raise[2] = {0, 0};
    int nseg = 0;
    const int any_up = up2[0] > 0 || up2[1] > 0, any_down = down2[0] > 0 || down2[1] > 0;
    const int send_up = r + 1 < P && any_up, send_down = r > 0 && any_down;
    for (int col = 0; col < 2; col++) {
        if (send_up && up2[col] > 0) { /* my top planes -> the lower ghosts of rank+1 */
            const mg_geom3d* ng = &q->nb_geom[1][level];
            src[nseg] = plane_ptr(mg, L, field, col, L->own_hi - up2[col]);
            dst[nseg] = q->peer_arena[1] + q->nb_off[1][3 * level + fi] +
                        ((size_t)col * (size_t)ng->cstride + (size_t)(q->nb_own[1][2 * level] - up2[col]) * (size_t)ng->plane) * es;
            bytes[nseg++] = pb * up2[col];
            mg->halo_bytes += (long long)(pb * up2[col]);
        }
        if (send_down && down2[col] > 0) { /* my bottom planes -> the upper ghosts of rank-1 */
            const mg_geom3d* ng = &q->nb_geom[0][level];
            src[nseg] = plane_ptr(mg, L, field, col, L->own_lo);
            dst[nseg] = q->peer_arena[0] + q->nb_off[0][3 * level + fi] +
                        ((size_t)col * (size_t)ng->cstride + (size_t)q->nb_own[0][2 * level + 1] * (size_t)ng->plane) * es;
            bytes[nseg++] = pb * down2[col];
            mg->halo_bytes += (long long)(pb * down2[col]);
        }
    }
    if (send_up) raise[1] = q->peer_flags[1] + 0;    /* its "from below" word */
    if (send_down) raise[0] = q->peer_flags[0] + 32; /* its "from above" word */
    const int recv_below = r > 0 && any_up, recv_above = r + 1 < P && any_down;
    if (xs == mg->core.stream) PROF_BEGIN(mg, level, MG_OP_OTHER);
    MG_LAUNCH(mg->core.launches, mgk_halo_exchange(xs, src, dst, bytes, raise, recv_below, recv_above, q->flags));
    if (xs == mg->core.stream) PROF_END(mg);
    return MG_OK;
}

/* depth_up / depth_down planes (<= MG_GHOST_LO / MG_GHOST_HI; 0 = nothing travels in that direction) */
static int exchange_on(mg3d_t* mg, int level, void* field, int colour_mask, int depth_up, int depth_down, cudaStream_t xs)
{
    mg_level3d* L = &mg->lv[level];
    if (!L->dist) return MG_OK;
    /* the direct NVLink path addresses the neighbour's v buffers and f inside its arena; anything else (the Jacobi scratch) goes through NCCL */
    if (mg->p2p.enabled && (field == L->vbuf[0] || field == L->vbuf[1] || field == L->f))
        return exchange_p2p(mg, level, field, colour_mask, depth_up, depth_down, xs);
    const size_t pe = (size_t)L->g.plane; /* elements per colour plane */
    const int r = mg->rank, P = mg->nranks;
    int st;
    if (xs == mg->core.stream) PROF_BEGIN(mg, level, MG_OP_OTHER);
    if ((st = mg_comm_group_start(mg->comm))) return st;
    for (int col = 0; col < 2; col++) {
        if (!(colour_mask & (1 << col))) continue;
        if (r + 1 < P) {
            if (depth_up > 0) {
                st = mg_comm_send(mg->comm, plane_ptr(mg, L, field, col, L->own_hi - depth_up), pe * depth_up, mg->core.dtype, r + 1, xs);
                mg->halo_bytes += (long long)(pe * depth_up * mg_esize(mg->core.dtype));
            }
            if (!st && depth_down > 0) st = mg_comm_recv(mg->comm, plane_ptr(mg, L, field, col, L->own_hi), pe * depth_down, mg->core.dtype, r + 1, xs);
        }
        if (!st && r > 0) {
            if (depth_down > 0) {
                st = mg_comm_send(mg->comm, plane_ptr(mg, L, field, col, L->own_lo), pe * depth_down, mg->core.dtype, r - 1, xs);
                mg->halo_bytes += (long long)(pe * depth_down * mg_esize(mg->core.dtype));
            }
            if (!st && depth_up > 0)
                st = mg_comm_recv(mg->comm, plane_ptr(mg, L, field, col, L->own_lo - depth_up), pe * depth_up, mg->core.dtype, r - 1, xs);
        }
        if (st) break;
    }
    int st2 = mg_comm_group_end(mg->comm);
    if (xs == mg->core.stream) PROF_END(mg);
    return st ? st : st2;
}

static int exchange(mg3d_t* mg, int level, void* field, int colour_mask, int depth_up, int depth_down)
{
    return exchange_on(mg, level, field, colour_mask, depth_up, depth_down, mg->core.stream);
}

/* one exchange with different depths for the two colours (one launch on the NVLink path, two grouped exchanges through NCCL) */
static int exchange2(mg3d_t* mg, int level, void* field, const int up2[2], const int down2[2])
{
    mg_level3d* L = &mg->lv[level];
    if (!L->dist) return MG_OK;
    if (mg->p2p.enabled && (field == L->vbuf[0] || field == L->vbuf[1] || field == L->f))
        return exchange_p2p2(mg, level, field, up2, down2, mg->core.stream);
    int st = MG_OK;
    for (int col = 0; col < 2 && !st; col++)
        if (up2[col] > 0 || down2[col] > 0) st = exchange_on(mg, level, field, 1 << col, up2[col], down2[col], mg->core.stream);
    return st;
}

/* The temporally blocked smoother writes the planes a rank owns into the OTHER v buffer and reads, of that buffer's ghost
   planes, nothing -- but a later pass out of it reads the Dirichlet points of colour 0 on its ghost planes (the exchange in
   front of a pass only moves colour 1).  Dirichlet values never change, so it is enough that whoever defines v on every stored
   plane (InitV, set_field, setToValue) gives the ghost planes of the other buffer the same values. */
static int mirror_v_ghosts(mg3d_t* mg, int level)
{
    mg_level3d* L = &mg->lv[level];
    if (!L->dist || !L->vbuf[1]) return MG_OK;
    void* other = L->vbuf[L->cur ^ 1];
    const size_t pb = (size_t)L->g.plane * mg_esize(mg->core.dtype);
    for (int col = 0; col < 2; col++) {
        if (L->own_lo > 0)
            MG_CUDA(cudaMemcpyAsync(plane_ptr(mg, L, other, col, 0), plane_ptr(mg, L, L->v, col, 0), pb * (size_t)L->own_lo, cudaMemcpyDeviceToDevice, mg->core.stream));
        if (L->g.nzl > L->own_hi)
            MG_CUDA(cudaMemcpyAsync(plane_ptr(mg, L, other, col, L->own_hi), plane_ptr(mg, L, L->v, col, L->own_hi),
                                    pb * (size_t)(L->g.nzl - L->own_hi), cudaMemcpyDeviceToDevice, mg->core.stream));
    }
    return MG_OK;
}

/* ghost planes of v as the colour-per-launch kernels, the fused residual+restrict and the prolongation expect them
   (2 below, 1 above, both colours): refreshed here if the temporally blocked smoother left them behind */
static int ensure_v_ghosts(mg3d_t* mg, int level)
{
    mg_level3d* L = &mg->lv[level];
    if (!L->dist || L->vg_valid) return MG_OK;
    int st = exchange(mg, level, L->v, 3, 2, 1);
    if (!st) L->vg_valid = 1;
    return st;
}

/* first agglomerated level below a distributed one: every rank computed the coarse planes under its own
   slab into its full-size array; gather them so that every rank holds the whole level.  The top plane
   n-1 (not covered by the equal shares) comes from the last rank when `top_from_last` is set, else the
   caller fills it. */
#define MG_TOP_NONE 0
#define MG_TOP_FROM_LAST 1
#define MG_TOP_ZERO 2
static int gather_level(mg3d_t* mg, int level, void* field, int top_mode)
{
    mg_level3d* L = &mg->lv[level];
    const int P = mg->nranks, m = (L->g.n - 1) / P;
    const size_t pe = (size_t)L->g.plane;
    int st = MG_OK, st2;
    if (mg->p2p.gather_p2p && field == L->f && top_mode == MG_TOP_ZERO) {
        /* the V-cycle's gather (the restricted residual): direct stores of this rank's share into every peer's copy of the level (two small launches instead of an NCCL
           all-gather: 0.03 against 0.09 ms for the 129^3 level on 8 GPUs) */
        const mg_p2p* q = &mg->p2p;
        const size_t es = mg_esize(mg->core.dtype), share = pe * (size_t)m * es;
        const void* src2[2];
        void* dst[MG_GATHER_MAX_PEERS][2];
        unsigned int* pblk[MG_GATHER_MAX_PEERS];
        int np = 0;
        for (int col = 0; col < 2; col++) src2[col] = plane_ptr(mg, L, field, col, mg->rank * m);
        for (int nr = 0; nr < P; nr++) {
            if (nr == mg->rank) continue;
            /* an agglomerated level is stored whole on every rank: same geometry, the rank's own arena offset */
            char* base = q->all_arena[nr] + q->all_off[((size_t)nr * mg->core.nlevels + level) * 3 + 1];
            for (int col = 0; col < 2; col++)
                dst[np][col] = base + ((size_t)col * (size_t)L->g.cstride + (size_t)(mg->rank * m) * (size_t)L->g.plane) * es;
            pblk[np++] = q->all_flags[nr];
            mg->halo_bytes += (long long)(2 * share);
        }
        PROF_BEGIN(mg, level, MG_OP_OTHER);
        MG_LAUNCH(mg->core.launches, mgk_gather_push(mg->core.stream, src2, (unsigned long long)share, dst, pblk, np, mg->rank, q->flags));
        if (mg->rank != P - 1) /* the Dirichlet plane n-1 of a restricted residual is +0: written locally (see below) */
            MG_LAUNCH(mg->core.launches, mgk3d_set(mg->core.stream, mg->core.dtype, field, L->g, 0.0, 1, L->g.n - 1, L->g.n));
        PROF_END(mg);
        return MG_OK;
    }
    PROF_BEGIN(mg, level, MG_OP_OTHER);
    /* both colour arrays in ONE NCCL group: one fused launch instead of two */
    st = mg_comm_group_start(mg->comm);
    for (int col = 0; col < 2 && !st; col++) {
        st = mg_comm_allgather_inplace(mg->comm, plane_ptr(mg, L, field, col, 0), pe * m, mg->core.dtype, mg->core.stream);
        mg->halo_bytes += (long long)(pe * m * mg_esize(mg->core.dtype));
    }
    st2 = mg_comm_group_end(mg->comm);
    if (!st) st = st2;
    if (!st && top_mode == MG_TOP_FROM_LAST) {
        st = mg_comm_group_start(mg->comm);
        for (int col = 0; col < 2 && !st; col++) {
            char* top = plane_ptr(mg, L, field, col, L->g.n - 1);
            if (mg->rank == P - 1) {
                for (int peer = 0; peer < P - 1 && !st; peer++) st = mg_comm_send(mg->comm, top, pe, mg->core.dtype, peer, mg->core.stream);
            } else {
                st = mg_comm_recv(mg->comm, top, pe, mg->core.dtype, P - 1, mg->core.stream);
            }
        }
        st2 = mg_comm_group_end(mg->comm);
        if (!st) st = st2;
    } else if (!st && top_mode == MG_TOP_ZERO && mg->rank != P - 1) {
        /* the restricted residual is +0 on the Dirichlet plane n-1 (injection of the zero boundary residual, N3/MultiGrid3D.cpp:113-119,
           :705): nothing to fetch, every rank but the last (which produced it) writes the zeros itself */
        int k = mgk3d_set(mg->core.stream, mg->core.dtype, field, L->g, 0.0, 1, L->g.n - 1, L->g.n);
        if (k < 0) st = mg_fail(MG_ERR_CUDA, "set launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        else mg->core.launches += k;
    }
    PROF_END(mg);
    return st;
}

/* ------------------------------------------------------------------------------------------------
 * CUDA IPC mapping of the z-neighbours' arenas and flag words (enables exchange_p2p).  Handles travel
 * through an NCCL all-gather.  If IPC / peer access is not available the NCCL send/recv path stays.
 * ---------------------------------------------------------------------------------------------- */
static int p2p_setup(mg3d_t* mg)
{
    mg_p2p* q = &mg->p2p;
    const int r = mg->rank, P = mg->nranks;
    /* what the neighbours' arenas look like: replay the allocation arithmetic for rank-1 and rank+1 */
    for (int k = 0; k < 2; k++) {
        const int nr = k == 0 ? r - 1 : r + 1;
        if (nr < 0 || nr >= P) continue;
        q->nb_off[k] = (size_t*)calloc(3 * (size_t)mg->core.nlevels, sizeof(size_t));
        q->nb_geom[k] = (mg_geom3d*)calloc((size_t)mg->core.nlevels, sizeof(mg_geom3d));
        q->nb_own[k] = (int*)calloc(2 * (size_t)mg->core.nlevels, sizeof(int));
        if (!q->nb_off[k] || !q->nb_geom[k] || !q->nb_own[k]) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
        size_t off = 0;
        for (int l = 0; l < mg->core.nlevels; l++) {
            int plan[5];
            mg3d_plan_level(mg->lv[l].g.n, P, nr, plan);
            set_geom(&q->nb_geom[k][l], mg->lv[l].g.n, mg->core.dtype, plan[1], plan[2]);
            q->nb_own[k][2 * l] = plan[3];
            q->nb_own[k][2 * l + 1] = plan[4];
            const size_t fb = mg_align256(2 * (size_t)q->nb_geom[k][l].cstride * mg_esize(mg->core.dtype));
            q->nb_off[k][3 * l] = off; off += fb;
            q->nb_off[k][3 * l + 1] = off; off += fb;
            q->nb_off[k][3 * l + 2] = off;
            if (level_uses_tma(mg->lv[l].g.n)) off += fb;
        }
    }
    q->all_arena = (char**)calloc((size_t)P, sizeof(char*));
    q->all_flags = (unsigned int**)calloc((size_t)P, sizeof(unsigned int*));
    q->all_off = (size_t*)calloc((size_t)P * 3 * (size_t)mg->core.nlevels, sizeof(size_t));
    if (!q->all_arena || !q->all_flags || !q->all_off) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    for (int nr = 0; nr < P; nr++) { /* the same allocation arithmetic for every rank of the job */
        size_t off = 0;
        for (int l = 0; l < mg->core.nlevels; l++) {
            int plan[5];
            mg_geom3d g;
            mg3d_plan_level(mg->lv[l].g.n, P, nr, plan);
            set_geom(&g, mg->lv[l].g.n, mg->core.dtype, plan[1], plan[2]);
            const size_t fb = mg_align256(2 * (size_t)g.cstride * mg_esize(mg->core.dtype));
            size_t* o = &q->all_off[((size_t)nr * mg->core.nlevels + l) * 3];
            o[0] = off; off += fb;
            o[1] = off; off += fb;
            o[2] = off;
            if (level_uses_tma(mg->lv[l].g.n)) off += fb;
        }
    }
    MG_CUDA(cudaMalloc((void**)&q->flags, MG_HALO_FLAG_WORDS * sizeof(unsigned int)));
    MG_CUDA(cudaMemsetAsync(q->flags, 0, MG_HALO_FLAG_WORDS * sizeof(unsigned int), mg->core.stream));
    /* all-gather {arena handle, flags handle} (64 B each) */
    cudaIpcMemHandle_t mine[2];
    int ok = 1; /* a rank without IPC still takes part in the collectives below, then everybody keeps NCCL */
    memset(mine, 0, sizeof mine);
    if (cudaIpcGetMemHandle(&mine[0], mg->arena_raw) != cudaSuccess || cudaIpcGetMemHandle(&mine[1], q->flags) != cudaSuccess) {
        cudaGetLastError();
        ok = 0;
    }
    const size_t hb = sizeof mine; /* 128 */
    unsigned char* d_all = NULL;
    MG_CUDA(cudaMalloc((void**)&d_all, hb * P));
    MG_CUDA(cudaMemcpyAsync(d_all + hb * r, mine, hb, cudaMemcpyHostToDevice, mg->core.stream));
    int st = mg_comm_allgather_inplace(mg->comm, d_all, hb / 4, MG_F32, mg->core.stream);
    if (st) { cudaFree(d_all); return st; }
    cudaIpcMemHandle_t* all = (cudaIpcMemHandle_t*)malloc(hb * P);
    if (!all) { cudaFree(d_all); return mg_fail(MG_ERR_NOMEM, "host allocation failed"); }
    cudaError_t e = cudaMemcpyAsync(all, d_all, hb * P, cudaMemcpyDeviceToHost, mg->core.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
    cudaFree(d_all);
    if (e != cudaSuccess) ok = 0;
    /* map every peer once (the z-neighbours for the halo exchanges, everybody for the agglomeration gather) */
    for (int nr = 0; nr < P && ok; nr++) {
        if (nr == r) {
            q->all_arena[nr] = (char*)mg->arena;
            q->all_flags[nr] = q->flags;
            continue;
        }
        void *pa = NULL, *pf = NULL;
        if (cudaIpcOpenMemHandle(&pa, all[2 * nr], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
            cudaIpcOpenMemHandle(&pf, all[2 * nr + 1], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            cudaGetLastError();
            ok = 0;
            break;
        }
        q->all_arena[nr] = (char*)pa + MG_ARENA_SLACK;
        q->all_flags[nr] = (unsigned int*)pf;
    }
    for (int k = 0; k < 2 && ok; k++) {
        const int nr = k == 0 ? r - 1 : r + 1;
        if (nr < 0 || nr >= P) continue;
        q->peer_arena[k] = q->all_arena[nr];
        q->peer_flags[k] = q->all_flags[nr];
    }
    free(all);
    /* every rank must agree on the transport: all-reduce the success bit */
    double* d2 = mg->d_scratch + 2 * MGK_NORM_MAX_PARTS;
    double h2[2] = {ok ? 0.0 : 1.0, 0.0};
    MG_CUDA(cudaMemcpyAsync(d2, h2, sizeof h2, cudaMemcpyHostToDevice, mg->core.stream));
    if ((st = mg_comm_allreduce_sum_max(mg->comm, d2, mg->core.stream))) return st;
    MG_CUDA(cudaMemcpyAsync(h2, d2, sizeof h2, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    q->enabled = h2[0] == 0.0;
    q->gather_p2p = q->enabled && P - 1 <= MG_GATHER_MAX_PEERS;
    return MG_OK;
}

static void p2p_teardown(mg3d_t* mg)
{
    mg_p2p* q = &mg->p2p;
    for (int k = 0; k < 2; k++) {
        free(q->nb_off[k]); free(q->nb_geom[k]); free(q->nb_own[k]);
    }
    if (mg->comm && q->flags) { /* nobody unmaps or frees while a neighbour may still be pushing */
        double* d2 = mg->d_scratch + 2 * MGK_NORM_MAX_PARTS;
        if (mg_comm_allreduce_sum_max(mg->comm, d2, mg->core.stream) == MG_OK) cudaStreamSynchronize(mg->core.stream);
    }
    for (int nr = 0; nr < mg->nranks; nr++) { /* unmap after that barrier */
        if (nr == mg->rank) continue;
        if (q->all_arena && q->all_arena[nr]) cudaIpcCloseMemHandle(q->all_arena[nr] - MG_ARENA_SLACK);
        if (q->all_flags && q->all_flags[nr]) cudaIpcCloseMemHandle(q->all_flags[nr]);
    }
    free(q->all_arena); free(q->all_flags); free(q->all_off);
    if (q->flags) cudaFree(q->flags);
    memset(q, 0, sizeof *q);
}

static int halo_error_check(mg3d_t* mg)
{
    if (!mg->p2p.enabled) return MG_OK;
    unsigned int err = 0;
    MG_CUDA(cudaMemcpyAsync(&err, mg->p2p.flags + 96, sizeof err, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    if (err) return mg_fail(MG_ERR_COMM, "halo exchange timed out waiting for a neighbour's flag (rank %d)", mg->rank);
    return MG_OK;
}

/* ------------------------------------------------------------------------------------------------ */

static int create_common(mg3d_t** out, const int sz[3], const double range[6], int dtype, int residual_mode, int rank,
                         int nranks, const void* uid)
{
    if (!out || !sz || !range) return mg_fail(MG_ERR_ARG, "null argument");
    *out = NULL;
    /* N3/Grid3D.cpp:10-29 asserts */
    if (sz[0] != sz[1] || sz[0] != sz[2]) return mg_fail(MG_ERR_ARG, "sizeX == sizeY == sizeZ required (got %d,%d,%d; N3/Grid3D.cpp:10-11): non-cubic grids go through mg3b_create", sz[0], sz[1], sz[2]);
    const int n = sz[0];
    if (n < 3 || ((n - 1) & (n - 2)) != 0) return mg_fail(MG_ERR_ARG, "size must be 2^k+1 with k >= 1 (got %d)", n);
    if (!(range[1] > range[0]) || !(range[3] > range[2]) || !(range[5] > range[4])) return mg_fail(MG_ERR_ARG, "range must satisfy b > a on every axis");
    if (dtype != MG_F32 && dtype != MG_F64) return mg_fail(MG_ERR_ARG, "dtype must be MG_F32 or MG_F64");
    if (residual_mode != MG_REF_COMPAT && residual_mode != MG_CORRECTED) return mg_fail(MG_ERR_ARG, "bad residual_mode");
    if (nranks < 1 || rank < 0 || rank >= nranks) return mg_fail(MG_ERR_ARG, "bad rank %d of %d", rank, nranks);
    if (nranks > 1) {
        if ((nranks & (nranks - 1)) != 0) return mg_fail(MG_ERR_ARG, "the number of GPUs must be a power of two (got %d)", nranks);
        int plan[5];
        mg3d_plan_level(n, nranks, rank, plan);
        if (!plan[0]) return mg_fail(MG_ERR_ARG, "grid %d^3 is too small for %d z-slabs (needs >= 8 planes per GPU and n >= 257, or MG_B200_DIST_MIN_N)", n, nranks);
        if (!uid) return mg_fail(MG_ERR_ARG, "multi-GPU handles need the NCCL unique id");
    }
    int st = mg_require_device();
    if (st) return st;

    mg3d_t* mg = (mg3d_t*)calloc(1, sizeof *mg);
    if (!mg) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    mg->core.dtype = dtype;
    mg->mode = residual_mode;
    mg->rank = rank;
    mg->nranks = nranks;
    mg->smoother = MG_SMOOTHER_AUTO;
    mg->omega = 6.0 / 7.0;
    mg->arith = MG_ARITH_EXACT;
    mg->full_correction = getenv("MG_B200_FULL_CORRECTION") != NULL;
    memcpy(mg->range, range, sizeof mg->range);
    mg->core.nlevels = mg_num_levels_for(n);
    mg->lv = (mg_level3d*)calloc((size_t)mg->core.nlevels, sizeof(mg_level3d));
    if (!mg->lv) { free(mg); return mg_fail(MG_ERR_NOMEM, "host allocation failed"); }

    size_t total = 0;
    int nl = n;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3d* L = &mg->lv[l];
        int plan[5];
        mg3d_plan_level(nl, nranks, rank, plan);
        L->dist = plan[0];
        set_geom(&L->g, nl, dtype, plan[1], plan[2]);
        L->own_lo = plan[3];
        L->own_hi = plan[4];
        L->vg_valid = 1;
        L->vg_deep = 1;
        level_coefs(dtype, nl, range, L->h, &L->c);
        total += (size_t)(level_uses_tma(nl) ? 3 : 2) * field_bytes(L, dtype);
        nl = (nl - 1) / 2 + 1; /* N3/MultiGrid3D.cpp:40-42 */
    }
    cudaError_t e = cudaMalloc(&mg->arena_raw, total + 2 * MG_ARENA_SLACK);
    if (e != cudaSuccess) {
        free(mg->lv); free(mg);
        return mg_fail(e == cudaErrorMemoryAllocation ? MG_ERR_NOMEM : MG_ERR_CUDA, "cudaMalloc of %zu bytes failed: %s", total, cudaGetErrorString(e));
    }
    mg->arena = (char*)mg->arena_raw + MG_ARENA_SLACK;
    char* p = (char*)mg->arena;
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3d* L = &mg->lv[l];
        L->v = p; p += field_bytes(L, dtype);
        L->f = p; p += field_bytes(L, dtype);
        L->vbuf[0] = L->v;
        if (level_uses_tma(L->g.n)) { L->vbuf[1] = p; p += field_bytes(L, dtype); }
    }
    if ((st = mg_core_init(&mg->core))) { mg3d_destroy(mg); return st; }
    if (cudaMalloc((void**)&mg->d_scratch, (2 * MGK_NORM_MAX_PARTS + 2) * sizeof(double)) != cudaSuccess ||
        cudaMalloc((void**)&mg->d_tables, 3 * (size_t)n * sizeof(double)) != cudaSuccess ||
        cudaMalloc((void**)&mg->d_flag, 256) != cudaSuccess || cudaMemsetAsync(mg->d_flag, 0, 256, mg->core.stream) != cudaSuccess) {
        int code = mg_fail(MG_ERR_CUDA, "stream/scratch setup failed: %s", cudaGetErrorString(cudaGetLastError()));
        mg3d_destroy(mg);
        return code;
    }
    if (nranks > 1) {
        if (cudaStreamCreateWithFlags(&mg->cstream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&mg->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&mg->ev_join, cudaEventDisableTiming) != cudaSuccess) {
            int code = mg_fail(MG_ERR_CUDA, "side stream setup failed: %s", cudaGetErrorString(cudaGetLastError()));
            mg3d_destroy(mg);
            return code;
        }
        st = mg_comm_create(&mg->comm, rank, nranks, uid);
        if (!st) st = p2p_setup(mg);
        if (st) { mg3d_destroy(mg); return st; }
    }
    /* TMA tensor maps for the levels large enough to fill the z-marching tiles */
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3d* L = &mg->lv[l];
        if (!level_uses_tma(L->g.n)) continue;
        const int es = (int)mg_esize(dtype);
        for (int b = 0; b < 2 && !st; b++) {
            for (int col = 0; col < 2 && !st; col++) {
                char* base = plane_ptr(mg, L, L->vbuf[b], col, 0);
                st = mg_tma_make_colour_map(L->tmap_v[b][col], dtype, base, &L->g, MGK3D_TMA_BOX_I(es), MGK3D_TMA_BOX_Y);
                if (!st) st = mg_tma_make_colour_map(L->tmap_rr[b][col], dtype, base, &L->g, MGK3D_RR_BOX_I(es), MGK3D_RR_BOX_Y);
                if (!st) st = mg_tma_make_colour_map(L->tmap_fu[b][col], dtype, base, &L->g, MGK3D_FU_BOX_I(es), MGK3D_FU_BOX_Y);
                if (!st && col == 1) st = mg_tma_make_colour_map(L->tmap_pp[b], dtype, base, &L->g, MGK3D_PP_BOX_I(es), MGK3D_PP_BOX_Y);
            }
        }
        for (int col = 0; col < 2 && !st; col++) {
            st = mg_tma_make_colour_map(L->tmap_ff[col], dtype, plane_ptr(mg, L, L->f, col, 0), &L->g, MGK3D_FU_BOX_I(es), MGK3D_FU_BOX_Y);
            if (!st) st = mg_tma_make_colour_map(L->tmap_pf[col], dtype, plane_ptr(mg, L, L->f, col, 0), &L->g, MGK3D_PP_BOX_I(es), MGK3D_PP_BOX_Y);
        }
        if (st) { mg3d_destroy(mg); return st; }
    }
    /* a level below one with tensor maps is the coarse operand of that level's fused prolongation */
    for (int l = 1; l < mg->core.nlevels && !st; l++) {
        mg_level3d* L = &mg->lv[l];
        if (!level_uses_tma(mg->lv[l - 1].g.n)) continue;
        const int es = (int)mg_esize(dtype);
        for (int b = 0; b < 2 && !st; b++) {
            if (!L->vbuf[b]) continue;
            for (int col = 0; col < 2 && !st; col++)
                st = mg_tma_make_colour_map(L->tmap_pc[b][col], dtype, plane_ptr(mg, L, L->vbuf[b], col, 0), &L->g, MGK3D_PP_CBOX_I(es), MGK3D_PP_CBOX_Y);
        }
        if (st) { mg3d_destroy(mg); return st; }
    }
    /* pad elements of the layout are never used by a kernel, but keep them defined */
    if (cudaMemsetAsync(mg->arena_raw, 0, total + 2 * MG_ARENA_SLACK, mg->core.stream) != cudaSuccess) {
        int code = mg_fail(MG_ERR_CUDA, "arena clear failed: %s", cudaGetErrorString(cudaGetLastError()));
        mg3d_destroy(mg);
        return code;
    }
    st = mg3d_init_problem(mg);
    if (st) { mg3d_destroy(mg); return st; }
    *out = mg;
    return MG_OK;
}

int mg3d_create(mg3d_t** out, const int sz[3], const double range[6], int dtype, int residual_mode)
{
    return create_common(out, sz, range, dtype, residual_mode, 0, 1, NULL);
}

int mg3d_create_dist(mg3d_t** out, const int sz[3], const double range[6], int dtype, int residual_mode, int rank,
                     int nranks, const void* nccl_unique_id)
{
    return create_common(out, sz, range, dtype, residual_mode, rank, nranks, nccl_unique_id);
}

int mg3d_destroy(mg3d_t* mg)
{
    if (!mg) return MG_OK;
    if (mg->core.stream) cudaStreamSynchronize(mg->core.stream);
    /* captured slab cycles hold NCCL operations: their graphs go before the communicator (mg_core_free's second call
       finds the cache empty) */
    mg_graphs_free(&mg->core.graphs);
    p2p_teardown(mg); /* its barrier runs on the handle's stream, which the core destroys */
    if (mg->comm) mg_comm_destroy(mg->comm);
    if (mg->cstream) { cudaStreamSynchronize(mg->cstream); cudaStreamDestroy(mg->cstream); }
    if (mg->ev_fork) cudaEventDestroy(mg->ev_fork);
    if (mg->ev_join) cudaEventDestroy(mg->ev_join);
    mg_core_free(&mg->core);
    if (mg->arena_raw) cudaFree(mg->arena_raw);
    if (mg->d_scratch) cudaFree(mg->d_scratch);
    if (mg->d_tables) cudaFree(mg->d_tables);
    if (mg->d_flag) cudaFree(mg->d_flag);
    if (mg->xstream) {
        cudaStreamSynchronize(mg->xstream);
        for (int i = 0; i < 2; i++) { cudaEventDestroy(mg->ev_copied[i]); cudaEventDestroy(mg->ev_packed[i]); }
        cudaStreamDestroy(mg->xstream);
    }
    if (mg->staging) cudaFree(mg->staging);
    for (int l = 0; mg->lv && l < mg->core.nlevels; l++)
        if (mg->lv[l].jscratch) cudaFree(mg->lv[l].jscratch);
    for (int l = 0; mg->pcg && l < mg->core.nlevels; l++) mg_pcg_vecs_free(&mg->pcg[l]);
    free(mg->pcg);
    free(mg->lv);
    free(mg);
    return MG_OK;
}

int mg3d_num_levels(const mg3d_t* mg) { return mg ? mg->core.nlevels : 0; }
int mg3d_level_size(const mg3d_t* mg, int level) { return (mg && level >= 0 && level < mg->core.nlevels) ? mg->lv[level].g.n : 0; }
double mg3d_level_h(const mg3d_t* mg, int level) { return (mg && level >= 0 && level < mg->core.nlevels) ? mg->lv[level].h[0] : 0.0; }
void* mg3d_stream(mg3d_t* mg) { return mg ? (void*)mg->core.stream : NULL; }
long long mg3d_kernel_launches(const mg3d_t* mg) { return mg ? mg->core.launches : 0; }
long long mg3d_halo_bytes(const mg3d_t* mg) { return mg ? mg->halo_bytes : 0; }

int mg3d_owned_range(const mg3d_t* mg, int level, int* z_begin, int* z_count)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    const mg_level3d* L = &mg->lv[level];
    if (z_begin) *z_begin = L->g.z0 + L->own_lo;
    if (z_count) *z_count = L->own_hi - L->own_lo;
    return MG_OK;
}

int mg3d_set_smoother(mg3d_t* mg, int smoother, int sweeps_per_pass)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    if (smoother < MG_SMOOTHER_AUTO || smoother > MG_SMOOTHER_PIPE) return mg_fail(MG_ERR_ARG, "bad smoother %d", smoother);
    /* sweeps per HBM pass is a property of the implementation: the temporally blocked smoothers do two, the others one;
       MG_SMOOTHER_AUTO picks per level and call, so it takes either value */
    const int two = smoother == MG_SMOOTHER_FUSED || smoother == MG_SMOOTHER_PIPE;
    if (smoother == MG_SMOOTHER_AUTO ? (sweeps_per_pass != 1 && sweeps_per_pass != 2) : sweeps_per_pass != (two ? 2 : 1))
        return mg_fail(MG_ERR_ARG, "sweeps_per_pass %d is not what smoother %d does (%s)", sweeps_per_pass, smoother,
                       smoother == MG_SMOOTHER_AUTO ? "1 or 2" : two ? "2" : "1");
    mg->smoother = smoother;
    return MG_OK;
}

int mg3d_set_arith(mg3d_t* mg, int arith)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    if (arith != MG_ARITH_EXACT && arith != MG_ARITH_FAST) return mg_fail(MG_ERR_ARG, "bad arithmetic mode %d", arith);
    mg->arith = arith;
    return MG_OK;
}

int mg3d_set_jacobi_weight(mg3d_t* mg, double omega)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    if (!(omega > 0.0 && omega <= 1.0)) return mg_fail(MG_ERR_ARG, "Jacobi weight %g outside (0,1]", omega);
    mg->omega = mg->core.dtype == MG_F32 ? (double)(float)omega : omega;
    mg_graphs_drop(&mg->core.graphs, MG_GRAPH_KEY_SMOOTHER, MG_SMOOTHER_JACOBI); /* captured cycles carry the old weight as a kernel argument */
    return MG_OK;
}

int mg3d_profile(mg3d_t* mg, int enable) { return mg_profile_enable(MG_CORE(mg), enable); }
int mg3d_profile_read(mg3d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls)
{
    return mg_profile_read(MG_CORE(mg), level, op, ms_total, kernel_launches, calls);
}

int mg3d_sync(mg3d_t* mg)
{
    int st = mg_sync(MG_CORE(mg));
    return st ? st : halo_error_check(mg);
}

/* dense host array (x fastest, idx = x + y*n + z*n*n) <-> colour-split device field, local planes [zl_lo, zl_hi) of the
   field <-> the start of the host array.  Chunks of planes travel through two dense staging slots on a copy stream while
   the repack kernel of the previous chunk runs on the handle's stream: the PCIe link never waits for a kernel, v and f
   uploads follow each other without a gap, and the staging memory is two chunks instead of a whole field. */
#define MG_XFER_CHUNK_BYTES ((size_t)96 << 20)

static int xfer_reserve(mg3d_t* mg, size_t plane_bytes, int* planes_per_chunk)
{
    int ppc = (int)(MG_XFER_CHUNK_BYTES / plane_bytes);
    if (ppc < 1) ppc = 1;
    const size_t need = 2 * (size_t)ppc * plane_bytes;
    if (mg->staging_bytes < need) {
        if (mg->staging) { MG_CUDA(cudaStreamSynchronize(mg->core.stream)); cudaFree(mg->staging); mg->staging = NULL; mg->staging_bytes = 0; }
        MG_CUDA(cudaMalloc(&mg->staging, need));
        mg->staging_bytes = need;
    }
    if (!mg->xstream) {
        MG_CUDA(cudaStreamCreateWithFlags(&mg->xstream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            MG_CUDA(cudaEventCreateWithFlags(&mg->ev_copied[i], cudaEventDisableTiming));
            MG_CUDA(cudaEventCreateWithFlags(&mg->ev_packed[i], cudaEventDisableTiming));
        }
    }
    *planes_per_chunk = ppc;
    return MG_OK;
}

static int copy_in(mg3d_t* mg, void* dev, const mg_geom3d* g, const void* host, int zl_lo, int zl_hi)
{
    const size_t pbytes = (size_t)g->n * g->n * mg_esize(mg->core.dtype);
    int ppc, st = xfer_reserve(mg, pbytes, &ppc);
    if (st) return st;
    /* the copy stream starts after whatever the handle's stream has queued that may still read the staging slots */
    MG_CUDA(cudaEventRecord(mg->ev_packed[0], mg->core.stream));
    MG_CUDA(cudaEventRecord(mg->ev_packed[1], mg->core.stream));
    int k = 0;
    for (int z = zl_lo; z < zl_hi; z += ppc, k++) {
        const int nz = zl_hi - z < ppc ? zl_hi - z : ppc, slot = k & 1;
        char* stg = (char*)mg->staging + (size_t)slot * ppc * pbytes;
        MG_CUDA(cudaStreamWaitEvent(mg->xstream, mg->ev_packed[slot], 0)); /* the slot's previous chunk has been repacked */
        MG_CUDA(cudaMemcpyAsync(stg, (const char*)host + (size_t)(z - zl_lo) * pbytes, (size_t)nz * pbytes, cudaMemcpyHostToDevice, mg->xstream));
        MG_CUDA(cudaEventRecord(mg->ev_copied[slot], mg->xstream));
        MG_CUDA(cudaStreamWaitEvent(mg->core.stream, mg->ev_copied[slot], 0));
        MG_LAUNCH(mg->core.launches, mgk3d_repack(mg->core.stream, mg->core.dtype, dev, *g, stg, 1, z, z + nz));
        MG_CUDA(cudaEventRecord(mg->ev_packed[slot], mg->core.stream));
    }
    return MG_OK;
}

static int copy_out(mg3d_t* mg, void* host, const void* dev, const mg_geom3d* g, int zl_lo, int zl_hi)
{
    const size_t pbytes = (size_t)g->n * g->n * mg_esize(mg->core.dtype);
    int ppc, st = xfer_reserve(mg, pbytes, &ppc);
    if (st) return st;
    MG_CUDA(cudaEventRecord(mg->ev_copied[0], mg->xstream));
    MG_CUDA(cudaEventRecord(mg->ev_copied[1], mg->xstream));
    int k = 0;
    for (int z = zl_lo; z < zl_hi; z += ppc, k++) {
        const int nz = zl_hi - z < ppc ? zl_hi - z : ppc, slot = k & 1;
        char* stg = (char*)mg->staging + (size_t)slot * ppc * pbytes;
        MG_CUDA(cudaStreamWaitEvent(mg->core.stream, mg->ev_copied[slot], 0)); /* the slot's previous chunk is on its way to the host */
        MG_LAUNCH(mg->core.launches, mgk3d_repack(mg->core.stream, mg->core.dtype, (void*)dev, *g, stg, 0, z, z + nz));
        MG_CUDA(cudaEventRecord(mg->ev_packed[slot], mg->core.stream));
        MG_CUDA(cudaStreamWaitEvent(mg->xstream, mg->ev_packed[slot], 0));
        MG_CUDA(cudaMemcpyAsync((char*)host + (size_t)(z - zl_lo) * pbytes, stg, (size_t)nz * pbytes, cudaMemcpyDeviceToHost, mg->xstream));
        MG_CUDA(cudaEventRecord(mg->ev_copied[slot], mg->xstream));
    }
    MG_CUDA(cudaStreamSynchronize(mg->xstream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return halo_error_check(mg); /* data computed from ghost planes a neighbour never delivered must not look like a result */
}

/* host_dense holds the planes this rank owns (mg3d_owned_range): the whole grid on one GPU */
int mg3d_set_field(mg3d_t* mg, int level, int field, const void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3d* L = &mg->lv[level];
    st = copy_in(mg, field_ptr(L, field), &L->g, host_dense, L->own_lo, L->own_hi);
    if (!st) st = exchange(mg, level, field_ptr(L, field), 3, MG_GHOST_LO, MG_GHOST_HI);
    if (st) return st;
    if (field == MG_FIELD_V) {
        L->vg_valid = L->vg_deep = 1;
        if ((st = mirror_v_ghosts(mg, level))) return st;
    }
    MG_CUDA(cudaStreamSynchronize(mg->core.stream)); /* host buffer may be reused by the caller */
    return MG_OK;
}

int mg3d_get_field(mg3d_t* mg, int level, int field, void* host_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3d* L = &mg->lv[level];
    return copy_out(mg, host_dense, field_ptr(L, field), &L->g, L->own_lo, L->own_hi);
}

/* sin(PI*coord) per axis for one level, computed with the host libm exactly like N3/Grid3D.cpp:88-92 and
   N3/Grid3D.cpp:146-150 (float coordinate, double sine), uploaded into mg->d_tables (x | y | z, n each) */
static int upload_sin_tables(mg3d_t* mg, int level)
{
    const double PI = 3.141592653589793; /* N3/inclusion.h:9 */
    const mg_level3d* L = &mg->lv[level];
    const int n = L->g.n;
    double* tab = (double*)malloc(3 * (size_t)n * sizeof(double));
    if (!tab) return mg_fail(MG_ERR_NOMEM, "host allocation failed");
    for (int a = 0; a < 3; a++)
        for (int i = 0; i < n; i++) {
            /* float x = x_a + posX*h_x;  sin(PI*x) in double */
            double x;
            if (mg->core.dtype == MG_F32) {
                float xf = (float)mg->range[2 * a] + i * (float)L->h[a];
                x = xf;
            } else {
                x = mg->range[2 * a] + i * L->h[a];
            }
            tab[(size_t)a * n + i] = sin(PI * x);
        }
    cudaError_t e = cudaMemcpyAsync(mg->d_tables, tab, 3 * (size_t)n * sizeof(double), cudaMemcpyHostToDevice, mg->core.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(mg->core.stream);
    free(tab);
    if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e));
    return MG_OK;
}

/* Grid3D::InitV / InitF on every level (N3/Grid3D.cpp:61-96); ghost planes are initialised like owned ones */
int mg3d_init_problem(mg3d_t* mg)
{
    if (!mg) return mg_fail(MG_ERR_ARG, "null handle");
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3d* L = &mg->lv[l];
        const int n = L->g.n;
        int st = upload_sin_tables(mg, l);
        if (st) return st;
        int k1 = mgk3d_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 1, 0, L->g.nzl);
        int k2 = mgk3d_init_f(mg->core.stream, mg->core.dtype, L->f, L->g, mg->d_tables, mg->d_tables + n, mg->d_tables + 2 * n, 0, L->g.nzl);
        if (k1 < 0 || k2 < 0) return mg_fail(MG_ERR_CUDA, "init launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        mg->core.launches += k1 + k2;
        cudaError_t e = cudaStreamSynchronize(mg->core.stream); /* d_tables is reused by the next level */
        if (e != cudaSuccess) return mg_fail(MG_ERR_CUDA, "init failed: %s", cudaGetErrorString(e));
    }
    /* The init kernels wrote the ghost planes locally.  With the direct-store halo transport a neighbour that
       is already past this point could push into them before those kernels ran here: a bidirectional
       exchange per distributed level is the handshake that orders the two (and it is cheap). */
    for (int l = 0; l < mg->core.nlevels; l++) {
        mg_level3d* L = &mg->lv[l];
        int st = exchange(mg, l, L->v, 3, MG_GHOST_LO, MG_GHOST_HI);
        if (!st) st = exchange(mg, l, L->f, 3, MG_GHOST_LO, MG_GHOST_HI);
        if (!st) st = mirror_v_ghosts(mg, l);
        if (st) return st;
        L->vg_valid = L->vg_deep = 1;
    }
    return MG_OK;
}

/* interior planes this rank updates, in local indices */
static void interior_range(const mg_level3d* L, int* lo, int* hi)
{
    const int first = 1 - L->g.z0, last = L->g.n - 2 - L->g.z0; /* local indices of global planes 1 and n-2 */
    *lo = L->own_lo > first ? L->own_lo : first;
    *hi = (L->own_hi - 1 < last ? L->own_hi - 1 : last) + 1;
}

/* Relax: ncycles x (red half-sweep, black half-sweep), N3/MultiGrid3D.cpp:489-567.  On a distributed
   level the boundary planes of the colour just updated go to the neighbours after every half-sweep. */
static int relax_launch(mg3d_t* mg, mg_level3d* L, int colour, int lo, int hi, int use_tma)
{
    if (hi <= lo) return MG_OK;
    if (use_tma)
        MG_LAUNCH(mg->core.launches, mgk3d_relax_colour_tma(mg->core.stream, mg->core.dtype, L->tmap_v[L->cur][colour ^ 1], L->v, L->f, L->g, L->c, colour, lo, hi));
    else
        MG_LAUNCH(mg->core.launches, mgk3d_relax_colour(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, colour, lo, hi));
    return MG_OK;
}

/* the kernel family that relaxes a level: PIPE (register-tiled) and FUSED (shared memory) are the temporally blocked
   smoothers, the COLOUR ones sweep one colour per launch */
typedef enum { MG_RELAX_JACOBI, MG_RELAX_PIPE, MG_RELAX_FUSED, MG_RELAX_COLOUR_TMA, MG_RELAX_COLOUR } mg_relax3d;
typedef struct {
    mg_relax3d relax;    /* PIPE and FUSED run pairs of sweeps; an odd last sweep runs as COLOUR_TMA */
    int tma;             /* residual+restrict, the residual norm and the one-colour sweeps read v through tensor maps */
    int tail;            /* the V-cycle from this level down is one launch of the coarse-tail kernel */
    int correct_colour1; /* a correction followed by red-black post-smoothing only needs the colour-1 points */
} mg_path3d;

/* The kernels that work on `level`: the only place that decides them.  Computed on every call from the smoother, the level's
   geometry and coefficients and MG_B200_FULL_CORRECTION, so a mg3d_set_smoother between two calls takes effect. */
static mg_path3d level_path(const mg3d_t* mg, int level)
{
    const mg_level3d* L = &mg->lv[level];
    const int s = mg->smoother;
    mg_path3d p;
    p.tma = level_uses_tma(L->g.n) && level + 1 < mg->core.nlevels && s != MG_SMOOTHER_COLOUR; /* the TMA residuals read level+1 */
    /* the scaled arithmetic of the pipelined pass is exact: the same power-of-two h^2 on every axis, inside its guard's range */
    const int pipe_exact = L->c.fast_den && L->c.hx2 == L->c.hy2 && L->c.hy2 == L->c.hz2 && mgk3d_pipe_exact_range(mg->core.dtype, L->c.hx2);
    p.relax = s == MG_SMOOTHER_JACOBI ? MG_RELAX_JACOBI
            : (s == MG_SMOOTHER_PIPE || s == MG_SMOOTHER_AUTO) && p.tma && pipe_exact && (!L->dist || L->own_hi - L->own_lo >= 8) ? MG_RELAX_PIPE
            : s == MG_SMOOTHER_FUSED && p.tma && !L->dist ? MG_RELAX_FUSED
            : p.tma ? MG_RELAX_COLOUR_TMA : MG_RELAX_COLOUR;
    p.tail = L->g.n <= MGK3D_TAIL_N && !L->dist && mg->core.nlevels - level <= MGK3D_TAIL_MAX_LEVELS && p.relax != MG_RELAX_JACOBI;
    p.correct_colour1 = p.relax != MG_RELAX_JACOBI && !mg->full_correction;
    return p;
}

/* 1 when relax_level(level, n > 0) takes the overlapped path: the boundary planes of the slab and their halo exchange
   run on the side stream while the interior planes are swept; every half-sweep ends with a join.  (A level the temporally
   blocked smoother handles exchanges once per pass, in front of it, on the main stream.) */
static int relax_overlaps(const mg3d_t* mg, int level)
{
    const mg_level3d* L = &mg->lv[level];
    const mg_relax3d r = level_path(mg, level).relax;
    int lo, hi;
    interior_range(L, &lo, &hi);
    return L->dist && !mg->core.prof.enabled && hi - lo >= 4 && (r == MG_RELAX_COLOUR_TMA || r == MG_RELAX_COLOUR);
}

/* A halo exchange whose ghost planes are first read by the boundary-plane kernel of the smoothing call that follows
   (an overlapped one: the caller checks relax_overlaps): it goes to the side stream, the main stream carries on with
   the interior sweep, and the join of that call's first half-sweep covers it.  Exchanges keep their global order:
   everything on the side stream is joined before the next exchange on the main stream. */
static int exchange_deferred(mg3d_t* mg, int level, void* field, int colour_mask, int depth_up, int down)
{
    MG_CUDA(cudaEventRecord(mg->ev_fork, mg->core.stream));
    MG_CUDA(cudaStreamWaitEvent(mg->cstream, mg->ev_fork, 0));
    return exchange_on(mg, level, field, colour_mask, depth_up, down, mg->cstream);
}

/* Weighted Jacobi, ncycles sweeps.  On the colour-split layout a sweep is two launches: the new colour-0 values go
   to a scratch array (colour 1 still needs the old ones), colour 1 is then updated in place (a point reads only
   its own old value of that array).  The scratch array IS the colour-0 array of the next sweep, so the roles of
   scratch and v alternate; an odd number of sweeps ends with one copy back.  4*B*N_l bytes per sweep (RB-GS: 3). */
static int relax_jacobi_level(mg3d_t* mg, int level, int ncycles)
{
    mg_level3d* L = &mg->lv[level];
    const size_t cbytes = (size_t)L->g.cstride * mg_esize(mg->core.dtype);
    int st;
    if (!L->jscratch) {
        MG_CUDA(cudaMalloc(&L->jscratch, cbytes));
        MG_CUDA(cudaMemsetAsync(L->jscratch, 0, cbytes, mg->core.stream));
    }
    if ((st = ensure_v_ghosts(mg, level))) return st;
    L->vg_deep = 0;
    char *red = (char*)L->v, *black = red + cbytes, *cur = red;
    const char *f_red = (const char*)L->f, *f_black = f_red + cbytes;
    for (int k = 0; k < ncycles; k++) {
        char* nxt = cur == red ? (char*)L->jscratch : red;
        PROF_BEGIN(mg, level, MG_OP_RELAX);
        MG_LAUNCH(mg->core.launches, mgk3d_jacobi_colour(mg->core.stream, mg->core.dtype, nxt, cur, black, f_red, L->g, L->c, mg->omega, 0, L->own_lo, L->own_hi));
        MG_LAUNCH(mg->core.launches, mgk3d_jacobi_colour(mg->core.stream, mg->core.dtype, black, black, cur, f_black, L->g, L->c, mg->omega, 1, L->own_lo, L->own_hi));
        PROF_END(mg);
        cur = nxt;
        if (L->dist) {
            /* `cur` as a field pointer with colour mask 1 addresses exactly that colour-0 array */
            if ((st = exchange(mg, level, cur == red ? L->v : (void*)cur, 1, 1, 1))) return st;
            if ((st = exchange(mg, level, L->v, 2, 1, 1))) return st;
        }
    }
    if (cur != red) {
        /* owned planes and the nearest ghost on each side (refreshed by the exchanges above).  Not the second lower
           ghost: the scratch never receives it, and a neighbour that is already one exchange ahead may have pushed
           its fresh value into v by now. */
        const int a = L->own_lo > 0 ? L->own_lo - 1 : 0, b = L->own_hi < L->g.nzl ? L->own_hi + 1 : L->g.nzl;
        const size_t off = (size_t)a * (size_t)L->g.plane * mg_esize(mg->core.dtype);
        MG_CUDA(cudaMemcpyAsync(red + off, cur + off, (size_t)(b - a) * (size_t)L->g.plane * mg_esize(mg->core.dtype), cudaMemcpyDeviceToDevice,
                                mg->core.stream));
    }
    return MG_OK;
}

/* 1 when VCycle's Interpolate + ApplyCorrection on `level` can ride on the first pass of the post-smoothing: that pass
   corrects the colour-1 points only.  (A PIPE level has tensor maps, so the coarser level has its tmap_pc.) */
static int correction_fuses(const mg3d_t* mg, int level, int v2)
{
    const mg_path3d p = level_path(mg, level);
    return v2 >= 2 && p.relax == MG_RELAX_PIPE && p.correct_colour1;
}

/* correct_first: the first two-sweep pass starts from v + Interpolate(v of level+1) on the colour-1 points (the caller has
   checked correction_fuses) */
static int relax_level_ex(mg3d_t* mg, int level, int ncycles, int correct_first)
{
    mg_level3d* L = &mg->lv[level];
    int lo, hi, st;
    interior_range(L, &lo, &hi);
    if (ncycles <= 0) return MG_OK;
    const mg_path3d p = level_path(mg, level);
    if (p.relax == MG_RELAX_JACOBI) return relax_jacobi_level(mg, level, ncycles);
    /* register-tiled temporally blocked smoother (the default where it applies): two full sweeps per pass, out of place.
       Bit-exact mode: the pass range-checks everything it touches; the conditional literal-arithmetic pass behind it only
       runs (and then recomputes the same output buffer from the untouched input) if that check failed. */
    if (p.relax == MG_RELAX_PIPE) {
        while (ncycles >= 2) {
            const void* maps3[3] = {L->tmap_pp[L->cur], L->tmap_pf[0], L->tmap_pf[1]};
            const void* maps4[4] = {L->tmap_fu[L->cur][0], L->tmap_fu[L->cur][1], L->tmap_ff[0], L->tmap_ff[1]};
            /* slab: four planes of colour 1 from each neighbour -- all the pass reads of v beyond the planes it owns (one
               exchange per two sweeps instead of four; the halo planes are swept redundantly, bit-identical on both sides) */
            if (L->dist && !L->vg_deep && (st = exchange(mg, level, L->v, 2, MG_GHOST_LO, MG_GHOST_HI))) return st;
            mg_level3d* C = correct_first ? &mg->lv[level + 1] : NULL;
            const void* cmaps[2] = {C ? C->tmap_pc[C->cur][0] : NULL, C ? C->tmap_pc[C->cur][1] : NULL};
            int elo = 0, ehi = 0; /* planes the pass reads of v: the owned ones and four on each side, inside the grid */
            if (C) {
                /* the halo planes of the slab are corrected here as well (the neighbour's own correction never reaches memory):
                   coarse planes up to two below and three above the coarse slab */
                if (C->dist) {
                    if ((st = exchange(mg, level + 1, C->v, 3, 2, 3))) return st;
                    C->vg_valid = 1;
                }
                const int first = 1 - L->g.z0, last = L->g.n - 2 - L->g.z0;
                elo = L->own_lo - 4 > first ? L->own_lo - 4 : first;
                ehi = (L->own_hi + 4 < last + 1 ? L->own_hi + 4 : last + 1);
                if (elo < 0) elo = 0;
                if (ehi > L->g.nzl) ehi = L->g.nzl;
            }
            PROF_BEGIN(mg, level, MG_OP_RELAX);
            MG_LAUNCH(mg->core.launches, mgk3d_relax_pipe2(mg->core.stream, mg->core.dtype, maps3, L->vbuf[L->cur], L->f, L->vbuf[L->cur ^ 1], L->g, L->c,
                                                      L->own_lo, L->own_hi, mg->arith == MG_ARITH_FAST, mg->d_flag, C ? cmaps : NULL, C ? &C->g : NULL));
            if (mg->arith != MG_ARITH_FAST) { /* conditional on the range guard; reads the same input planes, no exchange of its own */
                if (C) /* ... after the correction the pass applied on the fly has been applied to the input buffer for real */
                    MG_LAUNCH(mg->core.launches, mgk3d_interpolate(mg->core.stream, mg->core.dtype, L->v, L->g, C->v, C->g, 1, 2, elo, ehi, mg->d_flag));
                MG_LAUNCH(mg->core.launches, mgk3d_relax_fused2(mg->core.stream, mg->core.dtype, maps4, L->vbuf[L->cur ^ 1], L->g, L->c, L->own_lo, L->own_hi, mg->d_flag));
            }
            PROF_END(mg);
            correct_first = 0;
            L->cur ^= 1;
            L->v = L->vbuf[L->cur];
            L->vg_valid = L->vg_deep = 0; /* only the owned planes of the new buffer were written */
            ncycles -= 2;
        }
        if (ncycles <= 0) return MG_OK;
    }
    if ((st = ensure_v_ghosts(mg, level))) return st;
    L->vg_deep = 0; /* the sweeps below refresh one ghost plane per side only */
    /* the shared-memory version of the same idea (literal arithmetic; slower than four colour launches, kept as the
       exact fallback above and selectable for tests) */
    if (p.relax == MG_RELAX_FUSED) {
        while (ncycles >= 2) {
            const void* maps4[4] = {L->tmap_fu[L->cur][0], L->tmap_fu[L->cur][1], L->tmap_ff[0], L->tmap_ff[1]};
            PROF_BEGIN(mg, level, MG_OP_RELAX);
            MG_LAUNCH(mg->core.launches, mgk3d_relax_fused2(mg->core.stream, mg->core.dtype, maps4, L->vbuf[L->cur ^ 1], L->g, L->c, L->own_lo, L->own_hi, NULL));
            PROF_END(mg);
            L->cur ^= 1;
            L->v = L->vbuf[L->cur];
            ncycles -= 2;
        }
        if (ncycles <= 0) return MG_OK;
    }
    /* distributed level: the two boundary planes of the slab are swept first, their halo exchange then runs on
       the side stream while the interior planes are swept; the next half-sweep waits for both */
    const int overlap = relax_overlaps(mg, level);
    for (int k = 0; k < ncycles; k++)
        for (int colour = 0; colour < 2; colour++) {
            if (overlap) {
                /* boundary planes and interior planes are disjoint writes of the same colour: they run concurrently */
                MG_CUDA(cudaEventRecord(mg->ev_fork, mg->core.stream));
                MG_CUDA(cudaStreamWaitEvent(mg->cstream, mg->ev_fork, 0));
                MG_LAUNCH(mg->core.launches, mgk3d_relax_colour_pair(mg->cstream, mg->core.dtype, L->v, L->f, L->g, L->c, colour, lo, hi - 1));
                if ((st = exchange_on(mg, level, L->v, 1 << colour, 1, 1, mg->cstream))) return st;
                MG_CUDA(cudaEventRecord(mg->ev_join, mg->cstream));
                if ((st = relax_launch(mg, L, colour, lo + 1, hi - 1, p.tma))) return st;
                MG_CUDA(cudaStreamWaitEvent(mg->core.stream, mg->ev_join, 0));
                continue;
            }
            PROF_BEGIN(mg, level, MG_OP_RELAX);
            st = relax_launch(mg, L, colour, lo, hi, p.tma);
            PROF_END(mg);
            if (st) return st;
            if ((st = exchange(mg, level, L->v, 1 << colour, 1, 1))) return st;
        }
    return MG_OK;
}

static int relax_level(mg3d_t* mg, int level, int ncycles) { return relax_level_ex(mg, level, ncycles, 0); }

int mg3d_relax(mg3d_t* mg, int level, int ncycles)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (ncycles < 0) return mg_fail(MG_ERR_ARG, "ncycles < 0");
    return relax_level(mg, level, ncycles);
}

/* CalculateResidual -> host array of the planes this rank owns */
int mg3d_residual(mg3d_t* mg, int level, void* host_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!host_out) return mg_fail(MG_ERR_ARG, "null output");
    mg_level3d* L = &mg->lv[level];
    if ((st = ensure_v_ghosts(mg, level))) return st;
    void* r = NULL;
    MG_CUDA(cudaMalloc(&r, field_bytes(L, mg->core.dtype)));
    int k = mgk3d_residual(mg->core.stream, mg->core.dtype, L->v, L->f, r, L->g, L->c, mg->mode == MG_CORRECTED, L->own_lo, L->own_hi);
    if (k < 0) { cudaFree(r); return mg_fail(MG_ERR_CUDA, "residual launch failed: %s", cudaGetErrorString(cudaGetLastError())); }
    mg->core.launches += k;
    st = copy_out(mg, host_out, r, &L->g, L->own_lo, L->own_hi);
    cudaFree(r);
    return st;
}

static void coarse_share(const mg3d_t* mg, int fine_level, int* czl_lo, int* czl_hi);

/* the norm pass of mg3d_residual_norm: {sum of r^2, max |r|} of `level` into norm_out2 (all-reduced over the ranks of a
   distributed level); nothing is read back */
static double* norm_out2(mg3d_t* mg) { return mg->d_scratch + 2 * MGK_NORM_MAX_PARTS; }

static int residual_norm_enqueue(mg3d_t* mg, int level)
{
    mg_level3d* L = &mg->lv[level];
    int st;
    if ((st = ensure_v_ghosts(mg, level))) return st;
    double* out2 = norm_out2(mg);
    int k = -2;
    if (level_path(mg, level).tma) {
        /* large levels: the staging of the fused residual+restrict kernel; the coarse planes this rank restricts to
           lie over exactly the fine planes it owns */
        int clo, chi;
        coarse_share(mg, level, &clo, &chi);
        k = mgk3d_residual_norm_tma(mg->core.stream, mg->core.dtype, L->tmap_rr[L->cur][0], L->tmap_rr[L->cur][1], L->f, L->g, L->c,
                                    mg->mode == MG_CORRECTED, mg->lv[level + 1].g, clo, chi, mg->d_scratch, MGK_NORM_MAX_PARTS, out2);
        if (k == -1) return mg_fail(MG_ERR_CUDA, "residual norm launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        if (k > 0) mg->core.launches += k;
    }
    if (k == -2)
        MG_LAUNCH(mg->core.launches, mgk3d_residual_norm(mg->core.stream, mg->core.dtype, L->v, L->f, L->g, L->c, mg->mode == MG_CORRECTED,
                                                    L->own_lo, L->own_hi, mg->d_scratch, out2));
    if (L->dist && (st = mg_comm_allreduce_sum_max(mg->comm, out2, mg->core.stream))) return st;
    return MG_OK;
}

int mg3d_residual_norm(mg3d_t* mg, int level, double* l2, double* linf)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if ((st = residual_norm_enqueue(mg, level)) || (st = mg_read_norm(&mg->core, norm_out2(mg), l2, linf))) return st;
    return halo_error_check(mg);
}

/* coarse local planes this rank computes when restricting from fine level `fine_level` */
static void coarse_share(const mg3d_t* mg, int fine_level, int* czl_lo, int* czl_hi)
{
    const mg_level3d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    if (C->dist || !F->dist) {
        *czl_lo = C->own_lo;
        *czl_hi = C->own_hi;
    } else { /* first agglomerated level: the planes under my fine slab (C is stored whole: z0 = 0) */
        const int a = F->g.z0 + F->own_lo, b = F->g.z0 + F->own_hi;
        *czl_lo = a / 2;
        *czl_hi = (b - 1) / 2 + 1; /* the last rank's b = n makes this n_c: it also produces the top plane */
        if (mg->rank < mg->nranks - 1) *czl_hi = b / 2;
    }
}

/* Position-keyed additive checksum of a level's field over the whole grid (tests/golden_util.py:field_checksum is
   the same sum in numpy; tests/golden/hashes3d.json holds the reference CPU solver's values).  Every rank sums the
   planes it owns; distributed levels are combined over the ranks, so each rank returns the global value. */
int mg3d_field_checksum(mg3d_t* mg, int level, int field, unsigned long long* out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!out || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3d* L = &mg->lv[level];
    unsigned long long* d = (unsigned long long*)(mg->d_scratch + 2 * MGK_NORM_MAX_PARTS);
    MG_CUDA(cudaMemsetAsync(d, 0, sizeof *d, mg->core.stream));
    MG_LAUNCH(mg->core.launches, mgk3d_field_checksum(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, L->own_lo, L->own_hi, d));
    if (L->dist && (st = mg_comm_allreduce_u64_sum(mg->comm, d, mg->core.stream))) return st;
    MG_CUDA(cudaMemcpyAsync(mg->core.h_out2, d, sizeof *d, cudaMemcpyDeviceToHost, mg->core.stream));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    memcpy(out, mg->core.h_out2, sizeof *out);
    return halo_error_check(mg);
}

/* Grid3D::PrintDiff (N3/Grid3D.cpp:136-159) as a reduction: mean and max over ALL points of |realSol - approxSol|,
   realSol = (real)(sin(PI x) sin(PI y) sin(PI z)), the difference taken in the grid's own precision */
int mg3d_abs_error(mg3d_t* mg, int level, double* mean_abs, double* max_abs)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    mg_level3d* L = &mg->lv[level];
    const int n = L->g.n;
    if ((st = upload_sin_tables(mg, level))) return st;
    double* out2 = mg->d_scratch + 2 * MGK_NORM_MAX_PARTS;
    MG_LAUNCH(mg->core.launches, mgk3d_abs_error(mg->core.stream, mg->core.dtype, L->v, L->g, mg->d_tables, mg->d_tables + n, mg->d_tables + 2 * n,
                                            L->own_lo, L->own_hi, mg->d_scratch, out2));
    if (L->dist && (st = mg_comm_allreduce_sum_max(mg->comm, out2, mg->core.stream))) return st;
    if ((st = mg_read_out2(&mg->core, out2))) return st;
    if (mean_abs) *mean_abs = mg->core.h_out2[0] / ((double)n * n * n);
    if (max_abs) *max_abs = mg->core.h_out2[1];
    return halo_error_check(mg);
}

/* diagnostic: `reps` halo exchanges of (colour_mask, depth_up, depth_down) on the current v of `level`, back to back on the
   handle's stream -- for timing the transport (scripts/bench_halo.py); the data it moves is what the ghosts hold anyway */
int mg3d_halo_benchmark(mg3d_t* mg, int level, int colour_mask, int depth_up, int depth_down, int reps)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (depth_up < 0 || depth_up > MG_GHOST_LO || depth_down < 0 || depth_down > MG_GHOST_HI || reps < 0 || !(colour_mask & 3))
        return mg_fail(MG_ERR_ARG, "bad halo benchmark arguments");
    for (int i = 0; i < reps && !st; i++) st = exchange(mg, level, mg->lv[level].v, colour_mask & 3, depth_up, depth_down);
    return st;
}

/* what follows a restriction onto level+1: refresh ghosts (distributed) or gather (first agglomerated level) */
static int after_restrict(mg3d_t* mg, int fine_level, void* coarse_field, int defer, int top_mode)
{
    const mg_level3d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    if (C->dist && defer) return exchange_deferred(mg, fine_level + 1, coarse_field, 3, MG_GHOST_LO, MG_GHOST_HI);
    if (C->dist) return exchange(mg, fine_level + 1, coarse_field, 3, MG_GHOST_LO, MG_GHOST_HI);
    if (F->dist) return gather_level(mg, fine_level + 1, coarse_field, top_mode);
    return MG_OK;
}

int mg3d_restrict(mg3d_t* mg, int fine_level, int field)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level3d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    int lo, hi;
    coarse_share(mg, fine_level, &lo, &hi);
    if (field == MG_FIELD_V && (st = ensure_v_ghosts(mg, fine_level))) return st;
    PROF_BEGIN(mg, fine_level, MG_OP_OTHER);
    MG_LAUNCH(mg->core.launches, mgk3d_restrict(mg->core.stream, mg->core.dtype, field_ptr(F, field), F->g, field_ptr(C, field), C->g, lo, hi));
    PROF_END(mg);
    st = after_restrict(mg, fine_level, field_ptr(C, field), 0, MG_TOP_FROM_LAST);
    if (!st && field == MG_FIELD_V) C->vg_valid = C->vg_deep = 1;
    return st;
}

/* defer_f_halo: the coarse f ghosts are not read before the coarse level's residual (the smoother reads f at its own
   points only), so inside a V-cycle their exchange overlaps the first coarse half-sweep */
static int residual_restrict_level(mg3d_t* mg, int fine_level, int defer_f_halo)
{
    mg_level3d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    const mg_path3d p = level_path(mg, fine_level);
    int lo, hi, st;
    coarse_share(mg, fine_level, &lo, &hi);
    /* the fused kernel reads v two planes below the slab: only plane a-2 is stale after the smoother's exchanges */
    if (F->dist) {
        if (p.relax == MG_RELAX_PIPE && !F->vg_deep) {
            /* v does not change between here and the first pass of the post-smoothing (prolongation and correction ride on that
               pass), so the four colour-1 planes that pass needs from each neighbour travel now, in the same launch: one
               exchange fewer on the way up */
            const int up2[2] = {2, MG_GHOST_LO}, down2[2] = {F->vg_valid ? 0 : 1, MG_GHOST_HI};
            if ((st = exchange2(mg, fine_level, F->v, up2, down2))) return st;
            F->vg_deep = 1;
        } else if ((st = exchange(mg, fine_level, F->v, 3, 2, F->vg_valid ? 0 : 1)))
            return st;
        F->vg_valid = 1;
    }
    PROF_BEGIN(mg, fine_level, MG_OP_RESIDUAL_RESTRICT);
    if (p.tma) {
        const void* fmaps[2] = {F->tmap_pf[0], F->tmap_pf[1]};
        MG_LAUNCH(mg->core.launches, mgk3d_residual_restrict_tma(mg->core.stream, mg->core.dtype, F->tmap_rr[F->cur][0], F->tmap_rr[F->cur][1],
                                                            fmaps, F->f, F->g, F->c,
                                                            mg->mode == MG_CORRECTED, C->f, C->v, C->g, lo, hi));
    }
    else
        MG_LAUNCH(mg->core.launches, mgk3d_residual_restrict(mg->core.stream, mg->core.dtype, F->v, F->f, F->g, F->c, mg->mode == MG_CORRECTED,
                                                        C->f, C->v, C->g, lo, hi));
    if (F->dist && C->dist) {
        /* coarse v = 0 everywhere this rank stores it: the kernel above zeroed the planes it restricted to (all the planes the
           rank owns), the ghost planes are zeroed here -- and those of the other buffer too: see mirror_v_ghosts */
        MG_LAUNCH(mg->core.launches, mgk3d_set_ghosts(mg->core.stream, mg->core.dtype, C->v, C->g, 0.0, C->own_lo, C->own_hi));
        if (C->vbuf[1])
            MG_LAUNCH(mg->core.launches, mgk3d_set_ghosts(mg->core.stream, mg->core.dtype, C->vbuf[C->cur ^ 1], C->g, 0.0, C->own_lo, C->own_hi));
    } else if (F->dist) { /* first agglomerated level: the kernel zeroed this rank's share only, every rank holds the whole level */
        MG_LAUNCH(mg->core.launches, mgk3d_set(mg->core.stream, mg->core.dtype, C->v, C->g, 0.0, 1, 0, C->g.nzl));
    }
    C->vg_valid = C->vg_deep = 1;
    PROF_END(mg);
    return after_restrict(mg, fine_level, C->f, defer_f_halo, MG_TOP_ZERO);
}

int mg3d_residual_restrict(mg3d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return residual_restrict_level(mg, fine_level, 0);
}

/* colour_mask 3: the operator as the reference defines it.  colour_mask 2: only the colour-1 points -- what a V-cycle
   with nu2 >= 1 needs, because the red half-sweep that follows recomputes every interior colour-0 point from its
   colour-1 neighbours and f alone (N3/MultiGrid3D.cpp:532 never reads the point's own old value); the colour-0
   ghosts are refreshed by that half-sweep's own exchange. */
static int interpolate_level(mg3d_t* mg, int fine_level, int add, int colour_mask, int defer_halo)
{
    mg_level3d *F = &mg->lv[fine_level], *C = &mg->lv[fine_level + 1];
    int lo, hi, st;
    interior_range(F, &lo, &hi);
    if ((st = ensure_v_ghosts(mg, fine_level + 1))) return st; /* the last fine plane of a slab reads the coarse plane above */
    PROF_BEGIN(mg, fine_level, MG_OP_INTERPOLATE);
    MG_LAUNCH(mg->core.launches, mgk3d_interpolate(mg->core.stream, mg->core.dtype, F->v, F->g, C->v, C->g, add, colour_mask, lo, hi, NULL));
    PROF_END(mg);
    if (!F->dist) return MG_OK;
    /* The owned planes of the fine v changed: the neighbours' ghost copies are stale.  A level the temporally blocked
       smoother takes next fetches its (deeper) ghost planes itself, and whoever else reads ghost planes refreshes them
       first (ensure_v_ghosts); otherwise the colour that changed travels now. */
    F->vg_deep = 0;
    if (level_path(mg, fine_level).relax == MG_RELAX_PIPE || !F->vg_valid) {
        F->vg_valid = 0;
        return MG_OK;
    }
    if (defer_halo) return exchange_deferred(mg, fine_level, F->v, colour_mask, 1, 1);
    return exchange(mg, fine_level, F->v, colour_mask, 1, 1);
}

int mg3d_interpolate(mg3d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 0, 3, 0);
}

int mg3d_interpolate_correct(mg3d_t* mg, int fine_level)
{
    int st = mg_check_fine_level(MG_CORE(mg), fine_level);
    if (st) return st;
    return interpolate_level(mg, fine_level, 1, 3, 0);
}

int mg3d_set_to_value(mg3d_t* mg, int level, int field, double value, int modify_boundaries)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (field != MG_FIELD_V && field != MG_FIELD_F) return mg_fail(MG_ERR_ARG, "bad field");
    mg_level3d* L = &mg->lv[level];
    /* ghost planes take the same constant; the exchange is the neighbour handshake (see mg3d_init_problem) */
    MG_LAUNCH(mg->core.launches, mgk3d_set(mg->core.stream, mg->core.dtype, field_ptr(L, field), L->g, value, modify_boundaries, 0, L->g.nzl));
    st = exchange(mg, level, field_ptr(L, field), 3, MG_GHOST_LO, MG_GHOST_HI);
    if (!st && field == MG_FIELD_V) {
        L->vg_valid = L->vg_deep = 1;
        st = mirror_v_ghosts(mg, level);
    }
    return st;
}

/* VCycle, N3/MultiGrid3D.cpp:623-647.  CalculateResidual + Restrict + setToValue(coarse v, 0, true)
   are one kernel; Interpolate + ApplyCorrection are one kernel: no residual / error grid exists. */
static int vcycle_rec(mg3d_t* mg, int level, int v1, int v2)
{
    int st;
    const mg_path3d p = level_path(mg, level);
    if (p.tail) {
        /* the coarse tail: the whole recursion from here down in one launch of one CTA */
        mg_geom3d g[MGK3D_TAIL_MAX_LEVELS];
        mg_coef3d c[MGK3D_TAIL_MAX_LEVELS];
        void *v[MGK3D_TAIL_MAX_LEVELS], *f[MGK3D_TAIL_MAX_LEVELS];
        const int nlev = mg->core.nlevels - level;
        for (int l = 0; l < nlev; l++) {
            g[l] = mg->lv[level + l].g; c[l] = mg->lv[level + l].c;
            v[l] = mg->lv[level + l].v; f[l] = mg->lv[level + l].f;
        }
        PROF_BEGIN(mg, level, MG_OP_RELAX);
        MG_LAUNCH(mg->core.launches, mgk3d_vcycle_tail(mg->core.stream, mg->core.dtype, nlev, g, c, v, f, v1, v2, mg->mode == MG_CORRECTED));
        PROF_END(mg);
        return MG_OK;
    }
    st = relax_level(mg, level, v1);
    if (st) return st;
    if (level != mg->core.nlevels - 1) {
        if ((st = residual_restrict_level(mg, level, v1 > 0 && relax_overlaps(mg, level + 1)))) return st;
        if ((st = vcycle_rec(mg, level + 1, v1, v2))) return st;
        if (correction_fuses(mg, level, v2)) return relax_level_ex(mg, level, v2, 1);
        if ((st = interpolate_level(mg, level, 1, (v2 > 0 && p.correct_colour1) ? 2 : 3,
                                    v2 > 0 && relax_overlaps(mg, level))))
            return st;
    }
    return relax_level(mg, level, v2);
}

/* ---- the graph cache (mg_host_common.c) runs, captures and replays one cycle on `level` with fixed sweep counts ---- */

static int c3_cycle(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return vcycle_rec(x->h, x->level, x->v1, x->v2); }
static int c3_public(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return mg3d_vcycle(x->h, x->level, x->v1, x->v2); }
static int c3_norm(void* c) { mg_cycle_ctx* x = (mg_cycle_ctx*)c; return residual_norm_enqueue(x->h, x->level); }

/* [0] = which v buffer every level works on (bit l, levels < 32); [1] = the ghost-validity flags (bits 2l and 2l+1 =
   vg_valid, vg_deep, levels < 16; coarser levels load as valid and not deep).  A captured graph bakes in [0] (the
   temporally blocked smoothers ping-pong); [1] steers the exchanges of distributed levels.  Both are part of the cycle
   graph's key, and both are put back after a capture and set after a replay or a device solve, so that the next call
   finds the graph the hand-written loop would find. */
static void c3_save(void* c, unsigned out[2])
{
    const mg3d_t* mg = ((mg_cycle_ctx*)c)->h;
    out[0] = out[1] = 0;
    for (int l = 0; l < mg->core.nlevels && l < 32; l++) {
        out[0] |= (unsigned)mg->lv[l].cur << l;
        if (l < 16) out[1] |= ((unsigned)(mg->lv[l].vg_valid != 0) | ((unsigned)(mg->lv[l].vg_deep != 0) << 1)) << (2 * l);
    }
}

static void c3_load(void* c, const unsigned in[2])
{
    mg3d_t* mg = ((mg_cycle_ctx*)c)->h;
    for (int l = 0; l < mg->core.nlevels && l < 32; l++) {
        mg->lv[l].cur = (int)((in[0] >> l) & 1u);
        mg->lv[l].v = mg->lv[l].vbuf[mg->lv[l].cur];
        mg->lv[l].vg_valid = l < 16 ? (int)((in[1] >> (2 * l)) & 1u) : 1;
        mg->lv[l].vg_deep = l < 16 ? (int)((in[1] >> (2 * l + 1)) & 1u) : 0;
    }
}

static mg_cycle_ops cycle_ops(mg_cycle_ctx* x)
{
    mg3d_t* mg = x->h;
    const mg_cycle_ops ops = {x, mg->core.stream, &mg->core.launches, &mg->halo_bytes, c3_cycle, c3_public, c3_norm, norm_out2(mg), c3_save, c3_load};
    return ops;
}

/* graphs for cycles of up to MG_GRAPH_MAX_LAUNCHES launches */
static int graphs_on(const mg3d_t* mg, int level, int v1, int v2)
{
    return mg_graphs_on(&mg->core.graphs, mg->core.prof.enabled, 2LL * (v1 + v2) * (mg->core.nlevels - level) * 2);
}

/* (level, v1, v2, smoother, arith, buffer bits, ghost bits); a solve graph keys on the buffer bits only */
static void graph_key(mg_cycle_ctx* x, int with_ghosts, int key[MG_GRAPH_KEY])
{
    const mg3d_t* mg = x->h;
    unsigned state[2];
    c3_save(x, state);
    const int k[MG_GRAPH_KEY] = {x->level, x->v1, x->v2, mg->smoother, mg->arith, (int)state[0], with_ghosts ? (int)state[1] : 0};
    memcpy(key, k, sizeof k);
}

/* The first call with a key runs eagerly, the second captures the cycle into a CUDA graph, later calls replay it.  The
   P2P halo kernels keep their sequence counters in device memory, so their arguments are capture-stable; NCCL
   collectives are graph-capturable.  A cycle with an odd number of passes ends on the other buffers, and the next call
   finds (or captures) the graph that starts there. */
int mg3d_vcycle(mg3d_t* mg, int level, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative sweep count");
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = cycle_ops(&x);
    int key[MG_GRAPH_KEY];
    graph_key(&x, 1, key);
    return mg_graph_cycle(&mg->core.graphs, graphs_on(mg, level, v1, v2) ? key : NULL, &ops);
}

/* ---- tolerance-driven solve (mg_host_common.c builds and runs it) ---------------------------------------------- */

int mg3d_solve(mg3d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles, int* cycles_out, int* converged_out,
               double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_cycles, v1, v2);
    if (st) return st;
    mg_cycle_ctx x = {mg, level, v1, v2};
    const mg_cycle_ops ops = cycle_ops(&x);
    int key[MG_GRAPH_KEY];
    graph_key(&x, 0, key);
    /* A distributed solve stays host-driven: a conditional body may hold kernels, copies, memsets and nested graphs only,
       and the NCCL all-reduce of the norm is not known to stay inside that set.  Every rank checks the same all-reduced
       norm, so every rank stops after the same cycle. */
    const int device = mg->nranks == 1 && graphs_on(mg, level, v1, v2);
    st = mg_solve_run(&mg->core.graphs, device ? key : NULL, &ops, rtol, atol, max_cycles, cycles_out, converged_out, history);
    return st ? st : halo_error_check(mg);
}

/* ---- multigrid-preconditioned conjugate gradients (mg_host_common.c runs the loop, mg3d_cg.cu has the vector passes) ---- */

static void* p3_v(mg_cycle_ctx* x) { return ((mg3d_t*)x->h)->lv[x->level].v; }
/* a slab runs the V-cycle through the cycle-graph cache, as the host-driven distributed solve does */
static int p3_vcycle(mg_cycle_ctx* x)
{
    mg3d_t* mg = x->h;
    return mg->lv[x->level].dist ? mg3d_vcycle(mg, x->level, x->v1, x->v2) : vcycle_rec(mg, x->level, x->v1, x->v2);
}
static int p3_norm0(mg_cycle_ctx* x) { return residual_norm_enqueue(x->h, x->level); }
/* setToValue(v, 0, true) on the buffer the V-cycle starts from; on a slab the ghost planes too, behind the handshake
   exchange, and those of the other buffer (mirror_v_ghosts): the preconditioner's Dirichlet values are 0 */
static int p3_zero_v(mg_cycle_ctx* x) { return mg3d_set_to_value(x->h, x->level, MG_FIELD_V, 0.0, 1); }

/* ---- the slab hooks: the only communication of a distributed PCG outside its V-cycles ---- */
/* r' on the owned planes of f: the temporally blocked pass sweeps halo planes and reads f there, four deep */
static int p3_r_written(mg_cycle_ctx* x) { mg3d_t* mg = x->h; return exchange(mg, x->level, mg->lv[x->level].f, 3, MG_GHOST_LO, MG_GHOST_HI); }
/* the direction pass reads z on the planes next to the owned ones */
static int p3_z_ready(mg_cycle_ctx* x) { return ensure_v_ghosts(x->h, x->level); }
static int p3_allgather(mg_cycle_ctx* x, double* dd) { mg3d_t* mg = x->h; return mg_comm_allgather_inplace(mg->comm, dd, 4, MG_F64, mg->core.stream); }
static int p3_allreduce(mg_cycle_ctx* x, double* out2) { mg3d_t* mg = x->h; return mg_comm_allreduce_sum_max(mg->comm, out2, mg->core.stream); }
/* as mg3d_set_field_device after the owned planes of v are written: the caller's boundary values are back in every ghost
   plane of both buffers */
static int p3_v_restored(mg_cycle_ctx* x)
{
    mg3d_t* mg = x->h;
    mg_level3d* L = &mg->lv[x->level];
    int st = exchange(mg, x->level, L->v, 3, MG_GHOST_LO, MG_GHOST_HI);
    if (st) return st;
    L->vg_valid = L->vg_deep = 1;
    return mirror_v_ghosts(mg, x->level);
}

/* The first pcg on a level allocates on every rank.  A rank that failed alone would leave its peers waiting in the first
   exchange, so the ranks agree on the outcome first (one all-reduce); if any failed, every rank frees its vectors. */
static int pcg_alloc_agree(mg3d_t* mg, int level, int st)
{
    double* d = norm_out2(mg);
    mg->core.h_out2[0] = mg->core.h_out2[1] = st ? 1.0 : 0.0;
    MG_CUDA(cudaMemcpyAsync(d, mg->core.h_out2, 2 * sizeof(double), cudaMemcpyHostToDevice, mg->core.stream));
    int st2 = mg_comm_allreduce_sum_max(mg->comm, d, mg->core.stream);
    if (!st2) st2 = mg_read_out2(&mg->core, d);
    if (st2) return st2;
    if (mg->core.h_out2[1] == 0.0) return MG_OK;
    if (!st) mg_pcg_vecs_free(&mg->pcg[level]);
    return st ? st : mg_fail(MG_ERR_NOMEM, "PCG vectors: %g of %d ranks could not allocate theirs", mg->core.h_out2[0], mg->nranks);
}

int mg3d_pcg(mg3d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_iters, int* iters_out, int* converged_out,
             double* history)
{
    int st = mg_solve_check_args(MG_CORE(mg), level, rtol, atol, max_iters, v1, v2);
    if (st) return st;
    if (mg->mode != MG_CORRECTED) return mg_fail(MG_ERR_STATE, "pcg needs MG_CORRECTED: the MG_REF_COMPAT residual is not a symmetric operator");
    mg_level3d* L = &mg->lv[level];
    const int fresh = !mg->pcg || !mg->pcg[level].b;
    if (!mg->pcg) mg->pcg = (mg_pcg_vecs*)calloc((size_t)mg->core.nlevels, sizeof *mg->pcg);
    st = mg->pcg ? mg_pcg_vecs_alloc(&mg->pcg[level], field_bytes(L, mg->core.dtype), L->dist ? mg->nranks : 0, mg->core.stream)
                 : mg_fail(MG_ERR_NOMEM, "host allocation failed");
    if (fresh && mg->nranks > 1) st = pcg_alloc_agree(mg, level, st);
    if (st) return st;
    mg_pcg_ctx pc;
    memset(&pc, 0, sizeof pc);
    pc.cx.h = mg; pc.cx.level = level; pc.cx.v1 = v1; pc.cx.v2 = v2;
    pc.P = &mg->pcg[level];
    pc.dtype = mg->core.dtype;
    pc.stream = mg->core.stream;
    pc.launches = &mg->core.launches;
    pc.g.nx = pc.g.ny = pc.g.nz = L->g.n;
    pc.g.hp = L->g.hp; pc.g.plane = L->g.plane; pc.g.cstride = L->g.cstride;
    pc.g.z0 = L->g.z0; pc.g.nzl = L->g.nzl;
    pc.c = L->c;
    pc.f = L->f;
    pc.out2 = norm_out2(mg);
    pc.v = p3_v; pc.zero_v = p3_zero_v; pc.vcycle = p3_vcycle; pc.norm0 = p3_norm0;
    pc.save = c3_save; pc.load = c3_load;
    pc.own_lo = pc.wr_lo = 0;
    pc.own_hi = pc.wr_hi = L->g.nzl;
    if (L->dist) {
        pc.own_lo = L->own_lo; pc.own_hi = L->own_hi;
        pc.wr_lo = L->own_lo > 0 ? L->own_lo - 1 : 0;
        pc.wr_hi = L->own_hi < L->g.nzl ? L->own_hi + 1 : L->g.nzl;
        pc.rank = mg->rank; pc.nranks = mg->nranks;
        pc.r_written = p3_r_written; pc.z_ready = p3_z_ready; pc.allgather = p3_allgather; pc.allreduce = p3_allreduce;
        pc.v_restored = p3_v_restored;
    }
    int key[MG_GRAPH_KEY];
    graph_key(&pc.cx, 0, key);
    key[MG_GRAPH_KEY_KIND] = MG_GRAPH_PCG;
    /* a distributed handle stays host-driven, as mg3d_solve does (the NCCL collectives are not known to be legal inside a
       conditional body); every rank checks the same all-reduced norm and stops after the same iteration */
    const int device = mg->nranks == 1 && graphs_on(mg, level, v1, v2);
    st = mg_pcg_run(&pc, &mg->core.graphs, device ? key : NULL, rtol, atol, max_iters, iters_out, converged_out, history);
    return st ? st : halo_error_check(mg);
}

/* FullMultiGridVCycle, N3/MultiGrid3D.cpp:569-585 */
static int fmg_rec(mg3d_t* mg, int level, int v0, int v1, int v2)
{
    int st;
    if (level != mg->core.nlevels - 1) {
        mg_level3d *F = &mg->lv[level], *C = &mg->lv[level + 1];
        int lo, hi;
        coarse_share(mg, level, &lo, &hi);
        PROF_BEGIN(mg, level, MG_OP_OTHER);
        MG_LAUNCH(mg->core.launches, mgk3d_restrict(mg->core.stream, mg->core.dtype, F->f, F->g, C->f, C->g, lo, hi));
        PROF_END(mg);
        if ((st = after_restrict(mg, level, C->f, 0, MG_TOP_FROM_LAST))) return st;
        if ((st = fmg_rec(mg, level + 1, v0, v1, v2))) return st;
        if ((st = interpolate_level(mg, level, 0, 3, 0))) return st;
    } else {
        mg_level3d* L = &mg->lv[level];
        MG_LAUNCH(mg->core.launches, mgk3d_set(mg->core.stream, mg->core.dtype, L->v, L->g, 0.0, 0, 0, L->g.nzl));
    }
    for (int i = 0; i < v0; i++)
        if ((st = vcycle_rec(mg, level, v1, v2))) return st;
    return MG_OK;
}

int mg3d_fmg(mg3d_t* mg, int level, int v0, int v1, int v2)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (v0 < 0 || v1 < 0 || v2 < 0) return mg_fail(MG_ERR_ARG, "negative cycle/sweep count");
    return fmg_rec(mg, level, v0, v1, v2);
}

/* ---- reference-facing operators on HOST arrays (N3/MultiGrid3D.h:16-27) ---------------------- */

static int cubic(const int s[3], int* n)
{
    if (!s || s[0] != s[1] || s[0] != s[2] || s[0] < 3) return mg_fail(MG_ERR_ARG, "cubic size >= 3 required");
    *n = s[0];
    return MG_OK;
}

/* a cube is a box: the box engine's dense kernels (mg3d_box.cu), built from the same per-point functions as the cubic ones.
   A result must not look valid after a neighbour missed a halo flag: every call that hands data back checks that. */
int mg3d_restrict_host(mg3d_t* mg, const void* fine, const int fs[3], void* coarse, const int cs[3])
{
    int fn = 0, cn = 0, st;
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N3/MultiGrid3D.cpp:60-62 */
    const size_t nf = (size_t)fn * fn * fn, nc = (size_t)cn * cn * cn;
    void *df, *dc;
    if ((st = mg_tmp_begin(&mg->core, &df, nf, fine, &dc, nc, NULL))) return st;
    st = mg_tmp_finish(&mg->core, mgk3b_dense_restrict(mg->core.stream, mg->core.dtype, df, fs, dc, cs), coarse, dc, nc, df, dc);
    return st ? st : halo_error_check(mg);
}

int mg3d_interpolate_host(mg3d_t* mg, void* fine, const int fs[3], const void* coarse, const int cs[3])
{
    int fn = 0, cn = 0, st;
    if (!mg || !fine || !coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1"); /* N3/MultiGrid3D.cpp:196-198 */
    const size_t nf = (size_t)fn * fn * fn, nc = (size_t)cn * cn * cn;
    void *df, *dc;
    if ((st = mg_tmp_begin(&mg->core, &df, nf, fine, &dc, nc, coarse))) return st; /* the boundary of fine is kept */
    st = mg_tmp_finish(&mg->core, mgk3b_dense_interpolate(mg->core.stream, mg->core.dtype, df, fs, dc, cs), fine, df, nf, df, dc);
    return st ? st : halo_error_check(mg);
}

int mg3d_apply_correction_host(mg3d_t* mg, void* fine, const int fs[3], const void* error, const int es[3])
{
    int fn = 0, en = 0, st;
    if (!mg || !fine || !error) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(es, &en))) return st;
    if (fn != en) return mg_fail(MG_ERR_ARG, "fsize != esize"); /* N3/MultiGrid3D.cpp:660-662 */
    const size_t nf = (size_t)fn * fn * fn;
    void *df, *de;
    if ((st = mg_tmp_begin(&mg->core, &df, nf, fine, &de, nf, error))) return st;
    st = mg_tmp_finish(&mg->core, mgk3b_dense_apply_correction(mg->core.stream, mg->core.dtype, df, de, fs), fine, df, nf, df, de);
    return st ? st : halo_error_check(mg);
}

int mg3d_set_to_value_host(mg3d_t* mg, void* grid, const int s[3], double value, int modify_boundaries)
{
    int n = 0, st;
    if (!mg || !grid) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(s, &n))) return st;
    const size_t nn = (size_t)n * n * n;
    void *d, *unused;
    if ((st = mg_tmp_begin(&mg->core, &d, nn, grid, &unused, 0, NULL))) return st;
    st = mg_tmp_finish(&mg->core, mgk3b_dense_set(mg->core.stream, mg->core.dtype, d, s, value, modify_boundaries), grid, d, nn, d, NULL);
    return st ? st : halo_error_check(mg);
}

/* ---- the CUDA_TESI faces: the same operators on DEVICE arrays in the reference's dense layout (C3/MultiGrid3D.h:16-24,
        C3/Grid3D.h:11,26-27: d_v / d_f / device-pointer operands).  No host trip: a level's fields move with one repack
        kernel each way, the operators run in place on the caller's arrays. ---------------------------------------------- */

static int dense_in(mg3d_t* mg, void* dev, const mg_geom3d* g, const void* dense_dev, int zl_lo, int zl_hi)
{
    MG_LAUNCH(mg->core.launches, mgk3d_repack(mg->core.stream, mg->core.dtype, dev, *g, (void*)dense_dev, 1, zl_lo, zl_hi));
    return MG_OK;
}

static int dense_out(mg3d_t* mg, void* dense_dev, const void* dev, const mg_geom3d* g, int zl_lo, int zl_hi)
{
    MG_LAUNCH(mg->core.launches, mgk3d_repack(mg->core.stream, mg->core.dtype, (void*)dev, *g, dense_dev, 0, zl_lo, zl_hi));
    MG_CUDA(cudaStreamSynchronize(mg->core.stream)); /* the caller's next access may be on any stream (the reference uses the default one) */
    return halo_error_check(mg);
}

int mg3d_set_field_device(mg3d_t* mg, int level, int field, const void* dev_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!dev_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3d* L = &mg->lv[level];
    MG_CUDA(cudaDeviceSynchronize()); /* whatever produced the caller's array (any stream) is complete */
    st = dense_in(mg, field_ptr(L, field), &L->g, dev_dense, L->own_lo, L->own_hi);
    if (!st) st = exchange(mg, level, field_ptr(L, field), 3, MG_GHOST_LO, MG_GHOST_HI);
    if (st) return st;
    if (field == MG_FIELD_V) {
        L->vg_valid = L->vg_deep = 1;
        if ((st = mirror_v_ghosts(mg, level))) return st;
    }
    MG_CUDA(cudaStreamSynchronize(mg->core.stream));
    return MG_OK;
}

int mg3d_get_field_device(mg3d_t* mg, int level, int field, void* dev_dense)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!dev_dense || (field != MG_FIELD_V && field != MG_FIELD_F)) return mg_fail(MG_ERR_ARG, "bad field/pointer");
    mg_level3d* L = &mg->lv[level];
    return dense_out(mg, dev_dense, field_ptr(L, field), &L->g, L->own_lo, L->own_hi);
}

/* CalculateResidual(grid) -> caller-owned DEVICE array (C3/MultiGrid3D.cu:202-233) */
int mg3d_residual_device(mg3d_t* mg, int level, void* dev_dense_out)
{
    int st = mg_check_level(MG_CORE(mg), level);
    if (st) return st;
    if (!dev_dense_out) return mg_fail(MG_ERR_ARG, "null output");
    mg_level3d* L = &mg->lv[level];
    if ((st = ensure_v_ghosts(mg, level))) return st;
    void* r = NULL;
    MG_CUDA(cudaMalloc(&r, field_bytes(L, mg->core.dtype)));
    int k = mgk3d_residual(mg->core.stream, mg->core.dtype, L->v, L->f, r, L->g, L->c, mg->mode == MG_CORRECTED, L->own_lo, L->own_hi);
    if (k < 0) { cudaFree(r); return mg_fail(MG_ERR_CUDA, "residual launch failed: %s", cudaGetErrorString(cudaGetLastError())); }
    mg->core.launches += k;
    st = dense_out(mg, dev_dense_out, r, &L->g, L->own_lo, L->own_hi);
    cudaFree(r);
    return st;
}

static int device_done(mg3d_t* mg, int k)
{
    int st = mg_launch_done(&mg->core, k);
    return st ? st : halo_error_check(mg);
}

int mg3d_restrict_device(mg3d_t* mg, const void* d_fine, const int fs[3], void* d_coarse, const int cs[3])
{
    int fn = 0, cn = 0, st;
    if (!mg || !d_fine || !d_coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize()); /* the caller's arrays may have been produced on any stream */
    return device_done(mg, mgk3b_dense_restrict(mg->core.stream, mg->core.dtype, d_fine, fs, d_coarse, cs));
}

int mg3d_interpolate_device(mg3d_t* mg, void* d_fine, const int fs[3], const void* d_coarse, const int cs[3])
{
    int fn = 0, cn = 0, st;
    if (!mg || !d_fine || !d_coarse) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(cs, &cn))) return st;
    if (cn != (fn - 1) / 2 + 1) return mg_fail(MG_ERR_ARG, "csize != (fsize-1)/2+1");
    MG_CUDA(cudaDeviceSynchronize());
    return device_done(mg, mgk3b_dense_interpolate(mg->core.stream, mg->core.dtype, d_fine, fs, d_coarse, cs));
}

int mg3d_apply_correction_device(mg3d_t* mg, void* d_fine, const int fs[3], const void* d_error, const int es[3])
{
    int fn = 0, en = 0, st;
    if (!mg || !d_fine || !d_error) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(fs, &fn)) || (st = cubic(es, &en))) return st;
    if (fn != en) return mg_fail(MG_ERR_ARG, "fsize != esize");
    MG_CUDA(cudaDeviceSynchronize());
    return device_done(mg, mgk3b_dense_apply_correction(mg->core.stream, mg->core.dtype, d_fine, d_error, fs));
}

int mg3d_set_device(mg3d_t* mg, void* d_v, const int size_xyz[3], double value, int modify_border)
{
    int n = 0, st;
    if (!mg || !d_v) return mg_fail(MG_ERR_ARG, "null argument");
    if ((st = cubic(size_xyz, &n))) return st;
    MG_CUDA(cudaDeviceSynchronize());
    return device_done(mg, mgk3b_dense_set(mg->core.stream, mg->core.dtype, d_v, size_xyz, value, modify_border));
}

/* end to end with HOST buffers: v,f hold the planes this rank owns (the whole grid on one GPU) */
int mg3d_vcycle_host(mg3d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles)
{
    if (!mg || !v_host || !f_host) return mg_fail(MG_ERR_ARG, "null argument");
    if (v1 < 0 || v2 < 0 || cycles < 0) return mg_fail(MG_ERR_ARG, "negative count");
    mg_level3d* L = &mg->lv[0];
    int st = copy_in(mg, L->v, &L->g, v_host, L->own_lo, L->own_hi);
    if (!st) st = exchange(mg, 0, L->v, 3, MG_GHOST_LO, MG_GHOST_HI);
    if (!st) L->vg_valid = L->vg_deep = 1;
    if (!st) st = mirror_v_ghosts(mg, 0);
    if (!st) st = copy_in(mg, L->f, &L->g, f_host, L->own_lo, L->own_hi);
    if (!st) st = exchange(mg, 0, L->f, 3, MG_GHOST_LO, MG_GHOST_HI);
    for (int i = 0; i < cycles && !st; i++) st = vcycle_rec(mg, 0, v1, v2);
    if (!st) st = copy_out(mg, v_host, L->v, &L->g, L->own_lo, L->own_hi);
    return st;
}

/*
 * mg_launch.h -- internal C interface between the C host drivers (mg*_host.c) and the CUDA
 * translation units (mg*_kernels.cu).  Not part of the public ABI (that is include/mg_b200.h).
 *
 * 3D device layout (all levels, all fields): colour-split, x fastest.  A field is two arrays, one per
 * red-black colour c = (x+y+z)&1, each compacted along x:
 *     element (x,y,zl) lives at  base[c*cstride + zl*plane + y*hp + (x>>1)]
 *     hp = (n+1)/2 rounded up to 128 bytes, plane = hp*n, cstride = plane*nzl, base 256-byte aligned.
 * A half-sweep of one colour then touches only that colour's half of v and f (unit stride) and reads the
 * other colour's half of v: 12 B/point in fp64 instead of 24 B/point with interleaved colours.
 * A slab holds local planes zl = 0..nzl-1 which are the global planes z = z0 .. z0+nzl-1; on one
 * GPU z0 = 0 and nzl = n.  Multi-GPU slabs carry ghost planes at both ends.
 * 2D fields are pitched (element (x,y) at base[x + y*pitch]); the 1D hierarchy is one arena.
 *
 * Real-valued parameters travel as double; for MG_F32 they hold float values exactly (computed
 * in float on the host, widened) and the kernels narrow them back without rounding.
 */
#ifndef MG_LAUNCH_H
#define MG_LAUNCH_H

#include <cuda_runtime_api.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    int n;             /* global points per axis (cubic: sizeX = sizeY = sizeZ, N3/Grid3D.cpp:10-11) */
    int hp;            /* elements per half-row (one colour of one row) */
    long long plane;   /* elements per z-plane of ONE colour array = hp*n */
    long long cstride; /* elements between the two colour arrays = plane*nzl */
    int z0;            /* global z of local plane 0 */
    int nzl;           /* local planes stored */
} mg_geom3d;

/* coefficient block of one 3D level, all values exactly representable in the level's dtype */
typedef struct {
    double hx2, hy2, hz2; /* h*h per axis, N3/MultiGrid3D.cpp:498-500 */
    double cx, cy, cz;    /* hy2*hz2, hx2*hz2, hx2*hy2 */
    double den;           /* 2*(cx + cy + cz), N3/MultiGrid3D.cpp:532 */
    double rden;          /* RN(1/den) */
    double ihx2, ihy2, ihz2; /* 1/h^2 per axis (exact when h^2 is a power of two) */
    int fast_den;         /* den = 6*2^e: quotient by the 3-op exact sequence of mg_exact.cuh */
    int fast_h;           /* every h^2 is a power of two: x/h^2 == x*(1/h^2) exactly */
} mg_coef3d;

/* every launcher returns the number of kernels it launched (>= 0) or -1 on a launch error */

/* one colour of one RB Gauss-Seidel sweep, in place, on local planes [zl_lo, zl_hi) */
int mgk3d_relax_colour(cudaStream_t s, int dtype, void* v, const void* f, mg_geom3d g, mg_coef3d c, int colour,
                       int zl_lo, int zl_hi);
/* weighted Jacobi on one colour array: dst = own + omega*(GS(oth, f) - own) on the interior points of `colour`,
   local planes [zl_lo, zl_hi); dst == own works in place, otherwise dst also receives the non-interior points */
int mgk3d_jacobi_colour(cudaStream_t s, int dtype, void* dst, const void* own, const void* oth, const void* f, mg_geom3d g,
                        mg_coef3d c, double omega, int colour, int zl_lo, int zl_hi);
/* the same half-sweep on the two planes zl_a < zl_b only (the boundary planes of a slab) */
int mgk3d_relax_colour_pair(cudaStream_t s, int dtype, void* v, const void* f, mg_geom3d g, mg_coef3d c, int colour,
                            int zl_a, int zl_b);
/* same half-sweep with TMA-staged z-marching shared-memory tiles (mg3d_smooth_tma.cu); tmap_other is the
   128-byte CUtensorMap of the OTHER colour's v array built with box (MGK3D_TMA_BOX_I(esize), MGK3D_TMA_BOX_Y, 1) */
#define MGK3D_TMA_IT 128
#define MGK3D_TMA_YT 8
#define MGK3D_TMA_BOX_I(esize) (MGK3D_TMA_IT + 2 * (16 / (int)(esize)))
#define MGK3D_TMA_BOX_Y (MGK3D_TMA_YT + 2)
int mgk3d_relax_colour_tma(cudaStream_t s, int dtype, const void* tmap_other, void* v, const void* f, mg_geom3d g,
                           mg_coef3d c, int colour, int zl_lo, int zl_hi);
/* temporally blocked smoother (mg3d_smooth_fused.cu): TWO full RB sweeps in one pass over HBM, out of place.
   maps4 = tensor maps of {v_in colour 0, v_in colour 1, f colour 0, f colour 1} with box
   (MGK3D_FU_BOX_I(esize), MGK3D_FU_BOX_Y, 1); local planes [zl_lo, zl_hi) of v_out are written (a slab: the planes it owns;
   the input needs four valid planes of colour 1 on each side of them) */
#define MGK3D_FU_TI 32
#define MGK3D_FU_TY 16
#define MGK3D_FU_BOX_I(esize) (MGK3D_FU_TI + 2 * (16 / (int)(esize)))
#define MGK3D_FU_BOX_Y (MGK3D_FU_TY + 8)
/* cond: NULL = always run; otherwise {flag, done counter}: the pass runs only when *flag != 0 (raised by
   mgk3d_relax_pipe2) and the last CTA to finish clears both words */
int mgk3d_relax_fused2(cudaStream_t s, int dtype, const void* const maps4[4], void* v_out, mg_geom3d g, mg_coef3d c,
                       int zl_lo, int zl_hi, unsigned int* cond);
/* register-tiled temporally blocked smoother (mg3d_smooth_pipe.cu): TWO full RB sweeps per pass, out of place, 2.5*B*N
   bytes.  maps3 = tensor maps of {v_in colour 1, f colour 0, f colour 1} with box (MGK3D_PP_BOX_I(esize), MGK3D_PP_BOX_Y, 1).
   Needs c.fast_den and hx2 == hy2 == hz2.  arith 0: bit-exact (flag raised when the exactness range check fails: the
   caller follows up with mgk3d_relax_fused2(..., cond = flag)); arith 1: MG_ARITH_FAST */
#define MGK3D_PP_HXI 2
#define MGK3D_PP_HY 4
#ifndef MGK3D_PP_R
#define MGK3D_PP_R 2
#endif
#ifndef MGK3D_PP_NW
#define MGK3D_PP_NW 16
#endif
#define MGK3D_PP_PADL(esize) ((int)(esize) == 8 ? 0 : 2)
#define MGK3D_PP_BOX_I(esize) (32 + 2 * MGK3D_PP_PADL(esize))
#define MGK3D_PP_BOX_Y (MGK3D_PP_R * MGK3D_PP_NW)
/* the colour-1 sub-tile of the coarse planes is loaded MGK3D_PP_CSHIFT columns (64 bytes) further left, so that column c of the two
   colour sub-tiles -- which the even and the odd lanes of a warp read in the same instruction -- falls on different banks */
#define MGK3D_PP_CSHIFT(esize) (64 / (int)(esize))
#define MGK3D_PP_CBOX_I(esize) (((int)(esize) == 8 ? 18 : 20) + MGK3D_PP_CSHIFT(esize))
#define MGK3D_PP_CBOX_Y (MGK3D_PP_R * MGK3D_PP_NW / 2 + 1)
/* coarse_maps2 / gc: NULL, or the next coarser level's v (tensor maps of its two colour arrays with box (MGK3D_PP_CBOX_I(esize),
   MGK3D_PP_CBOX_Y, 1)) and geometry: prolongation + correction of the colour-1 points folded into the load stage of the pass */
int mgk3d_relax_pipe2(cudaStream_t s, int dtype, const void* const maps3[3], const void* v_in, const void* f, void* v_out,
                      mg_geom3d g, mg_coef3d c, int zl_lo, int zl_hi, int arith, unsigned int* flag, const void* const coarse_maps2[2],
                      const mg_geom3d* gc);
/* 1 when mgk3d_relax_pipe2 has a nonempty exactness range for h^2 = hx2 (otherwise it refuses to launch) */
int mgk3d_pipe_exact_range(int dtype, double hx2);
/* the coarse tail of a V-cycle in one launch (mg3d_tail.cu): V(v1,v2) on the sub-hierarchy g[0..nlev-1], g[0].n <=
   MGK3D_TAIL_N, every level resident in one CTA's shared memory */
#define MGK3D_TAIL_N 17
#define MGK3D_TAIL_MAX_LEVELS 4
int mgk3d_vcycle_tail(cudaStream_t s, int dtype, int nlev, const mg_geom3d* g, const mg_coef3d* c, void* const* v,
                      void* const* f, int v1, int v2, int corrected);
/* r = CalculateResidual, full array incl. zero boundary, local planes [zl_lo, zl_hi) */
int mgk3d_residual(cudaStream_t s, int dtype, const void* v, const void* f, void* r, mg_geom3d g, mg_coef3d c,
                   int corrected, int zl_lo, int zl_hi);
/* partial sums of r^2 and max|r| over local planes [zl_lo, zl_hi), residual computed on the fly;
   out2 = {sum, max} (device doubles), scratch >= 2*MGK_NORM_BLOCKS doubles */
#define MGK_NORM_BLOCKS 1184
#define MGK_NORM_MAX_PARTS 32768 /* partial pairs the scratch array of a handle has room for */
int mgk_norm_final(cudaStream_t s, const double* part, int nparts, double* out2);
/* the same norm with the TMA staging and register tiling of mgk3d_residual_restrict_tma (levels that have tensor maps);
   gc = geometry of the next coarser level, [czl_lo, czl_hi) = the coarse planes over the fine planes to be covered.
   Returns -2 without launching when more than max_parts partials would be needed. */
int mgk3d_residual_norm_tma(cudaStream_t s, int dtype, const void* tmap_v_c0, const void* tmap_v_c1, const void* f,
                            mg_geom3d gf, mg_coef3d c, int corrected, mg_geom3d gc, int czl_lo, int czl_hi,
                            double* scratch, int max_parts, double* out2);
int mgk3d_residual_norm(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom3d g, mg_coef3d c,
                        int corrected, int zl_lo, int zl_hi, double* scratch, double* out2);
/* coarse = Restrict(fine) on coarse local planes [czl_lo, czl_hi) */
int mgk3d_restrict(cudaStream_t s, int dtype, const void* fine, mg_geom3d gf, void* coarse, mg_geom3d gc,
                   int czl_lo, int czl_hi);
/* coarse_f = Restrict(CalculateResidual(v,f)), coarse_v = 0 (boundary included), fused: the fine
   residual only ever exists in shared memory */
int mgk3d_residual_restrict(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom3d gf, mg_coef3d c,
                            int corrected, void* coarse_f, void* coarse_v, mg_geom3d gc, int czl_lo, int czl_hi);
/* the same with TMA-staged z-marching tiles (mg3d_rr_tma.cu): tensor maps of the two colour arrays of the
   FINE v, built with box (MGK3D_RR_BOX_I(esize), MGK3D_RR_BOX_Y, 1) */
#define MGK3D_RR_CXT 32
#define MGK3D_RR_CYT 8
#define MGK3D_RR_BOX_Y (2 * MGK3D_RR_CYT + 3)
#define MGK3D_RR_BOX_I(esize) ((MGK3D_RR_CXT + 2 * (16 / (int)(esize))) / (16 / (int)(esize)) * (16 / (int)(esize)))
/* tmap_f: NULL, or the tensor maps of the two colour arrays of the fine f with the box of mgk3d_relax_pipe2 (L2 prefetch only) */
int mgk3d_residual_restrict_tma(cudaStream_t s, int dtype, const void* tmap_v_c0, const void* tmap_v_c1, const void* const tmap_f[2], const void* f,
                                mg_geom3d gf, mg_coef3d c, int corrected, void* coarse_f, void* coarse_v, mg_geom3d gc,
                                int czl_lo, int czl_hi);
/* fine interior = Interpolate(coarse) (add == 0) or fine interior += Interpolate(coarse) (add != 0);
   colour_mask 3 = every point, 2 = the colour-1 points only (see k_interp_octet) */
/* cond: NULL, or a device word: the launch does nothing unless it is nonzero (the exact fallback of mgk3d_relax_pipe2) */
int mgk3d_interpolate(cudaStream_t s, int dtype, void* fine, mg_geom3d gf, const void* coarse, mg_geom3d gc, int add,
                      int colour_mask, int zl_lo, int zl_hi, const unsigned int* cond);
/* setToValue */
int mgk3d_set(cudaStream_t s, int dtype, void* a, mg_geom3d g, double value, int modify_boundaries, int zl_lo,
              int zl_hi);
/* the same on every stored plane except [own_lo, own_hi): the ghost planes of a slab, boundary points included */
int mgk3d_set_ghosts(cudaStream_t s, int dtype, void* a, mg_geom3d g, double value, int own_lo, int own_hi);
/* Grid3D::InitF from per-axis tables sx,sy,sz (device doubles, n each) = sin(PI*coord) computed with
   the host libm exactly like the reference: f = (T)(-3*PI*PI*sx*sy*sz), N3/Grid3D.cpp:92 */
int mgk3d_init_f(cudaStream_t s, int dtype, void* f, mg_geom3d g, const double* sx, const double* sy,
                 const double* sz, int zl_lo, int zl_hi);

/* diagnostics (mg3d_diag.cu): *out += position-keyed checksum of local planes [zl_lo, zl_hi);
   {sum, max} of |sin(PI x)sin(PI y)sin(PI z) - v| from host-libm sine tables (N3/Grid3D.cpp:136-159) */
int mgk3d_field_checksum(cudaStream_t s, int dtype, const void* a, mg_geom3d g, int zl_lo, int zl_hi, unsigned long long* out);
int mgk3d_abs_error(cudaStream_t s, int dtype, const void* v, mg_geom3d g, const double* sx, const double* sy, const double* sz,
                    int zl_lo, int zl_hi, double* scratch, double* out2);

/* dense (reference layout, x fastest, zl_hi-zl_lo planes starting at `dense`) <-> colour-split field */
int mgk3d_repack(cudaStream_t s, int dtype, void* split, mg_geom3d g, void* dense, int to_device, int zl_lo, int zl_hi);

/* P2P halo exchange (mg_halo_p2p.cu), one launch: push up to 4 segments into peer memory, raise the peers'
   sequence flags, wait for the neighbours' pushes (bounded spin); sequence counters live in flag_block */
#define MG_HALO_FLAG_WORDS 384
#define MG_GATHER_MAX_PEERS 31
int mgk_halo_exchange(cudaStream_t s, const void* const src[4], void* const dst[4], const unsigned long long bytes[4],
                      unsigned int* const peer_flag[2], int wait_below, int wait_above, unsigned int* flag_block);
/* all-gather of one level field by direct stores into every peer's copy (two launches: ready handshake, push + done) */
int mgk_gather_push(cudaStream_t s, const void* const src2[2], unsigned long long bytes, void* const dst[][2], unsigned int* const peer_block[],
                    int npeers, int me, unsigned int* flag_block);

/* ---- tolerance-driven solve (mg_solve.cu) ---- */
/* device parameter block of one solve: the host writes everything above `k` before each launch, k_solve_check the rest */
typedef struct {
    double rtol, atol;
    double* hist;   /* device history: (l2, linf) of r_0, r_1, ...; room for hist_cap pairs */
    int max_cycles;
    int hist_cap;
    int k;          /* residuals checked so far: the cycles run are k - 1 */
    int done;       /* 1 once the stopping rule has fired */
    int converged;
    int pad_;
    double thr;     /* max(atol, rtol * ||r_0||_2), fixed by the first check */
} mg_solve_par;

/* one thread: l2 = sqrt(out2[0]), linf = out2[1] of the residual the norm pass has just written; appends them to the
   history, applies the stopping rule and, when nhandles > 0, sets the conditional handles h0 (and h1) to "continue" */
int mgk_solve_check(cudaStream_t s, const double* out2, mg_solve_par* par, int nhandles, cudaGraphConditionalHandle h0,
                    cudaGraphConditionalHandle h1);

/* ---- multigrid-preconditioned conjugate gradients (mg3d_cg.cu), cubic and box levels alike ---- */
/* a colour-split level of either 3D engine: element (x,y,zl) of colour c = (x+y+z0+zl)&1 at base[c*cstride + zl*plane + y*hp +
   (x>>1)]; the grid is nx*ny*nz points, local planes zl = 0..nzl-1 are the global planes z0.. (one GPU: z0 = 0, nzl = nz) */
typedef struct {
    int nx, ny, nz, hp;
    long long plane, cstride;
    int z0, nzl;
} mg_geom3cg;

/* the device scalar block of one PCG (doubles) */
#define MGK_PCG_RHO 0   /* z.r of the current iteration (after mgk3cg_dots: the previous one's is gone) */
#define MGK_PCG_BETA 1
#define MGK_PCG_ALPHA 2
#define MGK_PCG_FIRST 3 /* nonzero: the next mgk3cg_dots starts the recurrence (beta = 0) */
#define MGK_PCG_PI 4
#define MGK_PCG_SCALARS 8
#define MGK_PCG_BLOCKS 296 /* the fixed grid of the passes (two blocks per SM of a B200) */
/* partials of one iteration: the dots and the direction pass write two double-double sums per block (4*MGK_PCG_BLOCKS
   doubles each), the update pass the {sum r^2, max|r|} pair of mgk_norm_final (2*MGK_PCG_BLOCKS) */
#define MGK_PCG_DIR_PARTS (4 * MGK_PCG_BLOCKS)
#define MGK_PCG_UPD_PARTS (8 * MGK_PCG_BLOCKS)
#define MGK_PCG_PARTS (10 * MGK_PCG_BLOCKS)
/* every launcher covers local planes [zl_lo, zl_hi) (on one GPU: all of them) */
/* rho = z.r, sigma = z.d -> beta (two launches) */
int mgk3cg_dots(cudaStream_t s, int dtype, const void* z, const void* r, const void* d, mg_geom3cg g, int zl_lo, int zl_hi,
                double* part, double* sc);
/* p_out = z + beta*p_in, pi = p_out.(Laplacian p_out) -> alpha (two launches) */
int mgk3cg_dir(cudaStream_t s, int dtype, const void* z, const void* p_in, void* p_out, mg_geom3cg g, mg_coef3d c, int zl_lo,
               int zl_hi, double* part, double* sc);
/* x_out = x_in + alpha*p, r = b - Laplacian x_out (in place over the old r), d = new r - old r; {sum r^2, max|r|} partials
   for mgk_norm_final */
int mgk3cg_update(cudaStream_t s, int dtype, const void* x_in, const void* p, const void* b, void* r, void* x_out, void* d,
                  mg_geom3cg g, mg_coef3d c, const double* sc, int zl_lo, int zl_hi, double* part);
/* r = b - Laplacian x (zero on the Dirichlet points), and the scalar block marked for a first iteration */
int mgk3cg_residual(cudaStream_t s, int dtype, const void* x, const void* b, void* r, mg_geom3cg g, mg_coef3d c, double* sc,
                    int zl_lo, int zl_hi);

/* ---- 2D (pitched: element (x,y) at base[x + y*pitch]) ---- */
typedef struct {
    int n;
    int pitch;
} mg_geom2d;

typedef struct {
    double hx, hy, xa, ya; /* N2/Grid2D.cpp:24-35 */
    double A[4];           /* matrixA, N2/MultiGrid2D.cpp:45-60 */
    int alfa;
} mg_coef2d;

int mgk2d_relax_colour(cudaStream_t s, int dtype, void* v, const void* f, mg_geom2d g, mg_coef2d c, int colour);
/* levels with n <= MGK2D_SMALL_N: all `ncycles` RB sweeps in ONE launch of one CTA, v in shared memory */
#define MGK2D_SMALL_N 65
int mgk2d_relax_small(cudaStream_t s, int dtype, void* v, const void* f, mg_geom2d g, mg_coef2d c, int ncycles);
int mgk2d_residual(cudaStream_t s, int dtype, const void* v, const void* f, void* r, mg_geom2d g, mg_coef2d c);
int mgk2d_residual_norm(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom2d g, mg_coef2d c,
                        double* scratch, double* out2);
int mgk2d_restrict(cudaStream_t s, int dtype, const void* fine, mg_geom2d gf, void* coarse, mg_geom2d gc);
int mgk2d_residual_restrict(cudaStream_t s, int dtype, const void* v, const void* f, mg_geom2d gf, mg_coef2d c,
                            void* coarse_f, void* coarse_v, mg_geom2d gc);
int mgk2d_interpolate(cudaStream_t s, int dtype, void* fine, mg_geom2d gf, const void* coarse, mg_geom2d gc, int add);
int mgk2d_apply_correction(cudaStream_t s, int dtype, void* fine, const void* err, mg_geom2d g);
int mgk2d_set(cudaStream_t s, int dtype, void* a, mg_geom2d g, double value, int modify_boundaries);
int mgk2d_init_v(cudaStream_t s, int dtype, void* v, mg_geom2d g, mg_coef2d c);
/* sum |v - (2x^2-4xy+2y^2)| over all points, C2/Grid2D.cu:123-154 */
int mgk2d_abs_error_sum(cudaStream_t s, int dtype, const void* v, mg_geom2d g, mg_coef2d c, double* scratch,
                        double* out2);

/* ---- 1D: the whole hierarchy lives in one device arena; one persistent CTA runs whole cycles ---- */
#define MG1D_MAX_LEVELS 32
typedef struct {
    int nlevels;
    int n[MG1D_MAX_LEVELS];
    long long off_v[MG1D_MAX_LEVELS]; /* element offsets into the arena */
    long long off_f[MG1D_MAX_LEVELS];
    long long off_e[MG1D_MAX_LEVELS]; /* e1[j] = exp(x_j) + 1 computed with the host libm (N1/MultiGrid1D.cpp:101) */
    long long off_d[MG1D_MAX_LEVELS]; /* d[j]  = exp(x_j) + 1 + h */
    double h[MG1D_MAX_LEVELS];
} mg_hier1d;

int mgk1d_relax(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int ncycles);
int mgk1d_residual(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected, void* r_out);
int mgk1d_residual_norm(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected, double* out2);
/* level operators inside the arena: which = 0 Restrict(f) level->level+1, 1 Interpolate level+1 -> v of level,
   2 Interpolate + ApplyCorrection */
int mgk1d_level_op(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int which);
/* {sum, max} of |v - table| over n points, one block (table: the analytic solution from the host libm) */
int mgk1d_abs_error(cudaStream_t s, int dtype, const void* v, const void* table, int n, double* out2);
int mgk1d_restrict(cudaStream_t s, int dtype, const void* fine, int fn, void* coarse, int cn);
int mgk1d_residual_restrict(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int corrected);
int mgk1d_interpolate(cudaStream_t s, int dtype, void* fine, int fn, const void* coarse, int cn, int add);
int mgk1d_apply_correction(cudaStream_t s, int dtype, void* fine, const void* err, int n);
int mgk1d_set(cudaStream_t s, int dtype, void* a, int n, double value, int modify_boundaries);
/* whole V-cycles / FMG in ONE launch: a single persistent CTA walks the hierarchy (2 055 points at n=1025) */
int mgk1d_cycle(cudaStream_t s, int dtype, void* arena, mg_hier1d H, int level, int v0, int v1, int v2, int corrected,
                int fmg);

#ifdef __cplusplus
}
#endif
#endif

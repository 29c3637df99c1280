/*
 * mg_b200.h -- C ABI of the B200-native geometric multigrid engine.
 *
 * Drop-in boundary for the multigrid hot path of MisterPup/PDE-MultiGrid.  The reference exposes
 * this path as three C++ classes with all-public members and no FFI (SURVEY.md 8b):
 *     MultiGrid3D  NOCUDA_TESI/POISSON_3D(TESI)/MultiGrid3D.h:6-33   (GPU twin CUDA_TESI/CUDA Poisson 3D/MultiGrid3D.h:6-37)
 *     MultiGrid2D  NOCUDA_TESI/PDE Lyapunov 2D/MultiGrid2D.h:6-37    (GPU twin CUDA_TESI/CUDA Lyapunov 2D/MultiGrid2D.h:6-33)
 *     MultiGrid1D  NOCUDA_TESI/EQUAZIONE 1D/MultiGrid1D.h:6-31       (GPU twin CUDA_TESI/CUDA 1D/MultiGrid1D.h:6-31)
 * Every entry point below names the reference method it replaces.  include/compat/ holds header-
 * compatible C++ shim classes (same class, member and method names) built on this ABI, so the
 * reference's own main() files compile unchanged against libmg_b200.so (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: opaque handles, plain pointers and sizes, no C++ or torch types;
 *   - every call returns MG_OK (0) or an MG_ERR_* code; mg_last_error() gives the message of the
 *     last failure on the calling thread (the reference aborts through assert(), N3/MultiGrid3D.cpp:60-62);
 *   - host arrays use the reference layout: dense, x fastest, idx = x + y*sx + z*sx*sy
 *     (N3/MultiGrid3D.cpp:518-531); the engine keeps its own pitched layout on the device;
 *   - `dtype` selects float (what the reference is written in) or double (what BASELINE.json asks for);
 *   - `residual_mode`: MG_REF_COMPAT reproduces the reference residual bug-for-bug (sign defects at
 *     N3/MultiGrid3D.cpp:723 and N1/MultiGrid1D.cpp:210), MG_CORRECTED flips those signs;
 *   - there is NO CPU fallback: without a CUDA device every create() fails with MG_ERR_CUDA;
 *   - one handle = one host thread; work is enqueued on the handle's stream; getters and *_host calls
 *     synchronise, the rest is asynchronous until mg*_sync().
 */
#ifndef MG_B200_H
#define MG_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MG_OK 0
#define MG_ERR_ARG 1   /* bad argument / size mismatch (reference: assert) */
#define MG_ERR_CUDA 2  /* CUDA runtime failure, or no device */
#define MG_ERR_NOMEM 3
#define MG_ERR_STATE 4 /* call not valid in the handle's current state */
#define MG_ERR_COMM 5  /* NCCL / multi-GPU failure */

#define MG_F32 0
#define MG_F64 1

#define MG_REF_COMPAT 0
#define MG_CORRECTED 1

#define MG_FIELD_V 0 /* Grid?D::h_v  approximate solution / error */
#define MG_FIELD_F 1 /* Grid?D::h_f  right-hand side / restricted residual */

/* smoother implementation (results are bit-identical; the choice only affects speed) */
#define MG_SMOOTHER_AUTO 0   /* the fastest available per level and call: MG_SMOOTHER_PIPE for pairs of sweeps where it
                                applies, MG_SMOOTHER_TMA for the rest, plain kernels on the small levels */
#define MG_SMOOTHER_COLOUR 1 /* one colour per launch, in place, plain kernels */
#define MG_SMOOTHER_FUSED 2  /* two RB sweeps per HBM pass, all stages through shared memory, the reference's literal
                                arithmetic (slower than MG_SMOOTHER_TMA; it is the exact fallback of MG_SMOOTHER_PIPE) */
#define MG_SMOOTHER_JACOBI 3 /* weighted Jacobi (3D only): v += omega*(GS(v_old) - v_old), all points from old values.
                                Not in the reference (it only has red-black Gauss-Seidel): no parity contract with it */

#define MG_SMOOTHER_TMA 4    /* one colour per launch with TMA-staged z-marching tiles on the large levels (no temporal blocking) */
#define MG_SMOOTHER_PIPE 5   /* two RB sweeps per HBM pass, register-tiled z-pipeline (large, cubic, power-of-two-h levels on
                                one GPU; elsewhere as MG_SMOOTHER_TMA) */

/* arithmetic of the temporally blocked smoother (mg3d_set_arith) */
#define MG_ARITH_EXACT 0 /* every rounding of the reference reproduced: results bit-identical to NOCUDA_TESI (default) */
#define MG_ARITH_FAST 1  /* pairwise sums, FMA, multiplication by 1/6: within 1e-10 (fp64) / 1e-5 (fp32) relative */

/* operator classes of the per-operator device timers (mg?d_profile_read) */
#define MG_OP_RELAX 0             /* Relax */
#define MG_OP_RESIDUAL_RESTRICT 1 /* CalculateResidual + Restrict + setToValue(coarse v) */
#define MG_OP_INTERPOLATE 2       /* Interpolate (+ ApplyCorrection) */
#define MG_OP_OTHER 3             /* Restrict(f), setToValue, halo exchange ... */
#define MG_OP_COUNT 4

typedef struct mg3d_s mg3d_t;
typedef struct mg2d_s mg2d_t;
typedef struct mg1d_s mg1d_t;
typedef struct mg3b_s mg3b_t;

const char* mg_last_error(void);
const char* mg_version(void);
int mg_device_count(void); /* 0 when no CUDA device is usable */

/* ------------------------------------------------------------------ 3D Poisson ------------- */
/* MultiGrid3D::MultiGrid3D + InitGrids (N3/MultiGrid3D.cpp:5-47): builds numGrids=(int)log2(n-1)
   levels, n_l=(n_{l-1}-1)/2+1, and initialises every level like Grid3D's ctor (InitV: boundary 0,
   InitF: f=-3*PI*PI*sin(PI x)sin(PI y)sin(PI z), N3/Grid3D.cpp:61-96); interior v is zeroed. */
int mg3d_create(mg3d_t** out, const int finest_size_xyz[3], const double range[6], int dtype, int residual_mode);
/* same, on `nranks` GPUs (one process each): z-slab partition, halo exchange over NCCL.
   nccl_unique_id: 128 bytes from mg_comm_unique_id() on rank 0, broadcast by the caller. */
int mg3d_create_dist(mg3d_t** out, const int finest_size_xyz[3], const double range[6], int dtype, int residual_mode,
                     int rank, int nranks, const void* nccl_unique_id);
int mg_comm_unique_id(void* out128);
/* slab plan of a level with n points per axis (pure arithmetic, no GPU needed): out5 = {distributed?, global z of
   the first stored plane, stored planes, first owned local plane, one past the last owned local plane} */
int mg3d_plan_level(int n, int nranks, int rank, int out5[5]);
/* global planes [z_begin, z_begin + z_count) this rank owns on `level` (the whole level when it is not distributed);
   set_field / get_field / residual / vcycle_host move exactly these planes */
int mg3d_owned_range(const mg3d_t* mg, int level, int* z_begin, int* z_count);
/* diagnostic: `reps` halo exchanges (colour_mask bit c = colour c; depth_up planes to rank+1, depth_down planes to rank-1)
   of the current v of `level`, enqueued back to back: times the NVLink transport (scripts/bench_halo.py) */
int mg3d_halo_benchmark(mg3d_t* mg, int level, int colour_mask, int depth_up, int depth_down, int reps);
long long mg3d_halo_bytes(const mg3d_t* mg); /* bytes this rank has sent in halo exchanges and gathers so far */
int mg3d_destroy(mg3d_t* mg); /* ~MultiGrid3D */
int mg3d_num_levels(const mg3d_t* mg);         /* MultiGrid3D::numGrids */
int mg3d_level_size(const mg3d_t* mg, int level); /* grids3D[level]->sizeX */
double mg3d_level_h(const mg3d_t* mg, int level); /* grids3D[level]->h_x */
/* sweeps_per_pass must name what the implementation does: 2 for MG_SMOOTHER_FUSED / MG_SMOOTHER_PIPE, 1 for the
   others; MG_SMOOTHER_AUTO takes 1 or 2 */
int mg3d_set_smoother(mg3d_t* mg, int smoother, int sweeps_per_pass);
int mg3d_set_arith(mg3d_t* mg, int arith); /* MG_ARITH_EXACT (default) or MG_ARITH_FAST */
/* relaxation weight of MG_SMOOTHER_JACOBI, 0 < omega <= 1 (default 6/7, the optimal smoothing weight of the 7-point
   Laplacian); rounded to the handle's dtype */
int mg3d_set_jacobi_weight(mg3d_t* mg, double omega);
int mg3d_sync(mg3d_t* mg);
void* mg3d_stream(mg3d_t* mg); /* cudaStream_t the handle enqueues on (for event timing) */
long long mg3d_kernel_launches(const mg3d_t* mg); /* kernels launched by this handle so far */
/* per-level, per-operator device time: CUDA events recorded on the handle's stream around every
   operator call while enabled.  enable != 0 resets the counters and starts, 0 stops. */
int mg3d_profile(mg3d_t* mg, int enable);
int mg3d_profile_read(mg3d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls);

/* grids3D[level]->h_v / h_f  <->  host dense array of n_l^3 values (multi-GPU: the owned planes, n_l*n_l*z_count) */
int mg3d_set_field(mg3d_t* mg, int level, int field, const void* host_dense);
int mg3d_get_field(mg3d_t* mg, int level, int field, void* host_dense);
/* re-run Grid3D::InitV/InitF on every level (device side) and zero the interior of v */
int mg3d_init_problem(mg3d_t* mg);

int mg3d_relax(mg3d_t* mg, int level, int ncycles);                 /* Relax(grids3D[level], ncycles) */
int mg3d_residual(mg3d_t* mg, int level, void* host_out);           /* CalculateResidual(grids3D[level]) -> caller-owned n^3 */
int mg3d_residual_norm(mg3d_t* mg, int level, double* l2, double* linf); /* norms of that residual (the reference has none) */
/* Grid3D::PrintDiff (N3/Grid3D.cpp:136-159) as a device reduction: mean and max over all n^3 points of
   |realSol - approxSol|, realSol = (real)(sin(PI x)sin(PI y)sin(PI z)); all ranks return the global values */
int mg3d_abs_error(mg3d_t* mg, int level, double* mean_abs, double* max_abs);
/* position-keyed additive checksum (mod 2^64) of a whole level field, bit-pattern based: equal checksums <=> equal bits
   for all practical purposes; slab partial sums are combined over the ranks.  Used by bench.py to show that a run on N
   GPUs holds the bits of the reference CPU solver (tests/golden/hashes3d.json) without moving the field to the host. */
int mg3d_field_checksum(mg3d_t* mg, int level, int field, unsigned long long* out);
int mg3d_restrict(mg3d_t* mg, int fine_level, int field);           /* Restrict(fine->field, ..., coarse->field, ...) */
int mg3d_residual_restrict(mg3d_t* mg, int fine_level);             /* Restrict(CalculateResidual(fine), coarse->h_f) + setToValue(coarse->h_v,0,true), fused */
int mg3d_interpolate(mg3d_t* mg, int fine_level);                   /* Interpolate(fine->h_v, ..., coarse->h_v, ...) */
int mg3d_interpolate_correct(mg3d_t* mg, int fine_level);           /* Interpolate(tmp, coarse->h_v) + ApplyCorrection(fine->h_v, tmp), fused */
int mg3d_set_to_value(mg3d_t* mg, int level, int field, double value, int modify_boundaries); /* setToValue / Set */
int mg3d_vcycle(mg3d_t* mg, int level, int v1, int v2);             /* VCycle(gridID, v1, v2) */
int mg3d_fmg(mg3d_t* mg, int level, int v0, int v1, int v2);        /* FullMultiGridVCycle(gridID, v0, v1, v2) */
/* V-cycles VCycle(level, v1, v2) from the current v of `level` until
 *     ||r_k||_2 <= max(atol, rtol * ||r_0||_2)
 * or max_cycles cycles have run.  r_k is the residual after k cycles, the same residual and the same reduction as
 * mg3d_residual_norm(level) (the reference has no norm: SURVEY.md 8c).
 * cycles_out: cycles run (0 if r_0 already meets the target).  converged_out: 1 / 0.
 * history: NULL, or room for 2*(max_cycles+1) doubles, receives (l2, linf) of r_0 .. r_cycles.
 * A non-finite l2 stops the solve with converged = 0.  Not converging is not an error: MG_OK is returned.
 * rtol, atol >= 0, max_cycles >= 0, v1, v2 >= 0, otherwise MG_ERR_ARG and nothing runs.
 * Synchronous: returns when the solve has finished.  On one GPU the loop runs on the device (a CUDA graph with a WHILE
 * node: one launch and one wait per solve); distributed handles, MG_B200_NO_GRAPH and per-operator profiling drive it
 * from the host, one read-back per cycle.  Both give the same bits.  The mg3b / mg2d / mg1d versions are the same. */
int mg3d_solve(mg3d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles,
               int* cycles_out, int* converged_out, double* history);
/* Conjugate gradients preconditioned by one VCycle(level, v1, v2) per iteration (flexible, Polak-Ribiere: an RB
 * Gauss-Seidel V-cycle is not a symmetric operator), for Laplacian_h v = f on `level` with v's boundary values as the
 * Dirichlet data -- the operator of the MG_CORRECTED residual -- starting from the current v.  The preconditioner is
 * VCycle from v = 0 with f = r and uses the handle's smoother, arithmetic mode and Jacobi weight.  Stopping rule and
 * history as mg3d_solve, on the TRUE residual b - Laplacian_h x_k (the reference's residual expression, recomputed every
 * iteration): ||r_k||_2 <= max(atol, rtol * ||r_0||_2), a non-finite l2 (which is also how a breakdown such as
 * p.Laplacian p = 0 surfaces), or max_iters.  history[0] is mg3d_residual_norm(level) bit for bit.
 * iters_out counts iterations, one V-cycle each.  On return v of `level` holds the iterate, f of `level` is the caller's
 * bit for bit, v and f of the coarser levels hold preconditioner scratch (as after mg3d_vcycle); max_iters = 0, or an r_0
 * that already meets the target, leaves v and f as they were.
 * MG_ERR_ARG as mg3d_solve; MG_ERR_STATE on an MG_REF_COMPAT handle (its residual, N3/MultiGrid3D.cpp:723, is not a
 * symmetric operator) and on a distributed handle (nranks > 1); nothing runs in either case.
 * Memory: six fields of `level` (b, x and p twice, d), allocated by the first call on the level (MG_ERR_NOMEM before
 * anything runs if that fails) and freed by mg3d_destroy: 52 GB at 1025^3 fp64, on top of the 38 GB of the hierarchy.
 * The loop runs on the device like mg3d_solve's (DESIGN.md section 6b).  mg3b_pcg is the same on a box grid. */
int mg3d_pcg(mg3d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_iters,
             int* iters_out, int* converged_out, double* history);

/* reference-facing calls on HOST arrays (NOCUDA signatures, N3/MultiGrid3D.h:16-27): upload, run, download */
int mg3d_restrict_host(mg3d_t* mg, const void* fine, const int fsize_xyz[3], void* coarse, const int csize_xyz[3]);
int mg3d_interpolate_host(mg3d_t* mg, void* fine, const int fsize_xyz[3], const void* coarse, const int csize_xyz[3]);
int mg3d_apply_correction_host(mg3d_t* mg, void* fine, const int fsize_xyz[3], const void* error, const int esize_xyz[3]);
int mg3d_set_to_value_host(mg3d_t* mg, void* grid, const int size_xyz[3], double value, int modify_boundaries);
/* The CUDA_TESI faces of the same operators: operands are DEVICE arrays in the reference's dense layout
   (CUDA_TESI/CUDA Poisson 3D/MultiGrid3D.h:16-24: d_fine / d_coarse / d_v; Grid3D.h:26-27: d_v, d_f).  The reference
   passes the size triplets as device arrays too (Grid3D.h:11 d_sizeXYZ) and copies them back in every wrapper
   (MultiGrid3D.cu:68-72); here they are host ints -- the shim of include/compat/ does that copy. */
int mg3d_set_field_device(mg3d_t* mg, int level, int field, const void* dev_dense); /* grids3D[level]->d_v|d_f -> engine */
int mg3d_get_field_device(mg3d_t* mg, int level, int field, void* dev_dense);       /* engine -> grids3D[level]->d_v|d_f */
int mg3d_residual_device(mg3d_t* mg, int level, void* dev_dense_out);               /* CalculateResidual -> caller-owned device array */
int mg3d_restrict_device(mg3d_t* mg, const void* d_fine, const int fsize_xyz[3], void* d_coarse, const int csize_xyz[3]);
int mg3d_interpolate_device(mg3d_t* mg, void* d_fine, const int fsize_xyz[3], const void* d_coarse, const int csize_xyz[3]);
int mg3d_apply_correction_device(mg3d_t* mg, void* d_fine, const int fsize_xyz[3], const void* d_error, const int esize_xyz[3]);
int mg3d_set_device(mg3d_t* mg, void* d_v, const int size_xyz[3], double value, int modify_border); /* Set(d_v, d_sizeXYZ, value, modifyBorder) */
/* end-to-end: upload finest v,f -> `cycles` x VCycle(0,v1,v2) -> download finest v */
int mg3d_vcycle_host(mg3d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles);

/* ------------------------------------------------------------------ 3D Poisson, non-cubic grids ---- */
/* sizeX != sizeY != sizeZ (every one 2^k + 1).  The reference's constructor already takes three sizes and its hierarchy and
   operators are written per dimension (N3/MultiGrid3D.cpp:5-8, :19-47: numGrids = (int)log2(minSize - 1), every dimension
   halved per level), but Grid3D asserts them equal (N3/Grid3D.cpp:10-11; lifting that is the author's TODO, SURVEY.md 8f
   rank 4).  Same operators, same arithmetic, results bit-identical to the reference compiled with its assertions off
   (oracle/_ref ref3d_*x, tests/test_box3d_gpu.py); colour-split device layout like the cubic engine's, one GPU, no TMA / temporal
   blocking (DESIGN.md section 4). */
int mg3b_create(mg3b_t** out, const int finest_size_xyz[3], const double range[6], int dtype, int residual_mode);
int mg3b_destroy(mg3b_t* mg);
int mg3b_num_levels(const mg3b_t* mg);                               /* MultiGrid3D::numGrids */
int mg3b_level_size(const mg3b_t* mg, int level, int out_xyz[3]);    /* grids3D[level]->sizeXYZ */
int mg3b_level_h(const mg3b_t* mg, int level, double out_xyz[3]);    /* grids3D[level]->h_x, h_y, h_z */
int mg3b_sync(mg3b_t* mg);
void* mg3b_stream(mg3b_t* mg);
long long mg3b_kernel_launches(const mg3b_t* mg);
int mg3b_set_field(mg3b_t* mg, int level, int field, const void* host_dense); /* sizeX*sizeY*sizeZ values, x fastest */
int mg3b_get_field(mg3b_t* mg, int level, int field, void* host_dense);
int mg3b_init_problem(mg3b_t* mg);                                   /* Grid3D::InitV/InitF, N3/Grid3D.cpp:61-96 */
int mg3b_relax(mg3b_t* mg, int level, int ncycles);                  /* Relax */
int mg3b_residual(mg3b_t* mg, int level, void* host_out);            /* CalculateResidual -> caller-owned array */
int mg3b_residual_norm(mg3b_t* mg, int level, double* l2, double* linf);
int mg3b_restrict(mg3b_t* mg, int fine_level, int field);            /* Restrict(fine->field, coarse->field) */
int mg3b_residual_restrict(mg3b_t* mg, int fine_level);              /* Restrict(CalculateResidual(fine), coarse->h_f) + setToValue(coarse->h_v,0,true) */
int mg3b_interpolate(mg3b_t* mg, int fine_level);                    /* Interpolate */
int mg3b_interpolate_correct(mg3b_t* mg, int fine_level);            /* Interpolate + ApplyCorrection */
int mg3b_set_to_value(mg3b_t* mg, int level, int field, double value, int modify_boundaries);
int mg3b_vcycle(mg3b_t* mg, int level, int v1, int v2);              /* VCycle */
int mg3b_fmg(mg3b_t* mg, int level, int v0, int v1, int v2);         /* FullMultiGridVCycle */
int mg3b_solve(mg3b_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles,
               int* cycles_out, int* converged_out, double* history); /* as mg3d_solve */
int mg3b_pcg(mg3b_t* mg, int level, int v1, int v2, double rtol, double atol, int max_iters,
             int* iters_out, int* converged_out, double* history);   /* as mg3d_pcg */
int mg3b_vcycle_host(mg3b_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles);
/* the operators on caller-owned HOST arrays (N3/MultiGrid3D.h:16-27 with three different sizes) */
int mg3b_restrict_host(mg3b_t* mg, const void* fine, const int fsize_xyz[3], void* coarse, const int csize_xyz[3]);
int mg3b_interpolate_host(mg3b_t* mg, void* fine, const int fsize_xyz[3], const void* coarse, const int csize_xyz[3]);
int mg3b_apply_correction_host(mg3b_t* mg, void* fine, const int fsize_xyz[3], const void* error, const int esize_xyz[3]);
int mg3b_set_to_value_host(mg3b_t* mg, void* grid, const int size_xyz[3], double value, int modify_boundaries);

/* ------------------------------------------------------------------ 2D Lyapunov ------------ */
/* MultiGrid2D::MultiGrid2D + InitGrids + InitA (N2/MultiGrid2D.cpp:5-60); A4 = row-major 2x2 by value
   (the reference's InitA overflows its 2-float buffer, SURVEY.md App. B7); alfa is int as in the reference. */
int mg2d_create(mg2d_t** out, const int finest_size_xy[2], const double range[4], const double A4[4], int alfa,
                int dtype);
int mg2d_destroy(mg2d_t* mg);
int mg2d_num_levels(const mg2d_t* mg);
int mg2d_level_size(const mg2d_t* mg, int level);
double mg2d_level_h(const mg2d_t* mg, int level);
int mg2d_sync(mg2d_t* mg);
void* mg2d_stream(mg2d_t* mg);
long long mg2d_kernel_launches(const mg2d_t* mg);
int mg2d_profile(mg2d_t* mg, int enable);
int mg2d_profile_read(mg2d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls);
int mg2d_set_field(mg2d_t* mg, int level, int field, const void* host_dense);
int mg2d_get_field(mg2d_t* mg, int level, int field, void* host_dense);
int mg2d_init_problem(mg2d_t* mg); /* Grid2D::InitV/InitF, N2/Grid2D.cpp:50-80 */
int mg2d_relax(mg2d_t* mg, int level, int ncycles);
int mg2d_residual(mg2d_t* mg, int level, void* host_out);
int mg2d_residual_norm(mg2d_t* mg, int level, double* l2, double* linf);
int mg2d_restrict(mg2d_t* mg, int fine_level, int field);
int mg2d_residual_restrict(mg2d_t* mg, int fine_level);
int mg2d_interpolate(mg2d_t* mg, int fine_level);
int mg2d_interpolate_correct(mg2d_t* mg, int fine_level);
int mg2d_set_to_value(mg2d_t* mg, int level, int field, double value, int modify_boundaries);
int mg2d_vcycle(mg2d_t* mg, int level, int v1, int v2);
int mg2d_fmg(mg2d_t* mg, int level, int v0, int v1, int v2);
int mg2d_solve(mg2d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles,
               int* cycles_out, int* converged_out, double* history); /* as mg3d_solve */
int mg2d_mean_abs_error(mg2d_t* mg, double* mae); /* PrintMeanAbsoluteError, C2/Grid2D.cu:123-154 */
int mg2d_restrict_host(mg2d_t* mg, const void* fine, const int fsize_xy[2], void* coarse, const int csize_xy[2]);
int mg2d_interpolate_host(mg2d_t* mg, void* fine, const int fsize_xy[2], const void* coarse, const int csize_xy[2]);
int mg2d_apply_correction_host(mg2d_t* mg, void* fine, const int fsize_xy[2], const void* error, const int esize_xy[2]);
int mg2d_set_to_value_host(mg2d_t* mg, void* grid, const int size_xy[2], double value, int modify_boundaries);
int mg2d_vcycle_host(mg2d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles);
/* the CUDA_TESI faces (CUDA_TESI/CUDA Lyapunov 2D/MultiGrid2D.h:20-25, Grid2D.h:19-22): pitched DEVICE arrays given as
   (pointer, size, pitch in elements); the kernels run on the caller's arrays in place.  mg2d_level_device_ptr hands out
   a level's own field (what the twin's Grid2D::d_v / d_f / d_pitch are). */
int mg2d_level_device_ptr(mg2d_t* mg, int level, int field, void** ptr, int* pitch_elems);
int mg2d_restrict_device(mg2d_t* mg, const void* fine, int fsize, int f_pitch, void* coarse, int csize, int c_pitch);
int mg2d_interpolate_device(mg2d_t* mg, void* fine, int fsize, int f_pitch, const void* coarse, int csize, int c_pitch);
int mg2d_apply_correction_device(mg2d_t* mg, void* fine, int fsize, int f_pitch, const void* error, int esize, int e_pitch);
int mg2d_set_device(mg2d_t* mg, void* v, int size, int pitch, double value, int modify_border);
int mg2d_residual_device(mg2d_t* mg, int level, void* dev_out); /* pitched like the level itself */

/* ------------------------------------------------------------------ 1D equation ------------ */
/* MultiGrid1D::MultiGrid1D + InitGrids (N1/MultiGrid1D.cpp:5-31) */
int mg1d_create(mg1d_t** out, int finest_size, const double range[2], int dtype, int residual_mode);
int mg1d_destroy(mg1d_t* mg);
int mg1d_num_levels(const mg1d_t* mg);
int mg1d_level_size(const mg1d_t* mg, int level);
double mg1d_level_h(const mg1d_t* mg, int level);
int mg1d_sync(mg1d_t* mg);
void* mg1d_stream(mg1d_t* mg);
long long mg1d_kernel_launches(const mg1d_t* mg);
int mg1d_profile(mg1d_t* mg, int enable);
int mg1d_profile_read(mg1d_t* mg, int level, int op, double* ms_total, long long* kernel_launches, long long* calls);
int mg1d_set_field(mg1d_t* mg, int level, int field, const void* host_dense);
int mg1d_get_field(mg1d_t* mg, int level, int field, void* host_dense);
int mg1d_init_problem(mg1d_t* mg); /* Grid1D::InitV/InitF, N1/Grid1D.cpp:30-43 */
int mg1d_relax(mg1d_t* mg, int level, int ncycles);
int mg1d_residual(mg1d_t* mg, int level, void* host_out);
int mg1d_residual_norm(mg1d_t* mg, int level, double* l2, double* linf);
/* Grid1D::PrintDiffApproxReal (N1/Grid1D.cpp:46-60) as a device reduction: mean and max of |approxsol - realsol| */
int mg1d_abs_error(mg1d_t* mg, int level, double* mean_abs, double* max_abs);
int mg1d_restrict(mg1d_t* mg, int fine_level, int field);
int mg1d_residual_restrict(mg1d_t* mg, int fine_level);
int mg1d_interpolate(mg1d_t* mg, int fine_level);
int mg1d_interpolate_correct(mg1d_t* mg, int fine_level);
int mg1d_set_to_value(mg1d_t* mg, int level, int field, double value, int modify_boundaries);
int mg1d_vcycle(mg1d_t* mg, int level, int v1, int v2);
int mg1d_fmg(mg1d_t* mg, int level, int v0, int v1, int v2);
int mg1d_solve(mg1d_t* mg, int level, int v1, int v2, double rtol, double atol, int max_cycles,
               int* cycles_out, int* converged_out, double* history); /* as mg3d_solve */
int mg1d_restrict_host(mg1d_t* mg, const void* fine, int fsize, void* coarse, int csize);
int mg1d_interpolate_host(mg1d_t* mg, void* fine, int fsize, const void* coarse, int csize);
int mg1d_apply_correction_host(mg1d_t* mg, void* fine, int fsize, const void* error, int esize);
int mg1d_set_to_value_host(mg1d_t* mg, void* grid, int size, double value, int modify_boundaries);
int mg1d_vcycle_host(mg1d_t* mg, void* v_host, const void* f_host, int v1, int v2, int cycles);
/* the CUDA_TESI faces (CUDA_TESI/CUDA 1D/MultiGrid1D.h:16-23, Grid1D.h:15-18): DEVICE arrays */
int mg1d_level_device_ptr(mg1d_t* mg, int level, int field, void** ptr);
int mg1d_restrict_device(mg1d_t* mg, const void* fine, int fsize, void* coarse, int csize);
int mg1d_interpolate_device(mg1d_t* mg, void* fine, int fsize, const void* coarse, int csize);
int mg1d_apply_correction_device(mg1d_t* mg, void* fine, int fsize, const void* error, int esize);
int mg1d_set_device(mg1d_t* mg, void* d_v, int size, double value, int modify_boundaries);
int mg1d_residual_device(mg1d_t* mg, int level, void* dev_out);

#ifdef __cplusplus
}
#endif
#endif /* MG_B200_H */

// mg3d_rr_tma.cu -- fused CalculateResidual + Restrict (+ zero of the coarse v) for the large 3D levels,
// with TMA-staged z-marching shared-memory tiles.  Replaces, in one pass over HBM,
//     residual = CalculateResidual(fine)                       N3/MultiGrid3D.cpp:678-730
//     Restrict(residual, ..., coarse->h_f, ...)                N3/MultiGrid3D.cpp:50-184
//     setToValue(coarse->h_v, ..., 0, true)                    N3/MultiGrid3D.cpp:634
// The fine residual only ever exists in registers and shared memory.
//
// A CTA owns a (CXT x CYT) column of coarse points and marches along z, two FINE planes per iteration:
//   * the two colour sub-tiles of the fine v planes arrive by TMA (two cp.async.bulk.tensor.3d on one
//     mbarrier per plane) into a 6-slot ring, four planes ahead of their use; halo / out-of-domain
//     elements are zero-filled by the hardware;
//   * REGISTER TILING: thread (lane, warp) owns the 2x2 fine points under its coarse point -- half-index
//     cx0+lane (x = 2cx, 2cx+1, one point in each colour array) of rows 2cy, 2cy+1 -- and keeps their v
//     values of planes z-1, z, z+1 in registers.  Of the 7 stencil values of a residual, own value, D/U,
//     one of O/E and one of N/S are then registers; 3 shared-memory loads per point remain (the new
//     plane, the far O/E, the far N/S) instead of 7;
//   * the residuals of the thread's 2x2 column stay in registers for its own restriction (12 of the 27
//     taps); only the ones a neighbour needs go to a 3-slot ring of residual planes (parity-split in
//     x, unit-stride reads), from which the other 15 taps are loaded.  The residual row below and the
//     residual column left of the tile (81 points per plane) are computed by four warps the plain way;
//   * after every odd fine plane 2k+1 the coarse plane k is produced with the reference's exact grouping
//     of the 27 weights, and written together with coarse v = 0.
// The version before this one read every stencil value from shared memory: the LSU data pipe was the
// limiter (l1tex__data_pipe_lsu_wavefronts 76 % of peak, 815 M load wavefronts per launch at 1025^3;
// profiles/r1_residual_restrict_tma_ncu_full.txt).
// HBM traffic per fine point: v and f once (+ 19/16 x 36/32 halo re-reads that hit L2) and 2/8 coarse
// writes: the algorithmic 2*B*N_l + 2*B*N_{l+1} of SURVEY.md 8(d).
#include "mg3d_device.cuh"
#include "mg_tma.cuh"

using namespace mgx;
using namespace mg3;
using namespace mgtma;

namespace {

constexpr int CXT = MGK3D_RR_CXT;       // coarse points per tile in x
constexpr int CYT = MGK3D_RR_CYT;       // coarse points per tile in y
constexpr int VROWS = MGK3D_RR_BOX_Y;   // fine rows of a v tile: 2*CYT + 3
constexpr int RROWS = 2 * CYT + 1;      // fine rows of a residual plane tile
constexpr int RCOLS = CXT + 2;          // per-parity columns of a residual row (33 used, even pitch)
constexpr int RING = 6;   // v planes: z-1 .. z+2 live during a pair of planes + two in flight
constexpr int RRING = 3;  // residual planes: 2k-1, 2k, 2k+1
constexpr int NT = 256;
constexpr int RR_ZCHUNK_MAX = 16;  // coarse planes per CTA before tile_grid halves it to fill the SMs

template <typename T> struct VBox {
    static constexpr int A = 16 / sizeof(T);                      // TMA inner-coordinate alignment in elements
    static constexpr int W = (CXT + A + 1 + A - 1) / A * A;       // 36 doubles / 40 floats
};

// NORM = true turns the kernel into the residual-norm pass (sum r^2 in fp64 and max |r| over the fine planes 2cz, 2cz+1 of
// the chunk's coarse planes -- every fine plane exactly once over the grid): same staging and register tiling, no
// residual ring, no restriction, one partial per CTA in part[0 .. nblocks) / part[nblocks .. 2 nblocks).
template <typename T, bool FAST, bool NORM>
__global__ void __launch_bounds__(NT, 2)
k_residual_restrict_tma(const __grid_constant__ CUtensorMap map_c0, const __grid_constant__ CUtensorMap map_c1,
                        const __grid_constant__ CUtensorMap map_f0, const __grid_constant__ CUtensorMap map_f1, int f_prefetch,
                        const T* __restrict__ f, mg_geom3d gf, Coef3<T> c, int corrected, T* __restrict__ cf,
                        T* __restrict__ cv, mg_geom3d gc, int czl_lo, int czl_hi, int zchunk, double* __restrict__ part)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int A = VBox<T>::A, W = VBox<T>::W;
    constexpr int VSUB = VROWS * W;                                // one colour sub-tile
    constexpr uint32_t VSUB_BYTES = VSUB * sizeof(T);
    constexpr int VSUB_STRIDE = (VSUB_BYTES + 127) / 128 * 128 / sizeof(T);
    constexpr int VSLOT = 2 * VSUB_STRIDE;                         // both colours of one fine plane
    constexpr int RSLOT = RROWS * 2 * RCOLS;                       // residual plane: [row][x parity][col]
    T* vring = reinterpret_cast<T*>(smem_raw);
    T* rring = vring + (size_t)RING * VSLOT;
    uint64_t* bars = reinterpret_cast<uint64_t*>(rring + (size_t)RRING * RSLOT);

    const int tid = threadIdx.x;
    const int cx0 = blockIdx.x * CXT, cy0 = blockIdx.y * CYT;
    const int czl0 = czl_lo + blockIdx.z * zchunk;                 // coarse local planes [czl0, czl1)
    const int czl1 = min(czl0 + zchunk, czl_hi);
    const int n = gf.n;
    // fine GLOBAL planes whose residual is needed: 2*cz-1 .. 2*cz+1 for every coarse plane of the chunk
    const int zf0 = 2 * (gc.z0 + czl0) - 1, zf1 = 2 * (gc.z0 + czl1 - 1) + 1;
    const int fy0 = 2 * cy0 - 1;                                   // first fine row of the residual tile
    const int hi_org = cx0 - A;                                    // half-index of column 0 of a v sub-tile

    if (tid == 0) {
        prefetch_tensormap(&map_c0);
        prefetch_tensormap(&map_c1);
        for (int s = 0; s < RING; s++) mbar_init(&bars[s], 1);
        fence_barrier_init();
    }
    __syncthreads();

    // v plane p (global) lives in slot (p - pbase) % RING; planes pbase = zf0-1 .. zf1+1 are streamed
    const int pbase = zf0 - 1;
    auto issue = [&](int p) {
        const unsigned s = (unsigned)(p - pbase) % RING;
        T* dst = vring + (size_t)s * VSLOT;
        mbar_arrive_expect_tx(&bars[s], 2 * VSUB_BYTES);
        tma_load_3d(dst, &map_c0, &bars[s], hi_org, fy0 - 1, p - gf.z0);
        tma_load_3d(dst + VSUB_STRIDE, &map_c1, &bars[s], hi_org, fy0 - 1, p - gf.z0);
    };
    auto wait_plane = [&](int p) {
        const unsigned k = (unsigned)(p - pbase);
        mbar_wait(&bars[k % RING], (k / RING) & 1);
    };
    auto slot_of = [&](int p) -> const T* { return vring + ((unsigned)(p - pbase) % RING) * VSLOT; };
    // f is read with plain loads one plane ahead of its use; an L2 prefetch of its tile a few planes further ahead (TMA
    // prefetch, no shared memory, one thread) turns those loads into L2 hits
    auto prefetch_f = [&](int p) {
        const int pl = p - gf.z0;
        if (!f_prefetch || pl < 0 || pl >= gf.nzl || p > zf1) return;
        asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(&map_f0), "r"(cx0), "r"(fy0), "r"(pl) : "memory");
        asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(&map_f1), "r"(cx0), "r"(fy0), "r"(pl) : "memory");
    };
    if (tid == 0) {
        for (int p = pbase; p <= min(pbase + RING - 1, zf1 + 1); p++) issue(p);
        for (int p = zf0; p <= zf0 + RING; p++) prefetch_f(p);
    }

    static_assert(CXT == 32 && CYT == 8 && NT == 256, "thread mapping: one coarse point = one 2x2 fine column per thread");
    const int w = tid >> 5, lane = tid & 31;
    const int hp = gf.hp;
    // the thread's fine column: half-index hi = cx0 + lane; rows ya = 2*(cy0+w) (even, "row 0") and ya+1 ("row 1").
    // Element of a colour sub-tile: row y - (fy0-1), column hi - hi_org.
    const int Pa = (2 * w + 2) * W + lane + A, Pb = Pa + W;
    const int T2 = (2 * w + 1) * 2 * RCOLS + lane;  // residual-plane element of (row ya, odd x = 2hi-1)
    // Per-thread predicates live in one opaque bit mask (otherwise ptxas re-derives each of them from
    // blockIdx/threadIdx in every plane).
    enum : unsigned {
        F_X0 = 1u << 0, F_X1 = 1u << 1,   // x = 2hi / 2hi+1 is an interior column
        F_YA = 1u << 2, F_YB = 1u << 3,   // row ya / ya+1 is an interior row
        F_FA = 1u << 4, F_FB = 1u << 5,   // f needed in row ya / ya+1
        F_TACT = 1u << 8, F_TST0 = 1u << 9, F_T0 = 1u << 10, F_T1 = 1u << 11, F_TF = 1u << 12, F_TP = 1u << 13,  // edge pass
        F_CIN = 1u << 14, F_CBND = 1u << 15, F_CP = 1u << 16  // coarse point: inside the grid, on its boundary, (cx+cy)&1
    };
    unsigned fl = 0;
    int t_own, t_oth, t_r;
    const T *fp, *tfp;  // f of the thread's (hi, ya) / edge-pass point in plane zf0 (advanced by one plane per plane)
    long long c_base;
    {
        const int hi = cx0 + lane, ya = 2 * (cy0 + w);
        const bool xv0 = 2 * hi >= 1 && 2 * hi <= n - 2, xv1 = 2 * hi + 1 <= n - 2;
        const bool yva = ya >= 1 && ya <= n - 2, yvb = ya + 1 <= n - 2;
        fl |= (xv0 ? F_X0 : 0) | (xv1 ? F_X1 : 0) | (yva ? F_YA : 0) | (yvb ? F_YB : 0);
        fl |= (yva && (xv0 || xv1) ? F_FA : 0) | (yvb && (xv0 || xv1) ? F_FB : 0);  // f is only read where a residual is evaluated
        const long long zoff = (long long)(zf0 - gf.z0) * gf.plane;
        fp = f + (zoff + (long long)ya * hp + hi);

        // edge pass: the residual row below the tile (ly = 0: warps 0, 1 = colour 0, 1 at half-indices cx0..cx0+31)
        // and the half-index left of it (hl = 0, every (colour, row) pair: 34 lanes of warps 2, 3)
        int col, ly, hl;
        bool act;
        if (w < 2) { col = w; ly = 0; hl = lane + 1; act = true; }
        else {
            const int u = (w - 2) * 32 + lane;
            act = w < 4 && u < 2 * RROWS;
            col = (act && u >= RROWS) ? 1 : 0;
            ly = act ? u - col * RROWS : 0;
            hl = 0;
        }
        const int y = fy0 + ly, thi = cx0 - 1 + hl, cc = (ly + 1) * W + hl + A - 1;
        t_own = col * VSUB_STRIDE + cc;
        t_oth = (col ^ 1) * VSUB_STRIDE + cc;
        t_r = ly * 2 * RCOLS + hl;
        const bool tyv = act && y >= 1 && y <= n - 2;
        const bool tx0 = hl >= 1 && 2 * thi >= 1 && 2 * thi <= n - 2, tx1 = 2 * thi + 1 >= 1 && 2 * thi + 1 <= n - 2;
        fl |= (act ? F_TACT : 0) | (act && hl >= 1 ? F_TST0 : 0) | (tyv && tx0 ? F_T0 : 0) | (tyv && tx1 ? F_T1 : 0) |
              (tyv && (tx0 || tx1) ? F_TF : 0) | (((col + y) & 1) ? F_TP : 0);
        tfp = f + (zoff + (long long)col * gf.cstride + (long long)y * hp + thi);

        // the thread's coarse point: cx = cx0 + lane, cy = cy0 + w
        const int cx = cx0 + lane, cy = cy0 + w;
        fl |= (cx < gc.n && cy < gc.n ? F_CIN : 0) | ((cx == 0 || cx == gc.n - 1 || cy == 0 || cy == gc.n - 1) ? F_CBND : 0) |
              (((cx + cy) & 1) ? F_CP : 0);
        c_base = (long long)cy * gc.hp + (cx >> 1);
    }
    asm volatile("" : "+r"(fl));
    const long long f_c1 = gf.cstride;  // f offset of colour 1, in elements (row ya+1: + hp)

    const int nzl = gf.nzl;
    // f of plane z (fp/tfp point into that plane) -> dst[row*2 + colour], dst[4] = edge pass
    auto load_f = [&](int z, T (&dst)[5]) {
        const int zl = z - gf.z0;
        const unsigned m = (zl >= 0 && zl < nzl) ? fl : 0u;
        if (m & (F_FA | F_FB)) MG_CHK_SITE(gf, cx0 + lane, 2 * (cy0 + w) + ((m & F_FA) ? 0 : 1), zl);
        dst[0] = (m & F_FA) ? __ldg(fp) : T(0);
        dst[1] = (m & F_FA) ? __ldg(fp + f_c1) : T(0);
        dst[2] = (m & F_FB) ? __ldg(fp + hp) : T(0);
        dst[3] = (m & F_FB) ? __ldg(fp + f_c1 + hp) : T(0);
        dst[4] = (m & F_TF) ? __ldg(tfp) : T(0);
    };

    // v of the thread's column: vm/vc/vu[row*2 + colour] at planes z-1, z, z+1
    T vm[4], vc[4], vu[4];
    // residuals of the thread's column by [row*2 + x parity]: planes 2k-1, 2k, 2k+1
    T rm[4] = {T(0), T(0), T(0), T(0)}, rc[4], rp[4];
    T fcur[5], fnext[5];
    double nsum = 0.0, nmax = 0.0;  // NORM: this thread's share

    // residual of fine plane z (ZP = z & 1) for the thread's column and the edge pass; v ring slots of planes
    // z-1, z, z+1 must have landed.  Shifts the register window by one plane at the end.
    auto plane = [&](int z, auto ZPc, T (&res)[4], bool count) {
        constexpr int ZP = decltype(ZPc)::value;
        const T* sD = slot_of(z - 1);
        const T* sC = slot_of(z);
        const T* sU = slot_of(z + 1);
        T* rz = rring + ((unsigned)(z - zf0) % RRING) * RSLOT;
        vu[0] = sU[Pa]; vu[1] = sU[VSUB_STRIDE + Pa]; vu[2] = sU[Pb]; vu[3] = sU[VSUB_STRIDE + Pb];
        const unsigned vmask = (z >= 1 && z <= n - 2) ? fl : 0u;  // residual is zero on the boundary planes
#pragma unroll
        for (int r = 0; r < 2; r++)
#pragma unroll
            for (int col = 0; col < 2; col++) {
                const int q = (col + r + ZP) & 1;  // x parity of this colour in this row of this plane: compile time
                const int oth = col ^ 1;
                const int P = r ? Pb : Pa;
                const T side = sC[oth * VSUB_STRIDE + P + (q ? 1 : -1)];
                const T own_oth = vc[r * 2 + oth];
                const T O = q ? own_oth : side, E = q ? side : own_oth;
                const T N = r ? vc[0 * 2 + oth] : sC[oth * VSUB_STRIDE + Pa - W];
                const T S = r ? sC[oth * VSUB_STRIDE + Pb + W] : vc[1 * 2 + oth];
                const T val = residual_point<T, FAST>(O, E, N, S, vm[r * 2 + oth], vu[r * 2 + oth], vc[r * 2 + col], fcur[r * 2 + col], c, corrected);
                const bool ok = (vmask & (r ? F_YB : F_YA)) && (vmask & (q ? F_X1 : F_X0));
                res[r * 2 + q] = ok ? val : T(0);
            }
        if constexpr (NORM) {
            if (count) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const double rd = (double)res[j];
                    nsum += rd * rd;
                    nmax = max_nan(nmax, fabs(rd));
                }
            }
        } else {
        // what the neighbours' restrictions read: the odd-x points (thread lane+1) and row ya+1 (warp w+1)
        rz[T2 + 1] = res[1];                         // (ya,   2hi+1): parity array 0 at lane+1
        rz[T2 + 2 * RCOLS + 1] = res[3];             // (ya+1, 2hi+1)
        rz[T2 + 2 * RCOLS + RCOLS] = res[2];         // (ya+1, 2hi):   parity array 1 at lane
        if (w < 4) {  // warp-uniform: the edge pass, every stencil value from shared memory
            const int q = ((fl / F_TP) ^ z) & 1;
            T val = T(0);
            if (vmask & (q ? F_T1 : F_T0)) {
                const int o = t_oth;
                val = residual_point<T, FAST>(sC[o - 1 + q], sC[o + q], sC[o - W], sC[o + W], sD[o], sU[o], sC[t_own], fcur[4], c, corrected);
            }
            if (fl & (q ? F_TACT : F_TST0)) rz[t_r + (q ? 0 : RCOLS - 1)] = val;
        }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) { vm[j] = vc[j]; vc[j] = vu[j]; }
    };
    auto step_f = [&](int z) {  // fcur <- f of plane z (prefetched), fnext <- f of plane z+1
#pragma unroll
        for (int j = 0; j < 5; j++) fcur[j] = fnext[j];
        fp += gf.plane;
        tfp += gf.plane;
        if (z < zf1) load_f(z + 1, fnext);
    };

    // ---- prologue: the odd plane zf0 = 2*cz0 - 1 ----
    load_f(zf0, fnext);
    step_f(zf0);
    wait_plane(zf0 - 1);
    wait_plane(zf0);
    wait_plane(zf0 + 1);
    {
        const T *s0 = slot_of(zf0 - 1), *s1 = slot_of(zf0);
        vm[0] = s0[Pa]; vm[1] = s0[VSUB_STRIDE + Pa]; vm[2] = s0[Pb]; vm[3] = s0[VSUB_STRIDE + Pb];
        vc[0] = s1[Pa]; vc[1] = s1[VSUB_STRIDE + Pa]; vc[2] = s1[Pb]; vc[3] = s1[VSUB_STRIDE + Pb];
    }
    plane(zf0, std::integral_constant<int, 1>{}, rm, false);  // counted by the chunk below (or a ghost plane)
    __syncthreads();  // v slot of plane zf0-1 free
    if (tid == 0 && zf0 + RING - 1 <= zf1 + 1) issue(zf0 + RING - 1);

    // ---- pairs of planes (2cz, 2cz+1), then coarse plane cz ----
    for (int z = zf0 + 1; z < zf1; z += 2) {
        step_f(z);
        wait_plane(z + 1);
        plane(z, std::integral_constant<int, 0>{}, rc, true);
        step_f(z + 1);
        wait_plane(z + 2);
        plane(z + 1, std::integral_constant<int, 1>{}, rp, true);
        __syncthreads();  // residual planes z-1, z, z+1 complete in shared memory; v slots of planes z-1, z free
        if (tid == 0) {
            if (z + RING - 1 <= zf1 + 1) issue(z + RING - 1);
            if (z + RING <= zf1 + 1) issue(z + RING);
            prefetch_f(z + RING + 1);
            prefetch_f(z + RING + 2);
        }
        if constexpr (NORM) continue;
        const int cz = z >> 1, czl = cz - gc.z0;
        if (fl & F_CIN) {
            T out = T(0);  // boundary: injection of the zero boundary residual (N3/MultiGrid3D.cpp:113-119, :705)
            if (!((fl & F_CBND) || cz == 0 || cz == gc.n - 1)) {
                const unsigned s0 = (unsigned)(z - 1 - zf0) % RRING;
                const T* qm = rring + s0 * RSLOT + T2;                                 // plane z-1
                const T* qc = rring + (s0 == RRING - 1 ? 0u : s0 + 1) * RSLOT + T2;    // plane z
                const T* qp = rring + (s0 == 0 ? RRING - 1u : s0 - 1) * RSLOT + T2;    // plane z+1
                // centre (2cx, 2cy) = the thread's (row 0, even x).  dx, dy in {0, 1}: own registers; dx = -1: parity
                // array 0 at lane of rows ya-1 .. ya+1; dy = -1: row ya-1, even x: array 1 at lane, odd x: array 0 at lane+1
                out = restrict_point<T>([&](int dx, int dy, int dz) {
                    if (dx >= 0 && dy >= 0) return dz < 0 ? rm[dy * 2 + dx] : (dz == 0 ? rc[dy * 2 + dx] : rp[dy * 2 + dx]);
                    const T* pl = dz < 0 ? qm : (dz == 0 ? qc : qp);
                    if (dx < 0) return pl[dy * 2 * RCOLS];
                    return dx == 0 ? pl[-2 * RCOLS + RCOLS] : pl[-2 * RCOLS + 1];
                });
            }
            const long long ci = ((((fl / F_CP) ^ cz) & 1) ? gc.cstride : 0ll) + (long long)czl * gc.plane + c_base;
            MG_CHK_SITE(gc, (cx0 + lane) >> 1, cy0 + w, czl);
            cf[ci] = out;
            cv[ci] = T(0);  // setToValue(coarse->h_v, 0, true), N3/MultiGrid3D.cpp:634
        }
#pragma unroll
        for (int j = 0; j < 4; j++) rm[j] = rp[j];
        __syncthreads();  // the 3-slot residual ring: plane z-1 is overwritten by plane z+2
    }
    if constexpr (NORM) {
        __shared__ double sh[64];
        block_sum_max(nsum, nmax, sh);
        if (tid == 0) {
            const unsigned nb = gridDim.x * gridDim.y * gridDim.z;
            const unsigned bid = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
            part[bid] = nsum;
            part[nb + bid] = nmax;
        }
    }
}

template <typename T>
size_t smem_bytes_t()
{
    constexpr size_t vsub = ((size_t)VROWS * VBox<T>::W * sizeof(T) + 127) / 128 * 128;
    return RING * 2 * vsub + (size_t)RRING * RROWS * 2 * RCOLS * sizeof(T) + RING * sizeof(uint64_t);
}

static void tile_grid(const mg_geom3d& gc, int czl_lo, int czl_hi, dim3& grid, int& zchunk)
{
    const int planes = czl_hi - czl_lo;
    const int tiles_xy = ((gc.n + CXT - 1) / CXT) * ((gc.n + CYT - 1) / CYT);
    // coarse planes per CTA: every chunk re-reads two fine planes of halo and refills its ring.  16-24 measured best at 1025^3
    // (3.80 ms against 3.87 at 32, 4.28 at 64, 5.46 at 256: short chunks keep neighbouring tiles in step, and their shared halo rows in L2)
    zchunk = RR_ZCHUNK_MAX;
    while (zchunk > 8 && (long long)tiles_xy * ((planes + zchunk - 1) / zchunk) < 148 * 4) zchunk /= 2;
    grid = dim3((gc.n + CXT - 1) / CXT, (gc.n + CYT - 1) / CYT, (planes + zchunk - 1) / zchunk);
}

template <typename T, bool FAST, bool NORM>
int launch_k(cudaStream_t s, const CUtensorMap& m0, const CUtensorMap& m1, const CUtensorMap* mf, const T* f, mg_geom3d gf, mg_coef3d c, int corrected, T* cf,
             T* cv, mg_geom3d gc, int czl_lo, int czl_hi, dim3 grid, int zchunk, double* part)
{
    const size_t smem = smem_bytes_t<T>();
    MG_SET_SMEM_LIMIT((k_residual_restrict_tma<T, FAST, NORM>), smem_bytes_t<T>());
    k_residual_restrict_tma<T, FAST, NORM><<<grid, NT, smem, s>>>(m0, m1, mf ? mf[0] : m0, mf ? mf[1] : m1, mf != nullptr, f, gf, narrow<T>(c), corrected, cf, cv,
                                                                 gc, czl_lo, czl_hi, zchunk, part);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

template <typename T>
int launch(cudaStream_t s, const void* tmap_c0, const void* tmap_c1, const void* const tmap_f[2], const T* f, mg_geom3d gf, mg_coef3d c,
           int corrected, T* cf, T* cv, mg_geom3d gc, int czl_lo, int czl_hi)
{
    if (czl_hi <= czl_lo) return 0;
    static_assert(NT == CXT * CYT, "one coarse point per thread");
    dim3 grid;
    int zchunk;
    tile_grid(gc, czl_lo, czl_hi, grid, zchunk);
    CUtensorMap m0, m1, mf[2];
    memcpy(&m0, tmap_c0, sizeof m0);
    memcpy(&m1, tmap_c1, sizeof m1);
    const bool pf = tmap_f && tmap_f[0] && tmap_f[1];
    if (pf) { memcpy(&mf[0], tmap_f[0], sizeof m0); memcpy(&mf[1], tmap_f[1], sizeof m0); }
    if (c.fast_h) return launch_k<T, true, false>(s, m0, m1, pf ? mf : nullptr, f, gf, c, corrected, cf, cv, gc, czl_lo, czl_hi, grid, zchunk, nullptr);
    return launch_k<T, false, false>(s, m0, m1, pf ? mf : nullptr, f, gf, c, corrected, cf, cv, gc, czl_lo, czl_hi, grid, zchunk, nullptr);
}

template <typename T>
int launch_norm(cudaStream_t s, const void* tmap_c0, const void* tmap_c1, const T* f, mg_geom3d gf, mg_coef3d c, int corrected,
                mg_geom3d gc, int czl_lo, int czl_hi, double* part, int max_parts, int* nparts)
{
    dim3 grid;
    int zchunk;
    tile_grid(gc, czl_lo, czl_hi, grid, zchunk);
    const long long nb = (long long)grid.x * grid.y * grid.z;
    if (czl_hi <= czl_lo || nb > max_parts) return -2;  // the caller takes the plain kernel
    *nparts = (int)nb;
    CUtensorMap m0, m1;
    memcpy(&m0, tmap_c0, sizeof m0);
    memcpy(&m1, tmap_c1, sizeof m1);
    if (c.fast_h) return launch_k<T, true, true>(s, m0, m1, nullptr, f, gf, c, corrected, nullptr, nullptr, gc, czl_lo, czl_hi, grid, zchunk, part);
    return launch_k<T, false, true>(s, m0, m1, nullptr, f, gf, c, corrected, nullptr, nullptr, gc, czl_lo, czl_hi, grid, zchunk, part);
}

}  // namespace

extern "C" int mgk3d_residual_restrict_tma(cudaStream_t s, int dtype, const void* tmap_v_c0, const void* tmap_v_c1, const void* const tmap_f[2],
                                           const void* f, mg_geom3d gf, mg_coef3d c, int corrected, void* coarse_f, void* coarse_v, mg_geom3d gc,
                                           int czl_lo, int czl_hi)
{
    if (dtype == 0)
        return launch<float>(s, tmap_v_c0, tmap_v_c1, tmap_f, (const float*)f, gf, c, corrected, (float*)coarse_f, (float*)coarse_v, gc, czl_lo, czl_hi);
    return launch<double>(s, tmap_v_c0, tmap_v_c1, tmap_f, (const double*)f, gf, c, corrected, (double*)coarse_f, (double*)coarse_v, gc, czl_lo, czl_hi);
}

/* residual norm of the fine planes under the coarse planes [czl_lo, czl_hi) with the staging of the kernel above: partials into
   scratch[0 .. 2*nparts), then {sum r^2, max |r|} into out2.  Returns -2 (nothing launched) when the tiling needs more
   than max_parts partials. */
extern "C" int mgk3d_residual_norm_tma(cudaStream_t s, int dtype, const void* tmap_v_c0, const void* tmap_v_c1, const void* f,
                                       mg_geom3d gf, mg_coef3d c, int corrected, mg_geom3d gc, int czl_lo, int czl_hi,
                                       double* scratch, int max_parts, double* out2)
{
    int nparts = 0;
    const int k = dtype == 0
        ? launch_norm<float>(s, tmap_v_c0, tmap_v_c1, (const float*)f, gf, c, corrected, gc, czl_lo, czl_hi, scratch, max_parts, &nparts)
        : launch_norm<double>(s, tmap_v_c0, tmap_v_c1, (const double*)f, gf, c, corrected, gc, czl_lo, czl_hi, scratch, max_parts, &nparts);
    if (k < 0) return k;
    const int k2 = mgk_norm_final(s, scratch, nparts, out2);
    return k2 < 0 ? -1 : k + k2;
}

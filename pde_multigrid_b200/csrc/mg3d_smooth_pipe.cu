// mg3d_smooth_pipe.cu -- temporally blocked smoother, register-tiled: TWO full red-black Gauss-Seidel sweeps (four
// half-sweeps R1, B1, R2, B2) of MultiGrid3D::Relax (N3/MultiGrid3D.cpp:489-567) in ONE pass over HBM.
//
// HBM traffic per pass: the colour-1 ("black") half of v in, f in, both halves of v out = 2.5*B*N bytes for two
// sweeps; the four colour launches of mg3d_smooth_tma.cu move 6*B*N.  (The colour-0 half of v is never read: the
// first half-sweep overwrites every interior colour-0 point from its colour-1 neighbours and f alone, :532; only
// the Dirichlet points of colour 0 are fetched.)
//
// Organisation.  A CTA owns a column of LW x TYT (half-index x row) sites and marches along z; a site (i, y) holds
// the two points x = 2i, 2i+1 of the row.  A thread owns the sites (lane, R consecutive rows) and keeps, in REGISTERS,
// the z-window (3 planes) of every stage's output at its own sites, so of the six neighbours of an update
//     D, U          are registers (same site, planes z-1 / z+1 of the previous stage),
//     O or E        one is a register (the other point of the same site), the other comes from the x-neighbour lane,
//     N, S          one is a register (the thread's other row), the other comes from the neighbouring thread row,
// i.e. 2 shared-memory loads + 1 store per update instead of 7 + 1 in mg3d_smooth_fused.cu (whose shared-memory data
// pipe was the limiter).  The stages are skewed by ONE plane each: at step p (raw plane p arrives by TMA)
//     R1 @ p-1,  B1 @ p-2,  R2 @ p-3,  B2 @ p-4   -> plane p-4 is final and is stored (out of place).
// Stage s+1 needs the neighbours' stage-s values only on its own centre plane, which was published one step earlier,
// and its own stage-s value of the plane above straight from a register: ONE __syncthreads per step.
// Halo: four half-sweeps consume 4 points on every side of the tile (2 half-indices in x, 4 rows in y, 4 planes in z at
// the ends of a z chunk); values in the halo are computed redundantly and never stored.
//
// Arithmetic, bit-identical to the reference.  This kernel is only used when every h^2 is a power of two and
// hx = hy = hz (the reference problem on [0,1]^3): all weights are c = h^4, exact scalings, so with s6 the
// reference's left-to-right sum O+E+N+S+D+U
//     reference:  ((O c + E c + N c + S c + D c + U c) - f h^6) / (6 c)   ==   (s6 - f h^2) / 6     (ours)
// rounding for rounding (scaling by a power of two commutes with RN), and f h^2 is exact, so the subtraction is one
// FMA; the quotient by 6 is the Markstein sequence of mg_exact.cuh: 9 fp64 instructions per update instead of 20.
// The identity fails only if an intermediate of the reference underflows (or ours overflows): every value that enters
// or leaves a stage is range-checked with 4 integer instructions (zero, or magnitude in [2^lo, 2^hi]); a violation
// raises a flag in global memory and the host-enqueued fallback (mg3d_smooth_fused.cu with the literal arithmetic,
// conditional on that flag) recomputes the pass from the untouched input buffer.  tests/test_smoother_pipe_gpu.py.
// MG_ARITH_FAST (template ARITH = 1): pairwise sum and multiplication by 1/6, no range check -- 7 instructions, results
// within 1e-10 (fp64) / 1e-5 (fp32) of the reference instead of identical.
#include <type_traits>

#include "mg3d_device.cuh"
#include "mg_tma.cuh"

using namespace mgx;
using namespace mg3;
using namespace mgtma;

namespace {

constexpr int LW = 32;               // sites per row of the tile = one warp
constexpr int HXI = MGK3D_PP_HXI;    // halo in half-indices on each side (4 points)
constexpr int HY = MGK3D_PP_HY;      // halo rows on each side
constexpr int R = MGK3D_PP_R;        // rows per thread
constexpr int NWARP = MGK3D_PP_NW;   // warps = thread rows
constexpr int NT = 32 * NWARP;
constexpr int TYT = R * NWARP;       // rows of the tile incl. halo
constexpr int TXO = LW - 2 * HXI;    // output half-indices per tile
constexpr int TYO = TYT - 2 * HY;    // output rows per tile
constexpr int NRING = 6;             // slots per TMA ring (raw colour-1 v, f colour 0, f colour 1); steps are unrolled 6-fold
constexpr int PF = 3;                // planes of prefetch: at step p the copies of raw(p+3), f0(p+2), f1(p+1) are issued
constexpr int ZH = 4;                // z halo planes at each end of a chunk

template <typename T> struct PBox {
    static constexpr int PADL = MGK3D_PP_PADL(sizeof(T));  // columns left of lane 0 (keeps the TMA start 16-byte aligned)
    static constexpr int W = MGK3D_PP_BOX_I(sizeof(T));    // row stride = TMA box width
    static constexpr int SLOT = (W * TYT * (int)sizeof(T) + 127) / 128 * 128 / (int)sizeof(T);  // elements
    // slot map (in slots): [0,6) raw v colour 1, [6,12) f colour 0, [12,18) f colour 1, [18,24) exchange r1, b1, r2 (2 each)
    static constexpr int NSLOT = 3 * NRING + 6;
    static constexpr int GUARD = 2 * W;  // addressable elements in front of slot 0 and behind the last slot (edge lanes / rows)
};

struct PipeMaps {
    CUtensorMap vblack;  // colour-1 array of the input v, box (W, TYT, 1)
    CUtensorMap f[2];    // colour arrays of f, same box
    CUtensorMap cv[2];   // CORR: colour arrays of the next coarser level's v, box (CBox::CW, CROWS, 1)
};

// CORR: the coarse tile under a fine tile.  Fine half-index i IS the coarse x (x = 2i, 2i+1 -> X = i), so the tile needs coarse
// X = i0-HXI .. i0-HXI+LW (half-indices X >> 1 of the coarse colour arrays) and coarse rows (y0-HY)/2 .. +TYT/2.
constexpr int CROWS = TYT / 2 + 1;
constexpr int NCR = 4;  // coarse planes in flight: Z0, Z0+1 in use, two ahead
template <typename T> struct CBox {
    static constexpr int A = 16 / (int)sizeof(T);                 // TMA inner-coordinate alignment in elements
    static constexpr int CW = MGK3D_PP_CBOX_I(sizeof(T));         // 18 doubles / 20 floats of data + CSH
    static constexpr int CSH = MGK3D_PP_CSHIFT(sizeof(T));        // column shift of the colour-1 sub-tile (bank skew, mg_launch.h)
    static constexpr int CSUB = (CW * CROWS * (int)sizeof(T) + 127) / 128 * 128 / (int)sizeof(T);
    static constexpr int CSLOT = 2 * CSUB;
};

// range check of a value that enters a stage: +0, or lo <= |x| <= hi in exponent terms.  Everything else -- tiny, huge,
// non-finite, and -0 (whose sign the FMA chain of the quotient would lose) -- leaves a nonzero mark in acc.
__device__ __forceinline__ void guard(double x, unsigned lo, unsigned span, unsigned& acc)
{
    const unsigned h = (unsigned)__double2hiint(x);
    if ((h & 0x7fffffffu) - lo > span) acc |= h | (unsigned)__double2loint(x);
}
__device__ __forceinline__ void guard(float x, unsigned lo, unsigned span, unsigned& acc)
{
    const unsigned h = __float_as_uint(x);
    if ((h & 0x7fffffffu) - lo > span) acc |= h;
}

template <typename T, int ARITH>
__device__ __forceinline__ T gs_update(T own, T nbx, T N, T S, T D, T U, T f, T h2, T y6)
{
    if (ARITH == 0) {
        T s = add(own, nbx);  // O + E (commutative)
        s = add(s, N);
        s = add(s, S);
        s = add(s, D);
        s = add(s, U);
        const T t = fma_(-f, h2, s);  // f*h2 is exact
        if (sizeof(T) == 4) return div(t, T(6));
        const T q = mul(t, y6);
        const T r = fma_(T(-6), q, t);
        return fma_(r, y6, q);
    } else {
        const T s = ((own + nbx) + (N + S)) + (D + U);
        return fma_(-f, h2, s) * y6;
    }
}

// CORR: the pass starts from v + Interpolate(coarse v) on the interior colour-1 points instead of v -- the prolongation and
// ApplyCorrection of the V-cycle (N3/MultiGrid3D.cpp:186-335, :649-676) folded into the load stage of the post-smoothing
// pass: every raw colour-1 value is corrected once, in its ring slot, by the thread that owns the site, before anybody reads
// it.  (Colour 0 is not corrected at all: the first half-sweep overwrites it unread.)  Saves the separate prolongation
// kernel's read and write of the colour-1 array.
template <typename T, int ARITH, bool CORR>
__global__ void __launch_bounds__(NT, 1)
k_relax_pipe2(const __grid_constant__ PipeMaps maps, const T* __restrict__ v_in, T* __restrict__ v_out, mg_geom3d g, T h2, T y6,
              int zchunk, int zlo, int zhi, unsigned glo, unsigned gspan, unsigned int* __restrict__ flag, mg_geom3d gc)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int PADL = PBox<T>::PADL, W = PBox<T>::W, SLOT = PBox<T>::SLOT, NSLOT = PBox<T>::NSLOT, GUARD = PBox<T>::GUARD;
    constexpr uint32_t SLOT_BYTES = W * TYT * sizeof(T);
    // intermediates only need the range check where the exponent range is short (see guard_window): float
    constexpr bool CHECK_MID = ARITH == 0 && sizeof(T) == 4;
    constexpr int GUARD_AL = (GUARD * (int)sizeof(T) + 127) / 128 * 128 / (int)sizeof(T);
    T* base = reinterpret_cast<T*>(smem_raw) + GUARD_AL;  // slot 0
    constexpr int CSUB = CBox<T>::CSUB, CSLOT = CBox<T>::CSLOT, CW = CBox<T>::CW, CSH = CBox<T>::CSH;
    T* cring = base + (size_t)NSLOT * SLOT + GUARD_AL;    // CORR: NCR coarse planes, two colour sub-tiles each
    uint64_t* bars = reinterpret_cast<uint64_t*>(cring + (CORR ? (size_t)NCR * CSLOT : 0));  // NRING + NCR barriers

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = g.n, imax = (n - 1) / 2;
    const int i0 = blockIdx.x * TXO, y0 = blockIdx.y * TYO;
    const int zs = zlo + blockIdx.z * zchunk, ze = min(zs + zchunk, zhi);  // output planes [zs, ze), local indices
    const int pb = zs - ZH, nsteps = ze - zs + 2 * ZH;                  // raw planes pb .. pb+nsteps-1, one per step

    if (tid == 0) {
        prefetch_tensormap(&maps.vblack);
        prefetch_tensormap(&maps.f[0]);
        prefetch_tensormap(&maps.f[1]);
        for (int s = 0; s < NRING + (CORR ? NCR : 0); s++) mbar_init(&bars[s], 1);
        if (CORR) { prefetch_tensormap(&maps.cv[0]); prefetch_tensormap(&maps.cv[1]); }
        fence_barrier_init();
    }
    // Everything starts as zero: edge lanes and rows read one element / row outside their slot (results that depend on it are
    // never stored), the first steps read ring slots no copy has filled yet, and whatever the halo computes from that must
    // stay finite and inside the guard window.
    for (int k = tid; k < NSLOT * SLOT + 2 * GUARD_AL; k += NT) (base - GUARD_AL)[k] = T(0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // order these generic-proxy writes before the TMA writes
    __syncthreads();

    const int bx0 = i0 - HXI - PADL, by0 = y0 - HY;  // box origin
    // One group of copies per step, all first needed at the same later step, tracked by one mbarrier: issued at step m
    // (raw plane pb+m arrives) for step m+PF: raw v colour 1 of plane p+PF, f colour 0 of plane p+PF-1 (R1), f colour 1 of
    // plane p+PF-2 (B1).  Out-of-range coordinates zero-fill.
    auto issue = [&](int slot, int pn) {  // slot = (step index of the consumer) % NRING, pn = its raw plane
        mbar_arrive_expect_tx(&bars[slot], 3 * SLOT_BYTES);
        tma_load_3d(base + (size_t)slot * SLOT, &maps.vblack, &bars[slot], bx0, by0, pn);
        tma_load_3d(base + (size_t)(NRING + slot) * SLOT, &maps.f[0], &bars[slot], bx0, by0, pn - 1);
        tma_load_3d(base + (size_t)(2 * NRING + slot) * SLOT, &maps.f[1], &bars[slot], bx0, by0, pn - 2);
    };
    if (tid == 0)
        for (int k = 0; k < PF && k < nsteps; k++) issue(k, pb + k);
    // CORR: coarse plane Z (global) lives in slot (Z - Zb) % NCR; fine plane p reads Z0 = (z0 + p) >> 1 and, on odd planes, Z0 + 1
    const int Zb = (g.z0 + pb) >> 1, Zlast = ((g.z0 + pb + nsteps - 1) >> 1) + 1;
    const int cxh0 = ((i0 - HXI) >> 1) & ~(CBox<T>::A - 1), cy0c = (y0 - HY) >> 1;
    auto issue_coarse = [&](int Z) {
        const int s = (Z - Zb) & (NCR - 1);
        uint64_t* bar = &bars[NRING + s];
        mbar_arrive_expect_tx(bar, 2 * CW * CROWS * (uint32_t)sizeof(T));
        tma_load_3d(cring + (size_t)s * CSLOT, &maps.cv[0], bar, cxh0, cy0c, Z - gc.z0);
        tma_load_3d(cring + (size_t)s * CSLOT + CSUB, &maps.cv[1], bar, cxh0 - CSH, cy0c, Z - gc.z0);
    };
    if (CORR && tid == 0)
        for (int Z = Zb; Z <= min(Zb + NCR - 2, Zlast); Z++) issue_coarse(Z);

    // ---- per-thread constants -------------------------------------------------------------------------------
    // Site (lane, row r): half-index i, row y.  On plane z its colour-c point has x = 2i + ((c + y + z) & 1).  Steps are
    // unrolled six-fold, so relative to the first plane every parity is a compile-time bit XOR s0 = (y_row0 + z0 + pb) & 1.
    const int i = i0 - HXI + lane;
    const int tr0 = R * warp, yr0 = y0 - HY + tr0;
    const int s0 = (yr0 + g.z0 + pb) & 1;  // (yr0 is even: s0 is the same for every thread of the CTA)
    // CORR: element of the site's coarse corner (dx, dy, dz) inside a coarse slot: colour (ipar + Yt + Z + dx + dy) & 1,
    // column ((i + dx) >> 1) - cxh0, row Yt + dy - cy0c with Yt = yr0 / 2
    const int ipar = i & 1, ca0 = ((i >> 1) - cxh0) + ((yr0 >> 1) - cy0c) * CW, ct = (i + (yr0 >> 1)) & 1;
    const T* sb = base + tr0 * W + lane + PADL;   // own site of row 0 in slot 0; row r: + r*W; slot j: + j*SLOT
    const T* sP = sb + (2 * s0 - 1);              // x-neighbour of row r when ((r & 1) ^ CV) == 0 ...
    const T* sM = sb - (2 * s0 - 1);              // ... and when it is 1 (CV: see step())
    T* sw = base + tr0 * W + lane + PADL;
    // byte offset of the site inside a colour plane (Dirichlet loads and the stores; both are predicated on the point existing)
    unsigned goff[R];
    const long long pbytes = g.plane * (long long)sizeof(T);
    // mA: the point of the site with x parity s_r = s0 ^ (r & 1); mB: the other one.  bit r: interior in (x, y);
    // bit 8+r: exists and lies in the tile's output region (store predicate); bit 16+r: exists in the grid
    unsigned mA = 0, mB = 0;
    {
        const bool ex0 = i >= 0 && i <= imax, ex1 = i >= 0 && 2 * i + 1 <= n - 1;      // x = 2i / 2i+1 exists
        const bool in0 = i >= 1 && 2 * i <= n - 2, in1 = i >= 0 && 2 * i + 1 <= n - 2;   // ... is interior in x
#pragma unroll
        for (int r = 0; r < R; r++) {
            const int tr = tr0 + r, y = yr0 + r;
            goff[r] = (unsigned)((min(max(y, 0), n - 1) * g.hp + min(max(i, 0), imax)) * (int)sizeof(T));
            const bool y_in = y >= 0 && y <= n - 1, y_int = y >= 1 && y <= n - 2;
            const bool outr = tr >= HY && tr < HY + TYO && lane >= HXI && lane < HXI + TXO;
            const int sr = s0 ^ (r & 1);
            const bool exA = sr ? ex1 : ex0, exB = sr ? ex0 : ex1, inA = sr ? in1 : in0, inB = sr ? in0 : in1;
            if (y_int && inA) mA |= 1u << r;
            if (y_int && inB) mB |= 1u << r;
            if (y_in && exA && outr) mA |= 1u << (8 + r);
            if (y_in && exB && outr) mB |= 1u << (8 + r);
            if (y_in && exA) mA |= 1u << (16 + r);
            if (y_in && exB) mB |= 1u << (16 + r);
        }
    }
    // uniform plane pointers, advanced by one plane per step
    const char* va = (const char*)v_in + (long long)pb * pbytes;                 // input v colour 0 (Dirichlet points), plane p
    char* oa = (char*)v_out + (long long)(pb - 4) * pbytes;                      // output colour 0, plane p-4
    char* ob = (char*)(v_out + g.cstride) + (long long)(pb - 4) * pbytes;        // output colour 1, plane p-4

    // ---- register state: z-windows (3 planes) of the raw colour-1 values and of the outputs of R1, B1, R2 -----
    T wr[3][R], w1[3][R], w2[3][R], w3[3][R], rr_n[R];
#pragma unroll
    for (int s = 0; s < 3; s++)
#pragma unroll
        for (int r = 0; r < R; r++) wr[s][r] = w1[s][r] = w2[s][r] = w3[s][r] = T(0);
#pragma unroll
    for (int r = 0; r < R; r++) rr_n[r] = T(0);
    unsigned bad = 0;
    unsigned phase = 0;  // mbarrier parity of the ring: flips every NRING steps

    // One step = raw plane p = pb + m arrives; J6 = m % 6 is a template constant, so ring slots, exchange slots,
    // window rotation and parities are all compile-time.
    // FAST (compile-time): the tile with its halo lies strictly inside the grid in x and y and the planes p-4 .. p are all
    // interior and inside the chunk's pipeline steady state -- no Dirichlet points, no masks, no conditional copies.
    auto step = [&](auto Jc, auto Fc, int p) {
        constexpr int J6 = decltype(Jc)::value, J = J6 % 3, J1 = (J + 1) % 3, J2 = (J + 2) % 3;
        constexpr bool FAST = decltype(Fc)::value;
        constexpr int E = J6 & 1;          // exchange slot written for planes p-1 / p-3 (r1, r2) is E, for p-2 (b1) is E^1
        constexpr int CV = (J6 + 1) & 1;   // the updated point of row r has x parity s_r ^ CV in ALL four stages of this step
        const unsigned mU = CV ? mB : mA, mO = CV ? mA : mB;
        // the Dirichlet values of colour 0 on plane p-1, loaded one step ago
        T rkeep[R];
#pragma unroll
        for (int r = 0; r < R; r++) {
            rkeep[r] = FAST ? T(0) : rr_n[r];
            if (ARITH == 0 && !FAST) guard(rr_n[r], glo, gspan, bad);
        }
        if (!FAST) {
            const int zg = g.z0 + p;
            // Dirichlet points of colour 0 on plane p (parity s_r ^ CV ^ 1): exist and are not interior
            const unsigned mz = (p >= 0 && p < g.nzl) ? ((mO >> 16) & ~(((unsigned)(zg - 1) <= (unsigned)(n - 3)) ? mO : 0u)) : 0u;
#pragma unroll
            for (int r = 0; r < R; r++) {
                if ((mz >> r) & 1u) MG_CHK_SITE(g, i, yr0 + r, p);
                rr_n[r] = ((mz >> r) & 1u) ? __ldg((const T*)(va + goff[r])) : T(0);
            }
        }
        if (tid == 0 && (FAST || p - pb + PF < nsteps)) issue((J6 + PF) % NRING, p + PF);
        mbar_wait(&bars[J6], phase);
        constexpr int OFF_P = J6 * SLOT;                         // raw plane p
        constexpr int OFF_C = ((J6 + NRING - 1) % NRING) * SLOT; // raw plane p-1
        // the copy group of step m carries raw(p), f0(p-1), f1(p-2) in slot m % 6 of the three rings
        constexpr int F0A = (NRING + J6) * SLOT;                            // f colour 0, plane p-1
        constexpr int F0B = (NRING + (J6 + NRING - 2) % NRING) * SLOT;      // f colour 0, plane p-3 (group of step m-2)
        constexpr int F1A = (2 * NRING + J6) * SLOT;                        // f colour 1, plane p-2
        constexpr int F1B = (2 * NRING + (J6 + NRING - 2) % NRING) * SLOT;  // f colour 1, plane p-4 (group of step m-2)
        constexpr int XB = 3 * NRING;
        constexpr int X1W = (XB + 0 + E) * SLOT, X1R = (XB + 0 + (E ^ 1)) * SLOT;
        constexpr int X2W = (XB + 2 + (E ^ 1)) * SLOT, X2R = (XB + 2 + E) * SLOT;
        constexpr int X3W = (XB + 4 + E) * SLOT, X3R = (XB + 4 + (E ^ 1)) * SLOT;
        if constexpr (CORR) {
            static_assert(!CORR || R == 2, "the fused prolongation pairs the thread's even row (oy = 0) with its odd row (oy = 1)");
            const int zg = g.z0 + p, Z0 = zg >> 1, oz = zg & 1;
            if (tid == 0 && oz == 0 && Z0 + NCR - 2 <= Zlast && Z0 + NCR - 2 > Zb + NCR - 2) issue_coarse(Z0 + NCR - 2);
            const int k0 = Z0 - Zb;
            mbar_wait(&bars[NRING + (k0 & (NCR - 1))], (unsigned)(k0 >> 2) & 1u);
            if (oz) mbar_wait(&bars[NRING + ((k0 + 1) & (NCR - 1))], (unsigned)((k0 + 1) >> 2) & 1u);
            // Corner (dx, dy, dz) of the site = coarse point (i + dx, Yt + dy, Z0 + dz): colour (ct + dx + dy + dz + Z0) & 1 with the
            // per-thread bit ct = (i + Yt) & 1, column ((i + dx) >> 1), row Yt + dy.  Everything but ct is uniform over the CTA, so
            // each plane needs two pointers: corners with dx + dy even / odd.
            const T* q0 = cring + (size_t)(k0 & (NCR - 1)) * CSLOT + ca0;
            const T* q1 = cring + (size_t)((k0 + 1) & (NCR - 1)) * CSLOT + ca0;
            const int se = ((ct + Z0) & 1) * (CSUB + CSH), so = (CSUB + CSH) - se;  // colour sub-tile of plane Z0 for dx + dy even / odd
            const T *e0 = q0 + se, *o0 = q0 + so, *e1 = q1 + so, *o1 = q1 + se;  // plane Z0 + 1: colours swap
            const bool oxa = (((s0 ^ CV) & 1) != 0);  // x parity of the colour-1 point in the even row (the odd row has the other)
            T ea, eb;  // Interpolate at the colour-1 point of the even row (oy = 0) / the odd row (oy = 1), N3/MultiGrid3D.cpp:216-331
            if (!oz) {
                const T c000 = e0[0], c100 = o0[ipar], c010 = o0[CW];
                if (!oxa) {  // even row PPP, odd row DDP
                    ea = c000;
                    eb = mul(T(0.25f), add(add(add(c000, c100), c010), e0[CW + ipar]));
                } else {     // even row PDP, odd row DPP
                    ea = mul(T(0.5f), add(c000, c100));
                    eb = mul(T(0.5f), add(c000, c010));
                }
            } else {
                const T c000 = e0[0], c001 = e1[0];
                if (!oxa) {  // even row PPD, odd row DDD
                    ea = mul(T(0.5f), add(c000, c001));
                    T t8 = add(c000, c001);
                    t8 = add(t8, o1[ipar]);       // C(1,0,1)
                    t8 = add(t8, o0[ipar]);       // C(1,0,0)
                    t8 = add(t8, o0[CW]);         // C(0,1,0)
                    t8 = add(t8, o1[CW]);         // C(0,1,1)
                    t8 = add(t8, e1[CW + ipar]);  // C(1,1,1)
                    t8 = add(t8, e0[CW + ipar]);  // C(1,1,0)
                    eb = mul(T(0.125f), t8);
                } else {     // even row PDD, odd row DPD
                    ea = mul(T(0.25f), add(add(add(c001, o1[ipar]), c000), o0[ipar]));
                    eb = mul(T(0.25f), add(add(add(c000, c001), o0[CW]), o1[CW]));
                }
            }
            const unsigned mzc = FAST ? ~0u : ((unsigned)(zg - 1) <= (unsigned)(n - 3)) ? mU : 0u;  // colour 1 on plane p sits at parity s_r ^ CV
#pragma unroll
            for (int r = 0; r < R; r++) {
                const T rawv = sb[OFF_P + r * W];
                wr[J][r] = (FAST || ((mzc >> r) & 1u)) ? add(rawv, r ? eb : ea) : rawv;  // published at the end of the step
                if (ARITH == 0) guard(wr[J][r], glo, gspan, bad);
            }
        } else {
#pragma unroll
            for (int r = 0; r < R; r++) {
                wr[J][r] = sb[OFF_P + r * W];
                if (ARITH == 0) guard(wr[J][r], glo, gspan, bad);
            }
        }
        // One half-sweep stage on plane z for the thread's R sites: the colour being updated reads the other colour's
        // window (D, C, U = planes z-1, z, z+1 at the own sites), the neighbours on plane z in shared memory at OFF and
        // f at FOFF.  GF: first use of these f values -> range-check them, where they are used (f of boundary points is
        // never read by an update, and the reference problem has f = -0.0 on the faces x, y, z = 0).
        auto stage = [&](int z, auto offc, auto foffc, auto gfc, const T (&wD)[R], const T (&wC)[R], const T (&wU)[R], const T (&keep)[R],
                         T (&out)[R]) {
            constexpr int OFF = decltype(offc)::value, FOFF = decltype(foffc)::value;
            constexpr bool GF = decltype(gfc)::value;
            const int zg = g.z0 + z;
            const unsigned mz = FAST ? ~0u : ((unsigned)(zg - 1) <= (unsigned)(n - 3)) ? mU : 0u;
            T nbx[R], ff[R];
#pragma unroll
            for (int r = 0; r < R; r++) {
                nbx[r] = (((r & 1) ^ CV) ? sM : sP)[OFF + r * W];
                ff[r] = sb[FOFF + r * W];
            }
            const T nN = sb[OFF - W], nS = sb[OFF + R * W];
            T o[R];
#pragma unroll
            for (int r = 0; r < R; r++) {
                const T N = r == 0 ? nN : wC[r > 0 ? r - 1 : 0];
                const T S = r == R - 1 ? nS : wC[r < R - 1 ? r + 1 : 0];
                o[r] = gs_update<T, ARITH>(wC[r], nbx[r], N, S, wD[r], wU[r], ff[r], h2, y6);
            }
#pragma unroll
            for (int r = 0; r < R; r++) {
                out[r] = (FAST || ((mz >> r) & 1u)) ? o[r] : keep[r];
                if (ARITH == 0 && GF && (FAST || ((mz >> r) & 1u))) guard(ff[r], glo, gspan, bad);
                if (CHECK_MID) guard(out[r], glo, gspan, bad);
            }
        };
        using std::integral_constant;
        using GFY = integral_constant<bool, true>;
        using GFN = integral_constant<bool, false>;
        // R1 @ p-1: colour 0 from raw colour 1
        stage(p - 1, integral_constant<int, OFF_C>{}, integral_constant<int, F0A>{}, GFY{}, wr[J1], wr[J2], wr[J], rkeep, w1[J2]);
        // B1 @ p-2: colour 1 from R1
        stage(p - 2, integral_constant<int, X1R>{}, integral_constant<int, F1A>{}, GFY{}, w1[J], w1[J1], w1[J2], wr[J1], w2[J1]);
        // R2 @ p-3: colour 0 from B1
        stage(p - 3, integral_constant<int, X2R>{}, integral_constant<int, F0B>{}, GFN{}, w2[J2], w2[J], w2[J1], w1[J], w3[J]);
        // B2 @ p-4: colour 1 from R2; plane p-4 is final
        T b2[R];
        stage(p - 4, integral_constant<int, X3R>{}, integral_constant<int, F1B>{}, GFN{}, w3[J1], w3[J2], w3[J], w2[J2], b2);
        const int zo = p - 4;
        {
            // colour 0 was updated by R2 on plane p-3 at parity s_r ^ CV, so on plane p-4 it sits at the other parity (mO),
            // colour 1 at s_r ^ CV (mU); planes outside [zs, ze) belong to the z halo of the chunk
            const bool zok = FAST || (zo >= zs && zo < ze);
            const unsigned m0 = zok ? (mO >> 8) : 0u, m1 = zok ? (mU >> 8) : 0u;
#pragma unroll
            for (int r = 0; r < R; r++) {
                if (((m0 | m1) >> r) & 1u) MG_CHK_SITE(g, i, yr0 + r, zo);
                if ((m0 >> r) & 1u) __stcs((T*)(oa + goff[r]), w3[J2][r]);
                if ((m1 >> r) & 1u) __stcs((T*)(ob + goff[r]), b2[r]);
            }
        }
        // Publish this step's stage outputs (and, CORR, the corrected raw plane) for the neighbours' reads of the NEXT step.  All
        // shared-memory stores of a step come after all of its loads: the four stages only read what the previous step
        // published (different exchange slots), so the compiler is free to hoist every load and interleave the four stages.
#pragma unroll
        for (int r = 0; r < R; r++) {
            if (CORR) sw[OFF_P + r * W] = wr[J][r];
            sw[X1W + r * W] = w1[J2][r];
            sw[X2W + r * W] = w2[J1][r];
            sw[X3W + r * W] = w3[J][r];
        }
        va += pbytes; oa += pbytes; ob += pbytes;
        __syncthreads();
    };

    // steady-state steps m in [m_lo, m_hi]: planes p-4 .. p interior (global z in [1, n-2]) and stored (p-4 >= zs), the
    // copy group issued for step m+PF exists; interior tile in x, y
    const bool tile_fast = i0 - HXI >= 1 && 2 * (i0 - HXI + LW - 1) + 1 <= n - 2 && y0 - HY >= 1 && y0 - HY + TYT - 1 <= n - 2;
    const int m_lo = max(2 * ZH, 5 - g.z0 - pb), m_hi = min(n - 2 - g.z0 - pb, nsteps - 1 - PF);
    using std::integral_constant;
    for (int m = 0; m < nsteps; m += 6) {
        const int p = pb + m;
        if (tile_fast && m >= m_lo && m + 5 <= m_hi) {
            step(integral_constant<int, 0>{}, integral_constant<bool, true>{}, p);
            step(integral_constant<int, 1>{}, integral_constant<bool, true>{}, p + 1);
            step(integral_constant<int, 2>{}, integral_constant<bool, true>{}, p + 2);
            step(integral_constant<int, 3>{}, integral_constant<bool, true>{}, p + 3);
            step(integral_constant<int, 4>{}, integral_constant<bool, true>{}, p + 4);
            step(integral_constant<int, 5>{}, integral_constant<bool, true>{}, p + 5);
        } else {
            step(integral_constant<int, 0>{}, integral_constant<bool, false>{}, p);
            if (m + 1 < nsteps) step(integral_constant<int, 1>{}, integral_constant<bool, false>{}, p + 1);
            if (m + 2 < nsteps) step(integral_constant<int, 2>{}, integral_constant<bool, false>{}, p + 2);
            if (m + 3 < nsteps) step(integral_constant<int, 3>{}, integral_constant<bool, false>{}, p + 3);
            if (m + 4 < nsteps) step(integral_constant<int, 4>{}, integral_constant<bool, false>{}, p + 4);
            if (m + 5 < nsteps) step(integral_constant<int, 5>{}, integral_constant<bool, false>{}, p + 5);
        }
        phase ^= 1u;
    }
    if (ARITH == 0 && bad) atomicOr(flag, 1u);
}

template <typename T>
size_t smem_bytes_t(bool corr)
{
    const size_t guard_al = ((size_t)PBox<T>::GUARD * sizeof(T) + 127) / 128 * 128;
    return (size_t)PBox<T>::NSLOT * PBox<T>::SLOT * sizeof(T) + 2 * guard_al + (corr ? (size_t)NCR * CBox<T>::CSLOT * sizeof(T) : 0) +
           (NRING + NCR) * sizeof(uint64_t);
}

// Exponent window of the range check, h = 2^-k.  Where the scaled formula could differ from the reference:
//   * a product of the reference (x*h^4, f*h^6) must not lose bits to underflow: x nonzero on the grid 2^(e-p)
//     (p = significand bits - 1) needs e - p - 6k >= emin_subnormal;
//   * double only checks what ENTERS the pass (raw v, f, Dirichlet values).  Each stage can lose at most p + 3 bits of
//     magnitude to cancellation (a nonzero sum is a multiple of its inputs' grid, and f*h^2 sits 2k below f), so after four
//     stages values are >= 2^(lo - 2k - 3(p+3)) on the grid 2^(lo - 2k - 3(p+3) - p): with lo >= -857 + 6k every product
//     of the reference is still exact, and with lo >= -697 + 2k the Markstein residual stays normal (mg_exact.cuh);
//   * float has no exponent range to spare for that argument: every stage output is checked as well and the quotient is
//     the IEEE division, which leaves lo >= -126 + 6k for the products;
//   * hi, h <= 1 (k >= 0): four stages of sums of six can grow a value by less than 2^7;
//   * h > 1 (k < 0): the reference's products scale values UP, x*h^4 = x*2^(-4k) and f*h^6 = f*2^(-6k), and a stage adds
//     f*h^2/6 = f*2^(-2k)/6 to what it passes on.  With every checked value below 2^(hi+1), a stage value stays below
//     2^(hi+1-2k) (double: after the four stages; float checks each), so the reference's numerator
//     6*|x|*h^4 + |f|*h^6 stays below 2^(hi+4-6k): hi = hi(k=0) + 6k keeps it under 2^1014 (double) / 2^118 (float), where
//     neither it nor any partial sum or product can overflow.  Nothing of the reference underflows sooner than at
//     k = 0, and f*h^2 is no finer than f, so the lower bounds of k = 0 hold: lo = lo(k=0).
// Returns 0 when the window is empty: the pass would have nothing it may compute, so the level takes the literal kernels
// (mgk3d_pipe_exact_range).
template <typename T> int guard_window(double h2, unsigned* glo, unsigned* gspan);
template <> int guard_window<double>(double h2, unsigned* glo, unsigned* gspan)
{
    int e;
    frexp(h2, &e);  // h2 = 2^(e-1) = 2^(-2k)
    const int k = -(e - 1) / 2, kl = k > 0 ? k : 0, kh = k < 0 ? k : 0;
    const int a = -857 + 6 * kl, b = -697 + 2 * kl;
    const int lo = (a > b ? a : b) + 8, hi = 1010 + 6 * kh;
    if (lo > hi) return 0;
    const unsigned L = (unsigned)(lo + 1023) << 20, H = (((unsigned)(hi + 1023 + 1)) << 20) - 1;
    *glo = L;
    *gspan = H - L;
    return 1;
}
template <> int guard_window<float>(double h2, unsigned* glo, unsigned* gspan)
{
    int e;
    frexp(h2, &e);
    const int k = -(e - 1) / 2, kl = k > 0 ? k : 0, kh = k < 0 ? k : 0;
    const int lo = -126 + 6 * kl + 4, hi = 115 + 6 * kh;
    if (lo > hi) return 0;
    const unsigned L = (unsigned)(lo + 127) << 23, H = (((unsigned)(hi + 127 + 1)) << 23) - 1;
    *glo = L;
    *gspan = H - L;
    return 1;
}

template <typename T, int ARITH, bool CORR>
int launch_k(cudaStream_t s, const PipeMaps& m, const T* v_in, T* v_out, mg_geom3d g, mg_coef3d c, dim3 grid, int zchunk, int zlo, int zhi,
             unsigned int* flag, mg_geom3d gc)
{
    MG_SET_SMEM_LIMIT((k_relax_pipe2<T, ARITH, CORR>), smem_bytes_t<T>(CORR));
    unsigned glo = 0, gspan = 0;
    if (!guard_window<T>(c.hx2, &glo, &gspan)) return -1;
    const T y6 = T(1) / T(6);
    k_relax_pipe2<T, ARITH, CORR><<<grid, NT, smem_bytes_t<T>(CORR), s>>>(m, v_in, v_out, g, (T)c.hx2, y6, zchunk, zlo, zhi, glo, gspan, flag, gc);
    return cudaPeekAtLastError() == cudaSuccess ? 1 : -1;
}

template <typename T>
int launch(cudaStream_t s, const void* const maps3[3], const void* const cmaps2[2], const mg_geom3d* gc, const T* v_in, T* v_out, mg_geom3d g,
           mg_coef3d c, int zlo, int zhi, int arith, unsigned int* flag)
{
    if (zhi <= zlo) return 0;
    const int nz = zhi - zlo;
    PipeMaps m;
    memcpy(&m.vblack, maps3[0], sizeof(CUtensorMap));
    memcpy(&m.f[0], maps3[1], sizeof(CUtensorMap));
    memcpy(&m.f[1], maps3[2], sizeof(CUtensorMap));
    const bool corr = cmaps2 && cmaps2[0] && cmaps2[1] && gc;
    memcpy(&m.cv[0], corr ? cmaps2[0] : maps3[0], sizeof(CUtensorMap));
    memcpy(&m.cv[1], corr ? cmaps2[1] : maps3[0], sizeof(CUtensorMap));
    const mg_geom3d gcv = corr ? *gc : g;
    const int tx = ((g.n + 1) / 2 + TXO - 1) / TXO, ty = (g.n + TYO - 1) / TYO;
    // z chunks: every chunk pays 2*ZH planes of warm-up plus the pipeline depth; more chunks balance the waves of one-CTA SMs
    int sms = 148;
    {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms < 1) sms = 148;
    }
    int nchunk = 1;
    double best = 1e30;
    for (int k = 1; k <= 16; k++) {
        const int zc = (nz + k - 1) / k;
        if (k > 1 && zc < 8) break;
        const long long ctas = (long long)tx * ty * ((nz + zc - 1) / zc);
        const double cost = (double)((ctas + sms - 1) / sms) * (zc + 2 * ZH + 3);
        if (cost < best) { best = cost; nchunk = k; }
    }
    const int zchunk = (nz + nchunk - 1) / nchunk;
    dim3 grid(tx, ty, (nz + zchunk - 1) / zchunk);
    if constexpr (R != 2) {
        if (corr) return -1;
    } else if (corr) {
        if (arith) return launch_k<T, 1, true>(s, m, v_in, v_out, g, c, grid, zchunk, zlo, zhi, flag, gcv);
        return launch_k<T, 0, true>(s, m, v_in, v_out, g, c, grid, zchunk, zlo, zhi, flag, gcv);
    }
    if (arith) return launch_k<T, 1, false>(s, m, v_in, v_out, g, c, grid, zchunk, zlo, zhi, flag, gcv);
    return launch_k<T, 0, false>(s, m, v_in, v_out, g, c, grid, zchunk, zlo, zhi, flag, gcv);
}

}  // namespace

/* Local planes [zl_lo, zl_hi) of v_out are written (a slab: the planes it owns; v_in colour 1 and f need four valid planes
   on each side of them).  maps3: tensor maps of {v_in colour 1, f colour 0, f colour 1} with box (MGK3D_PP_BOX_I(esize), MGK3D_PP_BOX_Y, 1).
   Requires c.fast_den and hx2 == hy2 == hz2 (checked by the caller).  arith 0: bit-exact, *flag is raised when a value
   left the range in which the scaled formula is provably identical to the reference's (the caller enqueues the
   conditional literal-arithmetic pass after this one); arith 1: MG_ARITH_FAST.
   coarse_maps2 / gc: NULL, or the tensor maps of the two colour arrays of the next coarser level's v with box
   (MGK3D_PP_CBOX_I(esize), MGK3D_PP_CBOX_Y, 1) and that level's geometry: the pass then starts from
   v + Interpolate(coarse v) on the interior colour-1 points (prolongation + correction folded into the load stage). */
extern "C" int mgk3d_relax_pipe2(cudaStream_t s, int dtype, const void* const maps3[3], const void* v_in, const void* f, void* v_out,
                                 mg_geom3d g, mg_coef3d c, int zl_lo, int zl_hi, int arith, unsigned int* flag, const void* const coarse_maps2[2],
                                 const mg_geom3d* gc)
{
    (void)f;  // f only enters through its tensor maps
    if (dtype == 0) return launch<float>(s, maps3, coarse_maps2, gc, (const float*)v_in, (float*)v_out, g, c, zl_lo, zl_hi, arith, flag);
    return launch<double>(s, maps3, coarse_maps2, gc, (const double*)v_in, (double*)v_out, g, c, zl_lo, zl_hi, arith, flag);
}

/* 1 when the bit-exact pass has a nonempty range check for h^2 = hx2 (guard_window) */
extern "C" int mgk3d_pipe_exact_range(int dtype, double hx2)
{
    unsigned lo, span;
    return dtype == 0 ? guard_window<float>(hx2, &lo, &span) : guard_window<double>(hx2, &lo, &span);
}

"""CPU, gloo: the multi-GPU SCHEDULE of the distributed PCG (mg3d_pcg on a z-slab level, pde_multigrid_b200/csrc/
mg_host_common.c and mg3d_host.c; DESIGN.md section 6b).

Two or four processes hold the slabs mg3d_plan_level assigns them (the product's own partition arithmetic, through the C
ABI); everything outside a rank's stored planes is NaN.  They run the PCG with numpy stand-ins for the kernels and
exchange exactly where the C driver does:
  * prologue: r_0 on the owned planes of f, then f four planes deep each way,
  * per iteration: v <- 0 on every stored plane and the handshake exchange, the preconditioner, v (= z) two planes up and
    one down, the dots over the owned planes with their (hi, lo) sums all-gathered and added in rank order, p' and x'
    written on the owned planes and one more on each side (recomputed at the neighbours from z, p and x, never exchanged),
    r', d and f over the owned planes, f four planes deep each way, the norm partials combined over the ranks,
  * epilogue: the owned planes of x into v and of b into f, each followed by a full-depth exchange.
The stand-in preconditioner is partition-invariant like the V-cycle: four weighted-Jacobi sweeps from zero, the halo planes
swept redundantly (sweep k on the owned planes grown by 3 - k), so it reads f three planes into the ghosts and writes z on the
owned planes only; the ghost planes it leaves in v are stale (NaN here), as the temporally blocked smoother leaves them.
Every value a kernel writes only on the owned planes is NaN elsewhere, so a missing exchange or a too-narrow write range
puts a NaN into an owned plane.  The dots and the norm are exact sums (math.fsum of exact products, as (hi, lo) per rank),
so the owned planes and the history must equal the whole-grid run bit for bit."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

N = 65
ITERS = 8
SWEEPS = 4
OMEGA = 6.0 / 7.0
H2 = (1.0 / (N - 1)) ** 2
GHOST = 4  # MG_GHOST_LO / MG_GHOST_HI


class Slab:
    def __init__(self, plan, rank, world):
        self.rank, self.world = rank, world
        self.z0, self.nzl = plan["z0"], plan["nzl"]
        self.a, self.b = plan["z0"] + plan["own_lo"], plan["z0"] + plan["own_hi"]  # owned global planes
        self.stored = slice(self.z0, self.z0 + self.nzl)
        self.wr = (max(self.a - 1, self.z0), min(self.b + 1, self.z0 + self.nzl))  # write range of the p and x updates

    def field(self, value=np.nan):
        out = np.full((N, N, N), np.nan)
        out[self.stored] = value
        return out

    def poison_ghosts(self, arr):
        arr[self.z0:self.a] = np.nan
        arr[self.b:self.z0 + self.nzl] = np.nan

    def exchange(self, arr, depth_up, depth_down):
        """depth_up top owned planes -> the lower ghosts of rank+1, depth_down bottom owned planes -> the upper ghosts of rank-1"""
        if self.world == 1:
            return
        reqs, up, lo = [], None, None
        if self.rank + 1 < self.world:
            reqs.append(dist.isend(torch.from_numpy(arr[self.b - depth_up:self.b].copy()), self.rank + 1))
            up = torch.empty((depth_down, N, N), dtype=torch.float64)
            reqs.append(dist.irecv(up, self.rank + 1))
        if self.rank > 0:
            reqs.append(dist.isend(torch.from_numpy(arr[self.a:self.a + depth_down].copy()), self.rank - 1))
            lo = torch.empty((depth_up, N, N), dtype=torch.float64)
            reqs.append(dist.irecv(lo, self.rank - 1))
        for r in reqs:
            r.wait()
        if up is not None:
            arr[self.b:self.b + depth_down] = up.numpy()
        if lo is not None:
            arr[self.a - depth_up:self.a] = lo.numpy()

    def allgather(self, pairs):
        if self.world == 1:
            return [pairs]
        t = torch.tensor(pairs, dtype=torch.float64)
        out = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(out, t)
        return [o.tolist() for o in out]


# ---- numpy stand-ins for the kernels of csrc/mg3d_cg.cu, on planes [lo, hi) ------------------------------------

def interior(lo, hi):
    return max(lo, 1), min(hi, N - 1)


def residual(v, f, lo, hi):
    """f - Laplacian v on the interior points of planes [lo, hi), 0 on the Dirichlet points (shape (hi - lo, N, N))"""
    r = np.zeros((hi - lo, N, N))
    zl, zh = interior(lo, hi)
    if zh > zl:
        c = v[zl:zh, 1:-1, 1:-1]
        lap = (v[zl:zh, 1:-1, :-2] - 2 * c + v[zl:zh, 1:-1, 2:]) / H2 + (v[zl:zh, :-2, 1:-1] - 2 * c + v[zl:zh, 2:, 1:-1]) / H2 \
            + (v[zl - 1:zh - 1, 1:-1, 1:-1] - 2 * c + v[zl + 1:zh + 1, 1:-1, 1:-1]) / H2
        r[zl - lo:zh - lo, 1:-1, 1:-1] = f[zl:zh, 1:-1, 1:-1] - lap
    return r


def exact_terms(a, b):
    """the products a*b split exactly into p + e (Dekker)"""
    a, b = a.ravel(), b.ravel()
    p = a * b
    split = 134217729.0
    ca, cb = split * a, split * b
    ah, bh = ca - (ca - a), cb - (cb - b)
    al, bl = a - ah, b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p.tolist() + e.tolist()


def hi_lo(terms):
    """an exact sum as the pair (correctly rounded sum, exact remainder)"""
    hi = math.fsum(terms)
    return hi, math.fsum(terms + [-hi])


def combine(S, pairs):
    """this rank's (hi, lo) pairs all-gathered and added: the correctly rounded sums"""
    every = S.allgather([x for p in pairs for x in p])
    return [math.fsum([e[2 * k] for e in every] + [e[2 * k + 1] for e in every]) for k in range(len(pairs))]


def norm(S, r_own):
    s, = combine(S, [hi_lo(exact_terms(r_own, r_own))])
    m = float(np.max(np.abs(r_own)))
    if S.world > 1:
        t = torch.tensor([m], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        m = t.item()
    return math.sqrt(s), m


def precondition(S, v, f):
    """z from v = 0 on every stored plane: SWEEPS weighted-Jacobi sweeps, sweep k on the owned planes grown by
    SWEEPS - 1 - k; z lands on the owned planes of v, its ghost planes are stale"""
    w = v.copy()
    for k in range(SWEEPS):
        e = SWEEPS - 1 - k
        zl, zh = interior(S.a - e, S.b + e)
        nw = w.copy()
        gs = (w[zl:zh, 1:-1, :-2] + w[zl:zh, 1:-1, 2:] + w[zl:zh, :-2, 1:-1] + w[zl:zh, 2:, 1:-1] + w[zl - 1:zh - 1, 1:-1, 1:-1] +
              w[zl + 1:zh + 1, 1:-1, 1:-1] - f[zl:zh, 1:-1, 1:-1] * H2) / 6.0
        old = w[zl:zh, 1:-1, 1:-1]
        nw[zl:zh, 1:-1, 1:-1] = old + OMEGA * (gs - old)
        w = nw
    v[S.a:S.b] = w[S.a:S.b]
    S.poison_ghosts(v)


def pcg(S, v, f, rtol, skip=()):
    """the driver's schedule on this rank's slab; skip: steps left out to show that each one is needed"""
    a, b = S.a, S.b
    hist = [norm(S, residual(v, f, a, b))]
    B = f.copy()
    x = [v.copy(), S.field()]
    p = [S.field(0.0), S.field()]
    d = S.field(0.0)
    f[a:b] = residual(x[0], B, a, b)
    S.poison_ghosts(f)
    S.exchange(f, GHOST, GHOST)
    thr = rtol * hist[0][0]
    rho_prev, par, k = None, 0, 0
    while hist[-1][0] > thr and k < ITERS:
        cur, nxt = par, par ^ 1
        v[S.stored] = 0.0
        S.exchange(v, GHOST, GHOST)                      # the handshake behind the local ghost writes
        precondition(S, v, f)
        if "z" not in skip:
            S.exchange(v, 2, 1)
        z = v
        rho, sigma = combine(S, [hi_lo(exact_terms(z[a:b], f[a:b])), hi_lo(exact_terms(z[a:b], d[a:b]))])
        beta = 0.0 if rho_prev is None else sigma / rho_prev
        rho_prev = rho
        lo, hi = (a, b) if "write" in skip else S.wr
        ext = slice(max(a - 1, 0), min(b + 1, N))       # the neighbours the stencil reads, recomputed from z and p
        pn = np.full((N, N, N), np.nan)
        pn[ext] = z[ext] + beta * p[cur][ext]
        p[nxt][lo:hi] = pn[lo:hi]
        pi, = combine(S, [hi_lo(exact_terms(pn[a:b], -residual(pn, np.zeros((N, N, N)), a, b)))])
        alpha = rho / pi
        xn = x[cur].copy()
        xn[ext, 1:-1, 1:-1] = x[cur][ext, 1:-1, 1:-1] + alpha * p[nxt][ext, 1:-1, 1:-1]
        for zz in (0, N - 1):                            # Dirichlet planes keep x
            xn[zz] = x[cur][zz]
        x[nxt][lo:hi] = xn[lo:hi]
        rn = residual(xn, B, a, b)
        d[a:b] = rn - f[a:b]
        f[a:b] = rn
        S.poison_ghosts(f)
        if "f" not in skip:
            S.exchange(f, GHOST, GHOST)
        par = nxt
        k += 1
        hist.append(norm(S, rn))
    v[a:b] = x[par][a:b]
    S.exchange(v, GHOST, GHOST)
    f[a:b] = B[a:b]
    S.exchange(f, GHOST, GHOST)
    return k, np.array(hist)


def problem():
    """random interior v and f, random nonzero Dirichlet faces of v"""
    rng = np.random.default_rng(7)
    v = rng.uniform(-1.0, 1.0, (N, N, N))
    f = rng.uniform(-1.0, 1.0, (N, N, N))
    return v, f


def worker(rank, world, port, plan, skip, out_queue):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    S = Slab(plan, rank, world)
    v0, f0 = problem()
    v, f = S.field(), S.field()
    v[S.stored], f[S.stored] = v0[S.stored], f0[S.stored]
    k, hist = pcg(S, v, f, 1e-12, skip)
    out_queue.put((rank, S.a, S.b, S.stored, k, hist, v[S.stored].copy(), f[S.stored].copy()))
    dist.barrier()
    dist.destroy_process_group()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_slabs(mg, world, skip=()):
    plans = [mg.MultiGrid3D.plan_level(N, world, r) for r in range(world)]
    assert all(p["dist"] == 1 for p in plans)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=worker, args=(r, world, port, plans[r], skip, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted((q.get(timeout=240) for _ in range(world)), key=lambda g: g[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return got


@pytest.mark.parametrize("world", [2, 4])
def test_pcg_slab_schedule_gloo(mg, monkeypatch, world):
    monkeypatch.setenv("MG_B200_DIST_MIN_N", "65")  # distribute the small test grid (default threshold: n >= 257)
    v0, f0 = problem()
    whole = Slab(mg.MultiGrid3D.plan_level(N, 1, 0), 0, 1)
    v, f = v0.copy(), f0.copy()
    k_ref, hist_ref = pcg(whole, v, f, 1e-12)
    assert k_ref == ITERS and hist_ref[-1, 0] < 0.5 * hist_ref[0, 0]  # the iteration did something
    assert np.array_equal(f, f0)
    covered = 0
    for rank, a, b, stored, k, hist, vs, fs in run_slabs(mg, world):
        assert not np.isnan(vs[a - stored.start:b - stored.start]).any(), "a NaN reached the owned planes of rank %d" % rank
        assert k == k_ref and np.array_equal(hist, hist_ref), "rank %d: history differs from the whole-grid run" % rank
        # owned planes: the iterate; ghost planes: the neighbours' iterate, i.e. the caller's boundary values where they lie
        assert np.array_equal(vs, v[stored]), "rank %d: v differs from the whole-grid run" % rank
        assert np.array_equal(fs, f0[stored]), "rank %d: f is not the caller's" % rank
        covered += b - a
    assert covered == N


@pytest.mark.parametrize("skip", ["z", "f", "write"])
def test_each_exchange_and_the_write_range_is_needed(mg, monkeypatch, skip):
    """without the z exchange, the f exchange or the one-plane margin of the p and x updates, a NaN reaches the owned planes"""
    monkeypatch.setenv("MG_B200_DIST_MIN_N", "65")
    got = run_slabs(mg, 2, (skip,))
    assert any(np.isnan(vs[a - stored.start:b - stored.start]).any() or np.isnan(hist).any() for _, a, b, stored, _, hist, vs, _ in got)

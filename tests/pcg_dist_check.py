"""Multi-GPU check of the multigrid-preconditioned conjugate-gradient solve, run under torchrun (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node P --master-addr 127.0.0.1 --master-port 29561 tests/pcg_dist_check.py

The dots that steer a distributed PCG are the correctly rounded dot products of the whole level, so alpha and beta are the
single-GPU ones, and every vector update is pointwise or a partition-invariant stencil: the planes a rank owns must hold
the bits of the single-GPU pcg on every level.  Only the norm's sum of squares is added in another order (within 1e-12,
as tests/dist_check.py holds norms).  Every rank runs the distributed handle and, on its own GPU, a single-GPU handle.
129^3 runs with the slab threshold lowered to 65 (as tests/dist_check.py does), 257^3 with the default plan.
PCG_DIST_CHECK_RUNS="257:" (n:threshold, comma-separated) picks a subset."""
import ctypes
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pde_multigrid_b200 as mg  # noqa: E402
from pde_multigrid_b200._lib import MGError, MG_ERR_STATE  # noqa: E402

SMOOTHERS = (("default", mg.MG_SMOOTHER_AUTO), ("colour", mg.MG_SMOOTHER_COLOUR), ("jacobi", mg.MG_SMOOTHER_JACOBI))
SWEEPS = ((2, 2), (2, 1), (1, 1))


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    failures = []

    def new_uid():
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            raw = (ctypes.c_ubyte * 128)()
            mg._lib.check(mg.lib().mg_comm_unique_id(raw))
            buf.copy_(torch.tensor(list(raw), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        return bytes(buf.cpu().tolist())

    def same(a, b):
        return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))

    def fail(msg):
        failures.append("%s (rank %d/%d)" % (msg, rank, world))

    def agree_across_ranks(tag, r):
        mine = torch.tensor(np.concatenate([[r.cycles, float(r.converged)], r.history.ravel()]), device="cuda", dtype=torch.float64)
        n = torch.tensor([mine.numel()], device="cuda")
        every_n = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(every_n, n)
        if any(int(x.item()) != mine.numel() for x in every_n):
            fail("%s: ranks disagree on the number of iterations" % tag)
            return
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        if any(not same(e.cpu().numpy(), mine.cpu().numpy()) for e in every):
            fail("%s: ranks disagree on iterations / converged / history" % tag)

    def same_history(tag, hd, hs):
        if hd.shape != hs.shape:
            fail("%s: history lengths %d vs %d" % (tag, len(hd), len(hs)))
            return
        if not (np.all(np.abs(hd[:, 0] - hs[:, 0]) <= 1e-12 * np.abs(hs[:, 0])) and same(hd[:, 1], hs[:, 1])):
            fail("%s: history %r vs single GPU %r" % (tag, hd[:4], hs[:4]))

    def same_levels(tag, d, s, levels):
        for l in levels:
            zb, zc = d.owned_range(l)
            if not same(d.get_v(l), s.get_v(l)[zb:zb + zc]):
                fail("%s: v level %d differs from the single GPU" % (tag, l))
            if not same(d.get_f(l), s.get_f(l)[zb:zb + zc]):
                fail("%s: f level %d differs from the single GPU" % (tag, l))

    runs = [(129, "65"), (257, None)]
    if os.environ.get("PCG_DIST_CHECK_RUNS"):
        runs = [(int(a), b or None) for a, b in (r.split(":") for r in os.environ["PCG_DIST_CHECK_RUNS"].split(","))]
    for n, min_n in runs:
        if (n - 1) // world < 8:
            continue
        if min_n is None:
            os.environ.pop("MG_B200_DIST_MIN_N", None)
        else:
            os.environ["MG_B200_DIST_MIN_N"] = min_n
        for dtype in (np.float64, np.float32):
            d = mg.MultiGrid3D(n, dtype=dtype, residual_mode=mg.MG_CORRECTED, rank=rank, nranks=world, nccl_unique_id=new_uid())
            s = mg.MultiGrid3D(n, dtype=dtype, residual_mode=mg.MG_CORRECTED)
            zb, zc = d.owned_range(0)
            rtol = 1e-10 if dtype == np.float64 else 1e-5
            rng = np.random.default_rng(1000 + n)
            case = 0
            for sname, smoother in SMOOTHERS:
                d.set_smoother(smoother)
                s.set_smoother(smoother)
                for v1, v2 in SWEEPS:
                    case += 1
                    if case % 2:
                        start = "init_problem"
                        v0 = f0 = None
                    else:
                        # random interior v and f, random nonzero Dirichlet faces
                        start = "random"
                        v0 = rng.uniform(-1, 1, (n, n, n)).astype(dtype)
                        f0 = rng.uniform(-1, 1, (n, n, n)).astype(dtype)

                    def reset():
                        if v0 is None:
                            d.init_problem()
                            s.init_problem()
                        else:
                            d.set_v(0, v0[zb:zb + zc])
                            d.set_f(0, f0[zb:zb + zc])
                            s.set_v(0, v0)
                            s.set_f(0, f0)

                    tag = "n=%d %s %s V(%d,%d) %s" % (n, np.dtype(dtype).name, sname, v1, v2, start)
                    reset()
                    f_before = d.get_f(0)
                    norm0 = d.residual_norm(0)
                    rs = s.pcg(v1, v2, rtol=rtol, max_iters=40)
                    rd = d.pcg(v1, v2, rtol=rtol, max_iters=40)
                    if (rd.cycles, rd.converged) != (rs.cycles, rs.converged):
                        fail("%s: (%d, %s) vs single GPU (%d, %s)" % (tag, rd.cycles, rd.converged, rs.cycles, rs.converged))
                    agree_across_ranks(tag, rd)
                    if not same(rd.history[0], np.array(norm0)):
                        fail("%s: history[0] %r is not residual_norm %r" % (tag, rd.history[0], norm0))
                    same_history(tag, rd.history, rs.history)
                    same_levels(tag, d, s, range(d.numGrids))
                    if not same(d.get_f(0), f_before):
                        fail("%s: f of the level is not the caller's" % tag)
                    # what follows a pcg sees the same handles: ghost flags, both v buffers, boundary values
                    d.VCycle(0, v1, v2)
                    s.VCycle(0, v1, v2)
                    same_levels(tag + " then VCycle", d, s, [0])
                    sd, ss = d.solve(v1, v2, rtol=0.0, max_cycles=3), s.solve(v1, v2, rtol=0.0, max_cycles=3)
                    same_levels(tag + " then solve", d, s, range(d.numGrids))
                    if sd.cycles != ss.cycles:
                        fail("%s then solve: %d vs %d cycles" % (tag, sd.cycles, ss.cycles))
                    # tolerances at the geometric midpoints of the single-GPU history: the same stopping iteration
                    h = rs.history[:, 0]
                    for k in sorted({1, len(h) - 1}):
                        if k < 1 or k >= len(h) or not (h[k] > 0):
                            continue
                        mid = float(np.sqrt(h[k - 1] * h[k]) / h[0])
                        reset()
                        a = s.pcg(v1, v2, rtol=mid, max_iters=40)
                        b = d.pcg(v1, v2, rtol=mid, max_iters=40)
                        if (a.cycles, a.converged) != (b.cycles, b.converged):
                            fail("%s rtol %.3e: (%d, %s) vs single GPU (%d, %s)" % (tag, mid, b.cycles, b.converged, a.cycles, a.converged))
                        agree_across_ranks(tag + " midpoint", b)
            # a level every rank holds whole: the same iteration on every rank, no communication
            agg = [l for l in range(d.numGrids - 1) if d.owned_range(l)[1] == ((n - 1) >> l) + 1]
            if agg:
                l = agg[0]
                d.set_smoother(mg.MG_SMOOTHER_AUTO)
                s.set_smoother(mg.MG_SMOOTHER_AUTO)
                d.init_problem()
                s.init_problem()
                a, b = s.pcg(2, 2, rtol=rtol, max_iters=30, level=l), d.pcg(2, 2, rtol=rtol, max_iters=30, level=l)
                tag = "n=%d %s agglomerated level %d" % (n, np.dtype(dtype).name, l)
                if (a.cycles, a.converged) != (b.cycles, b.converged) or not same(a.history, b.history):
                    fail("%s: (%d, %s) vs single GPU (%d, %s)" % (tag, b.cycles, b.converged, a.cycles, a.converged))
                agree_across_ranks(tag, b)
                same_levels(tag, d, s, [l])
            elif n == 129:
                fail("n=129: no agglomerated level to run pcg on")
            d.close()
            s.close()
        # MG_REF_COMPAT: MG_ERR_STATE, nothing runs
        d = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_REF_COMPAT, rank=rank, nranks=world, nccl_unique_id=new_uid())
        v_before, f_before = d.get_v(0), d.get_f(0)
        try:
            d.pcg(2, 2, rtol=1e-8, max_iters=5)
            fail("n=%d: pcg on an MG_REF_COMPAT handle did not fail" % n)
        except MGError as e:
            if e.code != MG_ERR_STATE:
                fail("n=%d: MG_REF_COMPAT pcg failed with code %d, not MG_ERR_STATE" % (n, e.code))
        if not (same(d.get_v(0), v_before) and same(d.get_f(0), f_before)):
            fail("n=%d: the refused pcg changed v or f" % n)
        d.close()
    flag = torch.tensor([len(failures)], device="cuda")
    dist.all_reduce(flag)
    for f in failures[:20]:
        print("[rank %d] FAIL %s" % (rank, f), flush=True)
    if rank == 0:
        print("PCG_DIST_CHECK %s world=%d failures=%d" % ("OK" if flag.item() == 0 else "FAILED", world, int(flag.item())), flush=True)
    dist.destroy_process_group()
    return 1 if flag.item() else 0


if __name__ == "__main__":
    sys.exit(main())

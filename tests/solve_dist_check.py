"""Multi-GPU check of the tolerance-driven solve, run under torchrun (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node P --master-addr 127.0.0.1 --master-port 29547 tests/solve_dist_check.py

A distributed solve is host-driven and every rank checks the same all-reduced norm, so every rank must report the same
cycles and history, and the planes a rank owns must hold the bits of the single-GPU solve (RB Gauss-Seidel is
partition-invariant, SURVEY.md 8e).  129^3 runs with the slab threshold lowered to 65 (as tests/dist_check.py does),
257^3 with the default plan."""
import ctypes
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pde_multigrid_b200 as mg  # noqa: E402


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

    for n, min_n in ((129, "65"), (257, None)):
        if min_n is None:
            os.environ.pop("MG_B200_DIST_MIN_N", None)
        else:
            os.environ["MG_B200_DIST_MIN_N"] = min_n
        if (n - 1) // world < 8:
            continue
        d = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED, rank=rank, nranks=world, nccl_unique_id=new_uid())
        s = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        for v1, v2, rtol, cap in ((2, 2, 1e-8, 40), (2, 1, 1e-6, 40)):
            rd = d.solve(v1, v2, rtol=rtol, max_cycles=cap)
            rs = s.solve(v1, v2, rtol=rtol, max_cycles=cap)
            tag = "n=%d V(%d,%d) rank %d/%d" % (n, v1, v2, rank, world)
            if (rd.cycles, rd.converged) != (rs.cycles, rs.converged) or not same(rd.history, rs.history):
                failures.append("%s: (%d, %s) vs single GPU (%d, %s)" % (tag, rd.cycles, rd.converged, rs.cycles, rs.converged))
            # every rank the same decision and history
            mine = torch.tensor(np.concatenate([[rd.cycles, float(rd.converged)], rd.history.ravel()]), device="cuda")
            allh = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine)
            if any(not torch.equal(a, mine) for a in allh):
                failures.append("%s: ranks disagree on cycles / history" % tag)
            for l in range(d.numGrids):
                zb, zc = d.owned_range(l)
                if not same(d.get_v(l), s.get_v(l)[zb:zb + zc]):
                    failures.append("%s: v level %d differs from the single-GPU solve" % (tag, l))
        d.close()
        s.close()
    ok = torch.tensor([len(failures)], device="cuda")
    dist.all_reduce(ok)
    for f in failures:
        print("FAIL", f, flush=True)
    if rank == 0 and int(ok.item()) == 0:
        print("SOLVE_DIST_CHECK OK (%d ranks)" % world, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

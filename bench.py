#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native multigrid engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[3] at N=1, the configuration the metric is quoted on): 3D Poisson
1025^3 fp64, V(2,2) cycles on the reference problem (f = -3 pi^2 sin sin sin, v = 0 on the boundary).
A "step" is one V(2,2) cycle.  For N > 1 (launched by torchrun, one rank per GPU) the same 1025^3 grid
is z-slab partitioned over the ranks: strong scaling.

One JSON line on stdout (rank 0):
  value      V-cycles/s with all fields resident in HBM, CUDA events on the engine's stream, max over ranks
  e2e        the same metric through the C-ABI call with HOST buffers (mg3d_vcycle_host): pinned host
             v,f -> device, one V(2,2), v -> host, every step
  roofline   the dominant kernel (finest-level smoother launch): algorithmic bytes / live event time
  cpu_baseline  the reference CPU solver (oracle/_ref, compiled unmodified) on this box's host, bounded sample
  parity     after the timed region: InitV/InitF again, one V(2,2), and the position-keyed checksum of v on every level
             (mg3d_field_checksum, summed over the ranks) against tests/golden/hashes3d.json -- the numbers the reference
             CPU solver itself produced at this size (tests/golden/make_hash.py).  ok == true means: this run, on this many
             GPUs, holds the reference's bits.
  other_configs  (N=1) the remaining BASELINE.json configurations, measured in the same process: 1D N=1025, 2D Lyapunov
             1025^2, 3D 257^3, and a non-cubic 3D grid (1025 x 513 x 257); (N=8) the 2049^3 capacity run of configs[4]
`--impl reference` times that CPU solver as the measured arm instead (no GPU work at all): 513^3, K cycles.
`--dump-outputs DIR` (N=1) writes what the last timed V-cycle left to its caller: v on every level as DIR/v_level<l>.npy (a level of
more than 2^20 points as a fixed, seeded sample of 2^20 of them; 36 MB in all at 1025^3 fp64) and the level-0 residual norms
(l2, max) as DIR/residual_norm_level0.npy.  The inputs depend on the arguments only, so two builds can be compared file by file;
bench_outputs/ (e.g. --dump-outputs bench_outputs/<build>) is git-ignored for such dumps.
`--profile-traffic` re-measures roofline.traffic with ncu (one launch of the dominant kernel) into profiles/roofline_traffic.json.

Only this file's cpu_baseline / --impl reference legs touch oracle/; the GPU arm never does.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NU1 = NU2 = 2


def level_sizes(n):
    num = int(np.floor(np.log2(n - 1)))
    s = [n]
    for _ in range(1, num):
        s.append((s[-1] - 1) // 2 + 1)
    return s


def algorithmic_bytes_per_cycle(n, B, dim=3, nu1=NU1, nu2=NU2):
    """SURVEY.md 8(d): smoother reads v,f and writes v once per RB sweep; residual->restrict reads v,f
    and writes coarse f; coarse v zeroed; prolong+correct reads coarse v, reads+writes fine v."""
    N = [s ** dim for s in level_sizes(n)]
    tot = 0
    for l, Nl in enumerate(N):
        tot += (nu1 + nu2) * 3 * B * Nl
        if l + 1 < len(N):
            tot += 4 * B * Nl + 3 * B * N[l + 1]
    return tot


def updates_per_cycle(n, dim=3, nu1=NU1, nu2=NU2):
    return (nu1 + nu2) * sum((s - 2) ** dim for s in level_sizes(n))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        try:
            with open(self.path) as fh:
                for line in fh:
                    c = [x.strip() for x in line.split(",")]
                    if len(c) < 9:
                        continue
                    try:
                        sm.append(float(c[1]))
                        smax.append(float(c[2]))
                    except ValueError:
                        continue
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                         c[5:9]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            os.remove(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(smax), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def workload_name(n, B):
    tag = {257: " (BASELINE.json configs[2])", 1025: " (BASELINE.json configs[3])", 2049: " (BASELINE.json configs[4])"}.get(n, "")
    return "3D Poisson %d^3 %s V(%d,%d), reference problem%s, sign-corrected residual" % (n, "fp64" if B == 8 else "fp32", NU1, NU2, tag)


def golden_checksums(n, dtype_tag, mode="corrected"):
    """Checksums of v per level after each V(2,2) cycle, as the reference CPU solver produced them (or None)."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "hashes3d.json")) as fh:
            rec = json.load(fh).get("%d/%s/%s" % (n, dtype_tag, mode))
        return [c["checksum_v"] for c in rec["cycles"]] if rec else None
    except Exception:
        return None


def parity_block(eng, n, dtype_tag):
    """InitV/InitF, V(2,2) cycles, device checksum of v on every level against the reference's own run."""
    want = golden_checksums(n, dtype_tag)
    eng.init_problem()
    if want is None:
        return {"ok": None, "why": "the reference cannot run %d^3 (no golden checksum): see residual_l2 / closed form" % n}
    got, ok = [], True
    for cyc in want:
        eng.VCycle(0, NU1, NU2)
        cs = ["%016x" % eng.field_checksum(l) for l in range(eng.numGrids)]
        got.append(cs)
        ok = ok and cs == cyc
    return {"ok": bool(ok), "cycles": len(want), "checksum_v_level0": got[-1][0], "expected_level0": want[-1][0],
            "levels_compared": len(want[-1]),
            "what": "position-keyed additive checksum (mod 2^64) of the bit patterns of v on every level after each V(2,2) from "
                    "v=0, summed over the ranks' slabs on the device",
            "expected_from": "tests/golden/hashes3d.json: the reference NOCUDA_TESI solver compiled unmodified, run at this size "
                             "(tests/golden/make_hash.py)"}


DUMP_POINTS = 1 << 20


def dump_outputs(eng, out_dir, norms):
    """v of every level and (l2, max) of the level-0 residual, as the timed V-cycles left them.  A level of more than DUMP_POINTS
    points is sampled at DUMP_POINTS flat indices (x fastest) drawn by a generator seeded with the level number, so the same
    arguments always sample the same points."""
    os.makedirs(out_dir, exist_ok=True)
    for l in range(eng.numGrids):
        v = eng.get_v(l)
        if v.size > DUMP_POINTS:
            idx = np.sort(np.random.default_rng(l).choice(v.size, DUMP_POINTS, replace=False))
            v = v.reshape(-1)[idx]
        np.save(os.path.join(out_dir, "v_level%d.npy" % l), v)
    np.save(os.path.join(out_dir, "residual_norm_level0.npy"), np.array(norms, dtype=np.float64))


def bind_to_gpu_numa_node(torch, device_index):
    """Host-side plumbing of the end-to-end leg: run this process (and therefore first-touch and pin its host buffers) on the
    NUMA node the GPU hangs off, so that eight ranks do not pull their PCIe traffic across the socket interconnect.
    Returns (node, n_cpus) or (None, 0) when the topology cannot be read."""
    try:
        p = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as fh:
            node = int(fh.read().strip())
        if node < 0:
            return None, 0
        with open("/sys/devices/system/node/node%d/cpulist" % node) as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None, 0
        os.sched_setaffinity(0, cpus)
        return node, len(cpus)
    except Exception:
        return None, 0


def host_cpu_info():
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    return model, os.cpu_count()


def time_reference_cpu(n_sample, steps, warmup, dtype=np.float64, opt="O2"):
    """The reference's own CPU implementation of the path (NOCUDA_TESI VCycle(0,2,2), single-threaded as
    shipped), from oracle/_ref when it is present, else the plain-C port.  Returns seconds per cycle.
    opt="O0": the as-shipped build (the reference's CompileAndLink passes no optimisation flag)."""
    from oracle import port, ref
    if ref.available():
        o = ref.RefMG(3, dtype, corrected=True, n=n_sample, opt=opt)
        kind = "reference"
    else:
        o = port.PortMG(3, dtype, corrected=True, n=n_sample)
        kind = "port"
    for _ in range(warmup):
        o.vcycle(0, NU1, NU2)
    t0 = time.perf_counter()
    for _ in range(steps):
        o.vcycle(0, NU1, NU2)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    o.close()
    return dt, kind


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # the reference at the headline size needs ~40 GB and ~2 min per cycle (tests/golden/make_hash.py ran it once): the arm
    # samples 513^3 -- one level below, same code path, 1/8 of the points -- for --steps cycles and no warm-up
    n_sample = args.ref_n
    sec, kind = time_reference_cpu(n_sample, args.steps, 0)
    args.warmup = 0
    scale = updates_per_cycle(n_sample) / updates_per_cycle(args.n)
    value = scale / sec
    model, cores = host_cpu_info()
    sample = ("each step = one V(2,2) cycle of the reference NOCUDA_TESI solver (%s, g++ -O2, 1 thread: the reference is "
              "single-threaded) at %d^3 fp64, sign-corrected residual; V-cycles/s scaled to %d^3 by grid-point updates "
              "(x%.5f); the reference cannot use more host threads" % (kind, n_sample, args.n, scale))
    line = {
        "impl": "reference", "metric": "3D Poisson V(2,2) cycles/s", "value": value, "unit": "V-cycles/s",
        # ms_per_step is the wall time of one timed step of THIS run (a V(2,2) of the reference at the sample grid), so that
        # steps x ms_per_step is the time this process really spent; `value` is that rate scaled to the named workload by
        # grid-point updates (the factor is in `sample`), and ms_per_step_full_size_extrapolated is 1e3 / value
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "ms_per_step_full_size_extrapolated": sec * 1e3 / scale, "sample_scale": scale,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.n, 8), "sample_grid": n_sample, "host_cpu": model, "host_cores": cores},
        "grid_point_updates_per_s": updates_per_cycle(n_sample) / sec,
        "cpu_baseline": {"value": value, "unit": "V-cycles/s", "cores": 1, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "V-cycles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def _timed(torch, eng, fn, reps, warm=2):
    s = torch.cuda.ExternalStream(eng.stream)
    for _ in range(warm):
        fn()
    eng.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(reps):
        fn()
    e1.record(s)
    eng.sync()
    return e0.elapsed_time(e1) / reps


def other_configs(mg, torch, world, rank, uid, dist):
    """The BASELINE.json configurations that are not the headline, measured in this process so that the driver's record
    carries them: N=1: configs[0] 1D N=1025 (V(1000,1000) and FMG(2,1000,1000), N1/Poisson1DSolver.cpp:15-25), configs[1] 2D
    Lyapunov 1025^2 (V(2,2) and FMG(1,500,500), N2/LyapunovSolver.cpp:25-43), configs[2] 3D 257^3 fp64 V(2,2).  N=8:
    configs[4], 3D 2049^3 fp64 on 8 GPUs (the reference cannot run it: 32-bit indices)."""
    out = {}
    if world == 1:
        e = mg.MultiGrid1D(1025, dtype=np.float64)
        out["1d_n1025_f64"] = {"vcycle_1000_1000_ms": _timed(torch, e, lambda: e.VCycle(0, 1000, 1000), 5),
                               "fmg_2_1000_1000_ms": _timed(torch, e, lambda: (e.init_problem(), e.FullMultiGridVCycle(0, 2, 1000, 1000)), 3)}
        e.close()
        e = mg.MultiGrid2D(1025, dtype=np.float32)
        ms = _timed(torch, e, lambda: e.VCycle(0, 2, 2), 20)
        upd = 4 * sum((s - 2) ** 2 for s in level_sizes(1025))
        out["2d_lyapunov_1025_f32"] = {"vcycle_2_2_ms": ms, "vcycles_per_s": 1e3 / ms, "grid_point_updates_per_s": upd * 1e3 / ms,
                                       "fmg_1_500_500_ms": _timed(torch, e, lambda: (e.init_problem(), e.FullMultiGridVCycle(0, 1, 500, 500)), 2, warm=1)}
        e.close()
        e = mg.MultiGrid3D(257, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        ms = _timed(torch, e, lambda: e.VCycle(0, 2, 2), 50, warm=3)
        byt = algorithmic_bytes_per_cycle(257, 8)
        peak, _ = measured_peak_gbs()
        want = golden_checksums(257, "f64")
        e.init_problem()
        ok = True
        for cyc in want or []:
            e.VCycle(0, 2, 2)
            ok = ok and ["%016x" % e.field_checksum(l) for l in range(e.numGrids)] == cyc
        out["3d_257_f64"] = {"vcycle_2_2_ms": ms, "vcycles_per_s": 1e3 / ms, "grid_point_updates_per_s": updates_per_cycle(257) * 1e3 / ms,
                             "algorithmic_gbs": byt / ms / 1e6, "hbm_frac": byt / ms / 1e6 / peak, "parity_ok": bool(ok) if want else None}
        e.close()
        # SURVEY.md 8f rank 4: a non-cubic grid (the reference asserts them away, N3/Grid3D.cpp:10-11) through mg3b_*
        shape = (1025, 513, 257)
        e = mg.MultiGrid3DBox(shape, dtype=np.float64, residual_mode=mg.MG_CORRECTED)
        r0b = e.residual_norm(0)[0]
        ms = _timed(torch, e, lambda: e.VCycle(0, 2, 2), 5, warm=2)
        pts = shape[0] * shape[1] * shape[2]
        out["3d_box_1025x513x257_f64"] = {"vcycle_2_2_ms": ms, "vcycles_per_s": 1e3 / ms, "algorithmic_gbs": 149.8 * pts / ms / 1e6,
                                          "hbm_frac": 149.8 * pts / ms / 1e6 / peak, "residual_l2_initial": r0b,
                                          "residual_l2_after_7_cycles": e.residual_norm(0)[0],
                                          "note": "colour-split layout, one thread per point; no TMA staging / temporal blocking (DESIGN.md section 4)"}
        e.close()
    if world == 8:
        n = 2049
        import ctypes
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")  # a second communicator needs its own NCCL id
        if rank == 0:
            raw = (ctypes.c_ubyte * 128)()
            mg._lib.check(mg.lib().mg_comm_unique_id(raw))
            buf.copy_(torch.tensor(list(raw), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        uid = bytes(buf.cpu().tolist())
        e = mg.MultiGrid3D(n, dtype=np.float64, residual_mode=mg.MG_CORRECTED, rank=rank, nranks=world, nccl_unique_id=uid)
        r0 = e.residual_norm(0)[0]
        for _ in range(2):
            e.VCycle(0, NU1, NU2)
        e.sync()
        torch.cuda.synchronize()
        dist.barrier()
        s = torch.cuda.ExternalStream(e.stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        for _ in range(5):
            e.VCycle(0, NU1, NU2)
        e1.record(s)
        e.sync()
        t = torch.tensor([e0.elapsed_time(e1) / 5], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        r7 = e.residual_norm(0)[0]
        byt = algorithmic_bytes_per_cycle(n, 8)
        peak, _ = measured_peak_gbs()
        closed = 3.0 * np.pi ** 2 * ((n - 1) / 2.0) ** 1.5
        out["3d_2049_f64_8gpu"] = {"workload": workload_name(n, 8), "vcycle_2_2_ms": ms, "vcycles_per_s": 1e3 / ms,
                                   "grid_point_updates_per_s": updates_per_cycle(n) * 1e3 / ms,
                                   "hbm_frac_per_gpu": byt / ms / 1e6 / world / peak,
                                   "residual_l2_initial": r0, "closed_form_initial": closed, "initial_matches_closed_form": bool(abs(r0 - closed) <= 1e-10 * closed),
                                   "residual_l2_after_7_cycles": r7, "contraction_per_cycle": (r7 / r0) ** (1.0 / 7.0)}
        e.close()
    return out


def profile_traffic(args):
    """One launch of the dominant kernel under ncu (dram__bytes_read.sum + dram__bytes_write.sum), stored per
    (kernel, n, dtype, arithmetic) in profiles/roofline_traffic.json.  Needs a GPU; N=1 only."""
    kname = {"auto": "k_relax_pipe2", "pipe": "k_relax_pipe2", "tma": "k_relax_colour_tma"}[args.smoother]
    cmd = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum", "--clock-control", "none",
           "-k", "regex:" + kname, "-s", "1", "-c", "1", "--csv", sys.executable, os.path.join(ROOT, "scripts", "pipe_once.py"),
           str(args.n), args.dtype, "pipe" if kname == "k_relax_pipe2" else "tma"] + (["fast"] if args.arith == "fast" else [])
    out = subprocess.run(cmd, capture_output=True, text=True).stdout
    vals = {}
    for line in out.splitlines():
        c = [x.strip('"') for x in line.split('","')]
        if len(c) > 3 and c[-3] in ("dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__time_duration.sum"):
            unit, val = c[-2], float(c[-1].replace(",", ""))
            mult = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}.get(unit, 1)
            vals[c[-3]] = val * mult
    if len(vals) < 3:
        print(out[-2000:])
        raise SystemExit("ncu did not report the metrics")
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(path) as fh:
            tj = json.load(fh)
    except Exception:
        tj = {}
    tj.setdefault("kernels", {})["%s_n%d_%s_%s" % (kname, args.n, args.dtype, args.arith)] = {
        "dram_bytes_per_launch": vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"],
        "dram_bytes_read": vals["dram__bytes_read.sum"], "dram_bytes_write": vals["dram__bytes_write.sum"],
        "ms_under_ncu": vals["gpu__time_duration.sum"],
        "source": "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum, one launch of %s at %d^3 %s (bench.py --profile-traffic); "
                  "a property of the kernel and the grid, not re-measured in the run that prints it" % (kname, args.n, args.dtype)}
    with open(path, "w") as fh:
        json.dump(tj, fh, indent=1, sort_keys=True)
    print(json.dumps(tj["kernels"]))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", "--grid", dest="n", type=int, default=1025,
                    help="finest grid size per axis (2^k+1); under torchrun spell it --grid (torchrun treats --n as an abbreviation of its own options)")
    ap.add_argument("--dtype", default="f64", choices=["f32", "f64"])
    ap.add_argument("--cpu-n", type=int, default=257, help="grid of the bounded CPU-baseline sample of the GPU arm")
    ap.add_argument("--ref-n", type=int, default=513, help="grid the --impl reference arm runs")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--profile-traffic", action="store_true",
                    help="measure the dominant kernel's DRAM bytes per launch with ncu into profiles/roofline_traffic.json and exit")
    ap.add_argument("--arith", default="exact", choices=["exact", "fast"])
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--smoother", default="auto", choices=["auto", "colour", "tma", "fused", "pipe"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write v of every level and the level-0 residual "
                                                           "norms as DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)
    if args.profile_traffic:
        return profile_traffic(args)

    import torch
    import pde_multigrid_b200 as mg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if args.gpus > 1 and world == 1:
        raise SystemExit("--gpus %d needs one rank per GPU: launch with python -m torch.distributed.run "
                         "--nproc-per-node %d bench.py --gpus %d ..." % (args.gpus, args.gpus, args.gpus))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs runs on one GPU: each rank of a z-slab run holds only its own planes")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dist = None
    uid = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        import ctypes
        buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            raw = (ctypes.c_ubyte * 128)()
            mg._lib.check(mg.lib().mg_comm_unique_id(raw))
            buf.copy_(torch.tensor(list(raw), dtype=torch.uint8))
        dist.broadcast(buf, 0)
        uid = bytes(buf.cpu().tolist())

    np_dtype = np.float64 if args.dtype == "f64" else np.float32
    B = np.dtype(np_dtype).itemsize
    n = args.n
    eng = mg.MultiGrid3D(n, dtype=np_dtype, residual_mode=mg.MG_CORRECTED, rank=rank, nranks=world, nccl_unique_id=uid)
    if args.smoother != "auto":
        eng.set_smoother({"colour": mg.MG_SMOOTHER_COLOUR, "tma": mg.MG_SMOOTHER_TMA, "fused": mg.MG_SMOOTHER_FUSED,
                          "pipe": mg.MG_SMOOTHER_PIPE}[args.smoother])
    if args.arith == "fast":
        eng.set_arith(mg.MG_ARITH_FAST)
    stream = torch.cuda.ExternalStream(eng.stream)

    def barrier():
        eng.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    r0 = eng.residual_norm(0)
    for _ in range(args.warmup):
        eng.VCycle(0, NU1, NU2)
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = eng.kernel_launches
    hb0 = eng.halo_bytes
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        eng.VCycle(0, NU1, NU2)
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = eng.kernel_launches - l0
    halo_bytes = eng.halo_bytes - hb0
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    r1 = eng.residual_norm(0)
    if args.dump_outputs:
        dump_outputs(eng, args.dump_outputs, r1)

    # ---- second pass of the same K steps with the per-operator CUDA-event timers on (the timers need eager
    #      launches, the headline pass above replays the same kernels from a CUDA graph) ----
    eng._call("profile", 1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    p0.record(stream)
    for _ in range(args.steps):
        eng.VCycle(0, NU1, NU2)
    p1.record(stream)
    barrier()
    ms_step_profiled = p0.elapsed_time(p1) / args.steps
    eng._call("profile", 0)

    # ---- third figure (SURVEY.md 8d "norm pass accounting"): every cycle followed by the residual norm the parity
    #      runs report (one extra read of v and f on the finest level + a 16-byte read-back), host clock ----
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.VCycle(0, NU1, NU2)
        eng.residual_norm(0)
    barrier()
    ms_step_with_norm = (time.perf_counter() - t0) / args.steps * 1e3
    if dist is not None:
        t = torch.tensor([ms_step_with_norm], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step_with_norm = float(t.item())

    # ---- per-operator breakdown from the live event timers (this rank) ----
    import ctypes
    ops = {"relax": 0, "residual_restrict": 1, "interpolate_correct": 2, "other": 3}
    breakdown = []
    for l in range(eng.numGrids):
        row = {"level": l, "n": eng.level_size(l)}
        for name, op in ops.items():
            ms, kl, calls = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_longlong()
            eng._call("profile_read", ctypes.c_int(l), ctypes.c_int(op), ctypes.byref(ms), ctypes.byref(kl), ctypes.byref(calls))
            if calls.value:
                row[name] = {"ms": ms.value / args.steps, "launches": kl.value // args.steps}
        breakdown.append(row)

    peak, peak_src = measured_peak_gbs()
    bytes_cycle = algorithmic_bytes_per_cycle(n, B)
    N0 = n ** 3
    relax0 = breakdown[0].get("relax", {"ms": 0.0, "launches": 0})
    roofline = None
    if relax0["launches"]:
        # The dominant kernel is the finest-level smoother.  Default smoother: the temporally blocked pass, ONE kernel launch
        # = TWO full RB sweeps (k_relax_pipe2; the conditional exact-fallback launch behind it exits at once unless the range
        # guard fired and is timed with it).  Algorithmic bytes (SURVEY.md 8d): 3*B*N0 per RB sweep = read v, read f,
        # write v -- the pass moves fewer real bytes than that (2.5*B*N0 + halo for both sweeps), so achieved/peak can
        # exceed 1; `traffic` is what ncu saw it move.
        two_sweep = args.smoother in ("auto", "pipe") or (args.smoother == "fused" and world == 1)  # slabs take the pass too
        sweeps_per_launch = 2.0 if two_sweep else 0.5
        nlaunch = (NU1 + NU2) / sweeps_per_launch
        alg_per_launch = sweeps_per_launch * 3 * B * (N0 / world)
        avg_ms = relax0["ms"] / nlaunch
        achieved = alg_per_launch / (avg_ms * 1e-3) / 1e9
        kname = "k_relax_pipe2" if two_sweep and args.smoother != "fused" else ("k_relax_fused2" if two_sweep else "k_relax_colour_tma")
        traffic, traffic_src = None, None
        if world == 1:
            try:
                with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as fh:
                    ent = json.load(fh).get("kernels", {}).get("%s_n%d_%s_%s" % (kname, n, args.dtype, args.arith))
                if ent:
                    traffic, traffic_src = ent["dram_bytes_per_launch"], ent["source"]
            except Exception:
                pass
        roofline = {"bound": "hbm", "kernel": "%s: finest-level smoother, %g RB sweep(s) per launch" % (kname, sweeps_per_launch),
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "frac_of_nominal_8000_gbs": achieved / 8000.0, "traffic": traffic, "traffic_source": traffic_src,
                    "dram_gbs_on_traffic": (traffic / (avg_ms * 1e-3) / 1e9) if traffic else None,
                    "dram_frac_on_traffic": (traffic / (avg_ms * 1e-3) / 1e9 / peak) if traffic else None,
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_per_launch, "avg_launch_ms": avg_ms,
                    "launches_per_cycle": nlaunch, "kernel_launches_counted_per_cycle": relax0["launches"],
                    "share_of_step": relax0["ms"] / ms_step_profiled,
                    "measured_in": "second pass of the same %d steps with per-operator CUDA events on the engine's stream "
                                   "(%.3f ms/step eager; the headline pass replays the same kernels from a CUDA graph)" % (args.steps, ms_step_profiled)}

    parity = None if args.no_parity else parity_block(eng, n, args.dtype)

    # ---- end to end through the C-ABI call with HOST buffers (every rank moves the planes it owns) ----
    e2e = None
    if not args.no_e2e:
        zb, zc = eng.owned_range(0)
        cnt = zc * n * n
        numa_node, numa_cpus = bind_to_gpu_numa_node(torch, local_rank)
        hv = torch.zeros(cnt, dtype=torch.float64 if B == 8 else torch.float32).pin_memory()
        hf = torch.empty(cnt, dtype=hv.dtype).pin_memory()
        hf_np = hf.numpy().reshape(zc, n, n)
        hv_np = hv.numpy().reshape(zc, n, n)
        eng.init_problem()
        hf_np[...] = eng.get_f(0)
        eng.vcycle_host(hv_np, hf_np, NU1, NU2, 1)  # warm-up (allocates the staging buffer)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            eng.vcycle_host(hv_np, hf_np, NU1, NU2, 1)
        barrier()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        if dist is not None:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": 1.0 / dt, "unit": "V-cycles/s", "h2d_bytes_per_step": 2 * N0 * B, "d2h_bytes_per_step": N0 * B,
               "steps": args.e2e_steps, "ms_per_step": dt * 1e3, "pcie_gbs_per_gpu": 3 * N0 * B / world / dt / 1e9,
               "host_buffers": "pinned, allocated on the GPU's NUMA node %s (%d CPUs bound)" % (numa_node, numa_cpus) if numa_node is not None
                               else "pinned (the host exposes no NUMA node for the GPU -- a single-node VM: nothing to bind)",
               "call": "mg3d_vcycle_host (pinned host v,f -> device, VCycle(0,2,2), v -> host; every rank moves its own z-slab)",
               "timer": "host wall clock around the synchronous C-ABI call, barrier on both sides, max over ranks"}
        del hv, hf

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sec, kind = time_reference_cpu(args.cpu_n, args.cpu_steps, 0)
        scale = updates_per_cycle(args.cpu_n) / updates_per_cycle(n)
        as_shipped = None
        if kind == "reference":
            try:  # same sources without optimisation flags, as the reference's own build script compiles them
                sec0, _ = time_reference_cpu(args.cpu_n, 1, 0, opt="O0")
                as_shipped = {"value": scale / sec0, "unit": "V-cycles/s", "seconds_per_cycle_at_sample": sec0, "flags": "-O0"}
            except Exception:
                as_shipped = None
        cpu_baseline = {"value": scale / sec, "unit": "V-cycles/s", "cores": 1, "kind": kind, "as_shipped_O0": as_shipped,
                        "grid_point_updates_per_s": updates_per_cycle(args.cpu_n) / sec,
                        "sample": "%d V(2,2) cycles of the reference NOCUDA_TESI solver (g++ -O2, 1 thread: it is single-threaded) "
                                  "at %d^3 fp64, sign-corrected residual, %.2f s/cycle; V-cycles/s scaled to %d^3 by grid-point "
                                  "updates (x%.5f)" % (args.cpu_steps, args.cpu_n, sec, n, scale)}

    levels = eng.numGrids
    eng.close()
    eng = None
    other = None
    if not args.no_other_configs:
        try:
            other = other_configs(mg, torch, world, rank, uid, dist)
        except Exception as exc:  # the headline line must not die with a side measurement
            other = {"error": repr(exc)}
    if rank == 0:
        model, cores = host_cpu_info()
        value = 1e3 / ms_step
        line = {
            "metric": "3D Poisson V(2,2) cycles/s", "value": value, "unit": "V-cycles/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": workload_name(n, B), "levels": levels, "partition": "z-slabs x%d" % world,
                       "l2": "fields are %.1f GB per level-0 array, far larger than the 126 MB L2: no flush needed" % (N0 * B / 1e9),
                       "smoother": args.smoother, "arithmetic": args.arith, "host_cpu": model, "host_cores": cores},
            "grid_point_updates_per_s": updates_per_cycle(n) * value,
            "algorithmic_bytes_per_cycle": bytes_cycle,
            "hbm_roofline_cycle": {"achieved_gbs": bytes_cycle / (ms_step * 1e-3) / 1e9 / world, "peak_gbs": peak,
                                   "frac": bytes_cycle / (ms_step * 1e-3) / 1e9 / world / peak, "per": "GPU",
                                   "frac_of_nominal_8000_gbs": bytes_cycle / (ms_step * 1e-3) / 1e9 / world / 8000.0},
            # halo traffic of rank 0 against one direction of NVLink 5 (900 GB/s): the exchanges are latency-, not bandwidth-bound
            "nvlink_halo": (None if world == 1 else
                            {"bytes_per_cycle_rank0": int(halo_bytes) // max(args.steps, 1),
                             "achieved_gbs": halo_bytes / max(args.steps, 1) / (ms_step * 1e-3) / 1e9, "peak_gbs": 900.0,
                             "frac": halo_bytes / max(args.steps, 1) / (ms_step * 1e-3) / 1e9 / 900.0}),
            "residual_l2": {"before": r0[0], "after": r1[0]},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks, "parity": parity,
            "other_configs": other,
            "gpu_launches": int(launches), "halo_bytes_per_cycle_rank0": int(halo_bytes) // max(args.steps, 1),
            "ms_per_step_profiled_pass": ms_step_profiled,
            "with_per_cycle_norm": {"ms_per_step": ms_step_with_norm, "value": 1e3 / ms_step_with_norm, "unit": "V-cycles/s",
                                    "what": "V-cycle + residual_norm(0) per step, host clock (the norm is read back every cycle)"},
            "breakdown_ms_per_cycle": breakdown,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

#!/usr/bin/env python
"""bench.py -- BP4 CG throughput of the B200-native hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--degree P] [--s S] [--solver merged|plain]
                  [--mode weak|strong] [--sweep none|default|full] [--dump-outputs DIR]
  python bench.py --impl reference ...      # the reference algorithm's CPU restatement on host cores

A "step" is one call of the reference's `run_cg_solver` plugin (benchmark.h:193: x0 = 0,
ReductionControl(100, 1e-15, 1e-8)) on the synthetic BP4 problem; the metric is the
reference's own `dofs/s/it` column (benchmark.h:222): n_dofs * n_iterations / solver_time.

  value     device-timed (CUDA events on the solver's stream), right-hand side resident in HBM
  e2e       same call with HOST buffers: b uploaded and x downloaded inside the timed region
  roofline  dominant kernel (the cell kernel): algorithmic bytes (SURVEY 8d: 16 B/DoF + 300 B/cell
            for the operator, + 42.67 B per DoF whose vector updates run inside the loop) over the
            CUDA-event duration of its launches in the timed region, vs MEASURED_PEAKS.json;
            roofline.iteration = the whole merged iteration (58.67 B/DoF + 300 B/cell) over the
            device time of one iteration
  cpu_baseline  the CPU oracle (C/OpenMP restatement of the reference algorithm, kind "port": the
            real reference needs deal.II + p4est + MPI, absent here) on a bounded sample
  sweep     (N = 1) the other BASELINE.json configs, one timed solve each: Q3 s=15 plain, Q6 s=18
            merged, Q2..Q8 at ~100 M DoFs (merged; plain too with --sweep full)
Multi-GPU: --mode weak (default) runs s + log2(N) (fixed DoFs per GPU); --mode strong keeps s.
One JSON line on stdout (rank 0).

  --dump-outputs DIR  after the timed steps, rank 0 writes what the last of them returned to its
            caller (the end-to-end loop's last run_cg_solver call): DIR/x.npy, the solution of its owned
            DoFs (float64; above DUMP_MAX_ENTRIES entries a fixed, seeded sample of them), and
            DIR/iterations.npy.  The inputs depend on the arguments only, so two builds of the
            project can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "BP4 CG GDoF/s (DoFs x iterations / s)"
UNIT = "GDoF/s"
# BASELINE.json configs[3]: Q2..Q8 at ~100 M DoFs (SURVEY 8d)
DEGREE_SWEEP = [(2, 22), (3, 20), (4, 19), (5, 18), (6, 17), (7, 16), (8, 16)]
# --dump-outputs: 16 MB of float64 at most for the solution (Q4 s=18 has 51 M DoFs = 407 MB)
DUMP_MAX_ENTRIES = 1 << 21


def n_dofs_of(p, s):
    nr, rem = divmod(s, 3)
    n = [((2 if d < rem else 1) << nr) * p + 1 for d in range(3)]
    return 3 * n[0] * n[1] * n[2], (1 << s)


def algorithmic_bytes_per_iteration(p, s, merged=True):
    """SURVEY 8(d): merged = 7.333 doubles/DoF, plain = 17.333 doubles/DoF, + 300 B/cell metadata"""
    nd, nc = n_dofs_of(p, s)
    return (58.0 + 2.0 / 3.0 if merged else 138.0 + 2.0 / 3.0) * nd + 300.0 * nc


def cell_kernel_bytes(n_dofs, n_cells, n_private):
    """operator apply 16 B/DoF + 300 B/cell; the in-loop do_cg_update4b/3b add the remaining
    58.67 - 16 B/DoF of the merged iteration on the DoFs they cover"""
    return 16.0 * n_dofs + 300.0 * n_cells + (58.0 + 2.0 / 3.0 - 16.0) * n_private


def dump_outputs(out_dir, x, iterations):
    """--dump-outputs: x.npy (the solution, or the entries at DUMP_MAX_ENTRIES positions drawn with a
    fixed seed when it is longer) and iterations.npy, both float64"""
    import numpy as np
    if x.size > DUMP_MAX_ENTRIES:
        x = x[np.sort(np.random.default_rng(0).choice(x.size, DUMP_MAX_ENTRIES, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), np.asarray(x, dtype=np.float64))
    np.save(os.path.join(out_dir, "iterations.npy"), np.array([iterations], dtype=np.float64))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores():
    """physical cores this process may run on (SMT siblings counted once); torchrun's
    OMP_NUM_THREADS=1 is deliberately ignored: the CPU arm uses the whole host"""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1
    seen = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                seen.add(f.read().strip())
        except OSError:
            seen.add(str(c))
    return max(1, len(seen))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


class CpuArm:
    """the CPU oracle's CG (C/OpenMP restatement of the reference algorithm: even-odd, z-layer-wise
    cell kernel; merged variant with the vector updates per cell-batch range inside the loop,
    one chunk of ranges per thread) on this box's host cores"""

    def __init__(self, p, s, merged):
        from oracle import bp4_oracle as O
        from oracle import c_oracle
        c_oracle.build()
        self.lib = c_oracle.lib()
        self.cores = host_cores()
        self.lib.oracle_set_num_threads(self.cores)
        self.lib.oracle_set_fast(1)
        self.p, self.s, self.merged = p, s, merged
        self.rd = O.build_problem(p, s)[0]
        self.co = c_oracle.COracle(self.rd)
        self.prec = O.finish_inverse_diagonal(O.inverse_diagonal(self.rd))
        self.threads = self.lib.oracle_num_threads()

    def step(self, max_its):
        t0 = time.perf_counter()
        _, it, _ = self.co.cg(self.rd.rhs, self.prec, self.merged, max_steps=max_its, blocked=self.merged)
        return it, time.perf_counter() - t0


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port; the real reference cannot be
    built here) on this box's host cores: same metric, degree, mesh and solver; every step is a
    bounded sample (--cpu-iters CG iterations of the same problem instead of 100)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    s_gpu = args.s + (max(0, world.bit_length() - 1) if args.mode == "weak" else 0)
    s = min(s_gpu, args.cpu_s)          # the numpy set-up of the oracle needs ~0.2 kB per DoF
    merged = args.solver == "merged"
    arm = CpuArm(args.degree, s, merged)
    steps, warmup = args.steps, max(0, args.warmup)
    for _ in range(warmup):
        arm.step(min(args.cpu_iters, 3))
    its, sec = 0, 0.0
    for _ in range(steps):
        it, dt = arm.step(args.cpu_iters)
        its += it
        sec += dt
    nd, nc = n_dofs_of(args.degree, s)
    val = nd * its / sec * 1e-9
    sample = (f"degree {args.degree}, s={s} ({nc} cells, {nd} DoFs)"
              + (f" instead of s={s_gpu}" if s != s_gpu else "")
              + f"; {its // steps} CG iterations per step instead of 100; {arm.threads} OpenMP threads")
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
           "steps": steps, "warmup": warmup, "ms_per_step": sec / steps * 1e3,
           "higher_is_better": True, "scaling": args.mode, "vs_baseline": None, "dtype": "f64",
           "data": "synthetic", "config": workload_config(args, 1, s),
           "cpu_baseline": {"value": val, "unit": UNIT, "cores": arm.threads, "kind": "port", "sample": sample},
           "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def workload_config(args, n_gpus, s_run=None):
    s_run = args.s if s_run is None else s_run
    nd, nc = n_dofs_of(args.degree, s_run)
    plug = "benchmark_precond_merged" if args.solver == "merged" else "benchmark_precond"
    return {"workload": f"BP4 Q{args.degree} (q={args.degree + 2}) vector Laplace, curved mesh s={s_run}: "
                        f"{nc} cells, {nd} DoFs on {n_gpus} GPU(s), {plug} (ReductionControl(100,1e-15,1e-8), "
                        f"Jacobi, RHS i%8), Renumber(0,1,2)",
            "degree": args.degree, "s": s_run, "n_dofs": nd, "n_dofs_per_gpu": nd // n_gpus, "solver": args.solver,
            "parallelism": "single GPU" if n_gpus == 1 else
            f"domain decomposition over {n_gpus} GPUs (contiguous chunks of the cell order), ghost "
            f"exchange + 7-double all-reduce per iteration; {args.mode} scaling"
            + (f" s = {args.s} + log2(N)" if args.mode == "weak" else f" at fixed s = {args.s}"),
            "l2": "vectors (%.0f MB per GPU each) exceed the 126 MB L2; no flush needed" % (nd * 8 / 1e6 / n_gpus)}


def timed_solves(prob, stream, steps, barrier):
    """device time of `steps` plugin calls with the right-hand side resident in HBM"""
    import torch
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    iters = 0
    for _ in range(steps):
        _, it = prob.run_cg_solver(None, want_x=False)
        iters += it
    e1.record(stream)
    barrier()
    return e0.elapsed_time(e1), iters


def sweep_entry(name, p, s, solver, peak, local_rank):
    """one timed solve (after one warm-up solve) of another BASELINE config on this GPU"""
    import ctypes as C
    import torch
    from mf_data_locality_b200 import capi, host
    t0 = time.perf_counter()
    prob = host.Problem(p, s, plugin=solver, device=local_rank)
    setup = time.perf_counter() - t0
    ctx = C.c_void_p(prob.ctx_handle())
    sp = C.c_void_p()
    capi.lib().bp4_ctx_stream(ctx, C.byref(sp))
    stream = torch.cuda.ExternalStream(sp.value or 0, device=local_rank)
    prob.run_cg_solver(None, want_x=False)
    ms, iters = timed_solves(prob, stream, 1, torch.cuda.synchronize)
    nd, nc = prob.n_dofs, prob.n_cells_global
    byts = algorithmic_bytes_per_iteration(p, s, solver == "merged")
    it_ms = ms / max(iters, 1)
    out = {"config": name, "degree": p, "s": s, "solver": solver, "n_dofs": nd, "iterations": iters,
           "value": nd * iters / (ms * 1e-3) * 1e-9, "unit": UNIT, "ms_per_iteration": it_ms,
           "iteration_roofline_frac": byts / (it_ms * 1e-3) * 1e-9 / peak, "setup_seconds": setup,
           "steps": 1, "warmup": 1}
    prob.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--degree", type=int, default=4)
    ap.add_argument("--s", "--size", dest="s", type=int, default=18,
                    help="mesh size: 2^s cells (use --size under torchrun, whose own options shadow --s)")
    ap.add_argument("--mode", default="weak", choices=["weak", "strong"],
                    help="weak: s + log2(N) on N GPUs (fixed DoFs per GPU); strong: s on any N")
    ap.add_argument("--cpu-s", type=int, default=18, help="largest mesh of the CPU sample")
    ap.add_argument("--cpu-iters", type=int, default=10, help="CG iterations per CPU step (bounded sample)")
    ap.add_argument("--solver", default="merged", choices=["merged", "plain"])
    ap.add_argument("--sweep", default="default", choices=["none", "default", "full"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the solution and iteration count of the last timed solve to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from mf_data_locality_b200 import capi, host
    import ctypes as C

    # weak scaling: the mesh grows with the GPU count (s + log2 N: twice the cells per doubling,
    # SURVEY 8d config 5), partitioned along the renumbered cell order, one partition per GPU
    s_run = args.s + (max(0, world.bit_length() - 1) if args.mode == "weak" else 0)
    nccl_id = None
    if world > 1:
        idt = torch.tensor(list(capi.unique_id() if rank == 0 else bytes(128)), dtype=torch.uint8, device="cuda")
        dist.broadcast(idt, src=0)
        nccl_id = bytes(idt.cpu().tolist())
    prob = host.Problem(args.degree, s_run, plugin=args.solver, device=local_rank, n_ranks=world, rank=rank,
                        nccl_id=nccl_id)
    ctx = C.c_void_p(prob.ctx_handle())
    L = capi.lib()
    stream_ptr = C.c_void_p()
    L.bp4_ctx_stream(ctx, C.byref(stream_ptr))
    stream = torch.cuda.ExternalStream(stream_ptr.value or 0, device=local_rank)
    n_dofs = prob.n_dofs
    fused_flag, n_priv, n_units = C.c_int(), C.c_uint64(), C.c_uint64()
    L.bp4_fused_info(ctx, C.byref(fused_flag), C.byref(n_priv), C.byref(n_units))
    merged = args.solver == "merged"
    fused = merged and bool(fused_flag.value)
    nr_, pc_ = C.c_int(), C.c_int()
    L.bp4_comm_info(ctx, C.byref(nr_), C.byref(pc_))
    exchange = None if world == 1 else ("copy-engine peer copies into IPC-shared buffers, stream-memory-op flags"
                                        if pc_.value else "NCCL send/recv")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ------------------------------------------------------
    L.bp4_profile_enable(ctx, 1)        # on during the warm-up too: the timing events get created there
    for _ in range(args.warmup):
        prob.run_cg_solver(None, want_x=False)
    L.bp4_profile_reset(ctx)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_local, iters = timed_solves(prob, stream, args.steps, barrier)
    clocks = sampler.stop()
    ms = torch.tensor([ms_local], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    parts = {}
    for nm, kid in (("cells", capi.K_VMULT), ("cells_with_updates", capi.K_MERGED), ("pre", capi.K_PRE),
                    ("post", capi.K_POST), ("blas1", capi.K_BLAS1)):
        a_, b_ = C.c_double(), C.c_uint64()
        L.bp4_profile_get(ctx, kid, C.byref(a_), C.byref(b_))
        parts[nm] = {"ms_total": a_.value, "launches": int(b_.value)}
    kkey = "cells_with_updates" if fused else "cells"
    kms, kcnt = parts[kkey]["ms_total"], parts[kkey]["launches"]
    kernel_name = ("cell_kernel<P,CPB,true> (operator + in-loop do_cg_update4b/3b on range-private DoFs)" if fused
                   else "cell_kernel<P,CPB,false> (operator apply)")
    launches = C.c_uint64()
    L.bp4_launch_count(ctx, C.byref(launches))
    L.bp4_profile_enable(ctx, 0)
    value = n_dofs * iters / (total_ms * 1e-3) * 1e-9      # n_dofs is the global count

    # ---- end to end: host buffers through the plugin call --------------------------------
    b_host = torch.from_numpy(prob.rhs()).pin_memory()
    x_host = torch.empty(prob.n_owned, dtype=torch.float64).pin_memory()
    b_np, x_np = b_host.numpy(), x_host.numpy()
    it_c = C.c_uint()
    barrier()
    t0 = time.perf_counter()
    e2e_iters = 0
    for _ in range(args.steps):
        prob._chk(prob.l.bp4h_run_cg_solver(prob.h, b_np.ctypes.data_as(C.c_void_p),
                                           x_np.ctypes.data_as(C.c_void_p), C.byref(it_c)))
        e2e_iters += it_c.value
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = n_dofs * e2e_iters / float(dt.item()) * 1e-9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x_np, it_c.value)

    per_rank = None
    if world > 1:   # every rank's share of the iteration (the slowest one sets the pace)
        mine = {"rank": rank, "n_owned": prob.n_owned, "n_ghost": prob.n_ghost,
                "ms_per_iteration": {k: v["ms_total"] / max(iters, 1) for k, v in parts.items()},
                "launches_per_iteration": {k: v["launches"] / max(iters, 1) for k, v in parts.items()}}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    # per launch = per GPU: this rank's DoFs and cells
    alg_bytes = cell_kernel_bytes(prob.n_owned, prob.n_cells, int(n_priv.value) if fused else 0)
    # whole CG iteration against the same roof: SURVEY 8(d) bytes per iteration over the
    # device time of one iteration (all kernels, exchanges and the host round trip for the sums)
    it_bytes = algorithmic_bytes_per_iteration(args.degree, s_run, merged) * prob.n_owned / n_dofs
    it_ms = total_ms / max(iters, 1)
    # with the overlapped exchange a loop is three launches (cell partitions): per-loop time
    loops = max(iters, 1) * args.steps // args.steps if merged else max(kcnt, 1)
    avg_ms = kms / max(iters if merged else kcnt, 1)
    achieved = alg_bytes / (avg_ms * 1e-3) * 1e-9 if avg_ms > 0 else 0.0
    traffic, fp64 = None, None
    tpath = os.path.join(ROOT, "profiles", "kernel_counters.json")
    if os.path.exists(tpath):          # ncu captures of the committed kernels (scripts/ncu_counters.py)
        with open(tpath) as f:
            kc = json.load(f).get(f"q{args.degree}_{'fused' if fused else 'plain'}")
        if kc:
            traffic = kc.get("dram_bytes_per_dof", 0) * prob.n_owned or None
            ipd = kc.get("fp64_lane_instr_per_dof")
            if ipd and avg_ms > 0:
                pk = 148 * 64 * (clocks.get("sm_max_mhz") or 1965.0) * 1e6
                fp64 = {"instr_per_dof": ipd, "source": kc.get("source"), "peak_lane_instr_per_s": pk,
                        "frac": ipd * prob.n_owned / (avg_ms * 1e-3) / pk}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel": kernel_name, "kernels_in_timed_region": parts,
                "kernel_ms_avg": avg_ms, "kernel_launches": int(kcnt),
                "kernel_share_of_step": kms / total_ms if total_ms else None,
                "algorithmic_bytes_per_launch": alg_bytes,
                "fused": fused, "dofs_updated_in_loop": int(n_priv.value) if fused else 0,
                # second roof: the cell kernel is FP64-pipe bound (DESIGN.md section 5)
                "fp64_pipe": fp64,
                "iteration": {"algorithmic_bytes": it_bytes, "ms": it_ms,
                              "achieved": it_bytes / (it_ms * 1e-3) * 1e-9,
                              "frac": it_bytes / (it_ms * 1e-3) * 1e-9 / peak}}

    setup_seconds = prob.setup_seconds
    sweep = None
    if world == 1 and args.sweep != "none":
        prob.close()                     # free HBM before the larger configs
        torch.cuda.empty_cache()
        todo = [("configs[0] Q3 s=15 plain CG", 3, 15, "plain"), ("configs[2] Q6 s=18 merged CG", 6, 18, "merged")]
        todo += [(f"configs[3] Q{p} s={s} merged CG", p, s, "merged") for p, s in DEGREE_SWEEP]
        if args.sweep == "full":
            todo += [(f"configs[3] Q{p} s={s} plain CG", p, s, "plain") for p, s in DEGREE_SWEEP]
        sweep = []
        for name, p, s, solver in todo:
            try:
                sweep.append(sweep_entry(name, p, s, solver, peak, local_rank))
            except Exception as e:       # the sweep is reported, never required
                sweep.append({"config": name, "error": str(e)})

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            s_cpu = min(args.s, args.cpu_s)
            arm = CpuArm(args.degree, s_cpu, merged)
            arm.step(2)
            its, sec = arm.step(args.cpu_iters)
            nd_c, nc_c = n_dofs_of(args.degree, s_cpu)
            cpu = {"value": nd_c * its / sec * 1e-9, "unit": UNIT, "cores": arm.threads, "kind": "port",
                   "sample": f"CPU oracle (C/OpenMP restatement of the reference algorithm: even-odd, layer-wise "
                             f"cells; vector updates per cell-batch range inside the loop), degree {args.degree}, "
                             f"s={s_cpu} ({nc_c} cells, {nd_c} DoFs), {its} CG iterations instead of 100, {sec:.1f} s"}
        except Exception as e:  # the baseline is reported, never required
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
           "scaling": args.mode, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": workload_config(args, world, s_run), "iterations_per_step": iters // args.steps,
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(prob.n_owned * 8),
                   "d2h_bytes_per_step": int(prob.n_owned * 8)},
           "gpu_launches": int(launches.value), "clocks": clocks, "roofline": roofline,
           "cpu_baseline": cpu, "setup_seconds": setup_seconds, "ghost_exchange": exchange, "per_rank": per_rank,
           "sweep": sweep}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

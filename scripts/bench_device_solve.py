"""Host-driven against device-resident CG solves on one B200.

For each workload the host-driven plugin (benchmark_precond / benchmark_precond_merged) and its
device-resident counterpart (..._device) solve the benchmark's problem, alternated in one process
after a warm-up, 100 iterations each (tolerances 0: every solve runs to the cap).  Reports ms per
iteration, GDoF/s, the spread over the repeats and the rel-L2 difference of the two solutions.
`host_driven_kernel_ms_per_it` is the summed per-kernel event time of the host-driven solve (bp4_profile_*),
i.e. what the GPU is busy with; the gap to the device solve's time per iteration is what the
graph still spends between kernels.

usage: python scripts/bench_device_solve.py [--repeats N] [--out FILE] [--quick]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# configs[0] (Q3 s=15, plain) and a size below it; merged Q4 from small to the 51 M DoFs of configs[1]
WORKLOADS = [(3, 14, "plain"), (3, 15, "plain"), (4, 12, "merged"), (4, 15, "merged"), (4, 18, "merged")]
STEPS = 100


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed_solve(prob, ctx):
    ctx.synchronize()
    t0 = time.perf_counter()
    _, it = prob.run_cg_solver(want_x=False)
    ctx.synchronize()
    return time.perf_counter() - t0, it


def kernel_ms(ctx):
    from mf_data_locality_b200 import capi
    return sum(ctx.profile_get(k)[0] for k in (capi.K_VMULT, capi.K_MERGED, capi.K_PRE, capi.K_POST, capi.K_BLAS1))


def run(p, s, kind, repeats):
    from mf_data_locality_b200 import capi, host
    probs, ctxs = {}, {}
    for name in (kind, kind + "_device"):
        pr = host.Problem(p, s, plugin=name, device=0)
        pr.set_solver(STEPS, 0.0, 0.0)
        probs[name] = pr
        ctxs[name] = capi.Context.from_handle(pr.ctx_handle(), p, pr.n_cells, pr.n_owned, pr.n_ghost)
    n_dofs = probs[kind].n_dofs
    for name in probs:                                   # warm-up: modules, pools, the graph
        timed_solve(probs[name], ctxs[name])
    times = {name: [] for name in probs}
    for _ in range(repeats):
        for name in probs:
            t, it = timed_solve(probs[name], ctxs[name])
            assert it == STEPS, (name, it)
            times[name].append(t / it)
    # GPU-busy time per iteration of the host-driven solve (separate run: event timing costs host time)
    ctx = ctxs[kind]
    ctx.profile_reset()
    ctx.profile_enable(True)
    _, it = probs[kind].run_cg_solver(want_x=False)
    busy = kernel_ms(ctx) / it
    ctx.profile_enable(False)
    xs = {name: probs[name].run_cg_solver()[0] for name in probs}
    diff = float(np.linalg.norm(xs[kind] - xs[kind + "_device"]) / np.linalg.norm(xs[kind]))
    fused = ctxs[kind].fused_info()[0] if kind == "merged" else None
    for pr in probs.values():
        pr.close()
    row = {"degree": p, "s": s, "solver": kind, "n_dofs": n_dofs, "iterations": STEPS, "repeats": repeats,
           "in_loop_updates": fused, "x_rel_l2_host_vs_device": diff,
           "host_driven_kernel_ms_per_it": busy}
    for name, ts in times.items():
        ms = 1e3 * np.array(ts)
        key = "device" if name.endswith("_device") else "host"
        row[key] = {"ms_per_it_median": float(np.median(ms)), "ms_per_it_min": float(ms.min()),
                    "ms_per_it_max": float(ms.max()), "gdof_s_median": n_dofs / np.median(ms) / 1e6}
    row["speedup_median"] = row["host"]["ms_per_it_median"] / row["device"]["ms_per_it_median"]
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a check of the script)")
    a = ap.parse_args()
    from mf_data_locality_b200 import capi
    if capi.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    work = [(3, 8, "plain"), (4, 7, "merged")] if a.quick else WORKLOADS
    res = {"gpu": gpu_info(), "note": "ms per CG iteration over 100-iteration solves, host-driven vs "
           "device-resident solve alternated in one process; spread = min/max over the repeats",
           "workloads": []}
    for p, s, kind in work:
        row = run(p, s, kind, a.repeats)
        print(json.dumps(row), flush=True)
        res["workloads"].append(row)
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

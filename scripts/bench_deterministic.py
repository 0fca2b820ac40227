"""Default against deterministic mode (bp4_desc::deterministic) on one B200.

For each workload the two modes are alternated in one process after a warm-up, `--repeats` times:
  - ms per operator apply: 50 applies between two CUDA events on the context's stream;
  - ms per CG iteration of the host-driven plugin and of its device-resident counterpart
    (100-iteration solves, tolerances 0: every solve runs to the cap).
Reports medians and the min/max spread, the number of cell colours, and whether two solves of
the deterministic mode gave the same bits.

usage: python scripts/bench_deterministic.py [--repeats N] [--out FILE] [--quick]"""
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

# configs[0] (Q3 s=15, plain), configs[1] (Q4 s=18, merged) and configs[2] (Q6 s=18, merged)
WORKLOADS = [(3, 15, "plain"), (4, 18, "merged"), (6, 18, "merged")]
STEPS = 100
APPLIES = 50
MODES = ("default", "deterministic")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def apply_ms(ctx, src, dst):
    import torch
    st = torch.cuda.ExternalStream(ctx.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(APPLIES):
        ctx.vmult(dst, src)
    e1.record(st)
    e1.synchronize()
    return e0.elapsed_time(e1) / APPLIES


def solve_ms(prob, ctx):
    ctx.synchronize()
    t0 = time.perf_counter()
    _, it = prob.run_cg_solver(want_x=False)
    ctx.synchronize()
    assert it == STEPS, it
    return 1e3 * (time.perf_counter() - t0) / it


def stats(ms):
    ms = np.array(ms)
    return {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())}


def run(p, s, kind, repeats):
    from mf_data_locality_b200 import capi, host
    probs, ctxs, vecs = {}, {}, {}
    for mode in MODES:
        for name in (kind, kind + "_device"):
            pr = host.Problem(p, s, plugin=name, device=0, deterministic=mode == "deterministic")
            pr.set_solver(STEPS, 0.0, 0.0)
            probs[mode, name] = pr
            ctxs[mode, name] = capi.Context.from_handle(pr.ctx_handle(), p, pr.n_cells, pr.n_owned, pr.n_ghost)
        ctx = ctxs[mode, kind]
        v = np.random.default_rng(1).standard_normal(ctx.n_owned)
        vecs[mode] = (ctx.vector(data=v), ctx.vector())
    n_dofs = probs["default", kind].n_dofs
    on, n_colors, _ = ctxs["deterministic", kind].deterministic_info()
    assert on and not ctxs["default", kind].deterministic_info()[0]
    for key in probs:                                         # warm-up: modules, pools, the graphs
        solve_ms(probs[key], ctxs[key])
    for mode in MODES:
        apply_ms(ctxs[mode, kind], *vecs[mode])
    t_apply = {mode: [] for mode in MODES}
    t_solve = {key: [] for key in probs}
    for _ in range(repeats):
        for mode in MODES:
            t_apply[mode].append(apply_ms(ctxs[mode, kind], *vecs[mode]))
            for name in (kind, kind + "_device"):
                t_solve[mode, name].append(solve_ms(probs[mode, name], ctxs[mode, name]))
    xs = [probs["deterministic", kind + "_device"].run_cg_solver()[0] for _ in range(2)]
    for mode in MODES:
        for v in vecs[mode]:
            v.free()
    for pr in probs.values():
        pr.close()
    row = {"degree": p, "s": s, "solver": kind, "n_dofs": n_dofs, "n_colors": n_colors, "repeats": repeats,
           "deterministic_solves_bitwise_equal": bool(np.array_equal(xs[0].view(np.uint64), xs[1].view(np.uint64)))}
    for mode in MODES:
        row[mode] = {"apply_ms": stats(t_apply[mode]),
                     "host_driven_ms_per_it": stats(t_solve[mode, kind]),
                     "device_resident_ms_per_it": stats(t_solve[mode, kind + "_device"])}
    row["cost_median"] = {k: row["deterministic"][k]["median"] / row["default"][k]["median"]
                          for k in ("apply_ms", "host_driven_ms_per_it", "device_resident_ms_per_it")}
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a check of the script)")
    a = ap.parse_args()
    from mf_data_locality_b200 import capi
    if capi.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    work = [(3, 8, "plain"), (4, 7, "merged")] if a.quick else WORKLOADS
    res = {"gpu": gpu_info(),
           "note": "default vs deterministic mode alternated in one process, medians and min/max over the "
                   f"repeats; apply = {APPLIES} operator applies between CUDA events; CG = ms per iteration "
                   f"of {STEPS}-iteration solves (host clock around a synchronised solve)",
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

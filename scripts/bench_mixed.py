"""Mixed-precision against FP64 solves on one B200 (DESIGN.md 4.7).

1. Operator apply: the FP32 cell kernel (bp4_debug_vmult_f32) against the FP64 one (bp4_vmult),
   kernel time from the context's CUDA-event profile (BP4_K_VMULT: the cell loop only, not the
   rounding of the input and the widening of the output the debug hook adds), alternated in one
   process, median [min-max] over the repeats.
2. Time to solution: bp4_solve_cg_mixed against the device-resident bp4_solve_cg_merged to the same
   FP64 tolerance (reduce 1e-8 and 1e-10, tol 1e-15, max_steps large enough for both), blocking calls
   timed with a host clock (the call ends in a stream synchronisation), alternated in one process.
   Reports the FP64 iterations, the refinement steps and inner FP32 iterations, and the true
   residual |b - A x| / |b| of both results recomputed with the FP64 operator.

The problems are the benchmark's (the C++ host mirror's set-up, merged plugin); every working set is
far larger than the 126 MB L2.

The FP32 tuning choices (Cfg<P, QUAD, float>) and the inner reduction (kMixedInnerReduce) were chosen
by running this script against library builds that differ in one of them only, with --apply / --solve
restricted to the sizes of interest (DESIGN.md 4.7).

usage: python scripts/bench_mixed.py [--repeats N] [--out FILE] [--quick] [--apply P,S ...] [--solve P,S ...]
                                     [--reduce R ...]"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

APPLY = [(4, 18), (6, 18), (3, 15)]
SOLVE = [(4, 18), (3, 15)]
REDUCE = [1e-8, 1e-10]
APPLIES = 20


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v)}


def setup(p, s):
    from mf_data_locality_b200 import capi, host
    prob = host.Problem(p, s, plugin="merged", device=0)
    ctx = capi.Context.from_handle(prob.ctx_handle(), p, prob.n_cells, prob.n_owned, prob.n_ghost)
    return prob, ctx


def apply_ms(ctx, f, dst, src):
    """mean cell-kernel time of APPLIES calls of f (event-timed BP4_K_VMULT)"""
    from mf_data_locality_b200 import capi
    ctx.profile_reset()
    ctx.profile_enable(True)
    for _ in range(APPLIES):
        f(dst, src)
    ctx.synchronize()
    ms, n = ctx.profile_get(capi.K_VMULT)
    ctx.profile_enable(False)
    return ms / n


def bench_apply(p, s, repeats):
    prob, ctx = setup(p, s)
    n = prob.n_owned
    src = ctx.vector(data=np.random.default_rng(p).standard_normal(ctx.n_local))
    dst = ctx.vector()
    variants = {"fp64": ctx.vmult, "fp32": ctx.vmult_f32}
    for f in variants.values():                          # warm-up: modules, the float coefficients
        f(dst, src)
    t = {k: [] for k in variants}
    for _ in range(repeats):
        for k, f in variants.items():
            t[k].append(apply_ms(ctx, f, dst, src))
    ctx.vmult(dst, src)
    a64 = dst.download()[:n]
    ctx.vmult_f32(dst, src)
    a32 = dst.download()[:n]
    row = {"degree": p, "s": s, "n_dofs": prob.n_dofs, "repeats": repeats, "applies_per_repeat": APPLIES,
           "fp64_ms": spread(t["fp64"]), "fp32_ms": spread(t["fp32"]),
           "speedup_median": statistics.median(t["fp64"]) / statistics.median(t["fp32"]),
           "fp32_rel_l2_vs_fp64": float(np.linalg.norm(a32 - a64) / np.linalg.norm(a64))}
    for v in (src, dst):
        v.free()
    prob.close()
    return row


def true_rel_residual(ctx, x, b, n):
    ax = ctx.vector()
    ctx.vmult(ax, x)
    bh = b.download()[:n]
    r = float(np.linalg.norm(bh - ax.download()[:n]) / np.linalg.norm(bh))
    ax.free()
    return r


def bench_solve(p, s, repeats):
    from mf_data_locality_b200 import capi
    prob, ctx = setup(p, s)
    n = prob.n_owned
    b = ctx.vector(data=prob.rhs())
    prec = ctx.inverse_diagonal()
    x = ctx.vector()
    rows = []
    for reduce in REDUCE:
        def merged():
            return ctx.solve_cg(x, b, prec, merged=True, max_steps=20000, tol=1e-15, reduce=reduce)

        def mixed():
            return ctx.solve_cg_mixed(x, b, prec, max_steps=40000, tol=1e-15, reduce=reduce)

        variants = {"fp64_merged": merged, "mixed": mixed}
        out = {}
        for k, f in variants.items():                    # warm-up: the graphs
            x.zero()
            out[k] = f()
        t = {k: [] for k in variants}
        res = {}
        for _ in range(repeats):
            for k, f in variants.items():
                x.zero()
                ctx.synchronize()
                t0 = time.perf_counter()
                out[k] = f()
                t[k].append((time.perf_counter() - t0) * 1e3)
                assert out[k][0] == capi.SUCCESS, (k, out[k])
                res[k] = true_rel_residual(ctx, x, b, n)
        row = {"degree": p, "s": s, "n_dofs": prob.n_dofs, "reduce": reduce, "repeats": repeats,
               "fp64_merged_ms": spread(t["fp64_merged"]), "mixed_ms": spread(t["mixed"]),
               "speedup_median": statistics.median(t["fp64_merged"]) / statistics.median(t["mixed"]),
               "fp64_iterations": out["fp64_merged"][1], "mixed_refinements": out["mixed"][1],
               "mixed_inner_iterations": out["mixed"][2],
               "true_rel_residual": {k: res[k] for k in variants}}
        print(json.dumps(row), flush=True)
        rows.append(row)
    for v in (b, prec, x):
        v.free()
    prob.close()
    return rows


def main():
    global APPLY, SOLVE, REDUCE
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_mixed.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes, for a rehearsal of the script")
    ap.add_argument("--apply", nargs="*", help="operator sizes P,S (default: %s)" % APPLY)
    ap.add_argument("--solve", nargs="*", help="solve sizes P,S (default: %s)" % SOLVE)
    ap.add_argument("--reduce", nargs="*", type=float, help="reduction targets (default: %s)" % REDUCE)
    a = ap.parse_args()
    if a.quick:
        APPLY, SOLVE = [(4, 6), (3, 5)], [(4, 6)]
    pairs = lambda v: [tuple(int(t) for t in x.split(",")) for x in v]
    if a.apply is not None:
        APPLY = pairs(a.apply)
    if a.solve is not None:
        SOLVE = pairs(a.solve)
    if a.reduce is not None:
        REDUCE = a.reduce
    res = {"gpu": gpu_info(), "apply": [], "solve": []}
    for p, s in APPLY:
        row = bench_apply(p, s, a.repeats)
        print(json.dumps(row), flush=True)
        res["apply"].append(row)
    for p, s in SOLVE:
        res["solve"] += bench_solve(p, s, a.repeats)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()

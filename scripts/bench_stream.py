"""The context on the caller's stream and enqueued device-resident solves, on one B200.

  (a) ms per iteration of the host-driven merged CG recurrence (`ITERS` vmult_merged calls, host
      clock around synchronised calls) at Q4 s=18 on wrapped PyTorch tensors, with the context on
      PyTorch's current stream (Context.use_stream: no event pair per call) against the context on
      its own stream (an event pair per call orders it with torch);
  (b) `N_SOLVES` back-to-back device-resident solves of `SOLVE_STEPS` iterations each (tolerances 0)
      at Q3 s=14 (plain) and Q4 s=15 (merged): queued with bp4_solve_cg*_async and one synchronisation
      at the end, against as many blocking bp4_solve_cg* calls.  Total wall time, and host time until
      the last call returns;
  (c) ms per iteration of one `LONG_STEPS`-iteration device-resident merged solve at Q4 s=18, with this
      library and, given --baseline-lib (a libbp4.so built from the parent commit), with that one: the
      hot loop is the same code, so the times should agree within the spread.
The variants of each measurement alternate in one process after a warm-up; every number is the
median and [min, max] over `--repeats`.  The card's name, power limit and maximum SM clock are read
in the same run.

usage: python scripts/bench_stream.py [--repeats N] [--out FILE] [--baseline-lib PATH] [--quick]"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ITERS = 50
N_SOLVES = 20
SOLVE_STEPS = 20
LONG_STEPS = 200


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def stats(v):
    v = np.array(v)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max())}


def merged_ms(ctx, vecs, prec):
    """ITERS iterations of SolverCGFullMerge's recurrence from x = 0, g = -b, d = h = 0"""
    x, g, d, h, b = vecs
    for w in (x, d, h):
        w.zero()
    ctx.equ(g, -1.0, b)
    ctx.synchronize()
    alpha = beta = alpha_old = beta_old = 0.0
    t0 = time.perf_counter()
    for it in range(1, ITERS + 1):
        S = ctx.vmult_merged(x, g, d, h, prec, alpha, beta, alpha_old if it % 2 == 1 else 0.0, beta_old)
        alpha_old, beta_old = alpha, beta
        alpha = S[6] / S[0]
        beta = alpha * (S[4] + alpha * S[5]) / S[6]
    ms = 1e3 * (time.perf_counter() - t0) / ITERS
    assert math.isfinite(alpha) and math.isfinite(beta)
    return ms


def part_a(p, s, repeats):
    import torch
    from mf_data_locality_b200 import capi, host
    prob = host.Problem(p, s, plugin="merged", device=0)
    ctx = capi.Context.from_handle(prob.ctx_handle(), p, prob.n_cells, prob.n_owned, prob.n_ghost)
    nl = ctx.n_local
    rhs = np.zeros(nl)
    rhs[:prob.n_owned] = prob.rhs()
    mk = lambda a: ctx.wrap(torch.tensor(a, device="cuda:0"))   # noqa: E731
    vecs = [mk(np.zeros(nl)) for _ in range(4)] + [mk(rhs)]
    prec = ctx.inverse_diagonal(out=mk(np.zeros(prob.n_owned // 3)))
    cur = torch.cuda.current_stream()
    variants = {"own_stream": None, "current_stream": cur}
    times = {k: [] for k in variants}
    for rep in range(repeats + 1):                          # repeat 0 is the warm-up
        for k, st in variants.items():
            ctx.use_stream(st)
            t = merged_ms(ctx, vecs, prec)
            if rep:
                times[k].append(t)
    ctx.use_stream(None)
    fused = ctx.fused_info()[0]
    for v in vecs + [prec]:
        v.free()
    prob.close()
    res = {"degree": p, "s": s, "n_dofs": prob.n_dofs, "in_loop_updates": bool(fused), "iterations": ITERS,
           "ms_per_it": {k: stats(t) for k, t in times.items()}}
    res["current_minus_own_us"] = 1e3 * (res["ms_per_it"]["current_stream"]["median"] -
                                         res["ms_per_it"]["own_stream"]["median"])
    return res


def part_b(p, s, kind, repeats):
    import torch
    from mf_data_locality_b200 import capi, host
    L = capi.lib()
    merged = kind == "merged"
    prob = host.Problem(p, s, plugin=kind, device=0)
    ctx = capi.Context.from_handle(prob.ctx_handle(), p, prob.n_cells, prob.n_owned, prob.n_ghost)
    x, b = ctx.vector(), ctx.vector()
    b.upload(prob.rhs())
    prec = ctx.inverse_diagonal()
    blocking = L.bp4_solve_cg_merged if merged else L.bp4_solve_cg
    queued = L.bp4_solve_cg_merged_async if merged else L.bp4_solve_cg_async
    res_dev = torch.empty(3 * N_SOLVES, dtype=torch.float64, device="cuda:0")
    one = (C.c_byte * 24)()

    def run(q):
        x.zero()
        ctx.synchronize()
        t0 = time.perf_counter()
        for k in range(N_SOLVES):
            if q:
                rc = queued(ctx.h, x.h, b.h, prec.h, SOLVE_STEPS, 0.0, 0.0, C.c_void_p(res_dev.data_ptr() + 24 * k),
                            None)
            else:
                rc = blocking(ctx.h, x.h, b.h, prec.h, SOLVE_STEPS, 0.0, 0.0, one)
            assert rc == 0, L.bp4_last_error()
        t_host = time.perf_counter() - t0
        ctx.synchronize()
        return 1e3 * (time.perf_counter() - t0), 1e3 * t_host, x.download()[:prob.n_owned]

    times = {"blocking": {"wall": [], "host": []}, "queued": {"wall": [], "host": []}}
    xs = {}
    for rep in range(repeats + 1):
        for k in times:
            wall, h, xk = run(k == "queued")
            xs[k] = xk
            if rep:
                times[k]["wall"].append(wall)
                times[k]["host"].append(h)
    steps = res_dev.view(torch.int32).view(-1, 6)[:, 1].cpu().tolist()
    assert steps == [SOLVE_STEPS] * N_SOLVES, steps
    diff = float(np.linalg.norm(xs["queued"] - xs["blocking"]) / np.linalg.norm(xs["blocking"]))
    for v in (x, b, prec):
        v.free()
    prob.close()
    return {"degree": p, "s": s, "solver": kind, "n_dofs": prob.n_dofs, "solves": N_SOLVES,
            "iterations_per_solve": SOLVE_STEPS,
            "total_ms": {k: stats(t["wall"]) for k, t in times.items()},
            "host_ms_until_last_call_returns": {k: stats(t["host"]) for k, t in times.items()},
            "x_rel_l2_queued_vs_blocking": diff}


def load_baseline(path):
    """another build of libbp4.so, with the argument types the calls of part_c need; capi.Context
    drives it while capi._lib points to it"""
    L = C.CDLL(os.path.abspath(path))
    vp, d = C.c_void_p, C.c_double
    L.bp4_last_error.restype = C.c_char_p
    L.bp4_vec_alloc.argtypes = [vp, C.c_uint64, vp]
    L.bp4_vec_upload.argtypes = [vp, vp, vp, C.c_uint64]
    L.bp4_vec_download.argtypes = [vp, vp, vp, C.c_uint64]
    L.bp4_solve_cg_merged.argtypes = [vp, vp, vp, vp, C.c_uint, d, d, vp]
    return L


def part_c(p, s, repeats, baseline):
    from mf_data_locality_b200 import capi, host
    prob = host.Problem(p, s, plugin="merged", device=0)
    rc, rp = prob.ranges()
    arrays = (prob.entity_index(), prob.vertices(), prob.n_owned, prob.n_ghost, prob.constrained())
    rhs = prob.rhs()
    libs = {"this": capi.lib()}
    if baseline:
        libs["parent"] = load_baseline(baseline)
    setups = {}
    for name, lb in libs.items():
        capi._lib = lb
        ctx = capi.Context(p, *arrays, ranges=(rc, rp))
        setups[name] = (ctx, ctx.vector(), ctx.vector(data=np.concatenate([rhs, np.zeros(prob.n_ghost)])),
                        ctx.inverse_diagonal())
    times = {k: [] for k in libs}
    results = {}
    for rep in range(repeats + 1):
        for name, (ctx, x, b, pr) in setups.items():
            capi._lib = libs[name]
            x.zero()
            ctx.synchronize()
            t0 = time.perf_counter()
            r = ctx.solve_cg(x, b, pr, merged=True, max_steps=LONG_STEPS, tol=0.0, reduce=0.0)
            t = time.perf_counter() - t0
            assert r[1] == LONG_STEPS, r
            results[name] = r
            if rep:
                times[name].append(1e3 * t / LONG_STEPS)
    fused = {}
    for name, (ctx, x, b, pr) in setups.items():
        capi._lib = libs[name]
        fused[name] = ctx.fused_info()[0]
        for v in (x, b, pr):
            v.free()
        ctx.close()
    capi._lib = libs["this"]
    prob.close()
    out = {"degree": p, "s": s, "n_dofs": prob.n_dofs, "iterations": LONG_STEPS, "in_loop_updates": fused,
           "ms_per_it": {k: stats(t) for k, t in times.items()}}
    if "parent" not in libs:
        out["ms_per_it"]["parent"] = "not measured (no --baseline-lib)"
    else:
        out["last_value_rel_diff"] = abs(results["this"][2] - results["parent"][2]) / abs(results["parent"][2])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    ap.add_argument("--baseline-lib", default=None, help="libbp4.so of the parent commit for (c)")
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script)")
    a = ap.parse_args()
    from mf_data_locality_b200 import capi
    if capi.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    big, b_plain, b_merged = ((4, 7), (3, 6), (4, 6)) if a.quick else ((4, 18), (3, 14), (4, 15))
    res = {"gpu": gpu_info(), "repeats": a.repeats,
           "note": "variants alternated in one process after a warm-up; median and [min, max] over the repeats. "
                   "(a) host clock around synchronised host-driven merged iterations on wrapped tensors; "
                   "(b) host clock, from the first call to the synchronisation after the last solve (total) "
                   "and until the last call returned (host); (c) host clock around one blocking solve / "
                   "iterations"}
    res["a_wrapped_merged_iteration"] = part_a(*big, a.repeats)
    print(json.dumps(res["a_wrapped_merged_iteration"]), flush=True)
    res["b_back_to_back_solves"] = [part_b(*b_plain, "plain", a.repeats), part_b(*b_merged, "merged", a.repeats)]
    print(json.dumps(res["b_back_to_back_solves"]), flush=True)
    res["c_long_device_solve"] = part_c(*big, a.repeats, a.baseline_lib)
    print(json.dumps(res["c_long_device_solve"]), flush=True)
    text = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()

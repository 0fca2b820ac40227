"""Wrapped PyTorch tensors (capi.Context.wrap, bp4_vec_wrap) against the context's own vectors on one
B200, at Q4 s=18 with the merged plugin's context (in-loop vector updates, the default there).

  1. ms per operator apply (`APPLIES` applies between two CUDA events on the context's stream) and ms
     per iteration of the host-driven merged CG recurrence (`ITERS` vmult_merged calls, host clock
     around synchronised calls), on wrapped and on owned vectors, alternated `--repeats` times;
  2. end to end, from a CUDA tensor to a CUDA tensor holding A src: wrap + apply + free, against
     download to the host + upload + apply + download + copy back to the device (host clock, each
     ending in a device synchronise);
  3. host cost of one wrap + free: the C entry points alone, and capi.Context.wrap + Vector.free.
Reports medians and the min/max spread, the card's name and power limit, and the difference
between the applies on wrapped and owned vectors.

usage: python scripts/bench_vec_wrap.py [--repeats N] [--out FILE] [--quick]"""
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

APPLIES = 50
ITERS = 50
WRAPS = 2000


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def stats(ms):
    ms = np.array(ms)
    return {"median": float(np.median(ms)), "min": float(ms.min()), "max": float(ms.max())}


def apply_ms(ctx, dst, src):
    import torch
    st = ctx.torch_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(APPLIES):
        ctx.vmult(dst, src)
    e1.record(st)
    e1.synchronize()
    return e0.elapsed_time(e1) / APPLIES


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


def end_to_end_ms(ctx, src_t, dst_t, own):
    """A src_t into dst_t (CUDA tensors): wrap/apply/free, or through the host with owned vectors"""
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if own is None:
        s, d = ctx.wrap(src_t), ctx.wrap(dst_t)
        ctx.vmult(d, s)
        s.free()
        d.free()
    else:
        own[0].upload(src_t.cpu().numpy())
        ctx.vmult(own[1], own[0])
        dst_t.copy_(torch.from_numpy(own[1].download()))
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0)


def wrap_us(ctx, t):
    from mf_data_locality_b200 import capi
    L, h, n, p = capi.lib(), C.c_void_p(), C.c_uint64(t.numel()), C.c_void_p(t.data_ptr())
    t0 = time.perf_counter()
    for _ in range(WRAPS):
        L.bp4_vec_wrap(ctx.h, p, n, C.byref(h))
        L.bp4_vec_free(ctx.h, h)
    c_abi = 1e6 * (time.perf_counter() - t0) / WRAPS
    t0 = time.perf_counter()
    for _ in range(WRAPS):
        ctx.wrap(t).free()
    python = 1e6 * (time.perf_counter() - t0) / WRAPS
    return c_abi, python


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small size (a check of the script)")
    a = ap.parse_args()
    import torch
    from mf_data_locality_b200 import capi, host
    if capi.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    p, s = (4, 7) if a.quick else (4, 18)
    prob = host.Problem(p, s, plugin="merged", device=0)
    ctx = capi.Context.from_handle(prob.ctx_handle(), p, prob.n_cells, prob.n_owned, prob.n_ghost)
    nl = ctx.n_local
    rng = np.random.default_rng(1)
    v = rng.standard_normal(nl)
    rhs = np.zeros(nl)
    rhs[:prob.n_owned] = prob.rhs()
    prec_own = ctx.inverse_diagonal()
    sets = {}
    for kind in ("owned", "wrapped"):
        mk = (lambda x: ctx.vector(len(x), data=x)) if kind == "owned" else \
             (lambda x: ctx.wrap(torch.tensor(x, device="cuda:0")))
        prec = prec_own if kind == "owned" else ctx.inverse_diagonal(out=mk(np.zeros(prob.n_owned // 3)))
        sets[kind] = {"apply": (mk(np.zeros(nl)), mk(v)), "merged": [mk(np.zeros(nl)) for _ in range(4)] + [mk(rhs)],
                      "prec": prec}
    fused = ctx.fused_info()[0]
    src_t = torch.tensor(v, device="cuda:0")
    dst_t = torch.zeros(nl, dtype=torch.float64, device="cuda:0")
    own = (ctx.vector(), ctx.vector())
    # warm-up of every path
    for kind in sets:
        apply_ms(ctx, *sets[kind]["apply"])
        merged_ms(ctx, sets[kind]["merged"], sets[kind]["prec"])
    for o in (None, own):
        end_to_end_ms(ctx, src_t, dst_t, o)
    t_apply = {k: [] for k in sets}
    t_merged = {k: [] for k in sets}
    t_e2e = {"wrap": [], "host_round_trip": []}
    for _ in range(a.repeats):
        for kind in sets:
            t_apply[kind].append(apply_ms(ctx, *sets[kind]["apply"]))
            t_merged[kind].append(merged_ms(ctx, sets[kind]["merged"], sets[kind]["prec"]))
        t_e2e["wrap"].append(end_to_end_ms(ctx, src_t, dst_t, None))
        t_e2e["host_round_trip"].append(end_to_end_ms(ctx, src_t, dst_t, own))
    wr = [wrap_us(ctx, src_t) for _ in range(a.repeats)]
    got = sets["wrapped"]["apply"][0].tensor.cpu().numpy()
    want = sets["owned"]["apply"][0].download()
    rel = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    res = {"gpu": gpu_info(), "degree": p, "s": s, "n_dofs": prob.n_dofs, "vector_mb": 8 * nl / 1e6,
           "in_loop_updates": bool(fused), "repeats": a.repeats,
           "note": f"owned vs wrapped alternated in one process, medians and min/max over the repeats; apply = "
                   f"{APPLIES} applies between CUDA events; merged = ms per iteration of {ITERS} host-driven "
                   f"vmult_merged iterations (host clock); end_to_end = host clock from a CUDA tensor to a CUDA "
                   f"tensor holding A src, synchronised; wrap_free_us = host cost of one wrap + free over "
                   f"{WRAPS} pairs",
           "apply_ms": {k: stats(t) for k, t in t_apply.items()},
           "merged_ms_per_it": {k: stats(t) for k, t in t_merged.items()},
           "end_to_end_ms": {k: stats(t) for k, t in t_e2e.items()},
           "wrap_free_us": {"c_abi": stats([w[0] for w in wr]), "capi_python": stats([w[1] for w in wr])},
           "apply_wrapped_vs_owned_rel_l2": rel}
    for kind in sets:
        for vv in list(sets[kind]["apply"]) + sets[kind]["merged"] + [sets[kind]["prec"]]:
            vv.free()
    for vv in own:
        vv.free()
    prob.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

"""The mixed-precision solve (bp4_solve_cg_mixed, Context.solve_cg_mixed) and its FP32 operator
(bp4_debug_vmult_f32): the FP32 apply against the FP64 oracle, the FP64 stopping test on the true
residual recomputed with the FP64 operator, the agreement with the FP64 merged solve, the step-0 and
budget rules, the history, the enqueued form, launch counts, wrapped tensors and the refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bp4_oracle as O

from helpers import make_ctx, rel_l2, single

pytestmark = pytest.mark.gpu

F64 = torch.float64


def _prec(rd):
    return O.finish_inverse_diagonal(O.inverse_diagonal(rd))


def _setup(p, s, quadratic=False):
    rd = O.build_problem(p, s, quadratic=True)[0] if quadratic else single(p, s)[0]
    ctx = make_ctx(rd)
    vp = ctx.vector(rd.n_owned // 3, data=_prec(rd))
    return rd, ctx, vp


def _true_residual(ctx, rd, x, b):
    """|b - A x| with the FP64 operator, the difference and the norm on the host"""
    ax = ctx.vector()
    ctx.vmult(ax, ctx.vector(data=x))
    return float(np.linalg.norm(b - ax.download()[:rd.n_owned]))


F32_CASES = [pytest.param(p, s, q, id=f"Q{p}-{'quadratic' if q else 'trilinear'}")
             for p, s in [(2, 6), (3, 5), (4, 4), (5, 4), (6, 3), (7, 3), (8, 3)] for q in (False, True)]


@pytest.mark.parametrize("p,s,quadratic", F32_CASES)
def test_vmult_f32_matches_fp64_oracle(p, s, quadratic, bp4_lib):
    rd, ctx, _ = _setup(p, s, quadratic)
    v = np.random.default_rng(10 * p + s).standard_normal(rd.n_owned)
    dst = ctx.vector()
    ctx.vmult_f32(dst, ctx.vector(data=v))
    got = dst.download()[:rd.n_owned]
    want = O.vmult(rd, O.make_tables(p), v)
    assert rel_l2(got, want) <= 1e-5
    # constrained rows are the identity (of the input rounded to float)
    v32 = v.astype(np.float32).astype(np.float64)
    assert np.array_equal(got[rd.constrained], v32[rd.constrained])
    ctx.close()


SOLVE_CASES = [(2, 8), (3, 6), (4, 5), (6, 3), (8, 3)]


@pytest.mark.parametrize("p,s", SOLVE_CASES)
def test_mixed_reaches_the_fp64_tolerance(p, s, bp4_lib):
    """the true residual recomputed with the FP64 operator passes max(tol, reduce |r0|), and x agrees
    with the FP64 merged solve run to the same tolerance"""
    from mf_data_locality_b200 import capi
    rd, ctx, vp = _setup(p, s)
    vb = ctx.vector(data=rd.rhs)
    for reduce in (1e-8, 1e-10):
        x = ctx.vector()
        state, ref, inner, last, init = ctx.solve_cg_mixed(x, vb, vp, max_steps=5000, reduce=reduce)
        assert state == capi.SUCCESS, (state, ref, inner, last, init)
        assert init == pytest.approx(np.linalg.norm(rd.rhs), rel=1e-12)
        bound = max(1e-15, reduce * init)
        xm = x.download()[:rd.n_owned]
        res = _true_residual(ctx, rd, xm, rd.rhs)
        # (the recomputed residual differs from the solver's by the rounding of A x: ~1e-16 |A x|)
        assert res <= bound * (1 + 1e-3)
        assert res == pytest.approx(last, rel=1e-3)
        assert ref >= 1 and inner >= ref
        x64 = ctx.vector()
        st64, it64, last64, _ = ctx.solve_cg(x64, vb, vp, merged=True, max_steps=5000, reduce=reduce)
        assert st64 == capi.SUCCESS
        assert rel_l2(xm, x64.download()[:rd.n_owned]) <= 1e5 * reduce
    ctx.close()


def test_nonzero_start_zero_rhs_and_budget(bp4_lib):
    from mf_data_locality_b200 import capi
    rd, ctx, vp = _setup(4, 5)
    n = rd.n_owned
    vb = ctx.vector(data=rd.rhs)
    x0 = 0.1 * np.random.default_rng(3).standard_normal(n)
    x0[rd.constrained] = 0.0
    # a nonzero start vector: step 0 checks |b - A x0|
    x = ctx.vector(data=x0)
    state, ref, inner, last, init = ctx.solve_cg_mixed(x, vb, vp, max_steps=5000, reduce=1e-10)
    assert state == capi.SUCCESS
    assert init == pytest.approx(_true_residual(ctx, rd, x0, rd.rhs), rel=1e-10)
    assert _true_residual(ctx, rd, x.download()[:n], rd.rhs) <= 1e-10 * init * (1 + 1e-3)
    # a zero right-hand side ends at step 0 and leaves x untouched
    zero = ctx.vector()
    x00 = ctx.vector()
    assert ctx.solve_cg_mixed(x00, zero, vp, max_steps=100) == (capi.SUCCESS, 0, 0, 0.0, 0.0)
    assert not x00.download().any()
    # ... and so does max_steps = 0 (failure) on a nonzero one
    x = ctx.vector(data=x0)
    state, ref, inner, _, _ = ctx.solve_cg_mixed(x, vb, vp, max_steps=0)
    assert (state, ref, inner) == (capi.FAILURE, 0, 0)
    assert np.array_equal(x.download()[:n], x0)
    # a budget too small to converge: failure, and never more inner steps than allowed
    for max_steps in (1, 3, 7):
        x = ctx.vector()
        state, ref, inner, last, init = ctx.solve_cg_mixed(x, vb, vp, max_steps=max_steps, reduce=1e-10)
        assert state == capi.FAILURE and inner == max_steps and ref >= 1
    ctx.close()


def test_stagnation_and_nan(bp4_lib):
    """a target below what FP64 can attain ends with state 2 once a refinement step no longer lowers
    the true residual, before the budget is used up, and x holds the last iterate; a NaN residual
    ends the solve at step 0 with state 2 and leaves x untouched"""
    from mf_data_locality_b200 import capi
    rd, ctx, vp = _setup(3, 6)
    n = rd.n_owned
    vb = ctx.vector(data=rd.rhs)
    x = ctx.vector()
    hnd = ctx.solve_cg_mixed(x, vb, vp, max_steps=20000, tol=0.0, reduce=0.0, blocking=False, history=True)
    state, ref, inner, last, init = hnd.result()
    assert state == capi.FAILURE and inner < 20000 and ref >= 2
    hist = hnd.history.cpu().numpy()[:ref + 1]
    assert (np.diff(hist[:-1]) < 0).all() and hist[-1] >= hist[-2]     # the step that did not reduce
    assert last == hist[-1] and last <= 1e-12 * init
    res = _true_residual(ctx, rd, x.download()[:n], rd.rhs)            # x is that last iterate
    assert 0.0 < res <= 1e-12 * init
    # NaN in b: step 0 fails, x stays as it was
    bn = rd.rhs.copy()
    bn[7] = np.nan
    x = ctx.vector()
    state, ref, inner, last, _ = ctx.solve_cg_mixed(x, ctx.vector(data=bn), vp, max_steps=100)
    assert (state, ref, inner) == (capi.FAILURE, 0, 0) and np.isnan(last)
    assert not x.download().any()
    ctx.close()


def test_history_async_and_launches(bp4_lib):
    """history = the true residuals (the first and the last recomputed), the enqueued solve equals
    the blocking one, and a repeated solve adds exactly one launch"""
    from mf_data_locality_b200 import capi
    rd, ctx, vp = _setup(3, 6)
    n = rd.n_owned
    vb = ctx.vector(data=rd.rhs)
    xb = ctx.vector()
    rb = ctx.solve_cg_mixed(xb, vb, vp, max_steps=2000, reduce=1e-10)
    xa = ctx.vector()
    hnd = ctx.solve_cg_mixed(xa, vb, vp, max_steps=2000, reduce=1e-10, blocking=False, history=True)
    ra = hnd.result()
    assert ra[0] == rb[0] == capi.SUCCESS
    # FP32 and FP64 atomics: the same refinement, give or take a step at either end
    assert abs(ra[1] - rb[1]) <= 1 and abs(ra[2] - rb[2]) <= ra[1] + 2
    hist = hnd.history.cpu().numpy()
    ref = ra[1]
    assert hist[0] == ra[4] and hist[ref] == ra[3]
    assert np.isnan(hist[ref + 1:]).all()
    assert (np.diff(hist[:ref + 1]) < 0).all()
    assert hist[0] == pytest.approx(np.linalg.norm(rd.rhs), rel=1e-12)
    assert hist[ref] == pytest.approx(_true_residual(ctx, rd, xa.download()[:n], rd.rhs), rel=1e-3)
    # repeated solves re-use the cached graph: one launch each, whatever the arguments
    x = ctx.vector()
    ctx.solve_cg_mixed(x, vb, vp, max_steps=2000, reduce=1e-8)
    n0 = ctx.launch_count()
    x.zero()
    ctx.solve_cg_mixed(x, vb, vp, max_steps=50, reduce=1e-6)
    assert ctx.launch_count() - n0 == 1
    ctx.close()


def test_async_equals_blocking_bit_for_bit(bp4_lib):
    """on a mesh where every sum the solve forms has at most two terms (two cells, reductions of at
    most two blocks), the FP32 and FP64 atomics give one result in any order: the enqueued solve
    gives the blocking solve's result and x bit for bit"""
    rd, ctx, vp = _setup(3, 1)
    n = rd.n_owned
    rhs = np.random.default_rng(5).standard_normal(n)
    rhs[rd.constrained] = 0.0
    vb = ctx.vector(data=rhs)
    xb = ctx.vector()
    rb = ctx.solve_cg_mixed(xb, vb, vp, max_steps=500, reduce=1e-12)
    xa = ctx.vector()
    ra = ctx.solve_cg_mixed(xa, vb, vp, max_steps=500, reduce=1e-12, blocking=False).result()
    assert ra == rb
    assert np.array_equal(xa.download().view(np.uint64), xb.download().view(np.uint64))
    ctx.close()


def test_wrapped_tensors_on_the_current_stream(bp4_lib):
    """x, b and prec as PyTorch tensors on a non-default current stream, no synchronisation between
    the torch ops and the solve"""
    from mf_data_locality_b200 import capi
    rd, ctx, vp = _setup(4, 5)
    n = rd.n_owned
    xr = ctx.vector()
    want = ctx.solve_cg_mixed(xr, ctx.vector(data=rd.rhs), vp, max_steps=2000, reduce=1e-10)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        b = torch.from_numpy(rd.rhs).to("cuda:0", non_blocking=True) * 1.0
        p = torch.from_numpy(_prec(rd)).to("cuda:0")
        x = torch.zeros(ctx.n_local, dtype=F64, device="cuda:0")
        wx, wb, wp = ctx.wrap(x), ctx.wrap(b), ctx.wrap(p)
        got = ctx.solve_cg_mixed(wx, wb, wp, max_steps=2000, reduce=1e-10, blocking=False).result()
        xs = x[:n].cpu().numpy()
    assert got[0] == want[0] == capi.SUCCESS and abs(got[1] - want[1]) <= 1
    assert _true_residual(ctx, rd, xs, rd.rhs) <= 1e-10 * got[4] * (1 + 1e-3)
    assert rel_l2(xs, xr.download()[:n]) <= 1e-6
    for v in (wx, wb, wp):
        v.free()
    ctx.close()


def test_refusals(bp4_lib):
    from mf_data_locality_b200 import capi
    lib = capi.lib()
    rd = single(3, 5)[0]
    # the deterministic mode has no FP32 path
    det = capi.Context(rd.degree, rd.entity_index, rd.vertices, rd.n_owned, rd.n_ghost, rd.constrained,
                       deterministic=True)
    x, vb = det.vector(), det.vector(data=rd.rhs)
    vp = det.vector(rd.n_owned // 3, data=_prec(rd))
    with pytest.raises(capi.Bp4Error, match="error -4:.*deterministic"):
        det.solve_cg_mixed(x, vb, vp)
    with pytest.raises(capi.Bp4Error, match="error -4:.*deterministic"):
        det.vmult_f32(det.vector(), vb)
    det.close()
    ctx = make_ctx(rd)
    x, vb = ctx.vector(), ctx.vector(data=rd.rhs)
    vp = ctx.vector(rd.n_owned // 3, data=_prec(rd))
    # null result memory, and result / history memory the device cannot write
    assert lib.bp4_solve_cg_mixed_async(ctx.h, x.h, vb.h, vp.h, 10, 1e-15, 1e-8, None, None) == -1
    assert b"null" in lib.bp4_last_error()
    host = np.zeros(16)
    assert lib.bp4_solve_cg_mixed_async(ctx.h, x.h, vb.h, vp.h, 10, 1e-15, 1e-8, C.c_void_p(host.ctypes.data),
                                        None) == -1
    assert b"mapped pinned host memory" in lib.bp4_last_error()
    res = torch.empty(4, dtype=F64, device="cuda:0")
    assert lib.bp4_solve_cg_mixed_async(ctx.h, x.h, vb.h, vp.h, 10, 1e-15, 1e-8, C.c_void_p(res.data_ptr()),
                                        C.c_void_p(host.ctypes.data)) == -1
    assert b"history" in lib.bp4_last_error()
    with pytest.raises(ValueError, match="max_steps"):
        ctx.solve_cg_mixed(x, vb, vp, max_steps=10, blocking=False, history=torch.empty(10, dtype=F64, device="cuda:0"))
    # mapped pinned host memory is accepted
    pinned = torch.empty(4, dtype=F64).pin_memory()
    assert lib.bp4_solve_cg_mixed_async(ctx.h, x.h, vb.h, vp.h, 5, 1e-15, 1e-8, C.c_void_p(pinned.data_ptr()),
                                        None) == 0
    ctx.synchronize()
    ctx.close()

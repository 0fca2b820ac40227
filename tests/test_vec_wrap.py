"""Vectors on caller-owned device memory (bp4_vec_wrap, capi.Context.wrap): every operation gives on
wrapped PyTorch tensors what it gives on the context's own vectors (bit for bit in the deterministic
mode), bad pointers and tensors are refused before anything runs, the in-loop updates never read past
a vector's end, the tensors outlive their handles and the context, the device-solve cache stays flat,
and the calls are ordered with PyTorch's current stream without a synchronisation."""
import contextlib
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bp4_oracle as O

from helpers import gpu_cg_merged, gpu_cg_plain, make_ctx, rel_l2, single

F64 = torch.float64


def _ctx(rd, deterministic=False):
    from mf_data_locality_b200 import capi
    return capi.Context(rd.degree, rd.entity_index, rd.vertices, rd.n_owned, rd.n_ghost, rd.constrained,
                        ranges=(rd.range_cell_offset, rd.range_private_offset), coefficients=rd.coefficients,
                        deterministic=deterministic)


def _prec(rd):
    return O.finish_inverse_diagonal(O.inverse_diagonal(rd))


def _tensor(ctx, a):
    return torch.tensor(np.asarray(a, dtype=np.float64), device=f"cuda:{ctx.device}")


def _wrap(ctx, a):
    """a wrapped vector holding a copy of the host array a"""
    return ctx.wrap(_tensor(ctx, a))


def _host(v):
    return v.tensor.cpu().numpy() if v.tensor is not None else v.download()


def _same(a, b, det, tol=1e-12):
    if det:
        return np.array_equal(np.asarray(a).view(np.uint64), np.asarray(b).view(np.uint64))
    return rel_l2(np.asarray(a), np.asarray(b)) <= tol


def _sums_close(a, b, det):
    if det:
        return _same(np.atleast_1d(a), np.atleast_1d(b), True)
    return np.allclose(a, b, rtol=1e-11, atol=0)


@contextlib.contextmanager
def _wrapped_vectors(ctx):
    """ctx.vector() hands out wrapped tensors, so that the host-driven solvers of helpers.py run on them"""
    ctx.vector = lambda n=None, data=None: _wrap(ctx, np.zeros(ctx.n_local if n is None else n)
                                                 if data is None else data)
    try:
        yield
    finally:
        del ctx.vector


class _NoDevice:
    def __getattr__(self, name):
        raise AssertionError(f"{name} called: the tensor check must refuse before any library call")


# ---- without a GPU ----------------------------------------------------------------------------
def test_wrap_exported_and_null_context(bp4_lib):
    from mf_data_locality_b200 import capi
    assert hasattr(bp4_lib, "bp4_vec_wrap") and "bp4_vec_wrap" in capi.EXPORTS
    h = C.c_void_p()
    buf = (C.c_double * 4)()
    assert bp4_lib.bp4_vec_wrap(None, C.cast(buf, C.c_void_p), C.c_uint64(4), C.byref(h)) == -1
    assert b"null" in bp4_lib.bp4_last_error() and not h.value


def test_tensor_check_refuses_cpu_tensor(monkeypatch):
    from mf_data_locality_b200 import capi
    t = torch.zeros(6, dtype=F64)
    with pytest.raises(ValueError, match="cuda"):
        capi.check_tensor(t, 0)
    with pytest.raises(TypeError):
        capi.check_tensor(np.zeros(6), 0)
    monkeypatch.setattr(capi, "_lib", _NoDevice())
    ctx = capi.Context.from_handle(None, 4, 0, 6)
    with pytest.raises(ValueError, match="cuda"):
        ctx.wrap(t)


# ---- parity: wrapped tensors against the context's own vectors ----------------------------------
PARITY = [pytest.param(p, s, det, id=f"Q{p}-s{s}-{'det' if det else 'default'}")
          for p, s in [(2, 6), (3, 5), (4, 6)] for det in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("p,s,det", PARITY)
def test_apply_diagonal_blas1(p, s, det, bp4_lib):
    rd, _ = single(p, s)
    ctx = _ctx(rd, det)
    n, nl = rd.n_owned, rd.n_owned + rd.n_ghost
    rng = np.random.default_rng(p)
    a, b, c = (rng.standard_normal(nl) for _ in range(3))
    diag = rng.standard_normal(n // 3)
    res = {}
    for kind in ("owned", "wrapped"):
        mk = (lambda x: ctx.vector(len(x), data=x)) if kind == "owned" else (lambda x: _wrap(ctx, x))
        va, vb, vc, vd = mk(a), mk(b), mk(c), mk(diag)
        dst, inv = mk(np.zeros(nl)), mk(np.zeros(n // 3))
        r = {}
        ctx.vmult(dst, va)
        r["vmult"] = _host(dst)
        ctx.inverse_diagonal(out=inv)
        r["inverse_diagonal"] = _host(inv)
        ctx.equ(vc, -1.5, va)
        ctx.add(vc, 0.25, vb)
        ctx.sadd(vc, 2.0, -1.0, va)
        r["equ_add_sadd"] = _host(vc)
        r["dot"] = ctx.dot(va, vb)
        r["l2_norm"] = ctx.l2_norm(vc)
        r["add_and_dot"] = ctx.add_and_dot(vc, 0.5, vb, va)
        r["after_add_and_dot"] = _host(vc)
        r["all_zero"] = (ctx.all_zero(va), ctx.all_zero(vc.zero()))
        ctx.jacobi_vmult(dst, va, vd)
        r["jacobi"] = _host(dst)
        ctx.x_finalize_even(vb, va, vc, vd, 0.3, -0.7)
        r["x_finalize_even"] = _host(vb)
        res[kind] = r
    o, w = res["owned"], res["wrapped"]
    for k in ("vmult", "inverse_diagonal", "equ_add_sadd", "after_add_and_dot", "jacobi", "x_finalize_even"):
        assert _same(o[k], w[k], det), k
    for k in ("dot", "l2_norm", "add_and_dot"):
        assert _sums_close(o[k], w[k], det), k
    assert o["all_zero"] == w["all_zero"] == (False, True)
    ctx.close()


MERGED = [pytest.param(p, s, fused, det, id=f"Q{p}-{'inloop' if fused else 'streamed'}-{'det' if det else 'default'}")
          for p, s, fused, det in [(2, 6, False, False), (3, 5, False, False), (4, 6, False, False),
                                   (4, 6, True, False), (2, 6, False, True), (3, 5, False, True),
                                   (4, 6, False, True)]]


@pytest.mark.gpu
@pytest.mark.parametrize("p,s,fused,det", MERGED)
def test_vmult_merged(p, s, fused, det, bp4_lib):
    """all five vectors wrapped, in the three do_cg_update4b regimes; Q4 in-loop is the default form"""
    rd, _ = single(p, s)
    ctx = _ctx(rd, det)
    if p == 4 and not det:
        assert ctx.fused_info()[0] is True          # the fused default at Q4
    if not det:
        ctx.set_fused(fused)
    n, nl = rd.n_owned, rd.n_owned + rd.n_ghost
    prec = _prec(rd)
    rng = np.random.default_rng(p + 10)
    for (alpha, beta, alpha_old, beta_old) in [(0.0, 0.0, 0.0, 0.0), (0.7, 0.3, 0.0, 0.2), (0.7, 0.3, 0.4, 0.2)]:
        x, g, d, h = (rng.standard_normal(nl) for _ in range(4))
        out = {}
        for kind in ("owned", "wrapped"):
            mk = (lambda a: ctx.vector(len(a), data=a)) if kind == "owned" else (lambda a: _wrap(ctx, a))
            vs = [mk(a) for a in (x, g, d, h)]
            vp = mk(prec)
            S = ctx.vmult_merged(*vs, vp, alpha, beta, alpha_old, beta_old)
            out[kind] = (S, [_host(v)[:n] for v in vs])
        assert _sums_close(out["owned"][0], out["wrapped"][0], det)
        for vo, vw in zip(out["owned"][1], out["wrapped"][1]):
            assert _same(vo, vw, det)
    ctx.close()


SOLVES = [pytest.param(p, merged, det, id=f"Q{p}-{'merged' if merged else 'plain'}-{'det' if det else 'default'}")
          for p in (2, 3, 4) for merged in (True, False) for det in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("p,merged,det", SOLVES)
def test_solves(p, merged, det, bp4_lib):
    """host-driven and device-resident solves with x, b, prec (and the host-driven temporaries) wrapped"""
    from mf_data_locality_b200 import capi
    rd, _ = single(p, 6)
    ctx = _ctx(rd, det)
    prec = _prec(rd)
    host_cg = gpu_cg_merged if merged else gpu_cg_plain
    n = rd.n_owned
    for max_steps in (3, 100):
        ctl_o = O.ReductionControl(max_steps, 1e-15, 1e-8)
        xo = host_cg(ctx, rd.rhs, ctx.vector(n // 3, data=prec), ctl_o).download()[:n]
        ctl_w = O.ReductionControl(max_steps, 1e-15, 1e-8)
        with _wrapped_vectors(ctx):
            xw = host_cg(ctx, rd.rhs, ctx.vector(n // 3, data=prec), ctl_w)
        assert xw.tensor is not None
        xw = _host(xw)[:n]
        if det:
            assert ctl_o.last_step == ctl_w.last_step and _same(xo, xw, True)
        else:
            assert abs(ctl_o.last_step - ctl_w.last_step) <= 1 and rel_l2(xw, xo) <= 1e-8
        # device-resident
        x_own = ctx.vector()
        r_o = ctx.solve_cg(x_own, ctx.vector(data=rd.rhs), ctx.vector(n // 3, data=prec), merged=merged,
                           max_steps=max_steps)
        xw, bw, pw = _wrap(ctx, np.zeros(ctx.n_local)), _wrap(ctx, rd.rhs), _wrap(ctx, prec)
        r_w = ctx.solve_cg(xw, bw, pw, merged=merged, max_steps=max_steps)
        if max_steps < 100:
            assert r_o[0] == r_w[0] == capi.FAILURE and r_o[1] == r_w[1] == max_steps
            assert r_w[2] == pytest.approx(r_o[2], rel=1e-10)
            assert _same(x_own.download()[:n], _host(xw)[:n], det)
        elif det:
            assert r_o[:3] == r_w[:3] and _same(x_own.download()[:n], _host(xw)[:n], True)
        else:
            assert abs(r_o[1] - r_w[1]) <= 1 and rel_l2(_host(xw)[:n], x_own.download()[:n]) <= 1e-8
        for v in (xw, bw, pw):
            v.free()
    ctx.close()


# ---- in-loop runs that reach the end of the vector ------------------------------------------------
def _one_cell_q2(private_end):
    """one Q2 cell, one DoF node per entity (entity a -> node a), no constrained DoFs, one range"""
    from mf_data_locality_b200 import capi
    ei = (3 * np.arange(27, dtype=np.uint32)).reshape(1, 27)
    vt = np.array([[x, y, z] for z in (0., 1.) for y in (0., 1.) for x in (0., 1.)]).reshape(1, 8, 3)
    return capi.Context(2, ei, vt, 81, 0, None, ranges=([0, 1], [0, private_end]))


@pytest.mark.gpu
def test_private_runs_stop_before_the_end(bp4_lib):
    """a private run ending at n_owned would make the in-loop jobs read one element (and one prec
    entry) past the end: such a context streams the updates (n_private = 0); a run ending a node
    earlier keeps them, and the oracle meshes keep n_private = group_sizes[0] < n_owned"""
    from mf_data_locality_b200 import capi
    ctx = _one_cell_q2(81)
    assert ctx.fused_info()[1] == 0
    with pytest.raises(capi.Bp4Error):
        ctx.set_fused(True)
    ctx.close()
    ctx = _one_cell_q2(75)                          # odd end: the last piece reaches index 75 < 81
    assert ctx.fused_info()[1] == 75
    ctx.set_fused(True)
    rng = np.random.default_rng(5)
    x, g, d, h = (rng.standard_normal(81) for _ in range(4))
    prec = rng.uniform(0.5, 1.5, 27)
    out = []
    for mk in ((lambda a: ctx.vector(len(a), data=a)), (lambda a: _wrap(ctx, a))):
        vs = [mk(a) for a in (x, g, d, h)]
        S = ctx.vmult_merged(*vs, mk(prec), 0.7, 0.3, 0.4, 0.2)
        out.append((S, [_host(v) for v in vs]))
    np.testing.assert_allclose(out[1][0], out[0][0], rtol=1e-11)
    for vo, vw in zip(out[0][1], out[1][1]):
        assert rel_l2(vw, vo) <= 1e-12
    ctx.close()
    for p, s in [(2, 6), (3, 5), (4, 6)]:
        rd, _ = single(p, s)
        ctx = make_ctx(rd)
        assert ctx.fused_info()[1] == rd.group_sizes[0] < rd.n_owned
        ctx.close()


# ---- refusals ------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals(bp4_lib, monkeypatch):
    from mf_data_locality_b200 import capi
    rd, co = single(3, 5)
    ctx = make_ctx(rd)
    nl = ctx.n_local
    h = C.c_void_p()
    host = np.zeros(nl + 2)
    hp = host.ctypes.data + (-host.ctypes.data) % 16
    assert bp4_lib.bp4_vec_wrap(ctx.h, C.c_void_p(hp), C.c_uint64(nl), C.byref(h)) == -1
    assert b"device memory" in bp4_lib.bp4_last_error() and not h.value
    t = torch.zeros(nl + 2, dtype=F64, device="cuda:0")
    assert bp4_lib.bp4_vec_wrap(ctx.h, C.c_void_p(t.data_ptr() + 8), C.c_uint64(nl), C.byref(h)) == -1
    assert b"aligned" in bp4_lib.bp4_last_error() and not h.value
    assert bp4_lib.bp4_vec_wrap(ctx.h, None, C.c_uint64(nl), C.byref(h)) == -1
    # the context keeps working
    w = np.random.default_rng(1).standard_normal(rd.n_owned)
    src, dst = _wrap(ctx, w), _wrap(ctx, np.zeros(nl))
    ctx.vmult(dst, src)
    assert rel_l2(_host(dst), co.vmult(w)) <= 1e-12
    # the length checks apply to wrapped vectors as to owned ones
    short = ctx.wrap(torch.zeros(nl - 3, dtype=F64, device="cuda:0"))
    with pytest.raises(capi.Bp4Error, match="n_owned"):
        ctx.vmult(dst, short)
    # tensors the context cannot view are refused in Python, before any library call
    base = torch.zeros(2 * nl, dtype=F64, device="cuda:0")
    monkeypatch.setattr(capi, "_lib", _NoDevice())
    with pytest.raises(ValueError, match="float64"):
        ctx.wrap(torch.zeros(nl, dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError, match="contiguous"):
        ctx.wrap(base[::2])
    with pytest.raises(ValueError, match="aligned"):
        ctx.wrap(base[1:])
    monkeypatch.undo()
    ctx.close()


# ---- lifetime and memory -------------------------------------------------------------------------
@pytest.mark.gpu
def test_tensor_outlives_handle_and_context(bp4_lib):
    rd, co = single(3, 5)
    w = np.random.default_rng(2).standard_normal(rd.n_owned)
    want = co.vmult(w)
    ctx = make_ctx(rd)
    ts, td = _tensor(ctx, w), torch.zeros(ctx.n_local, dtype=F64, device="cuda:0")
    src, dst = ctx.wrap(ts), ctx.wrap(td)
    ctx.vmult(dst, src)
    src.free()
    dst.free()
    assert np.array_equal(ts.cpu().numpy(), w)
    assert rel_l2(td.cpu().numpy()[:rd.n_owned], want) <= 1e-12
    td2 = td * 2.0
    assert rel_l2(td2.cpu().numpy()[:rd.n_owned], 2 * want) <= 1e-12
    # the context goes first, the wrapped vectors are still live
    ctx = make_ctx(rd)
    ts, td = _tensor(ctx, w), torch.zeros(ctx.n_local, dtype=F64, device="cuda:0")
    src, dst = ctx.wrap(ts), ctx.wrap(td)
    ctx.vmult(dst, src)
    ctx.close()
    assert np.array_equal(ts.cpu().numpy(), w)
    assert rel_l2(td.cpu().numpy()[:rd.n_owned], want) <= 1e-12
    td.mul_(3.0)
    assert rel_l2(td.cpu().numpy()[:rd.n_owned], 3 * want) <= 1e-12
    src.free()
    dst.free()
    del ts, td
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_solve_cache_stays_flat(bp4_lib):
    """ten device-resident solves, each on a freshly wrapped x at a new address: device memory after
    the tenth is within one vector of what it was after the first (each cached solve holds three
    vectors of temporaries, so one cache entry per address would grow by 27 vectors)"""
    from mf_data_locality_b200 import capi, host
    prob = host.Problem(4, 20, plugin="merged", device=0)
    ctx = capi.Context.from_handle(prob.ctx_handle(), 4, prob.n_cells, prob.n_owned, prob.n_ghost)
    nl = ctx.n_local
    stride = nl + (nl & 1)                          # 16-byte aligned slices
    big = torch.zeros(10 * stride, dtype=F64, device="cuda:0")
    b = _wrap(ctx, prob.rhs())
    prec = ctx.inverse_diagonal()
    free = []
    for i in range(10):
        x = ctx.wrap(big[i * stride:i * stride + nl])
        state, it, _, _ = ctx.solve_cg(x, b, prec, merged=True, max_steps=5)
        assert it == 5
        x.free()
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info(0)[0])
    assert abs(free[-1] - free[0]) <= 8 * nl, [(f - free[0]) / (8 * nl) for f in free]
    b.free()
    prec.free()
    prob.close()


# ---- stream order ----------------------------------------------------------------------------------
def _slow_fill(t, values, heavy):
    """t = values, written by a kernel queued behind a long matrix product (0 * a finite number)"""
    t.copy_(values + 0.0 * (heavy @ heavy)[0, 0])


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["vmult", "vmult_merged"])
def test_ordered_with_the_current_stream(op, bp4_lib):
    """on a non-default stream, torch fills the inputs, the context computes, torch reads the
    outputs, with no synchronisation in between: the same bits as the synchronised run"""
    rd, _ = single(4, 6)
    ctx = _ctx(rd, deterministic=True)
    nl, n = ctx.n_local, rd.n_owned
    rng = np.random.default_rng(7)
    inputs = [torch.tensor(rng.standard_normal(nl), device="cuda:0") for _ in range(4)]
    prec = torch.tensor(_prec(rd), device="cuda:0")
    heavy = torch.rand(4096, 4096, dtype=F64, device="cuda:0")
    torch.cuda.synchronize()

    def run(sync):
        vecs = [torch.full((nl,), float("nan"), dtype=F64, device="cuda:0") for _ in range(4)]
        for t, a in zip(vecs, inputs):
            _slow_fill(t, a, heavy)
            if sync:
                torch.cuda.synchronize()
        wv = [ctx.wrap(t) for t in vecs]
        if op == "vmult":
            out = torch.full((nl,), float("nan"), dtype=F64, device="cuda:0")
            ctx.vmult(ctx.wrap(out), wv[0])
            sums = None
            res = [out]
        else:
            sums = ctx.vmult_merged(*wv, ctx.wrap(prec), 0.7, 0.3, 0.4, 0.2)
            res = vecs
        if sync:
            torch.cuda.synchronize()
        copies = [(r * 1.0) for r in res]          # torch reads the results on the current stream
        return [c.cpu().numpy()[:n] for c in copies], sums

    want, want_s = run(True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got, got_s = run(False)
    for a, b in zip(want, got):
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    if op == "vmult_merged":
        assert np.array_equal(want_s.view(np.uint64), got_s.view(np.uint64))
    ctx.close()

"""The context on the caller's CUDA stream (bp4_ctx_set_stream, Context.use_stream) and device-resident
solves queued without a host synchronisation (bp4_solve_cg*_async, solve_cg(blocking=False)): the same
bits as on the context's own stream and as the blocking solves in the deterministic mode, calls that
return while the stream is still busy, safe switches with pending work, clean refusals, the residual
history of every step, queued solves that build no new graph, and the C++ mirror's replayed
SolverControl history."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bp4_oracle as O

from helpers import gpu_cg_merged, gpu_cg_plain, make_ctx, rel_l2, single

pytestmark = pytest.mark.gpu

F64 = torch.float64
SLEEP = 400_000_000  # GPU clock cycles of torch.cuda._sleep: a fraction of a second


def _ctx(rd, det=True):
    from mf_data_locality_b200 import capi
    return capi.Context(rd.degree, rd.entity_index, rd.vertices, rd.n_owned, rd.n_ghost, rd.constrained,
                        ranges=(rd.range_cell_offset, rd.range_private_offset), coefficients=rd.coefficients,
                        deterministic=det)


def _prec(rd):
    return O.finish_inverse_diagonal(O.inverse_diagonal(rd))


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _workload(ctx, rd, det):
    """every kind of call once, on owned vectors, in whatever stream the context is on"""
    n, nl = rd.n_owned, ctx.n_local
    rng = np.random.default_rng(rd.degree)
    a, b, c = (rng.standard_normal(nl) for _ in range(3))
    prec = _prec(rd)
    va, vb, vc = ctx.vector(data=a), ctx.vector(data=b), ctx.vector(data=c)
    vp = ctx.vector(n // 3, data=prec)
    dst = ctx.vector()
    r = {}
    ctx.vmult(dst, va)
    r["vmult"] = dst.download()
    r["inverse_diagonal"] = ctx.inverse_diagonal().download()
    ctx.equ(vc, -1.5, va)
    ctx.add(vc, 0.25, vb)
    ctx.sadd(vc, 2.0, -1.0, va)
    r["blas1"] = vc.download()
    r["sums"] = [ctx.dot(va, vb), ctx.l2_norm(vc), ctx.add_and_dot(vc, 0.5, vb, va)]
    r["all_zero"] = (ctx.all_zero(va), ctx.all_zero(ctx.vector()))
    ctx.jacobi_vmult(dst, va, vp)
    r["jacobi"] = dst.download()
    for fused in ((False,) if det else (False, True)):
        if not det:
            ctx.set_fused(fused)
        vs = [ctx.vector(data=v) for v in (a, b, c, np.zeros(nl))]
        S = ctx.vmult_merged(*vs, vp, 0.7, 0.3, 0.4, 0.2)
        r[f"merged-{fused}"] = (S, [v.download()[:n] for v in vs])
    for merged in (True, False):
        x = ctx.vector()
        r[f"solve-{merged}"] = (ctx.solve_cg(x, ctx.vector(data=rd.rhs), vp, merged=merged), x.download())
    return r


CASES = [pytest.param(p, s, False, id=f"Q{p}") for p, s in [(2, 6), (3, 5), (4, 6)]] + \
        [pytest.param(3, 5, True, id="Q3-quadratic")]


@pytest.mark.parametrize("p,s,quadratic", CASES)
def test_caller_stream_gives_the_same_bits(p, s, quadratic, bp4_lib):
    """deterministic mode: every call on a torch stream (and on the legacy default stream) gives the
    bits it gives on the context's own stream"""
    rd = O.build_problem(p, s, quadratic=True)[0] if quadratic else single(p, s)[0]
    ctx = _ctx(rd)
    want = _workload(ctx, rd, True)
    for stream in (torch.cuda.Stream(), torch.cuda.default_stream()):
        ctx.use_stream(stream)
        assert ctx.stream() == (stream.cuda_stream or 1)
        with torch.cuda.stream(stream):
            got = _workload(ctx, rd, True)
        for k, w in want.items():
            if k.startswith("merged"):
                assert _same(w[0], got[k][0]) and all(_same(a, b) for a, b in zip(w[1], got[k][1])), k
            elif k.startswith("solve"):
                assert w[0] == got[k][0] and _same(w[1], got[k][1]), k
            elif k == "all_zero":
                assert w == got[k] == (False, True)
            else:
                assert _same(w, got[k]), k
    ctx.use_stream(None)
    ctx.close()


def test_in_loop_merged_on_caller_stream(bp4_lib):
    """the in-loop form (default at Q4, per-block atomics): the same results up to summation order"""
    rd, _ = single(4, 6)
    ctx = _ctx(rd, det=False)
    want = _workload(ctx, rd, False)
    s = torch.cuda.Stream()
    ctx.use_stream(s)
    with torch.cuda.stream(s):
        got = _workload(ctx, rd, False)
    for fused in (False, True):
        (sw, vw), (sg, vg) = want[f"merged-{fused}"], got[f"merged-{fused}"]
        np.testing.assert_allclose(sg, sw, rtol=1e-11)
        assert all(rel_l2(a, b) <= 1e-12 for a, b in zip(vg, vw))
    ctx.close()


def test_returns_while_the_stream_is_busy(bp4_lib, monkeypatch):
    """a wrapped vmult queued behind a long kernel on the caller's stream returns before the stream
    drains, with no event pair between the streams, and is right once it has drained"""
    rd, co = single(3, 5)
    ctx = make_ctx(rd)
    w = np.random.default_rng(3).standard_normal(rd.n_owned)
    ready = torch.tensor(np.concatenate([w, np.zeros(rd.n_ghost)]), dtype=F64, device="cuda:0")
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    ctx.use_stream(s)

    def no_event(*a, **k):
        raise AssertionError("wait_stream called on a context bound to the current stream")

    with torch.cuda.stream(s):
        src = torch.empty(ctx.n_local, dtype=F64, device="cuda:0")
        dst = torch.full((ctx.n_local,), float("nan"), dtype=F64, device="cuda:0")
        torch.cuda._sleep(SLEEP)
        src.copy_(ready)
        monkeypatch.setattr(torch.cuda.Stream, "wait_stream", no_event)
        vs, vd = ctx.wrap(src), ctx.wrap(dst)
        ctx.vmult(vd, vs)
        busy = not s.query()
        monkeypatch.undo()
    assert busy
    s.synchronize()
    assert rel_l2(dst.cpu().numpy()[:rd.n_owned], co.vmult(w)) <= 1e-12
    assert isinstance(ctx.torch_stream(), torch.cuda.Stream) and ctx.torch_stream() is s
    vs.free()
    vd.free()
    ctx.close()


def test_switch_with_pending_work_and_destroy(bp4_lib):
    """work queued on stream A, switch to B, free a pooled vector and take its buffer again on B:
    B waits for A on the device, so both results are right.  Destroying the context leaves the
    caller's streams working."""
    rd, co = single(3, 5)
    ctx = make_ctx(rd)
    rng = np.random.default_rng(4)
    w1, w2 = rng.standard_normal(rd.n_owned), rng.standard_normal(rd.n_owned)
    src1, src2 = ctx.vector(data=w1), ctx.vector(data=w2)
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    ctx.use_stream(a)
    with torch.cuda.stream(a):
        torch.cuda._sleep(SLEEP)
    tmp = ctx.vector()                      # zeroed on A, behind the sleep
    ctx.vmult(tmp, src1)
    out1 = ctx.vector()
    ctx.equ(out1, 1.0, tmp)
    ctx.use_stream(b)
    assert not a.query()                    # the switch did not wait on the host
    tmp.free()
    tmp2 = ctx.vector()                     # the pooled buffer of tmp, zeroed on B
    ctx.vmult(tmp2, src2)
    assert rel_l2(out1.download()[:rd.n_owned], co.vmult(w1)) <= 1e-12
    assert rel_l2(tmp2.download()[:rd.n_owned], co.vmult(w2)) <= 1e-12
    ctx.use_stream(a)
    ctx.vmult(tmp2, src1)
    ctx.close()
    for st in (a, b):
        with torch.cuda.stream(st):
            t = torch.arange(8, dtype=F64, device="cuda:0") * 2.0
        st.synchronize()
        assert t.cpu().tolist() == [2.0 * i for i in range(8)]


def test_refusals(bp4_lib):
    from mf_data_locality_b200 import capi
    lib = capi.lib()
    rd, co = single(3, 5)
    ctx = make_ctx(rd)
    x, vb = ctx.vector(), ctx.vector(data=rd.rhs)
    vp = ctx.vector(rd.n_owned // 3, data=_prec(rd))
    # a stream of another device
    if torch.cuda.device_count() > 1:
        other = torch.cuda.Stream(device=1)
        with pytest.raises(capi.Bp4Error, match="error -1:.*device 1"):
            ctx.use_stream(other)
    # result / history memory the device cannot write: pageable host memory
    host = np.zeros(16)
    for merged in (True, False):
        f = lib.bp4_solve_cg_merged_async if merged else lib.bp4_solve_cg_async
        assert f(ctx.h, x.h, vb.h, vp.h, 10, 1e-15, 1e-8, C.c_void_p(host.ctypes.data), None) == -1
        assert b"mapped pinned host memory" in lib.bp4_last_error()
        res = torch.empty(3, dtype=F64, device="cuda:0")
        assert f(ctx.h, x.h, vb.h, vp.h, 10, 1e-15, 1e-8, C.c_void_p(res.data_ptr()),
                 C.c_void_p(host.ctypes.data)) == -1
        assert b"history" in lib.bp4_last_error()
    # a history too small for max_steps + 1 (checkable for a tensor only)
    with pytest.raises(ValueError, match="max_steps"):
        ctx.solve_cg(x, vb, vp, max_steps=10, blocking=False, history=torch.empty(10, dtype=F64, device="cuda:0"))
    # mapped pinned host memory is accepted
    pinned = torch.empty(3, dtype=F64).pin_memory()
    assert lib.bp4_solve_cg_async(ctx.h, x.h, vb.h, vp.h, 5, 1e-15, 1e-8, C.c_void_p(pinned.data_ptr()), None) == 0
    ctx.synchronize()
    # synchronising and allocating calls while the bound stream is being captured
    s = torch.cuda.Stream()
    ctx.use_stream(s)
    y = torch.zeros(4, dtype=F64, device="cuda:0")
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    codes = {}
    with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
        y.add_(1.0)
        r = C.c_double()
        codes["dot"] = lib.bp4_dot(ctx.h, vb.h, vb.h, C.byref(r))
        codes["sync"] = lib.bp4_ctx_synchronize(ctx.h)
        codes["solve"] = lib.bp4_solve_cg_merged_async(ctx.h, x.h, vb.h, vp.h, 5, 1e-15, 1e-8,
                                                       C.c_void_p(pinned.data_ptr()), None)
        h = C.c_void_p()
        codes["alloc"] = lib.bp4_vec_alloc(ctx.h, C.c_uint64(30), C.byref(h))
        codes["switch"] = lib.bp4_ctx_set_stream(ctx.h, None)
        msg = lib.bp4_last_error()
    assert codes == {"dot": -4, "sync": -4, "solve": -4, "alloc": -4, "switch": -4}, codes
    assert b"captur" in msg
    g.replay()
    torch.cuda.synchronize()
    assert y.cpu().tolist() == [1.0] * 4
    # the context keeps working on the stream
    w = np.random.default_rng(1).standard_normal(rd.n_owned)
    dst = ctx.vector()
    ctx.vmult(dst, ctx.vector(data=w))
    assert rel_l2(dst.download()[:rd.n_owned], co.vmult(w)) <= 1e-12
    ctx.close()


def _host_history(ctx, rd, merged, max_steps, tol, reduce):
    ctl = O.ReductionControl(max_steps, tol, reduce)
    vp = ctx.vector(rd.n_owned // 3, data=_prec(rd))
    (gpu_cg_merged if merged else gpu_cg_plain)(ctx, rd.rhs, vp, ctl)
    return ctl


ASYNC = [pytest.param(merged, p, id=f"{'merged' if merged else 'plain'}-Q{p}") for merged in (True, False)
         for p in (2, 4)]


@pytest.mark.parametrize("merged,p", ASYNC)
def test_async_equals_blocking(merged, p, bp4_lib):
    """deterministic mode: the enqueued solve gives the blocking solve's result and x bit for bit,
    history[last_step] == last_value, the history equals the host-driven solver's residuals, and the
    entries after last_step stay untouched"""
    from mf_data_locality_b200 import capi
    rd, _ = single(p, 6)
    ctx = _ctx(rd)
    n = rd.n_owned
    vp = ctx.vector(n // 3, data=_prec(rd))
    x0 = np.random.default_rng(p).standard_normal(n)
    x0[rd.constrained] = 0.0
    cases = [("zero x", None, rd.rhs, 100), ("x0", x0, rd.rhs, 100), ("zero b", None, np.zeros(n), 100),
             ("max_steps 0", None, rd.rhs, 0)] + [(f"fail {k}", None, rd.rhs, k) for k in (1, 2, 3, 4)]
    for name, start, rhs, max_steps in cases:
        vb = ctx.vector(data=rhs)
        xb = ctx.vector() if start is None else ctx.vector(data=start)
        rb = ctx.solve_cg(xb, vb, vp, merged=merged, max_steps=max_steps)
        xa = ctx.vector() if start is None else ctx.vector(data=start)
        hnd = ctx.solve_cg(xa, vb, vp, merged=merged, max_steps=max_steps, blocking=False, history=True)
        ra = hnd.result()
        assert ra == rb, name
        assert _same(xa.download(), xb.download()), name
        hist = hnd.history.cpu().numpy()
        last = ra[1]
        assert _same(hist[last], ra[2]) and _same(hist[0], ra[3]), name
        assert np.isnan(hist[last + 1:]).all(), name
        if max_steps < 100:
            assert last == max_steps and ra[0] == capi.FAILURE, name
        if name == "zero b":
            assert ra == (capi.SUCCESS, 0, 0.0, 0.0) and not xa.download().any()
        if start is None and rhs is rd.rhs:
            ctl = _host_history(ctx, rd, merged, max_steps, 1e-15, 1e-8)
            assert ctl.last_step == last and _same(ctl.history, hist[:last + 1]), name
    ctx.close()


@pytest.mark.parametrize("merged", [True, False])
def test_queued_solves_build_no_graph(merged, bp4_lib):
    """three solves with different b, tolerances, result and history buffers queued back to back on
    a torch stream and one synchronisation: each equals its blocking counterpart, and the queue
    costs one launch per solve (no graph is built)"""
    rd, _ = single(3, 6)
    ctx = _ctx(rd)
    n = rd.n_owned
    s = torch.cuda.Stream()
    ctx.use_stream(s)
    vp = ctx.vector(n // 3, data=_prec(rd))
    rng = np.random.default_rng(9)
    bs = [rd.rhs, rng.standard_normal(n), rng.standard_normal(n)]
    for b in bs[1:]:
        b[rd.constrained] = 0.0
    args = [(1e-15, 1e-8, 100), (1e-15, 1e-4, 100), (1e-3, 0.0, 30)]
    vbs = [ctx.vector(data=b) for b in bs]
    xs = [ctx.vector() for _ in bs]
    want = []
    for x, vb, (tol, red, ms) in zip(xs, vbs, args):     # blocking: builds the three graphs
        want.append((ctx.solve_cg(x, vb, vp, merged=merged, tol=tol, reduce=red, max_steps=ms), x.download()))
        x.zero()
    ctx.synchronize()
    n0 = ctx.launch_count()
    with torch.cuda.stream(s):
        torch.cuda._sleep(SLEEP // 4)
        hs = [ctx.solve_cg(x, vb, vp, merged=merged, tol=tol, reduce=red, max_steps=ms, blocking=False, history=True)
              for x, vb, (tol, red, ms) in zip(xs, vbs, args)]
    assert ctx.launch_count() - n0 == 3
    assert not hs[-1].done()
    s.synchronize()
    for h, x, (r, xw) in zip(hs, xs, want):
        assert h.result() == r
        assert _same(x.download(), xw)
        assert len(h.history_values()) == r[1] + 1
    ctx.close()


@pytest.mark.parametrize("plugin,p", [("merged", 4), ("plain", 3)])
def test_mirror_history_equals_host_driven(plugin, p, bp4_lib, monkeypatch):
    """deterministic mode: the device plugin's replayed SolverControl holds, step for step, the
    residuals the host-driven plugin checked"""
    from mf_data_locality_b200 import host
    monkeypatch.setenv("BP4_DETERMINISTIC", "1")
    hist = {}
    for name in (plugin, plugin + "_device"):
        prob = host.Problem(p, 8, plugin=name, device=0)
        _, it = prob.run_cg_solver()
        hist[name] = prob.solver_history()
        assert len(hist[name]) == it + 1
        prob.close()
    assert 1 < len(hist[plugin]) <= 101
    assert _same(hist[plugin], hist[plugin + "_device"])

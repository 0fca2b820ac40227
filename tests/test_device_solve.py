"""Device-resident CG solves (bp4_solve_cg, bp4_solve_cg_merged): the whole iteration loop as
one CUDA graph, the scalars and the stopping test on the device.  Against the C oracle with the
tolerances of test_cg_merged_parity / test_cg_plain_parity, and against the host-driven solvers
on the same context."""
import os
import subprocess

import numpy as np
import pytest

from oracle import bp4_oracle as O

from helpers import gpu_cg_merged, gpu_cg_plain, make_ctx, rel_l2, single

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _setup(p, s, fused=None):
    rd, co = single(p, s)
    ctx = make_ctx(rd)
    if fused is not None:
        ctx.set_fused(fused)
    prec = O.finish_inverse_diagonal(O.inverse_diagonal(rd))
    return rd, co, ctx, prec, ctx.vector(rd.n_owned // 3, data=prec), ctx.vector(data=rd.rhs)


MERGED_CASES = [pytest.param(p, s, f, id=f"Q{p}-s{s}-{'inloop' if f else 'streamed'}")
                for p, s, f in [(2, 9, True), (3, 6, True), (4, 6, True), (2, 9, False), (3, 6, False),
                                (4, 6, False), (5, 7, False), (6, 6, False)]]


@pytest.mark.parametrize("p,s,fused", MERGED_CASES)
def test_merged_matches_oracle(p, s, fused, bp4_lib, c_oracle_lib):
    from mf_data_locality_b200 import capi
    rd, co, ctx, prec, vp, vb = _setup(p, s, fused)
    for reduce in (1e-8, 1e-10):
        x = ctx.vector()
        state, it, last, init = ctx.solve_cg(x, vb, vp, merged=True, reduce=reduce)
        xo, ito, _ = co.cg(rd.rhs, prec, merged=True, reduce=reduce)
        assert abs(it - ito) <= 1
        assert state == (capi.SUCCESS if it < 100 else capi.FAILURE)
        assert init == pytest.approx(np.linalg.norm(rd.rhs), rel=1e-12)
        assert rel_l2(x.download(), xo) <= (1e-8 if ito < 100 else 1e-6)
    ctx.close()


@pytest.mark.parametrize("p,s", [(3, 6), (4, 6)])
def test_plain_matches_oracle(p, s, bp4_lib, c_oracle_lib):
    rd, co, ctx, prec, vp, vb = _setup(p, s)
    for reduce in (1e-8, 1e-10):
        x = ctx.vector()
        _, it, _, _ = ctx.solve_cg(x, vb, vp, merged=False, reduce=reduce)
        xo, ito, _ = co.cg(rd.rhs, prec, merged=False, reduce=reduce)
        assert abs(it - ito) <= 1
        assert rel_l2(x.download(), xo) <= (1e-8 if ito < 100 else 1e-6)
    ctx.close()


SAME_CTX_CASES = [pytest.param(True, 4, True, id="merged-Q4-inloop"),
                  pytest.param(True, 3, False, id="merged-Q3-streamed"),
                  pytest.param(False, 3, None, id="plain-Q3")]


@pytest.mark.parametrize("merged,p,fused", SAME_CTX_CASES)
def test_same_as_host_driven_solver(merged, p, fused, bp4_lib):
    """forced failure after 1..4 steps (both parities of the merged solver's x fix-up), the full
    solve, and a nonzero start vector, against the host-driven recurrences on the same context"""
    from mf_data_locality_b200 import capi
    rd, _, ctx, prec, vp, vb = _setup(p, 7, fused)
    host_cg = gpu_cg_merged if merged else gpu_cg_plain
    for max_steps in (1, 2, 3, 4):
        ctl = O.ReductionControl(max_steps, 1e-15, 1e-8)
        xh = host_cg(ctx, rd.rhs, vp, ctl).download()
        x = ctx.vector()
        state, it, last, _ = ctx.solve_cg(x, vb, vp, merged=merged, max_steps=max_steps)
        assert state == capi.FAILURE and it == max_steps == ctl.last_step
        assert last == pytest.approx(ctl.last_value, rel=1e-10)
        assert rel_l2(x.download(), xh) <= 1e-12
    ctl = O.ReductionControl(100, 1e-15, 1e-8)
    xh = host_cg(ctx, rd.rhs, vp, ctl).download()
    x = ctx.vector()
    state, it, _, _ = ctx.solve_cg(x, vb, vp, merged=merged)
    assert abs(it - ctl.last_step) <= 1
    assert rel_l2(x.download(), xh) <= 1e-8
    # start vector x0 (zero on the Dirichlet rows, as a solution is): the same iterates as the
    # solve of A e = b - A x0 from zero, x = x0 + e
    x0 = np.random.default_rng(p).standard_normal(rd.n_owned)
    x0[rd.constrained] = 0.0
    ax0 = ctx.vector()
    ctx.vmult(ax0, ctx.vector(data=x0))
    r0 = rd.rhs - ax0.download()[:rd.n_owned]
    ctl = O.ReductionControl(100, 1e-15, 1e-8)
    xh = x0 + host_cg(ctx, r0, vp, ctl).download()[:rd.n_owned]
    x = ctx.vector(data=x0)
    state, it, _, init = ctx.solve_cg(x, vb, vp, merged=merged)
    assert init == pytest.approx(np.linalg.norm(r0), rel=1e-10)
    assert abs(it - ctl.last_step) <= 1
    assert rel_l2(x.download(), xh) <= 1e-8
    ctx.close()


@pytest.mark.parametrize("merged", [True, False])
def test_zero_rhs_ends_at_step_zero(merged, bp4_lib):
    from mf_data_locality_b200 import capi
    rd, _, ctx, prec, vp, _ = _setup(3, 6)
    x, b = ctx.vector(), ctx.vector()
    assert ctx.solve_cg(x, b, vp, merged=merged) == (capi.SUCCESS, 0, 0.0, 0.0)
    assert not x.download().any()
    ctx.close()


@pytest.mark.parametrize("merged", [True, False])
def test_no_host_work_per_iteration(merged, bp4_lib):
    """10 and 40 iterations cost the same number of launches from the host; a repeated solve
    re-uses the cached graph and gives the same iteration count"""
    rd, _, ctx, prec, vp, vb = _setup(3, 8)
    x = ctx.vector()
    ctx.solve_cg(x, vb, vp, merged=merged, max_steps=10, tol=0.0, reduce=0.0)   # builds the graph
    counts = []
    for max_steps in (10, 40):
        x.zero()
        n0 = ctx.launch_count()
        ctx.solve_cg(x, vb, vp, merged=merged, max_steps=max_steps, tol=0.0, reduce=0.0)
        counts.append(ctx.launch_count() - n0)
    assert counts[0] == counts[1]
    its = []
    for _ in range(2):
        x.zero()
        its.append(ctx.solve_cg(x, vb, vp, merged=merged)[1])
    assert its[0] == its[1] and 1 <= its[0] < 100
    ctx.close()


def test_errors(bp4_lib):
    from mf_data_locality_b200 import capi, host
    rd, _, ctx, prec, vp, vb = _setup(3, 5)
    with pytest.raises(capi.Bp4Error, match="error -1:.*n_owned"):
        ctx.solve_cg(ctx.vector(10), vb, vp)
    with pytest.raises(capi.Bp4Error, match="error -1:.*prec"):
        ctx.solve_cg(ctx.vector(), vb, ctx.vector(3), merged=False)
    ctx.close()
    # a partition of a two-rank mesh: its context carries a ghost-exchange plan
    prob = host.Problem(3, 6, n_ranks=2, rank=0, device=-1)
    ctx = capi.Context(3, prob.entity_index(), prob.vertices(), prob.n_owned, prob.n_ghost, prob.constrained(),
                       peers=prob.plan())
    vp = ctx.vector(prob.n_owned // 3, data=np.ones(prob.n_owned // 3))
    for merged in (True, False):
        with pytest.raises(capi.Bp4Error, match="error -4:.*one rank"):
            ctx.solve_cg(ctx.vector(), ctx.vector(), vp, merged=merged)
    ctx.close()
    prob.close()


@pytest.mark.parametrize("plugin,p", [("merged", 4), ("plain", 3)])
def test_device_plugin_matches_host_plugin(plugin, p, bp4_lib):
    from mf_data_locality_b200 import host
    rd, _ = single(p, 9)
    res = {}
    for name in (plugin, plugin + "_device"):
        prob = host.Problem(p, 9, plugin=name, device=0)
        res[name] = prob.run_cg_solver(rd.rhs)
        prob.close()
    (x, it), (xd, itd) = res[plugin], res[plugin + "_device"]
    assert abs(it - itd) <= 1
    assert rel_l2(xd, x) <= 1e-8


def test_device_plugin_cli_row(bp4_lib):
    exe = os.path.join(ROOT, "mf_data_locality_b200", "benchmark_precond_merged_device", "bench")
    out = subprocess.run([exe, "4", "6"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    cols = [c.strip() for c in out.stdout.strip().splitlines()[-1].split("|")]
    rd, _ = single(4, 6)
    assert cols[0] == "4" and cols[1] == "6" and int(cols[2]) == rd.n_cells and int(cols[3]) == rd.n_owned
    assert 1 <= int(cols[6]) <= 100

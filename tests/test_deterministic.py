"""Deterministic mode (bp4_desc::deterministic): the cell colouring, parity with the oracle and with
the default mode, bit-for-bit repeatable applies, diagonals, sums and solves, and host-driven solves
that equal the device-resident ones exactly (the same reductions give the same sums, and the scalar
kernel computes the host's scalars from equal sums)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import bp4_oracle as O

from helpers import gpu_cg_merged, gpu_cg_plain, make_ctx, rel_l2, single

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 0xFFFFFFFF


def det_ctx(rd):
    from mf_data_locality_b200 import capi
    return capi.Context(rd.degree, rd.entity_index, rd.vertices, rd.n_owned, rd.n_ghost, rd.constrained,
                        ranges=(rd.range_cell_offset, rd.range_private_offset), coefficients=rd.coefficients,
                        deterministic=True)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


def _prec(rd):
    return O.finish_inverse_diagonal(O.inverse_diagonal(rd))


# s % 3 != 0: a non-cubic box ([0,2]^r x [0,1]^(3-r))
COLOR_CASES = [(p, s, False) for p in (2, 3, 4) for s in (6, 7)] + \
              [(p, s, False) for p in (6, 8) for s in (3, 4)] + [(3, 7, True)]


@pytest.mark.parametrize("p,s,quadratic", COLOR_CASES)
def test_coloring(p, s, quadratic, bp4_lib):
    rd = O.build_problem(p, s, quadratic=True)[0] if quadratic else single(p, s)[0]
    ctx = det_ctx(rd)
    on, n_colors, colors = ctx.deterministic_info()
    assert on and 1 <= n_colors <= 8
    assert colors.shape == (rd.n_cells,) and colors.max() == n_colors - 1
    ei = np.asarray(rd.entity_index, dtype=np.uint32).reshape(-1, 27)
    for k in range(n_colors):
        e = ei[colors == k]
        e = e[e != INVALID]
        assert len(np.unique(e)) == len(e), f"two cells of colour {k} share an entity"
    ctx.close()
    ref = make_ctx(rd)
    assert ref.deterministic_info() == (False, 0, None)
    ref.close()


@pytest.mark.parametrize("p,s", [(2, 7), (3, 6), (4, 9), (5, 5), (6, 4), (7, 4), (8, 3)])
def test_vmult(p, s, bp4_lib, c_oracle_lib):
    """oracle parity, default-mode parity, five repeats and a second context: the same bits"""
    rd, co = single(p, s)
    v = np.random.default_rng(100 * p + s).standard_normal(rd.n_owned)
    outs = []
    for _ in range(2):
        ctx = det_ctx(rd)
        src, dst = ctx.vector(data=v), ctx.vector()
        for _ in range(5):
            ctx.vmult(dst, src)
            outs.append(dst.download())
        ctx.close()
    assert rel_l2(outs[0], co.vmult(v)) <= 1e-12
    assert np.array_equal(outs[0][rd.constrained], v[rd.constrained])
    ref = make_ctx(rd)
    src, dst = ref.vector(data=v), ref.vector()
    ref.vmult(dst, src)
    assert rel_l2(outs[0], dst.download()) <= 1e-13
    ref.close()
    for o in outs[1:]:
        assert same_bits(o, outs[0])


@pytest.mark.parametrize("p,s", [(2, 6), (3, 6), (4, 6), (5, 4), (6, 5), (8, 3)])
def test_inverse_diagonal(p, s, bp4_lib):
    from mf_data_locality_b200 import capi
    rd, _ = single(p, s)
    want = _prec(rd)
    per_node, per_dof = [], []
    for _ in range(2):
        ctx = det_ctx(rd)
        for _ in range(3):
            per_node.append(ctx.inverse_diagonal().download())
            v = ctx.vector()
            capi._chk(capi.lib().bp4_inverse_diagonal_vector(ctx.h, v.h))
            per_dof.append(v.download())
        ctx.close()
    assert rel_l2(per_node[0], want) <= 1e-12
    assert rel_l2(per_dof[0][0:rd.n_owned:3], want) <= 1e-12
    for a in per_node[1:]:
        assert same_bits(a, per_node[0])
    for a in per_dof[1:]:
        assert same_bits(a, per_dof[0])


@pytest.mark.parametrize("p,s", [(2, 7), (3, 6), (4, 7), (4, 9), (6, 4), (8, 4)])
def test_merged_sums(p, s, bp4_lib, c_oracle_lib):
    """the seven sums against the oracle; sums and vectors the same bits on repeats and on a second
    context, in each of the three do_cg_update4b regimes; the in-loop form is refused"""
    from mf_data_locality_b200 import capi
    rd, co = single(p, s)
    n = rd.n_owned
    prec = _prec(rd)
    prec3 = np.repeat(prec, 3)
    rng = np.random.default_rng(3)
    free = np.ones(n)
    free[rd.constrained] = 0.0
    inputs = [tuple(rng.standard_normal(n) * free for _ in range(4)) for _ in range(3)]
    regimes = [(0.0, 0.0, 0.0, 0.0), (0.7, 0.3, 0.0, 0.2), (0.7, 0.3, 0.4, 0.2)]
    runs = []
    for _ in range(2):
        ctx = det_ctx(rd)
        assert not ctx.fused_info()[0]
        with pytest.raises(capi.Bp4Error, match="error -4"):
            ctx.set_fused(True)
        vp = ctx.vector(n // 3, data=prec)
        for _ in range(2):
            res = []
            for (x, g, d, h), sc in zip(inputs, regimes):
                vs = [ctx.vector(data=a) for a in (x, g, d, h)]
                S = ctx.vmult_merged(*vs, vp, *sc)
                res.append((S, [v.download() for v in vs]))
            runs.append(res)
        ctx.close()
    for (x, g, d, h), sc, (S, vecs) in zip(inputs, regimes, runs[0]):
        x, g, d, h = x.copy(), g.copy(), d.copy(), h.copy()
        O.cg_update4b(h, x, g, d, prec3, *sc)
        dd = d.copy()
        dd[rd.constrained] = 0.0
        h[:] = co.vmult_cells(dd)
        np.testing.assert_allclose(S, O.cg_update3b(g, d, h, prec3), rtol=1e-11)
        for got, ref in zip(vecs, (x, g, d, h)):
            assert rel_l2(got, ref) <= 1e-12
    for run in runs[1:]:
        for (S, vecs), (S0, vecs0) in zip(run, runs[0]):
            assert same_bits(S, S0)
            for a, b in zip(vecs, vecs0):
                assert same_bits(a, b)


def test_reductions(bp4_lib):
    """dot, add_and_dot and l2_norm over ~1.6 M entries (the full grid of 8 blocks per SM): the same
    bits on repeats and on a second context, and close to numpy's sums"""
    rd, _ = single(4, 9)
    n = rd.n_owned
    rng = np.random.default_rng(11)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    runs = []
    for _ in range(2):
        ctx = det_ctx(rd)
        va, vb = ctx.vector(data=a), ctx.vector(data=b)
        for _ in range(3):
            g = ctx.vector(data=a)
            runs.append((ctx.dot(va, vb), ctx.l2_norm(va), ctx.add_and_dot(g, 0.5, vb, g)))
        ctx.close()
    assert runs[0][0] == pytest.approx(a @ b, rel=1e-11)
    assert runs[0][1] == pytest.approx(np.linalg.norm(a), rel=1e-13)
    assert runs[0][2] == pytest.approx((a + 0.5 * b) @ (a + 0.5 * b), rel=1e-12)
    for r in runs[1:]:
        assert same_bits(r, runs[0])


def _host_cg_from(ctx, x, b, prec, control, merged):
    """gpu_cg_merged / gpu_cg_plain from a start vector already in x, step 0 as the device solve
    takes it (g = A x - b)"""
    g, d, h = ctx.vector(), ctx.vector(), ctx.vector()
    ctx.vmult(g, x)
    ctx.add(g, -1.0, b)
    res = ctx.l2_norm(g)
    if control.check(0, res) != "iterate":
        return
    if merged:
        alpha = beta = alpha_old = beta_old = 0.0
        it = 0
        while True:
            it += 1
            S = ctx.vmult_merged(x, g, d, h, prec, alpha, beta, alpha_old if it % 2 == 1 else 0.0, beta_old)
            alpha_old, beta_old = alpha, beta
            alpha = S[6] / S[0]
            res = math.sqrt(S[3] + 2 * alpha * S[2] + alpha * alpha * S[1])
            if control.check(it, res) != "iterate":
                if it % 2 == 1:
                    ctx.add(x, alpha, d)
                else:
                    ctx.x_finalize_even(x, d, g, prec, alpha + alpha_old / beta_old, alpha_old / beta_old)
                return
            beta = alpha * (S[4] + alpha * S[5]) / S[6]
    ctx.jacobi_vmult(h, g, prec)
    ctx.equ(d, -1.0, h)
    gh = ctx.dot(g, h)
    it = 0
    while True:
        it += 1
        ctx.vmult(h, d)
        alpha = gh / ctx.dot(d, h)
        ctx.add(x, alpha, d)
        res = math.sqrt(abs(ctx.add_and_dot(g, alpha, h, g)))
        if control.check(it, res) != "iterate":
            return
        ctx.jacobi_vmult(h, g, prec)
        beta_den = gh
        gh = ctx.dot(g, h)
        ctx.sadd(d, gh / beta_den, -1.0, h)


@pytest.mark.parametrize("merged", [True, False], ids=["merged", "plain"])
@pytest.mark.parametrize("p", [3, 4])
def test_host_driven_equals_device_resident(merged, p, bp4_lib):
    """forced failure after 1..4 steps (both parities of the merged x fix-up), a full solve and a
    nonzero start vector: equal last_step, equal last_value, the same bits in x"""
    from mf_data_locality_b200 import capi
    rd, _ = single(p, 7)
    ctx = det_ctx(rd)
    prec = _prec(rd)
    vp, vb = ctx.vector(rd.n_owned // 3, data=prec), ctx.vector(data=rd.rhs)
    host_cg = gpu_cg_merged if merged else gpu_cg_plain
    for max_steps in (1, 2, 3, 4, 100):
        ctl = O.ReductionControl(max_steps, 1e-15, 1e-8)
        xh = host_cg(ctx, rd.rhs, vp, ctl).download()
        x = ctx.vector()
        state, it, last, _ = ctx.solve_cg(x, vb, vp, merged=merged, max_steps=max_steps)
        if max_steps < 100:
            assert state == capi.FAILURE
        assert it == ctl.last_step and last == ctl.last_value
        assert same_bits(x.download(), xh)
    assert state == capi.SUCCESS and 4 < it < 100
    x0 = np.random.default_rng(p).standard_normal(rd.n_owned)
    x0[rd.constrained] = 0.0
    ctl = O.ReductionControl(100, 1e-15, 1e-8)
    xh = ctx.vector(data=x0)
    _host_cg_from(ctx, xh, vb, vp, ctl, merged)
    x = ctx.vector(data=x0)
    state, it, last, init = ctx.solve_cg(x, vb, vp, merged=merged)
    assert init == ctl.initial and it == ctl.last_step and last == ctl.last_value
    assert same_bits(x.download(), xh.download())
    ctx.close()


@pytest.mark.parametrize("plugin,p", [("merged", 4), ("plain", 3)])
def test_device_plugin_equals_host_plugin(plugin, p, bp4_lib):
    from mf_data_locality_b200 import host
    rd, _ = single(p, 9)
    res = {}
    for name in (plugin, plugin + "_device"):
        prob = host.Problem(p, 9, plugin=name, device=0, deterministic=True)
        res[name] = prob.run_cg_solver(rd.rhs)
        prob.close()
    (x, it), (xd, itd) = res[plugin], res[plugin + "_device"]
    assert it == itd
    assert same_bits(x, xd)


def test_repeated_runs(bp4_lib):
    from mf_data_locality_b200 import host
    out = []
    for _ in range(2):
        prob = host.Problem(4, 9, plugin="merged", device=0, deterministic=True)
        out.append(prob.run_cg_solver())
        prob.close()
    assert out[0][1] == out[1][1]
    assert same_bits(out[0][0], out[1][0])


def test_environment_variable(bp4_lib):
    code = ("from oracle import bp4_oracle as O\n"
            "from mf_data_locality_b200 import capi\n"
            "rd = O.build_problem(2, 4)[0]\n"
            "ctx = capi.Context(2, rd.entity_index, rd.vertices, rd.n_owned, 0, rd.constrained)\n"
            "on, n, _ = ctx.deterministic_info()\n"
            "print(int(on), n)\n")
    env = dict(os.environ, BP4_DETERMINISTIC="1")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr
    on, n = out.stdout.split()
    assert on == "1" and 1 <= int(n) <= 8


def test_single_rank_only(bp4_lib):
    from mf_data_locality_b200 import capi
    rd, _ = single(3, 5)
    ctx = det_ctx(rd)
    nccl_id = (C.c_ubyte * 128)()
    assert capi.lib().bp4_comm_init(ctx.h, 0, 2, nccl_id) == -4
    assert b"one rank" in capi.lib().bp4_last_error()
    ctx.close()


@pytest.mark.parametrize("merged", [True, False])
def test_no_host_work_per_iteration(merged, bp4_lib):
    """10 and 40 iterations cost the same number of launches from the host"""
    rd, _ = single(3, 8)
    ctx = det_ctx(rd)
    vp, vb = ctx.vector(rd.n_owned // 3, data=_prec(rd)), ctx.vector(data=rd.rhs)
    x = ctx.vector()
    ctx.solve_cg(x, vb, vp, merged=merged, max_steps=10, tol=0.0, reduce=0.0)   # builds the graph
    counts = []
    for max_steps in (10, 40):
        x.zero()
        n0 = ctx.launch_count()
        ctx.solve_cg(x, vb, vp, merged=merged, max_steps=max_steps, tol=0.0, reduce=0.0)
        counts.append(ctx.launch_count() - n0)
    assert counts[0] == counts[1]
    ctx.close()

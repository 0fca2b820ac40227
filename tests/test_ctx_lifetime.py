"""Context lifetime: bp4_comm_init gives a context one communicator for its whole life."""
import ctypes as C

import numpy as np
import pytest

from helpers import make_ctx, rel_l2, single

pytestmark = pytest.mark.gpu


def test_second_comm_init_is_a_state_error(bp4_lib, c_oracle_lib):
    from mf_data_locality_b200 import capi
    rd, co = single(3, 5)
    ctx = make_ctx(rd)
    first, second = ((C.c_ubyte * 128).from_buffer_copy(capi.unique_id()) for _ in range(2))
    assert capi.lib().bp4_comm_init(ctx.h, 0, 1, first) == 0
    assert capi.lib().bp4_comm_init(ctx.h, 0, 1, second) == -4
    msg = capi.lib().bp4_last_error()
    assert b"already initialised (rank 0 of 1)" in msg
    # the first communicator stays in use: the sums of dot go through its all-reduce
    v = np.random.default_rng(7).standard_normal(rd.n_owned)
    src, dst = ctx.vector(data=v), ctx.vector()
    ctx.vmult(dst, src)
    got = dst.download()
    assert rel_l2(got, co.vmult(v)) <= 1e-12
    assert ctx.dot(src, dst) == pytest.approx(float(v @ got), rel=1e-12)
    src.free()
    dst.free()
    h, ctx.h = ctx.h, C.c_void_p()
    assert capi.lib().bp4_ctx_destroy(h) == 0
    assert capi.lib().bp4_last_error() == msg     # destruction leaves the last error alone

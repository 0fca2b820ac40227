"""The mixed-precision solve and the FP32 operator hook without a GPU: the new entry points are
exported and listed, and refuse null arguments loudly like the other entry points (there is no CPU
fallback)."""
import ctypes as C

import pytest

NEW = ["bp4_solve_cg_mixed", "bp4_solve_cg_mixed_async", "bp4_debug_vmult_f32"]


@pytest.fixture(scope="module")
def lib():
    from mf_data_locality_b200 import build, capi
    build.build_cuda()
    return capi.lib()


@pytest.mark.parametrize("name", NEW)
def test_exported_and_listed(lib, name):
    from mf_data_locality_b200 import capi
    assert hasattr(lib, name) and name in capi.EXPORTS


def test_mixed_solves_fail_loudly(lib):
    res = (C.c_double * 4)()
    hist = (C.c_double * 11)()
    assert lib.bp4_solve_cg_mixed(None, None, None, None, 10, 1e-15, 1e-8, res) == -1
    assert b"null" in lib.bp4_last_error()
    assert lib.bp4_solve_cg_mixed_async(None, None, None, None, 10, 1e-15, 1e-8, res, hist) == -1
    assert b"null" in lib.bp4_last_error()
    assert lib.bp4_solve_cg_mixed_async(None, None, None, None, 10, 1e-15, 1e-8, None, None) == -1


def test_vmult_f32_null_context(lib):
    assert lib.bp4_debug_vmult_f32(None, None, None) == -1
    assert b"null" in lib.bp4_last_error()


def test_no_context_without_device(lib):
    """the FP32 paths need a context, and a context needs a device"""
    import numpy as np
    from mf_data_locality_b200 import capi
    n = C.c_int(-1)
    if lib.bp4_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(capi.Bp4Error):
        capi.Context(3, np.zeros((1, 27), np.uint32), np.zeros((1, 8, 3)), 3)


def test_blocking_history_is_refused_before_any_call(monkeypatch):
    """the history comes with the enqueued form only; the refusal needs no library"""
    from mf_data_locality_b200 import capi

    class NoLib:
        def __getattr__(self, name):
            raise AssertionError(f"{name} called")

    monkeypatch.setattr(capi, "_lib", NoLib())
    ctx = capi.Context.from_handle(None, 3, 0, 3)
    with pytest.raises(ValueError, match="blocking=False"):
        ctx.solve_cg_mixed(None, None, None, history=True)

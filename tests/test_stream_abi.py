"""The caller's-stream binding and the enqueued solves without a GPU: the three entry points are
exported and declared, and refuse null arguments loudly like the other entry points (there is no CPU
fallback)."""
import ctypes as C

import pytest

NEW = ["bp4_ctx_set_stream", "bp4_solve_cg_async", "bp4_solve_cg_merged_async"]


@pytest.fixture(scope="module")
def lib():
    from mf_data_locality_b200 import build, capi
    build.build_cuda()
    return capi.lib()


@pytest.mark.parametrize("name", NEW)
def test_exported_and_listed(lib, name):
    from mf_data_locality_b200 import capi
    assert hasattr(lib, name) and name in capi.EXPORTS


def test_set_stream_null_context(lib):
    assert lib.bp4_ctx_set_stream(None, None) == -1
    assert b"null" in lib.bp4_last_error()


@pytest.mark.parametrize("name", ["bp4_solve_cg_async", "bp4_solve_cg_merged_async"])
def test_async_solves_fail_loudly(lib, name):
    res = (C.c_double * 3)()
    hist = (C.c_double * 11)()
    assert getattr(lib, name)(None, None, None, None, 10, 1e-15, 1e-8, res, hist) == -1
    assert b"null" in lib.bp4_last_error()
    assert getattr(lib, name)(None, None, None, None, 10, 1e-15, 1e-8, None, None) == -1


def test_blocking_history_is_refused_before_any_call(monkeypatch):
    """the history comes with the enqueued form only; the refusal needs no library"""
    from mf_data_locality_b200 import capi

    class NoLib:
        def __getattr__(self, name):
            raise AssertionError(f"{name} called")

    monkeypatch.setattr(capi, "_lib", NoLib())
    ctx = capi.Context.from_handle(None, 3, 0, 3)
    with pytest.raises(ValueError, match="blocking=False"):
        ctx.solve_cg(None, None, None, history=True)

"""Device-resident CG solves without a GPU: the two new entry points are exported, reject bad
arguments loudly (there is no CPU fallback) and the two new host plugins report their names."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from mf_data_locality_b200 import build, capi
    build.build_cuda()
    return capi.lib()


@pytest.mark.parametrize("name", ["bp4_solve_cg", "bp4_solve_cg_merged"])
def test_solve_entry_points_fail_loudly(lib, name):
    res = (C.c_byte * 32)()
    assert getattr(lib, name)(None, None, None, None, 100, 1e-15, 1e-8, res) == -1
    assert b"null" in lib.bp4_last_error()


def test_no_context_without_device(lib):
    """a solve needs a context, and a context needs a device"""
    import numpy as np
    from mf_data_locality_b200 import capi
    n = C.c_int(-1)
    if lib.bp4_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(capi.Bp4Error):
        capi.Context(3, np.zeros((1, 27), np.uint32), np.zeros((1, 8, 3)), 3)


def test_device_plugins_report_their_names():
    from mf_data_locality_b200 import build, host
    build.build_all()
    assert host.lib("plain_device").bp4h_plugin() == b"benchmark_precond_device"
    assert host.lib("merged_device").bp4h_plugin() == b"benchmark_precond_merged_device"

"""Deterministic mode without a GPU: the one-rank check comes before any device call, the new
entry point is exported, and the Python descriptor mirrors bp4_desc of include/bp4.h."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from mf_data_locality_b200 import build, capi
    build.build_cuda()
    return capi.lib()


def test_deterministic_with_peers_is_an_argument_error(lib):
    from mf_data_locality_b200 import capi
    ei = np.zeros((1, 27), np.uint32)
    vt = np.zeros((1, 8, 3))
    one = np.zeros(2, np.uint64)
    d = capi._Desc()
    d.degree, d.n_cells, d.n_owned = 3, 1, 3
    d.entity_index, d.vertices = capi._ptr(ei), capi._ptr(vt)
    d.n_peers, d.import_offset, d.export_offset = 1, capi._ptr(one), capi._ptr(one)
    d.deterministic = 1
    h = C.c_void_p()
    assert lib.bp4_ctx_create(C.byref(d), C.byref(h)) == -1
    assert b"one rank" in lib.bp4_last_error()
    assert not h.value


def test_deterministic_info_rejects_null_context(lib):
    assert lib.bp4_deterministic_info(None, None, None, None) == -1
    assert b"null" in lib.bp4_last_error()


def test_desc_matches_header():
    from mf_data_locality_b200 import capi
    src = open(os.path.join(ROOT, "include", "bp4.h")).read()
    body = re.search(r"typedef struct bp4_desc\s*\{(.*?)\}\s*bp4_desc;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = [re.findall(r"\w+", decl)[-1] for decl in body.split(";") if decl.strip()]
    assert [f[0] for f in capi._Desc._fields_] == names

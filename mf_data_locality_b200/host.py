"""ctypes binding of the C++ host mirror (libbp4_host_plain.so / libbp4_host_merged.so):
the reference's problem set-up (mesh, Renumber(0,1,2), LaplaceOperator::initialize) and its
`run_cg_solver` plugin, executed by the same C++ code as the `bench` executables."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_libs = {}


class HostError(RuntimeError):
    pass


def lib(plugin: str):
    """plugin: 'plain' (benchmark_precond), 'merged' (benchmark_precond_merged), or the same
    solvers with the iteration loop on the device, 'plain_device' (benchmark_precond_device) and
    'merged_device' (benchmark_precond_merged_device; one rank)"""
    if plugin not in _libs:
        path = os.path.join(_HERE, f"libbp4_host_{plugin}.so")
        if not os.path.exists(path):
            raise HostError(f"{path} is missing: run `python -m mf_data_locality_b200.build`")
        l = C.CDLL(path)
        l.bp4h_last_error.restype = C.c_char_p
        l.bp4h_plugin.restype = C.c_char_p
        l.bp4h_ctx.restype = C.c_void_p
        l.bp4h_ctx.argtypes = [C.c_void_p]
        l.bp4h_setup_seconds.restype = C.c_double
        l.bp4h_setup_seconds.argtypes = [C.c_void_p]
        l.bp4h_set_solver.argtypes = [C.c_uint, C.c_double, C.c_double]
        _libs[plugin] = l
    return _libs[plugin]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Problem:
    """BenchmarkProblem of host/benchmark.h.  device < 0 builds the tables only (no GPU)."""

    def __init__(self, degree, s, plugin="merged", n_ranks=1, rank=0, device=0, n_lanes=8,
                 batches_per_range=1, renumber=(0, 1, 2), nccl_id: bytes | None = None,
                 numbering_only=False, mapping_degree=1, deterministic=False):
        """nccl_id: the 128-byte ncclUniqueId shared by all ranks (needed when n_ranks > 1 and a
        device is used; see capi.unique_id()); deterministic: bit-reproducible operator, reductions
        and solves on one rank (bp4_desc::deterministic)"""
        self.l = lib(plugin)
        self.plugin = plugin
        opts = (C.c_int * 11)(n_ranks, rank, device, n_lanes, batches_per_range, *renumber,
                              1 if numbering_only else 0, mapping_degree, 1 if deterministic else 0)
        idbuf = (C.c_ubyte * 128).from_buffer_copy(nccl_id) if nccl_id else None
        self.h = C.c_void_p()
        self._chk(self.l.bp4h_create(C.c_int(degree), C.c_int(s), opts, idbuf, C.byref(self.h)))
        sz = (C.c_uint64 * 8)()
        self._chk(self.l.bp4h_sizes(self.h, sz))
        (self.n_cells, self.n_owned, self.n_ghost, self.n_dofs, self.n_cells_global, self.n_constrained,
         self.n_batches, self.n_ranges) = [int(v) for v in sz]
        self.degree, self.s, self.device = degree, s, device
        self.setup_seconds = self.l.bp4h_setup_seconds(self.h)

    def _chk(self, code):
        if code != 0:
            raise HostError(self.l.bp4h_last_error().decode())

    def close(self):
        if self.h:
            self.l.bp4h_destroy(self.h)
            self.h = C.c_void_p()

    def ctx_handle(self):
        return self.l.bp4h_ctx(self.h)

    def entity_index(self):
        out = np.empty((self.n_cells, 27), dtype=np.uint32)
        self._chk(self.l.bp4h_get_entity_index(self.h, _p(out)))
        return out

    def vertices(self):
        out = np.empty((self.n_cells, 8, 3))
        self._chk(self.l.bp4h_get_vertices(self.h, _p(out)))
        return out

    def coefficients(self):
        """[n_cells][27][3] geometry coefficients of a quadratic mapping, None for the tri-linear one"""
        n = C.c_uint64()
        self._chk(self.l.bp4h_get_coefficients(self.h, C.byref(n), None))
        if n.value == 0:
            return None
        out = np.empty((self.n_cells, 27, 3))
        self._chk(self.l.bp4h_get_coefficients(self.h, C.byref(n), _p(out)))
        return out

    def ranges(self):
        """(range_cell_offset, range_private_offset) as handed to bp4_ctx_create"""
        n = C.c_uint64()
        self._chk(self.l.bp4h_get_ranges(self.h, C.byref(n), None, None))
        rc = np.zeros(n.value, dtype=np.uint64)
        rp = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            self._chk(self.l.bp4h_get_ranges(self.h, C.byref(n), _p(rc), _p(rp)))
        return rc, rp

    def constrained(self):
        out = np.empty(self.n_constrained, dtype=np.uint32)
        self._chk(self.l.bp4h_get_constrained(self.h, _p(out)))
        return out

    def node_of_local(self):
        out = np.empty((self.n_owned + self.n_ghost) // 3, dtype=np.uint64)
        self._chk(self.l.bp4h_get_node_of_local(self.h, _p(out)))
        return out

    def rhs(self):
        out = np.empty(self.n_owned)
        self._chk(self.l.bp4h_get_rhs(self.h, _p(out)))
        return out

    def diagonal(self):
        out = np.empty(self.n_owned // 3)
        self._chk(self.l.bp4h_get_diagonal(self.h, _p(out)))
        return out

    def plan(self):
        """ghost exchange plan of the vector partitioner: peers, import/export offsets (DoFs),
        exported owned local DoF indices"""
        cnt = (C.c_uint64 * 2)()
        self._chk(self.l.bp4h_plan_sizes(self.h, cnt))
        npeer, nexp = int(cnt[0]), int(cnt[1])
        peers = np.zeros(npeer, dtype=np.int32)
        io = np.zeros(npeer + 1, dtype=np.uint64)
        eo = np.zeros(npeer + 1, dtype=np.uint64)
        ex = np.zeros(max(nexp, 1), dtype=np.uint32)
        self._chk(self.l.bp4h_get_plan(self.h, _p(peers), _p(io), _p(eo), _p(ex)))
        return {"rank": peers, "import_offset": io, "export_offset": eo, "export_index": ex[:nexp]}

    def set_solver(self, max_steps=100, abs_tol=1e-15, rel_tol=1e-8):
        self.l.bp4h_set_solver(max_steps, abs_tol, rel_tol)

    def run_cg_solver(self, b=None, want_x=True):
        """the plugin's run_cg_solver with x0 = 0; b = None keeps the benchmark's i % 8 RHS"""
        if b is not None:
            b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.empty(self.n_owned) if want_x else None
        it = C.c_uint()
        self._chk(self.l.bp4h_run_cg_solver(self.h, _p(b), _p(x), C.byref(it)))
        return x, it.value

    def solver_history(self):
        """the residual norms the last run_cg_solver checked at steps 0 .. last_step (the
        plugin's ReductionControl with its history data enabled)"""
        n = C.c_uint()
        self._chk(self.l.bp4h_solver_history(None, C.byref(n)))
        out = np.empty(n.value)
        self._chk(self.l.bp4h_solver_history(_p(out), C.byref(n)))
        return out

    def vmult(self, src=None, want_dst=True):
        if src is not None:
            src = np.ascontiguousarray(src, dtype=np.float64)
        dst = np.empty(self.n_owned) if want_dst else None
        self._chk(self.l.bp4h_vmult(self.h, _p(src), _p(dst)))
        return dst

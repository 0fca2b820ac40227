"""ctypes binding of the C ABI in include/bp4.h (libbp4.so).

This is the Python face of the drop-in boundary: tests/, bench.py and
__graft_entry__.smoke() drive the CUDA path exclusively through these calls.  There is
no CPU fallback -- loading fails loudly if the extension has not been built, and every
call raises Bp4Error when no CUDA device is present."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbp4.so")
INVALID = 0xFFFFFFFF

K_VMULT, K_MERGED, K_PRE, K_POST, K_BLAS1 = range(5)


class Bp4Error(RuntimeError):
    pass


class _Desc(C.Structure):
    _fields_ = [("degree", C.c_int), ("device", C.c_int), ("n_cells", C.c_uint64),
                ("n_owned", C.c_uint64), ("n_ghost", C.c_uint64),
                ("entity_index", C.c_void_p), ("vertices", C.c_void_p),
                ("n_constrained", C.c_uint64), ("constrained", C.c_void_p),
                ("n_peers", C.c_int), ("peer_rank", C.c_void_p), ("import_offset", C.c_void_p),
                ("export_offset", C.c_void_p), ("export_index", C.c_void_p),
                ("n_cells_before_comm", C.c_uint64), ("n_cells_comm", C.c_uint64),
                ("n_ranges", C.c_uint64), ("range_cell_offset", C.c_void_p),
                ("range_private_offset", C.c_void_p), ("coefficients", C.c_void_p),
                ("deterministic", C.c_int)]


_lib = None

EXPORTS = [
    "bp4_last_error", "bp4_device_count", "bp4_ctx_create", "bp4_ctx_destroy", "bp4_ctx_synchronize",
    "bp4_ctx_stream", "bp4_vec_alloc", "bp4_vec_free", "bp4_vec_size", "bp4_vec_set_zero",
    "bp4_vec_upload", "bp4_vec_download", "bp4_vec_device_ptr", "bp4_vmult", "bp4_vmult_merged",
    "bp4_vec_alloc_uninitialized", "bp4_debug_set_fused", "bp4_fused_info", "bp4_inverse_diagonal", "bp4_inverse_diagonal_vector", "bp4_extract_component", "bp4_jacobi_vmult", "bp4_x_finalize_even",
    "bp4_equ", "bp4_add", "bp4_sadd", "bp4_dot", "bp4_add_and_dot", "bp4_l2_norm", "bp4_all_zero",
    "bp4_comm_unique_id", "bp4_comm_init", "bp4_comm_info", "bp4_update_ghost_values", "bp4_compress_add",
    "bp4_profile_enable", "bp4_profile_reset", "bp4_profile_get", "bp4_launch_count",
    "bp4_solve_cg", "bp4_solve_cg_merged", "bp4_deterministic_info", "bp4_vec_wrap",
    "bp4_ctx_set_stream", "bp4_solve_cg_async", "bp4_solve_cg_merged_async",
    "bp4_solve_cg_mixed", "bp4_solve_cg_mixed_async", "bp4_debug_vmult_f32",
]

SUCCESS, FAILURE = 1, 2  # SolverControl::State of a device-resident solve
CUDA_STREAM_LEGACY = 1   # cudaStreamLegacy: the legacy default stream (a null stream means "the context's own")


class _SolveResult(C.Structure):
    _fields_ = [("state", C.c_int), ("last_step", C.c_uint), ("last_value", C.c_double),
                ("initial_value", C.c_double)]


class _MixedResult(C.Structure):
    _fields_ = [("state", C.c_int), ("refinements", C.c_uint), ("inner_steps", C.c_uint),
                ("last_value", C.c_double), ("initial_value", C.c_double)]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Bp4Error(f"{LIB_PATH} is missing: run `python -m mf_data_locality_b200.build` "
                           "(there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        _lib.bp4_last_error.restype = C.c_char_p
        d = C.c_double
        vp = C.c_void_p
        _lib.bp4_vmult_merged.argtypes = [vp, vp, vp, vp, vp, vp, d, d, d, d, vp]
        _lib.bp4_x_finalize_even.argtypes = [vp, vp, vp, vp, vp, d, d]
        _lib.bp4_equ.argtypes = [vp, vp, d, vp]
        _lib.bp4_add.argtypes = [vp, vp, d, vp]
        _lib.bp4_sadd.argtypes = [vp, vp, d, d, vp]
        _lib.bp4_add_and_dot.argtypes = [vp, vp, d, vp, vp, vp]
        _lib.bp4_vec_alloc.argtypes = [vp, C.c_uint64, vp]
        _lib.bp4_vec_upload.argtypes = [vp, vp, vp, C.c_uint64]
        _lib.bp4_vec_download.argtypes = [vp, vp, vp, C.c_uint64]
        _lib.bp4_vec_wrap.argtypes = [vp, vp, C.c_uint64, vp]
        for f in (_lib.bp4_solve_cg, _lib.bp4_solve_cg_merged):
            f.argtypes = [vp, vp, vp, vp, C.c_uint, d, d, vp]
        for f in (_lib.bp4_solve_cg_async, _lib.bp4_solve_cg_merged_async):
            f.argtypes = [vp, vp, vp, vp, C.c_uint, d, d, vp, vp]
        _lib.bp4_ctx_set_stream.argtypes = [vp, vp]
        _lib.bp4_solve_cg_mixed.argtypes = [vp, vp, vp, vp, C.c_uint, d, d, vp]
        _lib.bp4_solve_cg_mixed_async.argtypes = [vp, vp, vp, vp, C.c_uint, d, d, vp, vp]
        _lib.bp4_debug_vmult_f32.argtypes = [vp, vp, vp]
    return _lib


def _chk(code):
    if code != 0:
        raise Bp4Error(f"bp4 error {code}: {lib().bp4_last_error().decode()}")


def device_count() -> int:
    n = C.c_int(0)
    _chk(lib().bp4_device_count(C.byref(n)))
    return n.value


def unique_id() -> bytes:
    """ncclUniqueId for bp4_comm_init (call on rank 0, distribute to the other ranks)"""
    buf = (C.c_ubyte * 128)()
    _chk(lib().bp4_comm_unique_id(buf))
    return bytes(buf)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def check_tensor(t, device: int):
    """Raise TypeError / ValueError unless `t` can be wrapped by a context on CUDA device `device`:
    a contiguous, non-empty float64 CUDA tensor on that device whose data starts on a 16-byte
    boundary (the in-loop vector updates move 16-byte pieces from even indices)."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"expected a torch.Tensor, got {type(t).__name__}")
    if t.device.type != "cuda" or t.device.index != device:
        raise ValueError(f"tensor is on {t.device}, the context runs on cuda:{device}")
    if t.dtype != torch.float64:
        raise ValueError(f"tensor has dtype {t.dtype}, need torch.float64")
    if not t.is_contiguous():
        raise ValueError("tensor is not contiguous")
    if t.numel() == 0:
        raise ValueError("tensor is empty")
    if t.data_ptr() % 16:
        raise ValueError(f"tensor data at {t.data_ptr():#x} is not 16-byte aligned (a view at an odd offset?)")


class Vector:
    tensor = None  # the torch tensor a wrapped vector views (Context.wrap); None for owned memory

    def __init__(self, ctx: "Context", n: int):
        self.ctx, self.n = ctx, int(n)
        self.h = C.c_void_p()
        _chk(lib().bp4_vec_alloc(ctx.h, C.c_uint64(self.n), C.byref(self.h)))

    @classmethod
    def _view(cls, ctx: "Context", t):
        self = cls.__new__(cls)
        self.ctx, self.n, self.tensor = ctx, t.numel(), t
        self.h = C.c_void_p()
        _chk(lib().bp4_vec_wrap(ctx.h, C.c_void_p(t.data_ptr()), C.c_uint64(self.n), C.byref(self.h)))
        return self

    def upload(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        with _Ordered(self.ctx, (self,)):
            _chk(lib().bp4_vec_upload(self.ctx.h, self.h, _ptr(a), C.c_uint64(a.size)))
        self.ctx.synchronize()      # `a` may be a temporary
        return self

    def download(self, n=None):
        n = self.n if n is None else int(n)
        out = np.empty(n)
        with _Ordered(self.ctx, (self,)):
            _chk(lib().bp4_vec_download(self.ctx.h, self.h, _ptr(out), C.c_uint64(n)))
        return out

    def zero(self):
        with _Ordered(self.ctx, (self,)):
            _chk(lib().bp4_vec_set_zero(self.ctx.h, self.h))
        return self

    def free(self):
        """release the handle; a wrapped vector's tensor stays the caller's, with its contents"""
        if self.h:
            lib().bp4_vec_free(self.ctx.h, self.h)
            self.h = C.c_void_p()
        self.tensor = None


class _Ordered:
    """Orders a context call on wrapped vectors (and the extra tensors `ts`) with PyTorch's current
    stream, without a host synchronisation: the context's stream waits for the work queued so far
    on the current stream, and the current stream waits for the call.  When the context runs on
    the current stream itself (Context.use_stream) stream order does that, and no event is needed.
    Every tensor is then recorded on the current stream, which runs behind the call, so the
    caching allocator does not hand its memory out while the call is queued.  (Not on the
    context's own stream: the allocator records an event on each recorded stream when the tensor
    is freed, and close() destroys that stream while the tensor may live on.)  A call on owned
    vectors only does nothing here."""
    __slots__ = ("ctx", "ts", "cur", "same")

    def __init__(self, ctx: "Context", vecs, ts=()):
        self.ctx = ctx
        self.ts = [v.tensor for v in vecs if v is not None and v.tensor is not None] + list(ts)

    def __enter__(self):
        if self.ts:
            import torch
            self.cur = torch.cuda.current_stream(self.ctx.device)
            bound = self.ctx._bound
            self.same = bound is not None and bound.cuda_stream == self.cur.cuda_stream
            if not self.same:
                self.ctx.torch_stream().wait_stream(self.cur)

    def __exit__(self, *exc):
        if self.ts:
            if not self.same:
                self.cur.wait_stream(self.ctx.torch_stream())
            for t in self.ts:
                t.record_stream(self.cur)
        return False


class SolveHandle:
    """A device-resident solve queued by Context.solve_cg(blocking=False).  `result_tensor` (three
    float64 on the device, one bp4_solve_result) and `history` (None, or max_steps + 1 float64:
    the residual checked at steps 0 .. last_step, NaN after it) are written by the stream when
    the solve ends; reading them on the stream the solve was queued on, or after result(), needs
    no other synchronisation."""

    def __init__(self, result_tensor, history, event):
        self.result_tensor, self.history, self._event = result_tensor, history, event

    def done(self) -> bool:
        return self._event.query()

    def result(self):
        """wait for the solve; (state, last_step, last_value, initial_value) as the blocking call"""
        import struct
        self._event.synchronize()
        return struct.unpack("<iIdd", self.result_tensor.cpu().numpy().tobytes())

    def history_values(self):
        """the residuals of steps 0 .. last_step as a numpy array (waits for the solve)"""
        last = self.result()[1]
        return self.history[:last + 1].cpu().numpy()


class MixedSolveHandle(SolveHandle):
    """A mixed-precision solve queued by Context.solve_cg_mixed(blocking=False): `result_tensor`
    (four float64 on the device) holds one bp4_mixed_result, `history` the FP64 true residual of
    refinement steps 0 .. refinements."""

    def result(self):
        """wait for the solve; (state, refinements, inner_steps, last_value, initial_value)"""
        import struct
        self._event.synchronize()
        return struct.unpack("<iII4xdd", self.result_tensor.cpu().numpy().tobytes())


class Context:
    """Device-side operator: mirrors what LaplaceOperator::initialize holds
    (poisson_operator.h:101-293)."""
    _bound = None  # the torch.cuda.Stream bound with use_stream, None: the context's own stream

    def __init__(self, degree, entity_index, vertices, n_owned, n_ghost=0, constrained=None,
                 device=0, peers=None, ranges=None, partitions=None, coefficients=None,
                 deterministic=False):
        """ranges = (range_cell_offset, range_private_offset): cell-batch ranges of the loop and
        the DoF runs private to them (bp4_desc::n_ranges); partitions = (n_cells_before_comm,
        n_cells_comm) of the overlapped ghost exchange; deterministic = bit-reproducible results
        on one rank (bp4_desc::deterministic, also on with BP4_DETERMINISTIC=1)"""
        ei = np.ascontiguousarray(entity_index, dtype=np.uint32).reshape(-1, 27)
        vt = np.ascontiguousarray(vertices, dtype=np.float64).reshape(-1, 8, 3)
        assert len(ei) == len(vt)
        con = np.ascontiguousarray(constrained if constrained is not None else [], dtype=np.uint32)
        d = _Desc()
        d.degree, d.device = int(degree), int(device)
        d.n_cells, d.n_owned, d.n_ghost = len(ei), int(n_owned), int(n_ghost)
        d.entity_index, d.vertices = _ptr(ei), _ptr(vt)
        d.n_constrained, d.constrained = con.size, _ptr(con)
        keep = [ei, vt, con]
        if peers:
            pr = np.ascontiguousarray(peers["rank"], dtype=np.int32)
            io = np.ascontiguousarray(peers["import_offset"], dtype=np.uint64)
            eo = np.ascontiguousarray(peers["export_offset"], dtype=np.uint64)
            ex = np.ascontiguousarray(peers["export_index"], dtype=np.uint32)
            d.n_peers, d.peer_rank, d.import_offset = len(pr), _ptr(pr), _ptr(io)
            d.export_offset, d.export_index = _ptr(eo), _ptr(ex)
            keep += [pr, io, eo, ex]
        if ranges is not None:
            rc = np.ascontiguousarray(ranges[0], dtype=np.uint64)
            rp = np.ascontiguousarray(ranges[1], dtype=np.uint64)
            assert len(rc) == len(rp)
            d.n_ranges, d.range_cell_offset, d.range_private_offset = len(rc) - 1, _ptr(rc), _ptr(rp)
            keep += [rc, rp]
        if coefficients is not None:            # [n_cells][27][3]: genuinely quadratic cells
            cq = np.ascontiguousarray(coefficients, dtype=np.float64).reshape(-1, 27, 3)
            assert len(cq) == len(ei)
            d.coefficients = _ptr(cq)
            keep += [cq]
        if partitions is not None:
            d.n_cells_before_comm, d.n_cells_comm = int(partitions[0]), int(partitions[1])
        d.deterministic = 1 if deterministic else 0
        self.h = C.c_void_p()
        _chk(lib().bp4_ctx_create(C.byref(d), C.byref(self.h)))
        self.degree, self.n_cells = int(degree), len(ei)
        self.n_owned, self.n_ghost = int(n_owned), int(n_ghost)
        self.n_local = self.n_owned + self.n_ghost
        self.device = int(device)

    @classmethod
    def from_handle(cls, handle, degree, n_cells, n_owned, n_ghost=0, device=0):
        """view of a context owned by someone else (the C++ host's LaplaceOperator); close() is a no-op"""
        self = cls.__new__(cls)
        self.h = C.c_void_p(handle)
        self.device = int(device)
        self.degree, self.n_cells = int(degree), int(n_cells)
        self.n_owned, self.n_ghost = int(n_owned), int(n_ghost)
        self.n_local = self.n_owned + self.n_ghost
        self.borrowed = True
        return self

    # ---- lifetime -----------------------------------------------------------------
    def close(self):
        if self.h and not getattr(self, "borrowed", False):
            lib().bp4_ctx_destroy(self.h)
        self.h = C.c_void_p()
        self._torch_stream = None
        self._bound = None

    def synchronize(self):
        _chk(lib().bp4_ctx_synchronize(self.h))

    def stream(self) -> int:
        s = C.c_void_p()
        _chk(lib().bp4_ctx_stream(self.h, C.byref(s)))
        return s.value or 0

    def use_stream(self, stream):
        """Queue every call of the context on `stream`, a torch.cuda.Stream of its device (PyTorch's
        default stream included), or on the context's own stream again with None
        (bp4_ctx_set_stream).  The new stream first waits, on the device, for what the context
        queued on the old one.  While the context runs on PyTorch's current stream, calls on
        wrapped tensors need no event pair to be ordered with torch's work."""
        handle = None if stream is None else (stream.cuda_stream or CUDA_STREAM_LEGACY)
        _chk(lib().bp4_ctx_set_stream(self.h, C.c_void_p(handle)))
        self._bound = stream
        self._torch_stream = None

    def torch_stream(self):
        """the context's current stream as a torch.cuda stream object"""
        if self._bound is not None:
            return self._bound
        if getattr(self, "_torch_stream", None) is None:
            import torch
            self._torch_stream = torch.cuda.ExternalStream(self.stream(), device=torch.device("cuda", self.device))
        return self._torch_stream

    def vector(self, n=None, data=None) -> Vector:
        v = Vector(self, self.n_local if n is None else n)
        if data is not None:
            v.upload(data)
        return v

    def wrap(self, t) -> Vector:
        """A Vector that views the CUDA tensor t in place (bp4_vec_wrap): no copy.  t must be a
        contiguous float64 tensor on the context's device starting on a 16-byte boundary
        (check_tensor); anything else raises before any device call.  The Vector keeps t alive;
        its free() releases the handle only.  Calls on wrapped vectors are ordered with PyTorch's
        current stream, so t can be filled and read by torch ops without a synchronisation."""
        check_tensor(t, self.device)
        return Vector._view(self, t)

    # ---- operator -----------------------------------------------------------------
    def vmult(self, dst: Vector, src: Vector):
        with _Ordered(self, (dst, src)):
            _chk(lib().bp4_vmult(self.h, dst.h, src.h))

    def vmult_merged(self, x, g, d, h, prec, alpha, beta, alpha_old, beta_old):
        out = (C.c_double * 7)()
        with _Ordered(self, (x, g, d, h, prec)):
            _chk(lib().bp4_vmult_merged(self.h, x.h, g.h, d.h, h.h, prec.h, alpha, beta, alpha_old,
                                        beta_old, out))
        return np.array(out[:])

    def vmult_f32(self, dst: Vector, src: Vector):
        """developer hook: dst = A src with the FP32 cell kernel (src rounded to float, the result
        widened; bp4_debug_vmult_f32)"""
        with _Ordered(self, (dst, src)):
            _chk(lib().bp4_debug_vmult_f32(self.h, dst.h, src.h))

    def set_fused(self, on: bool):
        """developer hook: in-loop vector updates on (default with range tables) / off"""
        _chk(lib().bp4_debug_set_fused(self.h, C.c_int(1 if on else 0)))

    def fused_info(self):
        f, npriv, nu = C.c_int(), C.c_uint64(), C.c_uint64()
        _chk(lib().bp4_fused_info(self.h, C.byref(f), C.byref(npriv), C.byref(nu)))
        return bool(f.value), int(npriv.value), int(nu.value)

    def deterministic_info(self):
        """(on, n_colors, colors): whether the context runs in the deterministic mode, its number of
        cell colours and the colour of every cell in the caller's order (None when off)"""
        on, nc = C.c_int(), C.c_uint32()
        _chk(lib().bp4_deterministic_info(self.h, C.byref(on), C.byref(nc), None))
        colors = None
        if on.value:
            colors = np.zeros(self.n_cells, dtype=np.uint32)
            _chk(lib().bp4_deterministic_info(self.h, None, None, _ptr(colors)))
        return bool(on.value), int(nc.value), colors

    def inverse_diagonal(self, out=None) -> Vector:
        """1/diag per node (n_owned/3 entries) into `out`, or into a new vector"""
        v = Vector(self, self.n_owned // 3) if out is None else out
        with _Ordered(self, (v,)):
            _chk(lib().bp4_inverse_diagonal(self.h, v.h))
        return v

    def jacobi_vmult(self, dst, src, diag):
        with _Ordered(self, (dst, src, diag)):
            _chk(lib().bp4_jacobi_vmult(self.h, dst.h, src.h, diag.h))

    def x_finalize_even(self, x, d, g, prec, c1, c2):
        with _Ordered(self, (x, d, g, prec)):
            _chk(lib().bp4_x_finalize_even(self.h, x.h, d.h, g.h, prec.h, c1, c2))

    def solve_cg(self, x, b, prec, merged=True, max_steps=100, tol=1e-15, reduce=1e-8, blocking=True,
                 history=False):
        """CG solve of A x = b with the iteration loop on the device (bp4_solve_cg_merged, or
        bp4_solve_cg with merged=False) from the start vector in x; prec holds n_owned/3 inverse
        diagonal entries.  Returns (state, last_step, last_value, initial_value); hitting
        max_steps is state FAILURE, not an exception.
        blocking=False queues the solve without a host synchronisation (bp4_solve_cg*_async) and
        returns a SolveHandle; history=True (or a float64 CUDA tensor of at least max_steps + 1
        entries) also collects the residual of every checked step there."""
        if blocking:
            if history is not False:
                raise ValueError("history needs blocking=False")
            r = _SolveResult()
            f = lib().bp4_solve_cg_merged if merged else lib().bp4_solve_cg
            with _Ordered(self, (x, b, prec)):
                _chk(f(self.h, x.h, b.h, prec.h, max_steps, tol, reduce, C.byref(r)))
            return r.state, r.last_step, r.last_value, r.initial_value
        import torch
        dev = torch.device("cuda", self.device)
        res = torch.empty(3, dtype=torch.float64, device=dev)
        hist = None
        if history is True:
            hist = torch.full((max_steps + 1,), float("nan"), dtype=torch.float64, device=dev)
        elif history is not False:
            hist = history
            check_tensor(hist, self.device)
            if hist.numel() < max_steps + 1:
                raise ValueError(f"history has {hist.numel()} entries, the solve needs max_steps + 1 = {max_steps + 1}")
        f = lib().bp4_solve_cg_merged_async if merged else lib().bp4_solve_cg_async
        with _Ordered(self, (x, b, prec), [res] + ([hist] if hist is not None else [])):
            _chk(f(self.h, x.h, b.h, prec.h, max_steps, tol, reduce, C.c_void_p(res.data_ptr()),
                   C.c_void_p(hist.data_ptr()) if hist is not None else None))
            ev = torch.cuda.Event()
            ev.record(self.torch_stream())
        return SolveHandle(res, hist, ev)

    def solve_cg_mixed(self, x, b, prec, max_steps=1000, tol=1e-15, reduce=1e-8, blocking=True,
                       history=False):
        """Mixed-precision CG (bp4_solve_cg_mixed): FP64 refinement steps around an inner FP32
        merged CG, stopped by ReductionControl(max_steps, tol, reduce) on the FP64 true residual;
        max_steps caps the inner FP32 iterations.  Returns (state, refinements, inner_steps,
        last_value, initial_value).  blocking=False and history as in solve_cg; the history holds
        the true residual of refinement steps 0 .. refinements."""
        if blocking:
            if history is not False:
                raise ValueError("history needs blocking=False")
            r = _MixedResult()
            with _Ordered(self, (x, b, prec)):
                _chk(lib().bp4_solve_cg_mixed(self.h, x.h, b.h, prec.h, max_steps, tol, reduce, C.byref(r)))
            return r.state, r.refinements, r.inner_steps, r.last_value, r.initial_value
        import torch
        dev = torch.device("cuda", self.device)
        res = torch.empty(4, dtype=torch.float64, device=dev)
        hist = None
        if history is True:
            hist = torch.full((max_steps + 1,), float("nan"), dtype=torch.float64, device=dev)
        elif history is not False:
            hist = history
            check_tensor(hist, self.device)
            if hist.numel() < max_steps + 1:
                raise ValueError(f"history has {hist.numel()} entries, the solve needs max_steps + 1 = {max_steps + 1}")
        with _Ordered(self, (x, b, prec), [res] + ([hist] if hist is not None else [])):
            _chk(lib().bp4_solve_cg_mixed_async(self.h, x.h, b.h, prec.h, max_steps, tol, reduce,
                                                C.c_void_p(res.data_ptr()),
                                                C.c_void_p(hist.data_ptr()) if hist is not None else None))
            ev = torch.cuda.Event()
            ev.record(self.torch_stream())
        return MixedSolveHandle(res, hist, ev)

    # ---- BLAS-1 -------------------------------------------------------------------
    def equ(self, dst, a, src):
        with _Ordered(self, (dst, src)):
            _chk(lib().bp4_equ(self.h, dst.h, a, src.h))

    def add(self, dst, a, src):
        with _Ordered(self, (dst, src)):
            _chk(lib().bp4_add(self.h, dst.h, a, src.h))

    def sadd(self, dst, s, a, src):
        with _Ordered(self, (dst, src)):
            _chk(lib().bp4_sadd(self.h, dst.h, s, a, src.h))

    def dot(self, a, b) -> float:
        r = C.c_double()
        with _Ordered(self, (a, b)):
            _chk(lib().bp4_dot(self.h, a.h, b.h, C.byref(r)))
        return r.value

    def add_and_dot(self, g, a, h, w) -> float:
        r = C.c_double()
        with _Ordered(self, (g, h, w)):
            _chk(lib().bp4_add_and_dot(self.h, g.h, a, h.h, w.h, C.byref(r)))
        return r.value

    def l2_norm(self, v) -> float:
        r = C.c_double()
        with _Ordered(self, (v,)):
            _chk(lib().bp4_l2_norm(self.h, v.h, C.byref(r)))
        return r.value

    def all_zero(self, v) -> bool:
        r = C.c_int()
        with _Ordered(self, (v,)):
            _chk(lib().bp4_all_zero(self.h, v.h, C.byref(r)))
        return bool(r.value)

    # ---- measurement --------------------------------------------------------------
    def profile_enable(self, on=True):
        _chk(lib().bp4_profile_enable(self.h, C.c_int(1 if on else 0)))

    def profile_reset(self):
        _chk(lib().bp4_profile_reset(self.h))

    def profile_get(self, kernel_id):
        ms, n = C.c_double(), C.c_uint64()
        _chk(lib().bp4_profile_get(self.h, C.c_int(kernel_id), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def launch_count(self) -> int:
        n = C.c_uint64()
        _chk(lib().bp4_launch_count(self.h, C.byref(n)))
        return n.value

"""ctypes binding of libarrow_b200.so (the C ABI declared in include/arrow_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present the
calls raise.  Thin object wrappers (`Context`, `Csr`, `Dense`, `RowMap`) keep handles alive and
turn error codes into `ArrowError` with the library's message.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import (POINTER, byref, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p)
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libarrow_b200.so")

ACCUMULATE = 1
VARIANT_AUTO, VARIANT_DIRECT, VARIANT_SHFL, VARIANT_TMA, VARIANT_TILES = -1, 0, 1, 2, 3
IPC_HANDLE_BYTES = 80
DTYPE_CODES = {"float32": 0, "bfloat16": 1}      # ARROW_DTYPE_F32, ARROW_DTYPE_BF16


def dtype_name(dtype) -> str:
    """``"float32"`` or ``"bfloat16"`` for a dense-tile element type given as a name, a numpy dtype or a torch dtype;
    ValueError for anything else (products and sums are fp32 either way)."""
    if isinstance(dtype, str):
        name = dtype
    elif type(dtype).__module__ == "torch":
        name = str(dtype).replace("torch.", "")
    else:
        try:
            name = np.dtype(dtype).name
        except TypeError:
            name = str(dtype)
    if name not in DTYPE_CODES:
        raise ValueError(f"dense tiles hold float32 or bfloat16, not {dtype!r} (arithmetic is float32 in both)")
    return name


def to_bf16(X):
    """Host rows as a contiguous CPU ``torch.bfloat16`` tensor: a bf16 tensor is taken as it is, anything else is
    converted to float32 and rounded to nearest even (``Tensor.to(torch.bfloat16)``).  numpy has no bf16 type."""
    import torch
    if isinstance(X, torch.Tensor):
        t = X if X.dtype == torch.bfloat16 else X.to(torch.float32).to(torch.bfloat16)
    else:
        t = torch.from_numpy(np.ascontiguousarray(X, dtype=np.float32)).to(torch.bfloat16)
    return t.contiguous()

EXPORTS = [
    "arrow_b200_abi_version", "arrow_ctx_create", "arrow_ctx_destroy", "arrow_last_error", "arrow_sync",
    "arrow_device_info", "arrow_set_tuning", "arrow_set_option",
    "arrow_csr_upload", "arrow_csr_free", "arrow_csr_info", "arrow_csr_remap_columns",
    "arrow_map_upload", "arrow_map_free", "arrow_map_compose", "arrow_map_invert", "arrow_map_d2h",
    "arrow_dense_alloc", "arrow_dense_free", "arrow_dense_fill", "arrow_dense_h2d", "arrow_dense_d2h",
    "arrow_dense_copy", "arrow_dense_ptr", "arrow_dense_wrap", "arrow_host_alloc", "arrow_host_free",
    "arrow_dense_h2d_lane", "arrow_dense_d2h_lane", "arrow_lane_wait", "arrow_lane_sync", "arrow_set_lane",
    "arrow_event_record", "arrow_event_wait",
    "arrow_spmm", "arrow_spmm_add", "arrow_gather_rows", "arrow_gather_rows_multi",
    "arrow_ipc_export", "arrow_ipc_import", "arrow_peer_barrier",
    "arrow_timer_start", "arrow_timer_stop", "arrow_timer_elapsed_ms", "arrow_launch_count", "arrow_l2_flush",
    "arrow_ptrtable_upload", "arrow_ptrtable_free", "arrow_spmm_ex", "arrow_push_rows", "arrow_reduce_rows",
    "arrow_graph_begin", "arrow_graph_end", "arrow_graph_launch", "arrow_graph_free",
    "arrow_host_alloc_numa", "arrow_bind_thread_to_device_numa", "arrow_preload_kernels",
    "arrow_dense_alloc_dtype", "arrow_dense_dtype", "arrow_dense_put", "arrow_dense_get",
]
ABI_VERSION = 3          # ARROW_ABI_VERSION of include/arrow_b200.h this binding was written against


class ArrowError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libarrow_b200 error {code}: {message}")
        self.code = code


_lib = None


def load_library(build_if_missing: bool = True) -> ctypes.CDLL:
    """dlopen the in-tree library.  A missing or stale library (older than its sources) is rebuilt first when nvcc
    is available -- under a file lock and through a temporary file, so that the ranks of one ``torchrun`` never
    dlopen a half-written file (``build.build``).  A library whose ABI version differs from this binding is refused."""
    global _lib
    if _lib is not None:
        return _lib
    from . import build as _build
    if build_if_missing and _build.needs_build() and _build.can_build():
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} not built; run `python -m arrow_matrix_b200.build` (needs nvcc)")
    lib = ctypes.CDLL(LIB_PATH)
    lib.arrow_b200_abi_version.restype = c_int
    found = lib.arrow_b200_abi_version()
    if found != ABI_VERSION:
        raise ImportError(f"{LIB_PATH} exports ABI version {found}, this binding needs {ABI_VERSION}: rebuild it "
                          f"(`python -m arrow_matrix_b200.build --force`)")
    P = c_void_p
    I, I64 = c_int, c_int64
    pI, pI64 = POINTER(c_int), POINTER(c_int64)
    sig = {
        "arrow_b200_abi_version": (c_int, []),
        "arrow_ctx_create": (c_int, [I, P, POINTER(P)]),
        "arrow_ctx_destroy": (None, [P]),
        "arrow_last_error": (c_char_p, [P]),
        "arrow_sync": (c_int, [P]),
        "arrow_device_info": (c_int, [P, pI, pI64, pI64]),
        "arrow_set_tuning": (c_int, [P, I, I]),
        "arrow_set_option": (c_int, [P, I, I]),
        "arrow_csr_upload": (c_int, [P, I64, I64, I64, P, I, P, I, P, pI]),
        "arrow_csr_free": (c_int, [P, I]),
        "arrow_csr_info": (c_int, [P, I, pI64, pI64, pI64, pI64, pI64]),
        "arrow_csr_remap_columns": (c_int, [P, I, I, I64, pI]),
        "arrow_map_upload": (c_int, [P, P, I64, I64, pI]),
        "arrow_map_free": (c_int, [P, I]),
        "arrow_map_compose": (c_int, [P, I, I, pI]),
        "arrow_map_invert": (c_int, [P, I, I64, pI]),
        "arrow_map_d2h": (c_int, [P, I, P, I64]),
        "arrow_dense_alloc": (c_int, [P, I64, I, pI]),
        "arrow_dense_free": (c_int, [P, I]),
        "arrow_dense_fill": (c_int, [P, I, c_float]),
        "arrow_dense_h2d": (c_int, [P, I, I64, I64, P]),
        "arrow_dense_d2h": (c_int, [P, I, I64, I64, P]),
        "arrow_dense_copy": (c_int, [P, I, I64, I, I64, I64]),
        "arrow_dense_ptr": (c_int, [P, I, POINTER(P), pI64, pI]),
        "arrow_dense_wrap": (c_int, [P, P, I64, I, pI]),
        "arrow_dense_h2d_lane": (c_int, [P, I, I, I64, I64, P]),
        "arrow_dense_d2h_lane": (c_int, [P, I, I, I64, I64, P]),
        "arrow_lane_wait": (c_int, [P, I, I]),
        "arrow_lane_sync": (c_int, [P, I]),
        "arrow_set_lane": (c_int, [P, I]),
        "arrow_event_record": (c_int, [P, I, I]),
        "arrow_event_wait": (c_int, [P, I, I]),
        "arrow_host_alloc": (c_int, [c_size_t, POINTER(P)]),
        "arrow_host_free": (c_int, [P]),
        "arrow_spmm": (c_int, [P, I, I, I, I, I, I]),
        "arrow_spmm_add": (c_int, [P, I, I, I, I, I, I]),
        "arrow_gather_rows": (c_int, [P, I, I, I, I]),
        "arrow_gather_rows_multi": (c_int, [P, I, pI, pI64, I, I, I]),
        "arrow_ipc_export": (c_int, [P, I, P]),
        "arrow_ipc_import": (c_int, [P, P, I64, I, pI]),
        "arrow_peer_barrier": (c_int, [P, pI, I, I]),
        "arrow_timer_start": (c_int, [P, I]),
        "arrow_timer_stop": (c_int, [P, I]),
        "arrow_timer_elapsed_ms": (c_int, [P, I, POINTER(c_float)]),
        "arrow_launch_count": (c_int, [P, pI64]),
        "arrow_l2_flush": (c_int, [P]),
        "arrow_ptrtable_upload": (c_int, [P, pI, I, P, P, I64, pI]),
        "arrow_ptrtable_free": (c_int, [P, I]),
        "arrow_spmm_ex": (c_int, [P, I, I, I, I64, I, I, I, I, I]),
        "arrow_push_rows": (c_int, [P, pI, pI64, I, I, I]),
        "arrow_reduce_rows": (c_int, [P, I, I, pI, I, I64]),
        "arrow_graph_begin": (c_int, [P]),
        "arrow_graph_end": (c_int, [P, pI]),
        "arrow_graph_launch": (c_int, [P, I]),
        "arrow_graph_free": (c_int, [P, I]),
        "arrow_host_alloc_numa": (c_int, [c_size_t, I, POINTER(P)]),
        "arrow_bind_thread_to_device_numa": (c_int, [I, pI, pI]),
        "arrow_preload_kernels": (c_int, [P, I]),
        "arrow_dense_alloc_dtype": (c_int, [P, I64, I, I, pI]),
        "arrow_dense_dtype": (c_int, [P, I, pI]),
        "arrow_dense_put": (c_int, [P, I, I, I64, I64, P]),
        "arrow_dense_get": (c_int, [P, I, I, I64, I64, P]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)          # AttributeError here = the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a: Optional[np.ndarray]) -> c_void_p:
    return c_void_p(None) if a is None else c_void_p(a.ctypes.data)


class PinnedArray:
    """Page-locked host staging buffer exposed as a numpy array (freed on `close()`/GC)."""

    def __init__(self, shape, dtype=np.float32, numa_device: Optional[int] = None):
        """``numa_device`` given: the buffer is placed on the NUMA node that GPU hangs off (arrow_host_alloc_numa)."""
        lib = load_library()
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = c_void_p()
        if numa_device is None:
            rc = lib.arrow_host_alloc(c_size_t(max(nbytes, 16)), byref(p))
        else:
            rc = lib.arrow_host_alloc_numa(c_size_t(max(nbytes, 16)), int(numa_device), byref(p))
        if rc != 0:
            raise ArrowError(rc, (lib.arrow_last_error(None) or b"").decode())
        self._p = p
        buf = (ctypes.c_char * max(nbytes, 16)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self.array = None
            load_library().arrow_host_free(self._p)
            self._p = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PinnedTensor(PinnedArray):
    """Page-locked host staging buffer exposed as a CPU torch tensor (``tensor``), for element types numpy lacks:
    the bf16 rows ``ArrowEngine.stream_step`` moves for a bf16 engine."""

    def __init__(self, shape, dtype=None, numa_device: Optional[int] = None):
        import torch
        dtype = torch.bfloat16 if dtype is None else dtype
        itemsize = torch.empty(0, dtype=dtype).element_size()
        super().__init__(shape, np.dtype(f"u{itemsize}"), numa_device)
        self.tensor = torch.from_numpy(self.array).view(dtype)

    def close(self):
        self.tensor = None
        super().close()


def bind_thread_to_device_numa(device: int):
    """Pin the calling thread to the CPUs of the NUMA node ``device`` hangs off; returns ``(node, n_cpus)``
    (``(-1, 0)`` when the topology is unknown and nothing was changed)."""
    lib = load_library()
    node, n = c_int(-1), c_int(0)
    lib.arrow_bind_thread_to_device_numa(int(device), byref(node), byref(n))
    return node.value, n.value


class Context:
    """One device context = one stream = one host thread (arrow_b200.h)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self.lib = load_library()
        self._h = c_void_p()
        rc = self.lib.arrow_ctx_create(int(device), c_void_p(stream) if stream else c_void_p(None), byref(self._h))
        if rc != 0:
            raise ArrowError(rc, (self.lib.arrow_last_error(None) or b"").decode())
        self.device = int(device)

    # -- plumbing ---------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc != 0:
            raise ArrowError(rc, (self.lib.arrow_last_error(self._h) or b"").decode())

    def close(self):
        if self._h:
            self.lib.arrow_ctx_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        self._check(self.lib.arrow_sync(self._h))

    def preload_kernels(self, k: int):
        """load every kernel a step with ``k`` feature columns can launch, before any peer barrier is in flight"""
        self._check(self.lib.arrow_preload_kernels(self._h, int(k)))

    def device_info(self):
        sm, fr, tot = c_int(), c_int64(), c_int64()
        self._check(self.lib.arrow_device_info(self._h, byref(sm), byref(fr), byref(tot)))
        return sm.value, fr.value, tot.value

    def set_tuning(self, long_row_threshold: int, long_row_segment: int):
        self._check(self.lib.arrow_set_tuning(self._h, int(long_row_threshold), int(long_row_segment)))

    OPT_L2_HINTS_PLAIN, OPT_L2_HINTS_FUSED, OPT_BIG_TILES, OPT_SPMM_CTAS_PER_SM, OPT_PREFETCH = 1, 2, 3, 4, 5
    OPT_ROWS_PER_GROUP, OPT_SPMM_SM_LIMIT, OPT_PUSH_CTAS, OPT_BARRIER_TIMEOUT_MS, OPT_SMEM_CARVEOUT = 6, 7, 8, 9, 10
    OPT_FORCE_PREDICATED, OPT_TILE_KERNEL, OPT_PUSH_INTERLEAVE = 11, 12, 13

    def set_option(self, option: int, value: int):
        self._check(self.lib.arrow_set_option(self._h, int(option), int(value)))

    # -- sparse -----------------------------------------------------------------------------
    def csr_upload(self, n_rows: int, n_cols: int, indptr: np.ndarray, indices: np.ndarray,
                   data: Optional[np.ndarray]) -> "Csr":
        """`indptr` may be a slice of a larger row pointer; indices/data are the matching slices."""
        indptr = np.ascontiguousarray(indptr)
        if indptr.dtype not in (np.int32, np.int64):
            indptr = indptr.astype(np.int64)
        nnz = int(indptr[-1] - indptr[0]) if indptr.size else 0
        indices = np.ascontiguousarray(indices)
        if indices.dtype not in (np.int32, np.int64):
            indices = indices.astype(np.int64)
        if indices.size != nnz:
            raise ValueError(f"indices has {indices.size} entries, indptr spans {nnz}")
        if data is not None:
            data = np.ascontiguousarray(data, dtype=np.float32)
            if data.size != nnz:
                raise ValueError(f"data has {data.size} entries, indptr spans {nnz}")
        h = c_int()
        self._check(self.lib.arrow_csr_upload(self._h, int(n_rows), int(n_cols), nnz, _ptr(indptr), indptr.dtype.itemsize,
                                              _ptr(indices), indices.dtype.itemsize, _ptr(data), byref(h)))
        return Csr(self, h.value, int(n_rows), int(n_cols), nnz)

    def csr_from_scipy(self, A) -> "Csr":
        from scipy import sparse
        A = sparse.csr_matrix(A)
        return self.csr_upload(A.shape[0], A.shape[1], A.indptr, A.indices, A.data.astype(np.float32, copy=False))

    # -- maps -------------------------------------------------------------------------------
    def map_upload(self, m: np.ndarray, limit: int) -> "RowMap":
        m = np.ascontiguousarray(m, dtype=np.int64)
        h = c_int()
        self._check(self.lib.arrow_map_upload(self._h, _ptr(m), m.size, int(limit), byref(h)))
        return RowMap(self, h.value, m.size, int(limit))

    # -- dense ------------------------------------------------------------------------------
    def dense_alloc(self, rows: int, k: int, dtype="float32") -> "Dense":
        """zero-filled ``rows x k`` tile of ``dtype`` (float32 or bfloat16, see ``dtype_name``)"""
        dtype = dtype_name(dtype)
        h = c_int()
        if dtype == "float32":
            self._check(self.lib.arrow_dense_alloc(self._h, int(rows), int(k), byref(h)))
        else:
            self._check(self.lib.arrow_dense_alloc_dtype(self._h, int(rows), int(k), DTYPE_CODES[dtype], byref(h)))
        return Dense(self, h.value, int(rows), int(k), owned=True, dtype=dtype)

    def dense_wrap(self, device_ptr: int, rows: int, k: int) -> "Dense":
        h = c_int()
        self._check(self.lib.arrow_dense_wrap(self._h, c_void_p(device_ptr), int(rows), int(k), byref(h)))
        return Dense(self, h.value, int(rows), int(k), owned=False)

    def dense_from_host(self, X: np.ndarray) -> "Dense":
        X = np.ascontiguousarray(X, dtype=np.float32)
        d = self.dense_alloc(X.shape[0], X.shape[1])
        d.h2d(X)
        self.sync()
        return d

    def ipc_import(self, handle: bytes, rows: int, k: int) -> "Dense":
        assert len(handle) == IPC_HANDLE_BYTES
        buf = ctypes.create_string_buffer(handle, IPC_HANDLE_BYTES)
        h = c_int()
        self._check(self.lib.arrow_ipc_import(self._h, buf, int(rows), int(k), byref(h)))
        return Dense(self, h.value, int(rows), int(k), owned=False)

    # -- hot path ---------------------------------------------------------------------------
    def spmm(self, A: "Csr", X: "Dense", C: "Dense", rowmap: Optional["RowMap"] = None,
             accumulate: bool = False, variant: int = VARIANT_AUTO):
        self._check(self.lib.arrow_spmm(self._h, A.h, X.h, C.h, rowmap.h if rowmap is not None else -1,
                                        ACCUMULATE if accumulate else 0, int(variant)))

    def spmm_add(self, A: "Csr", X: "Dense", C: "Dense", add: "Dense", add_map: "RowMap", variant: int = VARIANT_AUTO):
        """C[r] = (A X)[r] + add[add_map[r]] (where add_map[r] >= 0)"""
        self._check(self.lib.arrow_spmm_add(self._h, A.h, X.h, C.h, add.h, add_map.h, int(variant)))

    def spmm_ex(self, A: "Csr", X: "Dense", C: Optional["Dense"] = None, X2: Optional["Dense"] = None, x_split: int = 0,
                out_table: Optional["PtrTable"] = None, add: Optional["Dense"] = None, add_map: Optional["RowMap"] = None,
                variant: int = VARIANT_AUTO):
        """Generalised product (``arrow_spmm_ex``): two-part X operand, row-pointer epilogue, gather-add."""
        self._check(self.lib.arrow_spmm_ex(self._h, A.h, X.h, X2.h if X2 is not None else -1, int(x_split),
                                           C.h if C is not None else -1, out_table.h if out_table is not None else -1,
                                           add.h if add is not None else -1, add_map.h if add_map is not None else -1,
                                           int(variant)))

    def ptrtable_upload(self, tiles: Sequence["Dense"], which: np.ndarray, row: np.ndarray) -> "PtrTable":
        which = np.ascontiguousarray(which, dtype=np.int32)
        row = np.ascontiguousarray(row, dtype=np.int64)
        assert which.shape == row.shape and which.ndim == 1
        n = len(tiles)
        hs = (c_int * n)(*[t.h for t in tiles])
        h = c_int()
        self._check(self.lib.arrow_ptrtable_upload(self._h, hs, n, _ptr(which), _ptr(row), which.size, byref(h)))
        return PtrTable(self, h.value, which.size)

    def push_rows(self, dsts: Sequence[Optional["Dense"]], item_bounds: Sequence[int], src: "Dense", m: "RowMap"):
        n = len(dsts)
        hs = (c_int * n)(*[(d.h if d is not None else -1) for d in dsts])
        bd = (c_int64 * (n + 1))(*[int(b) for b in item_bounds])
        self._check(self.lib.arrow_push_rows(self._h, hs, bd, n, src.h, m.h))

    def reduce_rows(self, srcs: Sequence["Dense"], rows: int, dst: Optional["Dense"] = None,
                    out_table: Optional["PtrTable"] = None):
        n = len(srcs)
        hs = (c_int * n)(*[s.h for s in srcs])
        self._check(self.lib.arrow_reduce_rows(self._h, dst.h if dst is not None else -1,
                                               out_table.h if out_table is not None else -1, hs, n, int(rows)))

    # -- graphs -----------------------------------------------------------------------------
    def graph_begin(self):
        self._check(self.lib.arrow_graph_begin(self._h))

    def graph_end(self) -> int:
        h = c_int()
        self._check(self.lib.arrow_graph_end(self._h, byref(h)))
        return h.value

    def graph_launch(self, g: int):
        self._check(self.lib.arrow_graph_launch(self._h, int(g)))

    def graph_free(self, g: int):
        self._check(self.lib.arrow_graph_free(self._h, int(g)))

    def gather_rows(self, dst: "Dense", src: "Dense", m: "RowMap", accumulate: bool = False):
        self._check(self.lib.arrow_gather_rows(self._h, dst.h, src.h, m.h, ACCUMULATE if accumulate else 0))

    def gather_rows_multi(self, dst: "Dense", srcs: Sequence["Dense"], row_bounds: Sequence[int], m: "RowMap",
                          accumulate: bool = False):
        n = len(srcs)
        hs = (c_int * n)(*[s.h for s in srcs])
        bd = (c_int64 * (n + 1))(*[int(b) for b in row_bounds])
        self._check(self.lib.arrow_gather_rows_multi(self._h, dst.h, hs, bd, n, m.h, ACCUMULATE if accumulate else 0))

    def peer_barrier(self, flag_tiles: Sequence["Dense"], rank: int):
        n = len(flag_tiles)
        hs = (c_int * n)(*[s.h for s in flag_tiles])
        self._check(self.lib.arrow_peer_barrier(self._h, hs, int(rank), n))

    # -- copy lanes -------------------------------------------------------------------------
    LANE_MAIN, LANE_H2D, LANE_D2H = 0, 1, 2

    def h2d_lane(self, lane: int, dst: "Dense", X, row0: int = 0):
        """``X``: float32 numpy rows for an fp32 tile, a contiguous CPU bf16 tensor for a bf16 tile"""
        if dst.dtype == "bfloat16":
            _check_bf16_host(X, dst.k)
            self._check(self.lib.arrow_dense_put(self._h, lane, dst.h, int(row0), X.shape[0], c_void_p(X.data_ptr())))
            return
        assert X.dtype == np.float32 and X.flags.c_contiguous and X.shape[1] == dst.k
        self._check(self.lib.arrow_dense_h2d_lane(self._h, lane, dst.h, int(row0), X.shape[0], _ptr(X)))

    def d2h_lane(self, lane: int, src: "Dense", out, row0: int = 0):
        if src.dtype == "bfloat16":
            _check_bf16_host(out, src.k)
            self._check(self.lib.arrow_dense_get(self._h, lane, src.h, int(row0), out.shape[0], c_void_p(out.data_ptr())))
            return
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.shape[1] == src.k
        self._check(self.lib.arrow_dense_d2h_lane(self._h, lane, src.h, int(row0), out.shape[0], _ptr(out)))

    def lane_wait(self, waiting_lane: int, signalling_lane: int):
        self._check(self.lib.arrow_lane_wait(self._h, waiting_lane, signalling_lane))

    def lane_sync(self, lane: int):
        self._check(self.lib.arrow_lane_sync(self._h, lane))

    def set_lane(self, lane: int):
        self._check(self.lib.arrow_set_lane(self._h, lane))

    def event_record(self, event: int, lane: int):
        self._check(self.lib.arrow_event_record(self._h, event, lane))

    def event_wait(self, event: int, lane: int):
        self._check(self.lib.arrow_event_wait(self._h, event, lane))

    # -- timing -----------------------------------------------------------------------------
    def timer_start(self, slot: int = 0):
        self._check(self.lib.arrow_timer_start(self._h, slot))

    def timer_stop(self, slot: int = 0):
        self._check(self.lib.arrow_timer_stop(self._h, slot))

    def timer_ms(self, slot: int = 0) -> float:
        ms = c_float()
        self._check(self.lib.arrow_timer_elapsed_ms(self._h, slot, byref(ms)))
        return float(ms.value)

    def launch_count(self) -> int:
        n = c_int64()
        self._check(self.lib.arrow_launch_count(self._h, byref(n)))
        return int(n.value)

    def l2_flush(self):
        self._check(self.lib.arrow_l2_flush(self._h))


class _Handle:
    def __init__(self, ctx: Context, h: int):
        self.ctx, self.h = ctx, h

    def _free(self, fn_name: str):
        if self.h >= 0 and self.ctx is not None and self.ctx._h:
            self.ctx._check(getattr(self.ctx.lib, fn_name)(self.ctx._h, self.h))     # a refused free keeps the handle
        self.h = -1


class Csr(_Handle):
    def __init__(self, ctx, h, n_rows, n_cols, nnz):
        super().__init__(ctx, h)
        self.n_rows, self.n_cols, self.nnz = n_rows, n_cols, nnz

    def info(self):
        v = [c_int64() for _ in range(5)]
        self.ctx._check(self.ctx.lib.arrow_csr_info(self.ctx._h, self.h, *[byref(x) for x in v]))
        return dict(zip(("n_rows", "n_cols", "nnz", "max_row_nnz", "n_long_rows"), (x.value for x in v)))

    def remap_columns(self, m: "RowMap", new_n_cols: int) -> "Csr":
        h = c_int()
        self.ctx._check(self.ctx.lib.arrow_csr_remap_columns(self.ctx._h, self.h, m.h, int(new_n_cols), byref(h)))
        out = Csr(self.ctx, h.value, self.n_rows, int(new_n_cols), self.nnz)
        out._parent = self           # shares indptr/values: keep the source alive
        return out

    def free(self):
        self._free("arrow_csr_free")


class RowMap(_Handle):
    def __init__(self, ctx, h, n, limit):
        super().__init__(ctx, h)
        self.n, self.limit = n, limit

    def compose(self, outer: "RowMap") -> "RowMap":
        h = c_int()
        self.ctx._check(self.ctx.lib.arrow_map_compose(self.ctx._h, self.h, outer.h, byref(h)))
        return RowMap(self.ctx, h.value, self.n, outer.limit)

    def invert(self, n_out: int) -> "RowMap":
        h = c_int()
        self.ctx._check(self.ctx.lib.arrow_map_invert(self.ctx._h, self.h, int(n_out), byref(h)))
        return RowMap(self.ctx, h.value, int(n_out), self.n)

    def to_host(self) -> np.ndarray:
        out = np.empty(self.n, dtype=np.int32)
        self.ctx._check(self.ctx.lib.arrow_map_d2h(self.ctx._h, self.h, _ptr(out), self.n))
        return out

    def free(self):
        self._free("arrow_map_free")


class PtrTable(_Handle):
    def __init__(self, ctx, h, n):
        super().__init__(ctx, h)
        self.n = n

    def free(self):
        self._free("arrow_ptrtable_free")


def _check_bf16_host(t, k: int):
    import torch
    if not (isinstance(t, torch.Tensor) and t.dtype == torch.bfloat16 and t.device.type == "cpu" and t.is_contiguous()
            and t.dim() == 2 and t.shape[1] == k):
        raise ValueError(f"a bf16 tile moves rows as a contiguous CPU torch.bfloat16 tensor of [rows x {k}]")


class Dense(_Handle):
    def __init__(self, ctx, h, rows, k, owned, dtype="float32"):
        super().__init__(ctx, h)
        self.rows, self.k, self.owned, self.dtype = rows, k, owned, dtype

    def h2d(self, X, row0: int = 0):
        """Upload rows starting at ``row0``.  A bf16 tile takes a CPU bf16 tensor, or float32 data that is rounded on the
        host to nearest even (``to_bf16``)."""
        if self.dtype == "bfloat16":
            X = to_bf16(X)
            _check_bf16_host(X, self.k)
            self.ctx._check(self.ctx.lib.arrow_dense_put(self.ctx._h, 0, self.h, int(row0), X.shape[0], c_void_p(X.data_ptr())))
            self._keep = X
            return
        X = np.ascontiguousarray(X, dtype=np.float32)
        if X.ndim != 2 or X.shape[1] != self.k:
            raise ValueError(f"expected [rows x {self.k}] fp32, got {X.shape}")
        self.ctx._check(self.ctx.lib.arrow_dense_h2d(self.ctx._h, self.h, int(row0), X.shape[0], _ptr(X)))
        self._keep = X                  # async copy: keep the host array alive until the next sync

    def d2h(self, out=None, row0: int = 0, rows: Optional[int] = None, sync: bool = True):
        """Download rows: a float32 numpy array, or a CPU bf16 tensor for a bf16 tile (``out`` of the same kind)."""
        rows = self.rows - row0 if rows is None else rows
        if self.dtype == "bfloat16":
            import torch
            if out is None:
                out = torch.empty((rows, self.k), dtype=torch.bfloat16)
            _check_bf16_host(out, self.k)
            assert out.shape[0] == rows
            self.ctx._check(self.ctx.lib.arrow_dense_get(self.ctx._h, 0, self.h, int(row0), int(rows), c_void_p(out.data_ptr())))
            if sync:
                self.ctx.sync()
            return out
        if out is None:
            out = np.empty((rows, self.k), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.shape == (rows, self.k)
        self.ctx._check(self.ctx.lib.arrow_dense_d2h(self.ctx._h, self.h, int(row0), int(rows), _ptr(out)))
        if sync:
            self.ctx.sync()
        return out

    def fill(self, v: float = 0.0):
        self.ctx._check(self.ctx.lib.arrow_dense_fill(self.ctx._h, self.h, float(v)))

    def copy_from(self, src: "Dense", dst_row0: int = 0, src_row0: int = 0, rows: Optional[int] = None):
        rows = min(self.rows - dst_row0, src.rows - src_row0) if rows is None else rows
        self.ctx._check(self.ctx.lib.arrow_dense_copy(self.ctx._h, self.h, int(dst_row0), src.h, int(src_row0), int(rows)))

    def device_ptr(self) -> int:
        p = c_void_p()
        self.ctx._check(self.ctx.lib.arrow_dense_ptr(self.ctx._h, self.h, byref(p), None, None))
        return int(p.value)

    def ipc_export(self) -> bytes:
        buf = ctypes.create_string_buffer(IPC_HANDLE_BYTES)
        self.ctx._check(self.ctx.lib.arrow_ipc_export(self.ctx._h, self.h, buf))
        return buf.raw

    def free(self):
        self._free("arrow_dense_free")

"""``ArrowSlimMPI`` for B200: the operator one process exposes for its block-rows of one level.

Mirrors the surface of the reference's ``ArrowSlimMPI`` (``arrow/arrow_slim_mpi.py:25-440``) -- same
method names, argument meaning and aliasing rules -- but a process owns *all* block-rows of its
GPU instead of exactly one, tiles live on the device, and the sparse blocks are uploaded once
(no per-iteration ``_sp2cp``, ``arrow/common/sp2cp.py:6-16``).  The arithmetic happens in
``libarrow_b200.so``; there is no CPU path (``device='cpu'`` raises).
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from . import _lib
from .arrow_matrix import ArrowMatrix


class ArrowSlimMPI(ArrowMatrix):
    """Level ``level`` of a decomposition as seen by this process; backed by an ``ArrowEngine``."""

    def __init__(self, comm, owner=None, level: int = 0):
        self.comm = comm
        self.column_comm = comm
        self.tiles_per_side = 0
        self._owner = owner            # ArrowDecompositionMPI holding the engine
        self._level = level
        self._host_X: Optional[np.ndarray] = None

    # -- engine access ------------------------------------------------------------------------------
    @property
    def _engine(self):
        eng = self._owner._engine if self._owner is not None else None
        if eng is None:
            raise RuntimeError("sparse blocks not loaded yet: call load_sparse_matrix_from_blocks(blocks) first")
        return eng

    def spmm(self, device: str = 'gpu'):
        """This level's arrow product on its current features (``_arrow_spmm``, arrow_slim_mpi.py:246-280)."""
        _require_gpu(device)
        self._engine.spmm_level(self._level)

    def result_tile(self, out=None):
        """Host copy of this process's result rows (a CPU bf16 tensor after ``zero_rhs(dtype=torch.bfloat16)``); pass a
        (pinned) ``out`` of the same kind to avoid an allocation per call."""
        return self._engine.result(self._level, out)

    @property
    def C_i(self) -> np.ndarray:
        """Host copy of this process's result rows (the reference's ``B.C_i`` attribute)."""
        return self.result_tile()

    def feature_tile(self) -> np.ndarray:
        return self._engine.features(self._level)

    def set_features(self, X) -> None:
        """Upload this process's feature rows (level 0).  The reference keeps a reference to ``X``
        (arrow_slim_mpi.py:285-293); here the rows are copied to the device at call time.  With bf16 tiles ``X`` may be
        a CPU bf16 tensor; float32 rows are rounded to nearest even."""
        assert X is not None
        if self._level != 0:
            raise ValueError("features enter at level 0; deeper levels receive them through the exchange")
        eng = self._engine
        if getattr(eng, "dtype", "float32") == "bfloat16":
            eng.set_features(X)
        else:
            eng.set_features(np.ascontiguousarray(X, dtype=np.float32))

    def load_sparse_matrix_from_blocks(self, blocks) -> None:
        """``blocks`` is what ``ArrowDecompositionMPI.load_decomposition_new`` returned."""
        self._owner._build_engine(blocks)
        self.tiles_per_side = self._engine.n_blocks[self._level]

    def zero_rhs(self, number_of_rows_per_rank: int, number_of_columns: int, dtype=np.float32) -> None:
        """Zero the tiles (arrow_slim_mpi.py:354-394).  ``dtype`` is the element type of the feature and result tiles:
        float32 (default) or bfloat16 (``torch.bfloat16`` / ``"bfloat16"``: half the bytes per row, arithmetic still
        float32, one GPU only); switching re-allocates the tiles."""
        assert number_of_rows_per_rank >= 1 and number_of_columns >= 1
        try:
            dtype = _lib.dtype_name(dtype)
        except ValueError:
            raise ValueError(f"the B200 path stores features as float32 or bfloat16 and computes in float32 "
                             f"(like the reference's benchmark, arrow_bench.py:21), not {dtype!r}") from None
        if dtype == "bfloat16" and self.comm.Get_size() > 1:
            raise NotImplementedError("bf16 feature tiles run on one GPU; the N-GPU engine in bf16 (sharded fused step, "
                                      "exchange protocol, NCCL) is a follow-up -- use float32 with more than one rank")
        eng = self._engine
        if number_of_columns != eng.k or number_of_rows_per_rank != eng.width:
            raise ValueError(f"engine was initialised for width={eng.width}, k={eng.k}")
        if hasattr(eng, "set_dtype"):
            eng.set_dtype(dtype)
        eng.zero_rhs()

    def is_column_rank(self) -> bool:
        return True

    def allgather_result(self, C: np.ndarray) -> np.ndarray:
        """Fill the caller's ``(tiles_per_side*width) x k`` array with the whole level's result (every process)."""
        assert C is not None
        eng = self._engine
        mine = eng.result(self._level)
        parts = self.comm.allgather(mine) if self.comm.Get_size() > 1 else [mine]
        full = np.concatenate(parts) if len(parts) > 1 else parts[0]
        if C.shape != full.shape or C.dtype != np.float32:
            raise ValueError(f"C must be float32 of shape {full.shape}")
        C[:] = full
        return C

    def set_features_slice_from_features(self, X: np.ndarray) -> None:
        """Take this process's rows out of the full level-0 feature matrix."""
        eng = self._engine
        r0 = eng.plan.levels[0].r0 if hasattr(eng, "plan") else 0
        self.set_features(X[r0:r0 + eng.local_rows_of(0)])

    @staticmethod
    def column_subgroup(tiles_per_side, group):
        return group

    @staticmethod
    def row_subgroup(tiles_per_side, group):
        return group


def _require_gpu(device: str):
    if device != 'gpu':
        raise NotImplementedError(
            f"device={device!r}: arrow_matrix_b200 only implements the B200 path (device='gpu'); "
            "there is deliberately no CPU fallback -- run the reference for --device cpu")

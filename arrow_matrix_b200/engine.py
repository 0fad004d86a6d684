"""Single-GPU arrow SpMM engine: device-resident levels + the per-iteration step.

This is the B200 replacement for the body of ``ArrowDecompositionMPI.step()``
(``arrow/arrow_dec_mpi.py:283-307``) and ``ArrowSlimMPI._ad_spmm[_gpu]``
(``arrow/arrow_slim_mpi.py:78-244``) when one GPU holds every block-row of every level.  The
reference maps one MPI rank to one block-row and refuses to run with fewer ranks
(``arrow/arrow_bench.py:70-78``); here ranks and block-rows are decoupled.

Two execution modes, same results:

* ``exchange`` -- literal protocol: forward gather level by level, one SpMM per level, backward
  gather-add level by level.  Every level's tiles exist on the device exactly as the reference's
  ranks would hold them, including the ``X is C`` aliasing and the stale rows behind the
  sentinel (``arrow_dec_mpi.py:438, 544-545``).
* ``fused`` -- the forward permutation is folded into each level's column indices (they address
  level-0 rows directly) and the backward scatter-add into the SpMM epilogue
  (``C_0[map_j[r]] += ...``); no gather kernel runs and levels > 0 never materialise their tiles.
  Chosen automatically when no non-zero of a level reads a row behind the sentinel (then both
  modes are mathematically identical); otherwise the engine stays in ``exchange`` mode.

Feature and result tiles are float32 (default) or bfloat16 (``dtype``, ``set_dtype``); CSR values and all arithmetic stay
float32, and every stored bf16 row is rounded once to nearest even (DESIGN.md, numerics of bf16 tiles).  bf16 host
rows are CPU ``torch.bfloat16`` tensors.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from . import decomp


class _LevelState:
    __slots__ = ("rows", "n_blocks", "csr", "csr_fused", "to_prev", "to_next_dev", "to_prev_dev", "cmap_dev",
                 "bufs", "xi", "ci", "nnz", "dropped", "cbuf")

    def __init__(self):
        self.csr = self.csr_fused = None
        self.to_prev = None
        self.to_prev_dev = self.to_next_dev = self.cmap_dev = None
        self.bufs = [None, None]
        self.xi = self.ci = 0
        self.cbuf = None


class ArrowEngine:
    """All levels of one decomposition resident on one GPU."""

    def __init__(self, decomposition: Sequence[Tuple[decomp.Level, np.ndarray]], width: int, k: int,
                 block_diagonal: bool = True, device: int = 0, mode: str = "auto", stream: Optional[int] = None,
                 variant: int = _lib.VARIANT_AUTO, n_blocks: Optional[Sequence[int]] = None,
                 ctx: Optional[_lib.Context] = None, fused_style: str = "gather", dtype="float32"):
        if mode not in ("auto", "fused", "exchange"):
            raise ValueError(f"mode must be auto|fused|exchange, got {mode!r}")
        self.ctx = ctx if ctx is not None else _lib.Context(device, stream)
        self.width, self.k, self.variant = int(width), int(k), variant
        self.dtype = _lib.dtype_name(dtype)
        if fused_style not in ("gather", "scatter"):
            raise ValueError("fused_style must be 'gather' or 'scatter'")
        self.fused_style = fused_style
        self.block_diagonal = block_diagonal
        self.L = len(decomposition)
        if self.L == 0:
            raise ValueError("empty decomposition")
        self.n_blocks = [decomp.number_of_blocks(B, width) for B, _ in decomposition] if n_blocks is None \
            else [int(b) for b in n_blocks]
        self.perms, self.to_prev, self.to_next, self.sentinel = decomp.prepare_permutations(
            [p for _, p in decomposition], self.n_blocks, width)
        self.levels: List[_LevelState] = []
        fused_ok = True
        cmap_prev = None                      # level j-1 row -> level-0 row (host, int64, -1 invalid)
        for j, (B, _) in enumerate(decomposition):
            st = _LevelState()
            st.n_blocks = self.n_blocks[j]
            st.rows = st.n_blocks * width
            ip, idx, dat, dropped = decomp.arrow_rows(B, width, st.n_blocks, block_diagonal, 0, st.rows)
            st.dropped = dropped
            st.nnz = int(ip[-1])
            st.csr = self.ctx.csr_upload(st.rows, st.rows, ip, idx, dat)
            if j > 0:
                tp = self.to_prev[j][: st.rows]
                prev_rows = self.levels[j - 1].rows
                st.to_prev = tp
                st.to_prev_dev = self.ctx.map_upload(tp, prev_rows)
                st.to_next_dev = st.to_prev_dev.invert(prev_rows)          # level j-1 row -> level j row
                valid = tp < prev_rows
                safe = np.where(valid, tp, 0)
                if j == 1:
                    cmap = np.where(valid, tp, -1)
                else:
                    cmap = np.where(valid, cmap_prev[safe], -1)
                cmap_prev = cmap
                # fused mode needs every referenced column to be routed all the way from level 0
                if np.any(cmap[idx] < 0):
                    fused_ok = False
                st.cmap_dev = self.ctx.map_upload(cmap, self.levels[0].rows)
            else:
                cmap_prev = np.arange(st.rows, dtype=np.int64)
            self.levels.append(st)
        if mode == "fused" and not fused_ok:
            raise ValueError("fused mode requested but a level reads rows behind the sentinel; use mode='exchange'")
        self.mode = ("fused" if fused_ok else "exchange") if mode == "auto" else mode
        self.fused_ok = fused_ok
        self._alloc_buffers()
        self.total_nnz = sum(st.nnz for st in self.levels)
        self.ctx.sync()

    # -- buffers ---------------------------------------------------------------------------------
    def _alloc_buffers(self):
        for j, st in enumerate(self.levels):
            if j == 0 or self.mode == "exchange":
                st.bufs = [self._tile(st.rows), self._tile(st.rows)]
                st.xi, st.ci = 0, 0             # zero_rhs: X and C both zero (arrow_slim_mpi.py:354-394)
            if j > 0 and self.mode == "fused":
                st.csr_fused = st.csr.remap_columns(st.cmap_dev, self.levels[0].rows)
                if self.fused_style == "gather":
                    st.cbuf = self._tile(st.rows)     # this level's result tile, written once per step

    def _tile(self, rows: int) -> _lib.Dense:
        return self.ctx.dense_alloc(rows, self.k, self.dtype)

    @property
    def itemsize(self) -> int:
        """bytes per feature element"""
        return 2 if self.dtype == "bfloat16" else 4

    def set_mode(self, mode: str):
        """Switch between 'fused' and 'exchange' (re-allocates level tiles; features are reset)."""
        if mode == self.mode:
            return
        if mode == "fused" and not self.fused_ok:
            raise ValueError("fused mode is not valid for this decomposition")
        self._release_buffers()
        self.mode = mode
        self._alloc_buffers()

    def set_dtype(self, dtype):
        """Switch the feature / result tiles between float32 and bfloat16 (re-allocates level tiles and streaming slots
        like ``set_mode``; features are reset to zero)."""
        dtype = _lib.dtype_name(dtype)
        if dtype == self.dtype:
            return
        self._release_buffers()
        self.dtype = dtype
        self._alloc_buffers()

    def _release_buffers(self):
        if hasattr(self, "_slots"):                 # streaming slots hold level-0 tiles of the old mode
            self.stream_drain()
            for b in self._slots[1]:
                b.free()
            self.levels[0].bufs = list(self._slots[0])
            del self._slots
        for st in self.levels:
            for b in st.bufs:
                if b is not None:
                    b.free()
            st.bufs = [None, None]
            if st.csr_fused is not None:
                st.csr_fused.free()
                st.csr_fused = None
            if st.cbuf is not None:
                st.cbuf.free()
                st.cbuf = None

    @property
    def n_rows(self) -> int:
        return self.levels[0].rows

    # -- features / results (level-0 row order, like the reference's per-rank tiles) -----------------
    def set_features(self, X, sync: bool = True):
        """Level-0 feature tiles, concatenated (``B.set_features`` on every level-0 rank).  A bf16 engine takes a CPU
        bf16 tensor, or float32 rows it rounds to nearest even."""
        st = self.levels[0]
        if X.shape != (st.rows, self.k):
            raise ValueError(f"expected features of shape {(st.rows, self.k)}, got {X.shape}")
        if st.xi == st.ci:                      # X aliases C: keep the result tile intact, like a rebind
            st.xi = 1 - st.ci
        st.bufs[st.xi].h2d(X)
        if sync:
            self.ctx.sync()

    def rewind_features(self):
        """Point level 0 back at the tile the last ``set_features`` filled (no copy), so the next ``step()``
        multiplies the same features again instead of chaining -- the benchmark's "fresh X every iteration"
        (``arrow_bench.py:113-116``) without a host round trip.  ``step()`` never writes that tile."""
        st = self.levels[0]
        if st.xi == st.ci:
            st.xi = 1 - st.ci

    def features_buffer(self) -> _lib.Dense:
        st = self.levels[0]
        return st.bufs[st.xi]

    def result_buffer(self, level: int = 0) -> _lib.Dense:
        st = self.levels[level]
        if st.bufs[0] is None:
            if st.cbuf is not None:             # fused/gather keeps every level's aggregated result tile
                return st.cbuf
            raise RuntimeError("level tiles are not materialised in fused/scatter mode; use mode='exchange'")
        return st.bufs[st.ci]

    def result(self, level: int = 0, out: Optional[np.ndarray] = None) -> np.ndarray:
        return self.result_buffer(level).d2h(out)

    # -- small uniform API shared with the sharded engine (used by the reference-facing classes) ----------
    def local_rows_of(self, level: int) -> int:
        return self.levels[level].rows

    def zero_rhs(self):
        """``zero_rhs`` on every rank of every level (arrow_slim_mpi.py:354-394)."""
        for st in self.levels:
            for b in st.bufs:
                if b is not None:
                    b.fill(0.0)
            st.xi = st.ci = 0

    def features(self, level: int = 0, out: Optional[np.ndarray] = None) -> np.ndarray:
        st = self.levels[level]
        if st.bufs[st.xi] is None:
            raise RuntimeError("level tiles are not materialised in fused mode; use mode='exchange'")
        return st.bufs[st.xi].d2h(out)

    def spmm_level(self, level: int):
        """One level's arrow product on its current features (``B.spmm()`` of that level)."""
        self.ensure_level_tiles()
        st = self.levels[level]
        out = 1 - st.xi
        self.ctx.spmm(st.csr, st.bufs[st.xi], st.bufs[out], variant=self.variant)
        st.ci = out

    def ensure_level_tiles(self):
        """Materialise per-level tiles (exchange mode) keeping level 0's current tiles."""
        if self.mode == "exchange":
            return
        st0 = self.levels[0]
        keep = [b.d2h() for b in st0.bufs]
        xi, ci = st0.xi, st0.ci
        self.set_mode("exchange")
        st0 = self.levels[0]
        for b, h in zip(st0.bufs, keep):
            b.h2d(h)
        st0.xi, st0.ci = xi, ci
        self.ctx.sync()

    def sync(self):
        if hasattr(self, "_slots"):
            self.stream_drain()
        self.ctx.sync()

    # -- the iteration ----------------------------------------------------------------------------------
    def propagate_features(self):
        """Forward exchange (``_propagate_features_forwards``, arrow_dec_mpi.py:507-550)."""
        if self.mode == "fused":
            return
        for j in range(1, self.L):
            st, prev = self.levels[j], self.levels[j - 1]
            self.ctx.gather_rows(st.bufs[st.ci], prev.bufs[prev.xi], st.to_prev_dev)      # C_i[perm] = recvbuf (:544)
            st.xi = st.ci                                                                 # set_features(C_i) (:545)

    def spmm(self):
        """Every level's arrow product (``B.spmm``, arrow_slim_mpi.py:246-280 + :78-155)."""
        if self.mode == "fused":
            st0 = self.levels[0]
            x = st0.bufs[st0.xi]
            out = 1 - st0.xi
            if self.fused_style == "gather":
                # deepest level first; every level writes its tile once and ADDS the deeper level's rows that map onto
                # its own (C_j[r] += C_{j+1}[to_next_j[r]]): the reference's backward aggregation as an epilogue gather
                for j in range(self.L - 1, 0, -1):
                    st = self.levels[j]
                    if j == self.L - 1:
                        self.ctx.spmm(st.csr_fused, x, st.cbuf, variant=self.variant)
                    else:
                        nxt = self.levels[j + 1]
                        self.ctx.spmm_add(st.csr_fused, x, st.cbuf, nxt.cbuf, nxt.to_next_dev, variant=self.variant)
                if self.L > 1:
                    nxt = self.levels[1]
                    self.ctx.spmm_add(st0.csr, x, st0.bufs[out], nxt.cbuf, nxt.to_next_dev, variant=self.variant)
                else:
                    self.ctx.spmm(st0.csr, x, st0.bufs[out], variant=self.variant)
            else:
                self.ctx.spmm(st0.csr, x, st0.bufs[out], variant=self.variant)
                for st in self.levels[1:]:
                    self.ctx.spmm(st.csr_fused, x, st0.bufs[out], rowmap=st.cmap_dev, accumulate=True,
                                  variant=self.variant)
            st0.ci = out
            return
        for st in self.levels:
            out = 1 - st.xi
            self.ctx.spmm(st.csr, st.bufs[st.xi], st.bufs[out], variant=self.variant)     # C_i = A @ X_i: fresh tile
            st.ci = out

    def aggregate(self):
        """Backward exchange (``_aggregate_features_backwards``, arrow_dec_mpi.py:404-440)."""
        if self.mode == "fused":
            st0 = self.levels[0]
            st0.xi = st0.ci                                                               # X := A X  (:289, :438)
            return
        for j in range(self.L - 1, 0, -1):
            st, prev = self.levels[j], self.levels[j - 1]
            # C_{j-1}[to_prev[r]] += C_j[r], written as a gather-add over level j-1 rows (to_prev is injective)
            self.ctx.gather_rows(prev.bufs[prev.ci], st.bufs[st.ci], st.to_next_dev, accumulate=True)
            prev.xi = prev.ci                                                             # set_features(C_i) (:438)

    def step(self):
        """One ``ArrowDecompositionMPI.step()``; stream-ordered, does not synchronise."""
        self.propagate_features()
        self.spmm()
        self.aggregate()

    # -- streaming iteration for host-resident features ------------------------------------------------------
    def stream_step(self, X_host: np.ndarray, out_host: np.ndarray):
        """Enqueue one full iteration on host data: upload ``X_host`` -> ``step()`` -> download level-0 result
        into ``out_host``.  Returns immediately; uploads, compute and downloads of consecutive calls overlap
        (side copy streams ordered with events, two device slots).  Both arrays must be pinned
        (``_lib.PinnedArray``; for a bf16 engine the ``tensor`` of a ``_lib.PinnedTensor``) and must stay untouched until ``stream_drain()``; use at least two
        (X, out) pairs in rotation.  Results are identical to ``set_features(X); step(); result()``."""
        st = self.levels[0]
        if X_host.shape != (st.rows, self.k) or out_host.shape != (st.rows, self.k):
            raise ValueError(f"expected host arrays of shape {(st.rows, self.k)}")
        ctx = self.ctx
        if not hasattr(self, "_slots"):
            # slot 0 re-uses the engine's own level-0 tiles, slot 1 gets two more
            self._slots = [list(st.bufs), [self._tile(st.rows), self._tile(st.rows)]]
            self._slot_i = 0
        s = self._slot_i % 2
        slot = self._slots[s]
        self._slot_i += 1
        EV_H2D, EV_MAIN, EV_D2H = 3 * s, 3 * s + 1, 3 * s + 2      # per-slot events
        ctx.event_wait(EV_MAIN, ctx.LANE_H2D)      # the compute two calls ago has finished reading slot[0]
        ctx.h2d_lane(ctx.LANE_H2D, slot[0], X_host)
        ctx.event_record(EV_H2D, ctx.LANE_H2D)
        ctx.event_wait(EV_H2D, ctx.LANE_MAIN)      # features are on the device
        ctx.event_wait(EV_D2H, ctx.LANE_MAIN)      # slot[1]'s previous result has been downloaded
        st.bufs = slot
        st.xi, st.ci = 0, 1                        # X = uploaded tile, C = the slot's second tile
        self.step()
        ctx.event_record(EV_MAIN, ctx.LANE_MAIN)
        ctx.event_wait(EV_MAIN, ctx.LANE_D2H)
        ctx.d2h_lane(ctx.LANE_D2H, st.bufs[st.ci], out_host)
        ctx.event_record(EV_D2H, ctx.LANE_D2H)

    def stream_drain(self):
        ctx = self.ctx
        ctx.lane_sync(ctx.LANE_H2D)
        ctx.sync()
        ctx.lane_sync(ctx.LANE_D2H)

    # -- accounting (SURVEY.md 8d) ------------------------------------------------------------------------
    def flops_per_step(self) -> float:
        return 2.0 * self.total_nnz * self.k

    def algorithmic_bytes_per_step(self) -> float:
        """Per level nnz*8 + (R+1)*4 + U*k*e + R*k*e (U = R = active rows, e = bytes per feature element), plus the
        exchanges (forward 2 passes, backward 3 passes over the routed rows) -- the figure a fused
        implementation still reports against."""
        e = self.itemsize
        total = 0.0
        for j, st in enumerate(self.levels):
            total += st.nnz * 8 + (st.rows + 1) * 4 + 2.0 * st.rows * self.k * e
            if j > 0:
                m = int(np.count_nonzero(st.to_prev < self.levels[j - 1].rows))
                total += 5.0 * m * self.k * e
        return total

    def _launch_level_as_in_step(self, j: int, src, dst):
        st = self.levels[j]
        if self.mode == "fused" and self.fused_style == "gather" and j + 1 < self.L:
            nxt = self.levels[j + 1]
            self.ctx.spmm_add(st.csr, src, dst, nxt.cbuf, nxt.to_next_dev, variant=self.variant)
        else:
            self.ctx.spmm(st.csr, src, dst, variant=self.variant)

    def time_level_spmm(self, j: int, iters: int, warmup: int = 3) -> float:
        """Average duration (ms) of level ``j``'s launch exactly as ``step()`` issues it (level 0 of the fused/gather
        path includes the epilogue gather-add of level 1's tile), CUDA events on the engine's stream."""
        st = self.levels[j]
        if j > 0 and self.mode == "fused":
            raise ValueError("levels > 0 are timed through step() in fused mode")
        src = st.bufs[st.xi]
        scratch = self._tile(st.rows)
        for _ in range(warmup):
            self._launch_level_as_in_step(j, src, scratch)
        self.ctx.timer_start(5)
        for _ in range(iters):
            self._launch_level_as_in_step(j, src, scratch)
        self.ctx.timer_stop(5)
        ms = self.ctx.timer_ms(5) / iters
        scratch.free()
        return ms

    def level_bytes(self, j: int) -> float:
        """algorithmic bytes of level ``j``'s launch: nnz*8 + (R+1)*4 + R*k*e (X) + R*k*e (C), e = bytes per feature
        element, plus -- when the launch carries the epilogue gather-add -- one read of the routed rows of the deeper
        level's tile (the other two passes of the reference's backward exchange do not exist in this launch)"""
        st = self.levels[j]
        e = self.itemsize
        b = st.nnz * 8 + (st.rows + 1) * 4 + 2.0 * st.rows * self.k * e
        if self.mode == "fused" and self.fused_style == "gather" and j + 1 < self.L:
            nxt = self.levels[j + 1]
            b += float(np.count_nonzero(nxt.to_prev < st.rows)) * self.k * e
        return b

    def close(self):
        self.ctx.close()

"""``bench_spmm`` -- the driver behind the ``spmm_arrow`` entry point (reference ``arrow/arrow_bench.py:12-137``).

Same signature and flow: (synthesise) -> load -> initialize -> load blocks -> zero_rhs -> iterations of
[fresh features on level 0, barrier, timed ``step()``] -> logs.  Differences: the synthetic input is our
arrow-shaped generator instead of an igraph Barabasi-Albert graph + decomposition (igraph is unavailable),
and any number of GPUs >= 1 works (the reference needs one rank per block-row, ``:70-78``).
"""
from __future__ import annotations

import os
import sys
import time
from typing import Optional

import numpy as np

from . import comm as comm_mod
from . import _lib, graphio, synth, wb_logging
from .arrow_dec_mpi import ArrowDecompositionMPI


def bench_spmm(path: Optional[str], width: int, n_features: int, iterations: int, blocked: bool, device: str,
               p_per_side=3, ba_neighbors: int = 5, wandb_api_key: str = None, datatype=np.float32, slim=False,
               npy_format=True, comm=None, verbose: bool = True, synthetic: str = "arrow"):
    assert width > 0
    comm = comm if comm is not None else comm_mod.world_comm()
    rank = comm.Get_rank()

    if path is None:
        path = 'tmp/test_ba' + "_" + str(p_per_side) + "_" + str(ba_neighbors)
        if rank == 0:
            os.makedirs("tmp", exist_ok=True)
            if synthetic == "ba":
                # the reference's route (arrow_bench.py:33-34): Barabasi-Albert graph -> arrow_decomposition(g, width, 3)
                from .decomposition import arrow_decomposition
                A = synth.barabasi_albert(p_per_side * width, ba_neighbors, 503)
                dec = arrow_decomposition(A, width, 3, block_diagonal=blocked, seed=503)
            else:
                head = max(1, min(3, ba_neighbors // 2))
                dec = synth.synth_decomposition(p_per_side, width, levels=2 if p_per_side > 1 else 1, seed=503,
                                                head_nnz=head, diag_nnz=max(1, ba_neighbors * 2 - head))
            graphio.save_decomposition_new(dec, path, width, block_diagonal=blocked)
            print("DATASET GENERATED -- ", p_per_side * width, " vertices")
        comm.Barrier()

    name = "Arrow_B200_v0.1"
    if blocked:
        name += "_BlockDiagonal"
    if slim:
        name += "_Slim"
    wb_logging.wandb_init(comm, path, n_features, iterations, device, name, width, wandb_api_key)

    # `datatype` is the element type of the feature tiles (float32 or bfloat16); matrix values load as float32 either way
    feature_dtype = _lib.dtype_name(datatype)
    blocks, n_blocks, to_prev, to_next = ArrowDecompositionMPI.load_decomposition_new(
        comm, path, width, blocked, np.float32, slim=slim, use_npy=npy_format)
    if blocks is not None and verbose:
        print("RANK loaded decomposition", rank, n_blocks, flush=True)
    comm.Barrier()
    if np.sum(n_blocks) == 0:
        print("ERROR: Empty Matrix. Check that the file exists and all parameters match (width, block diagonal).",
              file=sys.stderr)
        return None

    arrow = ArrowDecompositionMPI.initialize(comm, n_blocks, to_prev, to_next, width, n_features, device, blocked, slim)
    rng = np.random.default_rng(42 + rank)
    comm.Barrier()
    times = []
    if arrow is not None:
        wb_logging.log({"actual_ranks": comm.Get_size()})
        tic = time.perf_counter()
        arrow.B.load_sparse_matrix_from_blocks(blocks)
        arrow.B.zero_rhs(width, n_features, dtype=feature_dtype)
        arrow.synchronize()
        comm.Barrier()
        wb_logging.log({"init_time": time.perf_counter() - tic})
        rows_local = arrow._engine.local_rows_of(0)
        for i in range(iterations):
            X_p0 = 2 * rng.random((rows_local, n_features), dtype=np.float32) - 1    # arrow_bench.py:115 (bf16: rounded on upload)
            arrow.B.set_features(X_p0)
            comm.Barrier()
            fail = False
            try:
                wb_logging.set_iteration_data({"iteration": i})
                tic = time.perf_counter()
                arrow.step()
                arrow.synchronize()
                toc = time.perf_counter()
                wb_logging.log({"spmm_time": toc - tic})
                times.append(toc - tic)
                if verbose:
                    print("RANK", rank, "Iteration", i, " -- ", toc - tic, "s", flush=True)
            except Exception as e:     # noqa: BLE001 - mirrors the reference's collective abort (:128-134)
                print("RANK", rank, "EXCEPTION", e, flush=True)
                fail = True
            if comm.allreduce_lor(fail):
                print("RANK", rank, "FAILED")
                break
    wb_logging.finish(comm)
    comm.Barrier()
    return dict(arrow=arrow, times=times)

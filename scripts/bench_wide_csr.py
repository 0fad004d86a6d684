"""SpMM launch time of a CSR block with more than 2^32 non-zeros against a 150M-non-zero block of the same recipe.

Both blocks follow the recipe of tests/test_gpu_wide_csr.py: 2^24 columns, row lengths uniform in [0, 258] (129 on
average), each row's columns one contiguous run starting at a hashed column, all values 1.  The large block has 2^25
rows (about 4.33e9 non-zeros, 35 GB of CSR on the device), the small one 1.16M rows (about 150M non-zeros).  For each
block and dtype (fp32, bf16) at k = 16 one JSON line: ms per `arrow_spmm` launch (CUDA events over `--iters` launches
after `--warmup`), the algorithmic bytes nnz*8 + rows*4 + 2*rows*k*e (e = bytes per feature element) and GB/s, and the
rate in non-zeros per ns.  The X tile (2^24 x 16) exceeds the L2 in both dtypes.  The card's name and power limit are
read in the same process.

    python scripts/bench_wide_csr.py --out DIR          # writes DIR/r04_wide_csr.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from arrow_matrix_b200 import _lib

N_COLS, MEAN_LEN, K = 1 << 24, 129, 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")] if q else ("unknown", "unknown", "unknown")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def block(n_rows, seed=7):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 2 * MEAN_LEN + 1, n_rows).astype(np.int64)
    indptr = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(lens, out=indptr[1:])
    start = (np.arange(n_rows, dtype=np.int64) * 2654435761) % N_COLS
    indices = np.empty(int(indptr[-1]), dtype=np.int32)
    step = 1 << 19
    for r0 in range(0, n_rows, step):
        r1 = min(n_rows, r0 + step)
        a, b = int(indptr[r0]), int(indptr[r1])
        shift = np.repeat(start[r0:r1] - (indptr[r0:r1] - a), lens[r0:r1])
        indices[a:b] = (np.arange(b - a, dtype=np.int64) + shift) % N_COLS
    return indptr, indices


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, metavar="DIR", help="directory that receives r04_wide_csr.jsonl")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    ctx = _lib.Context(0)
    info = card()
    X = np.random.default_rng(11).integers(-64, 65, (N_COLS, K)).astype(np.float32)
    lines = []
    for name, n_rows in (("150M", 1_162_790), ("4.3G", 1 << 25)):
        t0 = time.time()
        indptr, indices = block(n_rows)
        nnz = int(indptr[-1])
        A = ctx.csr_upload(n_rows, N_COLS, indptr, indices, None)
        del indices
        build_s = time.time() - t0
        for dtype, e in (("float32", 4), ("bfloat16", 2)):
            Xd = ctx.dense_alloc(N_COLS, K, dtype)
            Xd.h2d(X)
            C = ctx.dense_alloc(n_rows, K, dtype)
            ctx.sync()
            for _ in range(args.warmup):
                ctx.spmm(A, Xd, C)
            ctx.timer_start(0)
            for _ in range(args.iters):
                ctx.spmm(A, Xd, C)
            ctx.timer_stop(0)
            ms = ctx.timer_ms(0) / args.iters
            nbytes = nnz * 8 + n_rows * 4 + 2 * n_rows * K * e
            rec = dict(block=name, rows=n_rows, cols=N_COLS, nnz=nnz, k=K, dtype=dtype, ms=round(ms, 4),
                       algo_bytes=nbytes, gbps=round(nbytes / ms / 1e6, 1), nnz_per_ns=round(nnz / ms / 1e6, 3),
                       iters=args.iters, host_build_upload_s=round(build_s, 1), **info)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
            C.free()
            Xd.free()
        A.free()
        ctx.sync()
    with open(os.path.join(args.out, "r04_wide_csr.jsonl"), "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()

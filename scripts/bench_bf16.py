"""fp32 against bf16 feature tiles on the G2 workload of bench.py (10M rows, width 10 000, 2 levels, seed 503).

For every k the two dtypes run alternately in one process on the same decomposition (one engine each, both resident),
so both see the same card, clocks and neighbours.  Per dtype and k one JSON line: device-resident step time (CUDA events,
``rewind_features``, warm-up), the level-0 launch as the step issues it with its algorithmic bytes at the tile's element
size, and the full-size rank-1 parity property as ``verified``; at k = 128 also ``step_stream`` per step with pinned
host buffers.  The card's name and power limit are read in the same process.

    python scripts/bench_bf16.py --out DIR          # writes DIR/r03_bf16_steps.jsonl
"""
import argparse
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

import bench
from arrow_matrix_b200 import _lib
from arrow_matrix_b200.engine import ArrowEngine


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")] if q else ("unknown", "unknown", "unknown")
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def rank1_u(n):
    """u bf16-representable (one draw for every k: the float64 reference S u is computed once)"""
    u = 2.0 * np.random.default_rng(9001).random(n, dtype=np.float32) - 1.0
    return torch.from_numpy(u).to(torch.bfloat16).float().numpy()


def rank1_features(u, k):
    """X = u v^T with v powers of two: exactly rank 1 in both dtypes"""
    v = (2.0 ** np.random.default_rng(k).integers(-2, 3, k)).astype(np.float32)
    return v, u[:, None] * v[None, :]


def verified(eng, y, v, X):
    """the step on X = u v^T returns (S u) v^T within one bf16 (or fp32) rounding per store point"""
    eng.set_features(X if eng.dtype == "float32" else _lib.to_bf16(X))
    eng.step()
    got = eng.result()
    got = got.float().numpy() if eng.dtype == "bfloat16" else got
    ref_max = float(np.abs(y).max() * np.abs(v).max())
    levels = sum(float(torch.as_tensor(eng.result(j)).float().abs().max()) for j in range(1, eng.L))
    u_rel = 2.0 ** -8 if eng.dtype == "bfloat16" else 2.0 ** -23
    err = 0.0
    for c in range(0, len(v), 16):                       # column blocks keep the float64 temporaries small
        err = max(err, float(np.abs(got[:, c:c + 16] - np.outer(y, v[c:c + 16])).max()))
    return bool(err <= u_rel * (ref_max + levels) + 1e-5 * ref_max), err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=1000)
    ap.add_argument("--width", type=int, default=10000)
    ap.add_argument("--levels", type=int, default=2)
    ap.add_argument("--ks", type=str, default="16,32,64,128")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of fp32 / bf16 per k")
    ap.add_argument("--stream-steps", type=int, default=8)
    ap.add_argument("--out", type=str, required=True, help="directory for r03_bf16_steps.jsonl")
    args = ap.parse_args()
    a = types.SimpleNamespace(workload="g2", blocks=args.blocks, width=args.width, levels=args.levels, perm="random")
    dec = bench.build_decomposition(a)
    info = card()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r03_bf16_steps.jsonl")
    y = None
    with open(path, "w") as out:
        for k in [int(x) for x in args.ks.split(",")]:
            engs = {d: ArrowEngine(dec, args.width, k, dtype=d) for d in ("float32", "bfloat16")}
            n = engs["float32"].n_rows
            if y is None:
                u = rank1_u(n)
                y, state_free = bench.expected_step_on_vector(dec, args.width, u.astype(np.float64))
                assert state_free
            v, X = rank1_features(u, k)
            res = {d: {"step_ms": [], "level0_ms": []} for d in engs}
            for d, e in engs.items():
                res[d]["verified"], res[d]["max_abs_err"] = verified(e, y, v, X)
                e.set_features(X if d == "float32" else _lib.to_bf16(X))
            for _ in range(args.rounds):
                for d, e in engs.items():
                    res[d]["step_ms"].append(bench.time_steps(e, e.ctx, e.ctx.sync, args.steps, args.warmup))
                    res[d]["level0_ms"].append(e.time_level_spmm(0, args.steps))
            for d, e in engs.items():
                r = res[d]
                step_ms, l0_ms = float(np.median(r["step_ms"])), float(np.median(r["level0_ms"]))
                line = {"dtype": d, "k": k, "rows": n, "width": args.width, "levels": args.levels, "mode": e.mode,
                        "step_ms": step_ms, "step_ms_all": r["step_ms"],
                        "level0_ms": l0_ms, "level0_ms_all": r["level0_ms"],
                        "level0_algorithmic_bytes": e.level_bytes(0),
                        "level0_GBps": e.level_bytes(0) / l0_ms / 1e6,
                        "step_algorithmic_bytes": e.algorithmic_bytes_per_step(),
                        "gflops": e.flops_per_step() / step_ms / 1e6,
                        "verified": r["verified"], "max_abs_err": r["max_abs_err"],
                        "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, **info}
                if k == 128:
                    line["stream_ms_per_step"] = stream_ms(e, X, args.stream_steps)
                print(json.dumps(line), flush=True)
                out.write(json.dumps(line) + "\n")
            for e in engs.values():
                e.close()
            del X


def stream_ms(eng, X, steps):
    """``stream_step`` per step (host clock around ``steps`` pipelined calls and the final drain), pinned host pairs"""
    import time
    n, k = X.shape
    if eng.dtype == "bfloat16":
        hx = [_lib.PinnedTensor((n, k)) for _ in range(2)]
        hc = [_lib.PinnedTensor((n, k)) for _ in range(2)]
        xs = [p.tensor for p in hx]
        cs = [p.tensor for p in hc]
        src = _lib.to_bf16(X)
        for t in xs:
            t.copy_(src)
    else:
        hx = [_lib.PinnedArray((n, k)) for _ in range(2)]
        hc = [_lib.PinnedArray((n, k)) for _ in range(2)]
        xs = [p.array for p in hx]
        cs = [p.array for p in hc]
        for t in xs:
            t[:] = X
    for i in range(2):                                   # warm-up: both slots
        eng.stream_step(xs[i], cs[i])
    eng.stream_drain()
    t0 = time.perf_counter()
    for i in range(steps):
        eng.stream_step(xs[i % 2], cs[i % 2])
    eng.stream_drain()
    ms = (time.perf_counter() - t0) * 1e3 / steps
    for p in hx + hc:
        p.close()
    return ms


if __name__ == "__main__":
    main()

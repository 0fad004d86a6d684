#!/usr/bin/env python
"""Benchmark of the iterated arrow-decomposed SpMM hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # the B200 engine (torchrun for N > 1)
    python bench.py --impl reference --steps K --warmup W     # the reference's CPU arithmetic on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR   # also writes what the last timed step computed

``--dump-outputs`` lets two builds be compared output for output: the inputs depend only on the arguments (seeded
generators), and the files hold the level-0 result of the last timed step at k and at k = 16 (at most 36 MiB).

A step is one ``ArrowDecompositionMPI.step()`` (forward exchange -> per-level arrow SpMM -> backward
scatter-add) over the synthetic decomposition G2 of SURVEY.md 8d: 10M rows, width 10 000, two levels,
~10 nnz/row, k = 128 fp32 features, uniformly random level-1 permutation (seed 503).  Every rank goes through the
public path: level files on disk -> ``load_decomposition_new`` -> ``initialize`` -> ``load_sparse_matrix_from_blocks``.
Prints ONE JSON line.

* ``value``        GFLOP/s = 2 * sum(nnz) * k / time, features and matrices resident in HBM, CUDA-event timed, max over ranks
* ``e2e``          same metric with HOST buffers: every step uploads the features from pinned memory and downloads the
                   result tile (``step_stream``: copies of consecutive steps overlap the compute; the blocking
                   ``set_features / step / result_tile`` sequence of the reference is reported next to it)
* ``roofline``     level-0 arrow SpMM launch alone: algorithmic bytes / CUDA-event time vs the measured HBM peak
                   (N > 1: the slowest rank's launch and that rank's bytes)
* ``exposed_comm_ms`` (N > 1) step time minus the time of the same launches with every cross-GPU effect removed
* ``k16``          the k = 16 half of the metric on the same decomposition (device resident + roofline)
* ``cpu_baseline`` the reference's CPU path (oracle port of SciPy's kernel on host threads), bounded sample
* ``verified``     full-size parity property on rank-1 random features (sensitive to columns, maps and broadcasts)
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks", type=int, default=1000, help="block-rows of level 0 (x width = rows)")
    ap.add_argument("--width", type=int, default=10000)
    ap.add_argument("--k", type=int, default=128)
    ap.add_argument("--levels", type=int, default=2)
    ap.add_argument("--perm", type=str, default="random", choices=["random", "local", "identity"])
    ap.add_argument("--workload", type=str, default="g2", choices=["g2", "ba"],
                    help="g2 = the synthetic arrow decomposition of SURVEY 8d (default, BASELINE.json's workload); ba = a "
                         "Barabasi-Albert graph run through this repository's arrow decomposition (the reference's own "
                         "synthetic route, arrow_bench.py:24-41): skewed degrees, hub rows, a dense head")
    ap.add_argument("--vertices", type=int, default=1000000, help="--workload ba: vertices")
    ap.add_argument("--ba-m", type=int, default=5, help="--workload ba: edges per new vertex")
    ap.add_argument("--mode", type=str, default="auto", choices=["auto", "fused", "exchange"])
    ap.add_argument("--exchange", type=str, default="p2p", choices=["p2p", "p2p-direct", "nccl"],
                    help="multi-GPU exchange-mode transport (mode=exchange): NVLink peer pulls (default) or NCCL all-to-all")
    ap.add_argument("--overlap", type=int, default=1, help="multi-GPU: 0 = one lane, 1 = the exchange chain of the deeper levels runs beside the level-0 SpMM (default)")
    ap.add_argument("--graphs", type=int, default=1, help="multi-GPU fused step replayed as one CUDA graph (default 1)")
    ap.add_argument("--ctas", type=str, default="", help="main,side resident SpMM CTAs per SM while both lanes run (multi-GPU)")
    ap.add_argument("--l2-hints", type=str, default="", help="plain,fused L2 hint masks of the tile kernel (e.g. 3,0)")
    ap.add_argument("--prefetch", type=int, default=-1, help="tile kernel bulk-prefetch switch (ARROW_OPT_PREFETCH); -1 = library default")
    ap.add_argument("--fused-style", type=str, default="gather", choices=["gather", "scatter"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-k16", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the full-size parity property")
    ap.add_argument("--cpu-sample-blocks", type=int, default=0)
    ap.add_argument("--dump-outputs", type=str, default="", metavar="DIR",
                    help="write the level-0 result of the last timed step (k and k = 16) as DIR/result_k<k>.npy, float32, "
                         "rows in level-0 order: all rows, or a fixed seeded sample of them when the result is larger")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes what the B200 engine computed (--impl b200)")
    return a


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        load = [x for x in sm if mx and x > 0.5 * mx] or sm
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_name(a):
    if a.workload == "ba":
        return (f"Barabasi-Albert graph, {a.vertices} vertices, m={a.ba_m} (seed 503) -> arrow decomposition of this repository, "
                f"width {a.width}, at most {a.levels} levels, k={a.k} fp32")
    return (f"G2 synthetic arrow decomposition: {a.blocks * a.width} rows, width {a.width}, {a.levels} levels, "
            f"~10 nnz/row, k={a.k} fp32, level-1 permutation {a.perm} (seed 503)")


def build_decomposition(a, blocks=None):
    from arrow_matrix_b200 import synth
    if a.workload == "ba":
        from arrow_matrix_b200.decomposition import arrow_decomposition
        n = a.vertices if blocks is None else min(a.vertices, blocks * a.width)
        A = synth.barabasi_albert(n, a.ba_m, seed=503)
        return arrow_decomposition(A, a.width, max_number_of_levels=a.levels, block_diagonal=True, seed=1)
    return synth.synth_decomposition(blocks or a.blocks, a.width, levels=a.levels, perm_kind=a.perm, seed=503)


def traffic_from_profile(a, k):
    """dram bytes per launch of the level-0 SpMM from the committed ncu capture (profiles/), if it matches (N = 1 only)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        return t.get(f"blocks{a.blocks}_w{a.width}_k{k}")
    except Exception:
        return None


def host_info():
    """what the CPU arm ran on: the driver's boxes differ (round 1: 18.7 vs 77.9 GFLOP/s on '128 cores')"""
    info = {"cpu_count": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        info["numa_nodes"] = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()])
    except Exception:
        pass
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    info["cpu"] = line.split(":", 1)[1].strip()
                    break
    except Exception:
        pass
    try:
        a = np.ones(1 << 27, dtype=np.float32)           # 512 MB
        b = np.zeros_like(a)
        b[::1024] = 1.0                                   # pages touched before the clock starts
        t0 = time.perf_counter()
        np.copyto(b, a)
        info["one_thread_copy_GBps"] = round(2 * a.nbytes / (time.perf_counter() - t0) / 1e9, 1)
    except Exception:
        pass
    return info


# ----------------------------------------------------------------------------------------------------------
def run_reference(a):
    """The reference's CPU implementation of the path on this box's host cores (rank 0 only).  Like the reference's
    own driver (arrow_bench.py:113-126) the features are in place before the clock starts: only ``step()`` is timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_parallel
    from arrow_matrix_b200 import synth
    cores = os.cpu_count() or 1
    try:
        cores = min(cores, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    blocks = a.cpu_sample_blocks or (a.blocks if cores >= 64 else min(a.blocks, 250) if cores >= 16 else min(a.blocks, 100))
    dec = build_decomposition(a, blocks)
    ref = cpu_parallel.CpuArrowReference(dec, a.width, a.k, n_threads=cores)
    rng = np.random.default_rng(42)
    X = synth.generate_dense_matrix(ref.rows[0], a.k, np.float32, rng)
    ref.set_features(X)
    for _ in range(a.warmup):
        ref.step()
    times = []
    for _ in range(a.steps):
        t0 = time.perf_counter()
        ref.step()
        times.append(time.perf_counter() - t0)
    dt = float(np.mean(times))
    gflops = ref.flops_per_step() / dt / 1e9
    sample = (f"{blocks} of {a.blocks} block-rows of the same generator ({blocks * a.width} rows), full step "
              f"(gather, 2 products, scatter-add), {a.steps} timed steps, features in place before the clock starts")
    line = {"impl": "reference", "metric": "iterated SpMM GFLOP/s (k=%d)" % a.k, "value": gflops, "unit": "GFLOP/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(a)},
            "run": {"cpu_path": "oracle port of scipy csr_matvecs + row gather/scatter-add on host threads (the reference's "
                                "arithmetic; the literal reference needs mpi4py and >= 1500 MPI ranks)",
                    "host": host_info(), "ms_min": min(times) * 1e3, "ms_max": max(times) * 1e3},
            "cpu_baseline": {"value": gflops, "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": gflops, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    ref.close()


# ----------------------------------------------------------------------------------------------------------
# full-size parity property: one step on rank-1 random features
# ----------------------------------------------------------------------------------------------------------
def expected_step_on_vector(decomposition, width, u, block_diagonal=True):
    """float64 result column of ONE step applied to the vector ``u`` (level-0 row order): forward exchange through the
    level maps, every level's arrow blocks, backward scatter-add -- host arithmetic on the CSR arrays only, one sparse
    mat-vec per level.  Returns ``(y, state_free)``; ``state_free`` is False when some non-zero reads a row behind the
    sentinel (that row keeps the previous iteration's value, arrow_dec_mpi.py:544) and the property does not apply."""
    from scipy import sparse
    from arrow_matrix_b200 import decomp
    L = len(decomposition)
    n_blocks = [decomp.number_of_blocks(B, width) for B, _ in decomposition]
    _, to_prev, _, _ = decomp.prepare_permutations([p for _, p in decomposition], n_blocks, width)
    rows = [int(b) * width for b in n_blocks]
    x = [np.asarray(u, dtype=np.float64)[: rows[0]]]
    fed = [np.ones(rows[0], dtype=bool)]                    # rows whose value this iteration defines (chain down to level 0)
    for j in range(1, L):
        tp = to_prev[j][: rows[j]]
        valid = tp < rows[j - 1]
        safe = np.where(valid, tp, 0)
        fed.append(valid & fed[j - 1][safe])
        x.append(np.where(fed[j], x[j - 1][safe], 0.0))
    c = []
    state_free = True
    for j, (B, _) in enumerate(decomposition):
        ip, idx, dat, _ = decomp.arrow_rows(B, width, n_blocks[j], block_diagonal, 0, rows[j])
        # a row behind the sentinel keeps the previous iteration's value (arrow_dec_mpi.py:544): it only matters -- and
        # makes the result depend on history -- if some non-zero READS it (real decompositions have such rows but no reader)
        if idx.size and not bool(fed[j][idx].all()):
            state_free = False
        vals = np.ones(idx.size) if dat is None else np.asarray(dat, dtype=np.float64)
        c.append(sparse.csr_matrix((vals, idx, ip), shape=(rows[j], rows[j])) @ x[j])
    for j in range(L - 1, 0, -1):
        tp = to_prev[j][: rows[j]]
        valid = tp < rows[j - 1]
        c[j - 1][tp[valid]] += c[j][valid]                  # the maps are injective
    return c[0], state_free


def expected_ones_step(decomposition, width, block_diagonal=True):
    """round-1 property (all-ones features), kept for its tests: the row sums pushed through the maps"""
    from arrow_matrix_b200 import decomp
    n0 = decomp.number_of_blocks(decomposition[0][0], width) * width
    return expected_step_on_vector(decomposition, width, np.ones(n0), block_diagonal)


def rank1_vectors(n_rows, k):
    """u (per row, U[-1,1)) and v (per feature column, U[0.5,1.5): no column is insensitive) -- same on every rank"""
    u = 2.0 * np.random.default_rng(9001).random(n_rows) - 1.0
    v = 0.5 + np.random.default_rng(9002).random(k)
    return u, v


def verify_rank1_step(eng, decomposition, width, row0, hostX, hostC, comm, tol=1e-5):
    """Full-size parity property, outside every timed region: features ``X[r, c] = u[r] * v[c]`` with random u and v --
    every row differs, so a wrong column index, a wrong exchange map or a stale broadcast changes the result (the
    all-ones property of round 1 could not see those) -- and the step must return ``(S u) v^T`` where ``S`` is the
    whole iteration in float64.  Never raises: a failure of the check itself is reported in the JSON line, and every
    rank takes part in the same collectives whatever happens locally (the step is collective at N > 1)."""
    name = "one step on rank-1 random features X = u v^T == (step(u) in float64) v^T"
    expected, state_free, problem = None, None, None
    k = hostX.array.shape[1]
    try:
        from arrow_matrix_b200 import decomp
        n_rows = decomp.number_of_blocks(decomposition[0][0], width) * width
        u, v = rank1_vectors(n_rows, k)
        expected, state_free = expected_step_on_vector(decomposition, width, u)
    except Exception as e:     # noqa: BLE001
        problem = f"{type(e).__name__}: {e}"
    try:
        state = comm.allgather((problem, state_free))
    except Exception as e:     # noqa: BLE001
        return {"property": name, "error": f"{type(e).__name__}: {e}"}
    if any(p for p, _ in state):
        return {"property": name, "error": next(p for p, _ in state if p)}
    if not all(sf for _, sf in state):
        return {"property": name, "skipped": "rows behind the sentinel make the result state dependent"}
    rel = float("nan")
    try:
        n = hostX.array.shape[0]
        for a0 in range(0, n, 1 << 20):
            a1 = min(n, a0 + (1 << 20))
            hostX.array[a0:a1] = (u[row0 + a0: row0 + a1, None] * v[None, :]).astype(np.float32)
        eng.set_features(hostX.array)
        eng.step()
        got = eng.result(0, hostC.array)
        scale = max(float(np.max(np.abs(expected))) * float(np.max(np.abs(v))), 1e-30)
        err = 0.0
        for a0 in range(0, n, 1 << 20):                      # chunks: no 10 GB float64 temporary
            a1 = min(n, a0 + (1 << 20))
            want = expected[row0 + a0: row0 + a1, None] * v[None, :]
            err = max(err, float(np.max(np.abs(got[a0:a1].astype(np.float64) - want))))
        rel = err / scale
    except Exception as e:     # noqa: BLE001
        problem = f"{type(e).__name__}: {e}"
    try:
        outcome = comm.allgather((problem, rel))
    except Exception as e:     # noqa: BLE001
        return {"property": name, "error": f"{type(e).__name__}: {e}"}
    if any(p for p, _ in outcome):
        return {"property": name, "error": next(p for p, _ in outcome if p)}
    worst = float(max(r for _, r in outcome))
    return {"property": name, "rows": int(expected.size), "max_rel_err": worst, "tolerance": tol, "ok": bool(worst <= tol)}


def verify_ones_step(eng, decomposition, width, row0, hostX, hostC, comm, tol=1e-5):
    """round-1 property (all-ones features); superseded by ``verify_rank1_step`` in the bench line, kept as a test helper"""
    name = "one step on all-ones features == row sums of every level pushed through the exchange maps"
    expected, state_free = expected_ones_step(decomposition, width)
    if not state_free:
        return {"property": name, "skipped": "rows behind the sentinel make the result state dependent"}
    hostX.array[:] = 1.0
    eng.set_features(hostX.array)
    eng.step()
    got = eng.result(0, hostC.array)
    n = got.shape[0]
    scale = max(float(np.max(np.abs(expected))), 1e-30)
    err = 0.0
    for a0 in range(0, n, 1 << 20):
        a1 = min(n, a0 + (1 << 20))
        err = max(err, float(np.max(np.abs(got[a0:a1].astype(np.float64) - expected[row0 + a0: row0 + a1, None]))))
    worst = float(max(comm.allgather(err / scale)))
    return {"property": name, "rows": int(expected.size), "max_rel_err": worst, "tolerance": tol, "ok": bool(worst <= tol)}


# ----------------------------------------------------------------------------------------------------------
def max_over_ranks(dist, torch, x):
    if dist is None:
        return float(x)
    t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def time_steps(eng, ctx, barrier, steps, warmup, step_fn=None):
    """device-resident step time in ms (CUDA events on this rank's stream; the caller takes the max over ranks)"""
    fn = step_fn or eng.step
    for _ in range(warmup):
        eng.rewind_features()
        fn()
    barrier()
    ctx.timer_start(0)
    for _ in range(steps):
        eng.rewind_features()
        fn()
    ctx.timer_stop(0)
    barrier()
    return ctx.timer_ms(0) / steps


DUMP_MAX_ROWS = 1 << 16          # 32 MB at k = 128
DUMP_MAX_BYTES = 32 << 20        # per file: the k and k = 16 results stay below 64 MB together
DUMP_SEED = 1009


def dump_rows(n_rows, k):
    """level-0 rows that ``--dump-outputs`` writes: every row, or a sorted sample drawn with a fixed seed, so that two
    runs with the same arguments write the same rows"""
    m = min(n_rows, DUMP_MAX_ROWS, DUMP_MAX_BYTES // (4 * k))
    if m == n_rows:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n_rows, m, replace=False))


def dump_result(directory, name, eng, host_out, row0, n_rows, comm):
    """``directory/name.npy``: the level-0 result tile the last step left on the device (what ``B.result_tile()``
    returns), rows of ``dump_rows`` in level-0 order.  Collective: every rank sends its rows of the sample, rank 0 writes."""
    got = eng.result(0, host_out)
    rows = dump_rows(n_rows, got.shape[1])
    mine = rows[(rows >= row0) & (rows < row0 + got.shape[0])]
    parts = sorted(comm.allgather((row0, got[mine - row0])), key=lambda p: p[0])
    if comm.Get_rank() == 0:
        os.makedirs(directory, exist_ok=True)
        np.save(os.path.join(directory, name + ".npy"), np.concatenate([p for _, p in parts]))


def level0_roofline(a, eng, k, world, dist, torch, steps):
    """the dominant launch alone; at N > 1 the slowest rank's launch against that rank's own algorithmic bytes"""
    peak, peak_src = measured_peak_gbs()
    kms = eng.time_level_spmm(0, steps)
    kb = eng.level_bytes(0)
    if dist is not None:
        mine = torch.tensor([kms, kb], device="cuda", dtype=torch.float64)
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        kms, kb = max((float(t[0]), float(t[1])) for t in allv)
    if not kms:
        return None
    return {"bound": "hbm", "achieved": kb / kms / 1e6, "peak": peak, "unit": "GB/s", "frac": kb / kms / 1e6 / peak,
            "traffic": traffic_from_profile(a, k) if world == 1 else None,
            "kernel": "k_spmm_tiles level 0 (one launch%s)" % ("" if world == 1 else ", slowest rank's shard"), "kernel_ms": kms,
            "algorithmic_bytes_per_launch": kb, "peak_source": peak_src}


def build_engine(a, comm, base, k, local_rank):
    from arrow_matrix_b200.arrow_dec_mpi import ArrowDecompositionMPI
    blocks, n_blocks, to_prev, to_next = ArrowDecompositionMPI.load_decomposition_new(comm, base, a.width, True, slim=True)
    arrow = ArrowDecompositionMPI.initialize(comm, n_blocks, to_prev, to_next, a.width, k, 'gpu', True, True, mode=a.mode,
                                             exchange=a.exchange, overlap=a.overlap)
    arrow._fused_style = a.fused_style
    arrow.B.load_sparse_matrix_from_blocks(blocks)
    arrow.B.zero_rhs(a.width, k)
    eng = arrow._engine
    ctx = eng.ctx
    if a.l2_hints:
        hp, hf = (int(x) for x in a.l2_hints.split(","))
        ctx.set_option(ctx.OPT_L2_HINTS_PLAIN, hp)
        ctx.set_option(ctx.OPT_L2_HINTS_FUSED, hf)
    if a.prefetch >= 0:
        ctx.set_option(ctx.OPT_PREFETCH, a.prefetch)
    if a.ctas and hasattr(eng, "main_ctas"):
        eng.main_ctas, eng.side_ctas = (int(x) for x in a.ctas.split(","))
    return arrow, eng, blocks


def run_b200(a):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 engine has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    from arrow_matrix_b200 import _lib, graphio, synth
    # staging buffers and the thread that fills them live next to the GPU (two-socket box: GPUs 0-3 / 4-7)
    numa_node, numa_cpus = _lib.bind_thread_to_device_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from arrow_matrix_b200 import comm as comm_mod

    t_setup = time.time()
    comm = comm_mod.world_comm()
    # the public path: files on disk -> load_decomposition_new -> initialize -> load blocks (every rank maps the same files).
    # The files go to a directory of this run, removed when it exits: the source tree may be read-only.
    tag = f"ba_{a.vertices}_{a.ba_m}" if a.workload == "ba" else f"{a.blocks}_{a.perm}"
    files_dir = None
    if rank == 0:
        files_dir = tempfile.mkdtemp(prefix="arrow_b200_bench_")
        atexit.register(shutil.rmtree, files_dir, ignore_errors=True)
    base = os.path.join(comm.bcast(files_dir), f"bench_{tag}_{a.width}_{a.levels}")
    if rank == 0:
        dec0 = build_decomposition(a)
        graphio.save_decomposition_new(dec0, base, a.width, block_diagonal=True)
        del dec0
    comm.Barrier()
    arrow, eng, blocks = build_engine(a, comm, base, a.k, local_rank)
    dec = blocks.decomposition                 # memory-mapped level files (for the full-size property check)
    ctx = eng.ctx
    fused_n = hasattr(eng, "fp") and eng.fp is not None
    if fused_n and a.graphs:
        eng.use_graphs = True
    rows_local = eng.local_rows if hasattr(eng, "local_rows") else eng.levels[0].rows
    row0 = eng.plan.levels[0].r0 if hasattr(eng, "plan") else 0
    rng = np.random.default_rng(42 + rank)
    hostX = _lib.PinnedArray((rows_local, a.k), numa_device=local_rank)
    hostC = _lib.PinnedArray((rows_local, a.k), numa_device=local_rank)
    hostX.array[:] = 2 * rng.random((rows_local, a.k), dtype=np.float32) - 1
    eng.set_features(hostX.array)
    ctx.sync()
    t_setup = time.time() - t_setup

    def barrier():
        if dist is not None:
            dist.barrier()
        eng.sync()

    # ---- device-resident throughput -------------------------------------------------------------------------
    warm = max(a.warmup, 3)
    for _ in range(warm):
        eng.rewind_features()
        eng.step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    try:
        launches0 = ctx.launch_count()
        ms_step = time_steps(eng, ctx, barrier, a.steps, 0)
        launches = ctx.launch_count() - launches0
    finally:
        clocks = sampler.stop() if rank == 0 else None      # no nvidia-smi left running if a step fails
    n_rows = int(eng.n_blocks[0]) * a.width
    if a.dump_outputs:
        dump_result(a.dump_outputs, f"result_k{a.k}", eng, hostC.array, row0, n_rows, comm)
    ms_step = max_over_ranks(dist, torch, ms_step)
    flops = eng.flops_per_step()
    alg_bytes = eng.algorithmic_bytes_per_step()

    # ---- exposed communication (N > 1): the same launches with every cross-GPU effect removed ------------------
    exposed = None
    if world > 1 and not fused_n:
        # literal protocol (mode=exchange): compute-only = every level's local SpMM launch, back to back, nothing else
        def only_spmm():
            xi, ci = list(eng.xi), list(eng.ci)
            eng.spmm()
            eng.xi, eng.ci = xi, ci
        dry_ms = max_over_ranks(dist, torch, time_steps(eng, ctx, barrier, a.steps, 2, step_fn=only_spmm))
        exposed = {"exposed_comm_ms": max(ms_step - dry_ms, 0.0), "compute_only_ms": dry_ms,
                   "how": "step time minus the time of the per-level SpMM launches alone (max over ranks each)"}
    if fused_n and world > 1:
        dry_ms = max_over_ranks(dist, torch, time_steps(eng, ctx, barrier, a.steps, 2, step_fn=lambda: eng._step_fused(dry=True)))
        exposed = {"exposed_comm_ms": max(ms_step - dry_ms, 0.0), "compute_only_ms": dry_ms,
                   "how": "step time minus the time of the same launches without push, barriers, head reductions and with "
                          "every routed row stored locally (max over ranks each)"}

    # ---- dominant kernel alone: level-0 arrow SpMM -----------------------------------------------------------
    roof = level0_roofline(a, eng, a.k, world, dist, torch, a.steps)

    # ---- end to end through the public classes with host buffers --------------------------------------------
    e2e = None
    if not a.no_e2e:
        n_e2e = max(4, min(a.steps, 10))
        nbytes = rows_local * a.k * 4
        # two (features, result) pairs of pinned host buffers in rotation; uploads / compute / downloads of
        # consecutive iterations overlap on copy lanes (PCIe is full duplex) -- every step still moves its
        # own bytes up and down
        hx = [hostX, _lib.PinnedArray((rows_local, a.k), numa_device=local_rank)]
        hc = [hostC, _lib.PinnedArray((rows_local, a.k), numa_device=local_rank)]
        hx[1].array[:] = hostX.array
        for i in range(2):
            arrow.step_stream(hx[i % 2].array, hc[i % 2].array)
        arrow.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(n_e2e):
            arrow.step_stream(hx[i % 2].array, hc[i % 2].array)
        arrow.synchronize()
        barrier()
        dt = max_over_ranks(dist, torch, (time.perf_counter() - t0) / n_e2e)
        # the reference's own call sequence, blocking: set_features -> step -> result_tile
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            arrow.B.set_features(hostX.array)
            arrow.step()
            arrow.B.result_tile(out=hostC.array)
        barrier()
        dt_block = max_over_ranks(dist, torch, (time.perf_counter() - t0) / 2)
        e2e = {"value": flops / dt / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": int(nbytes) * world, "d2h_bytes_per_step": int(nbytes) * world,
               "ms_per_step": dt * 1e3, "steps": n_e2e,
               "api": "ArrowDecompositionMPI.step_stream(X_host, out_host) x N + synchronize() (pinned host buffers, copies overlap compute)",
               "pcie_GBps_per_gpu_per_direction": nbytes / dt / 1e9,
               "blocking_ms_per_step": dt_block * 1e3, "blocking_value": flops / dt_block / 1e9,
               "blocking_api": "B.set_features / step / B.result_tile (the reference's call sequence)",
               "numa": {"node": numa_node, "cpus_bound": numa_cpus}}
        for h in hx[1:] + hc[1:]:
            h.close()

    # ---- full-size parity property (untimed; all ranks take part in the step) ----------------------------------
    verified = None
    if not a.no_verify:
        use_graphs = getattr(eng, "use_graphs", False)
        verified = verify_rank1_step(eng, dec, a.width, row0, hostX, hostC, comm)
        verified["through_graph_replay"] = bool(use_graphs)

    mode = eng.mode + ("/" + eng.fused_style if getattr(eng, "fused_style", None) and eng.mode == "fused" else "")
    total_nnz = int(eng.total_nnz)

    # ---- the k = 16 half of the metric, same decomposition ---------------------------------------------------
    k16 = None
    if not a.no_k16 and a.k != 16:
        hostX.close(); hostC.close()
        eng.close()
        del arrow, eng
        arrow16, eng16, _ = build_engine(a, comm, base, 16, local_rank)
        if hasattr(eng16, "fp") and eng16.fp is not None and a.graphs:
            eng16.use_graphs = True
        x16 = _lib.PinnedArray((rows_local, 16), numa_device=local_rank)
        c16 = _lib.PinnedArray((rows_local, 16), numa_device=local_rank)
        x16.array[:] = 2 * rng.random((rows_local, 16), dtype=np.float32) - 1
        eng16.set_features(x16.array)
        eng16.ctx.sync()

        def barrier16():
            if dist is not None:
                dist.barrier()
            eng16.sync()
        ms16 = max_over_ranks(dist, torch, time_steps(eng16, eng16.ctx, barrier16, a.steps, warm))
        if a.dump_outputs:
            dump_result(a.dump_outputs, "result_k16", eng16, c16.array, row0, n_rows, comm)
        roof16 = level0_roofline(a, eng16, 16, world, dist, torch, a.steps)
        ver16 = None if a.no_verify else verify_rank1_step(eng16, dec, a.width, row0, x16, c16, comm)
        k16 = {"metric": "iterated SpMM GFLOP/s (k=16)", "value": eng16.flops_per_step() / ms16 / 1e6, "unit": "GFLOP/s",
               "ms_per_step": ms16, "hbm_gbs_effective": eng16.algorithmic_bytes_per_step() / ms16 / 1e6,
               "roofline": roof16, "verified": ver16}
        eng16.close()

    # ---- CPU baseline (rank 0, bounded sample) -----------------------------------------------------------------
    cpu = None
    if rank == 0 and not a.no_cpu and world == 1:
        from oracle import cpu_parallel
        cores = os.cpu_count() or 1
        _lib.bind_thread_to_device_numa(-1)                     # undo the NUMA pinning: the CPU arm uses every core and node
        try:
            cores = len(os.sched_getaffinity(0))
        except Exception:
            pass
        sb = a.cpu_sample_blocks or min(a.blocks, 100 if cores < 32 else 250)
        sdec = build_decomposition(a, sb)
        ref = cpu_parallel.CpuArrowReference(sdec, a.width, a.k, n_threads=cores)
        ref.set_features(synth.generate_dense_matrix(ref.rows[0], a.k, np.float32, np.random.default_rng(1)))
        dt = ref.time_steps(3, warmup=1)
        cpu = {"value": ref.flops_per_step() / dt / 1e9, "unit": "GFLOP/s", "cores": cores, "kind": "port",
               "sample": f"{sb} of {a.blocks} block-rows of the same generator, 3 full steps on {cores} host threads "
                         f"({dt * 1e3:.0f} ms/step)"}
        ref.close()

    if rank == 0:
        line = {"metric": "iterated SpMM GFLOP/s (k=%d)" % a.k, "value": flops / ms_step / 1e6, "unit": "GFLOP/s",
                "n_gpus": world, "steps": a.steps, "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_name(a)},
                "run": {"mode": mode, "overlap": int(bool(a.overlap)) if world > 1 else 0, "graph_replay": bool(fused_n and a.graphs),
                        "l2": "inputs larger than L2 (features 5.12 GB per pass at the default size); no flush",
                        "total_nnz": total_nnz, "setup_s": round(t_setup, 1),
                        "input": "level files on disk -> ArrowDecompositionMPI.load_decomposition_new / initialize / load_sparse_matrix_from_blocks on every rank"},
                "hbm_gbs_effective": alg_bytes / ms_step / 1e6, "algorithmic_bytes_per_step": alg_bytes,
                "roofline": roof, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "verified": verified, "k16": k16}
        if exposed is not None:
            line.update(exposed)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)

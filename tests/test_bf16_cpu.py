"""CPU tests of bf16 feature tiles: host rounding, dtype arguments, the one-GPU restriction, the C-ABI additions."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import torch

from arrow_matrix_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rne_bits(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 round-to-nearest-even on the bit pattern (NaN handled by the caller)"""
    b = x.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)


def test_host_rne_matches_torch_bit_for_bit():
    one = np.float32(1.0)
    ulp = np.float32(2.0 ** -7)                 # bf16 spacing at 1
    special = np.array([
        one + ulp / 2,                          # tie between 1 and 1 + ulp: to even (1)
        one + 3 * ulp / 2,                      # tie between 1 + ulp and 1 + 2 ulp: to even (1 + 2 ulp)
        one + ulp / 2 + np.float32(2.0 ** -23),  # just above the tie: up
        -(one + ulp / 2), -(one + 3 * ulp / 2),
        0.0, -0.0,
        1e-40, -1e-40, 2.0 ** -133, np.float32(1.1754942e-38),     # fp32 subnormals
        np.finfo(np.float32).max,               # rounds to +inf
        np.inf, -np.inf, 65504.0, 3.0, 255.5, 257.0,
    ], dtype=np.float32)
    rng = np.random.default_rng(3)
    with np.errstate(all="ignore"):              # magnitudes from subnormal to overflow on purpose
        rand = np.concatenate([rng.standard_normal(20000).astype(np.float32) * np.float32(10.0) ** rng.integers(-40, 38, 20000),
                               rng.integers(0, 2 ** 32, 20000, dtype=np.uint64).astype(np.uint32).view(np.float32)])
    x = np.concatenate([special, rand])
    got = _lib.to_bf16(x.reshape(-1, 1))
    assert got.dtype == torch.bfloat16 and got.is_contiguous()
    got_bits = got.view(torch.int16).numpy().view(np.uint16).ravel()
    ref_torch = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(got_bits, ref_torch)
    nan = np.isnan(x)
    assert np.array_equal(got_bits[~nan], _rne_bits(x[~nan]))
    assert np.all(np.isnan(got.float().numpy().ravel()[nan]))              # NaN stays NaN
    assert nan.sum() > 0
    assert got_bits[0] == 0x3F80 and got_bits[1] == 0x3F82 and got_bits[2] == 0x3F81
    assert got_bits[5] == 0x0000 and got_bits[6] == 0x8000                  # signed zeros kept
    assert got_bits[11] == 0x7F80                                           # FLT_MAX -> +inf
    # a bf16 tensor passes through untouched; other tensors go through float32
    t = torch.randn(5, 3).to(torch.bfloat16)
    assert torch.equal(_lib.to_bf16(t).view(torch.int16), t.view(torch.int16))
    d = torch.randn(5, 3, dtype=torch.float64)
    assert torch.equal(_lib.to_bf16(d).view(torch.int16), d.float().to(torch.bfloat16).view(torch.int16))


def test_dtype_arguments():
    for d in ("float32", np.float32, np.dtype("float32"), torch.float32):
        assert _lib.dtype_name(d) == "float32"
    for d in ("bfloat16", torch.bfloat16):
        assert _lib.dtype_name(d) == "bfloat16"
    for d in (np.float64, "float16", torch.float16, np.int32, "bf16", torch.float64):
        with pytest.raises(ValueError):
            _lib.dtype_name(d)
    from arrow_matrix_b200.arrow_slim_mpi import ArrowSlimMPI
    from arrow_matrix_b200.comm import SelfComm
    B = ArrowSlimMPI(SelfComm())                # no engine: the dtype is checked first
    for d in (np.float64, torch.float16, "int8"):
        with pytest.raises(ValueError):
            B.zero_rhs(8, 4, dtype=d)
    with pytest.raises(RuntimeError, match="sparse blocks not loaded"):
        B.zero_rhs(8, 4, dtype=torch.bfloat16)


def test_cli_dtype_flag(monkeypatch):
    from arrow_matrix_b200 import arrow_bench, cli
    seen = {}
    monkeypatch.setattr(arrow_bench, "bench_spmm", lambda *a, **kw: seen.update(kw))
    cli.main(["-w", "8", "--dtype", "bfloat16"])
    assert seen["datatype"] == "bfloat16"
    cli.main(["-w", "8"])
    assert seen["datatype"] == "float32"
    with pytest.raises(SystemExit):
        cli.main(["-w", "8", "--dtype", "float64"])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _two_rank_worker(rank, world, port, q):
    try:
        sys.path.insert(0, ROOT)
        import torch.distributed as dist
        dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
        from arrow_matrix_b200 import synth
        from arrow_matrix_b200.arrow_dec_mpi import ArrowDecompositionMPI
        from arrow_matrix_b200.comm import world_comm
        from arrow_matrix_b200.sharded import ShardPlan, ShardedArrowEngine
        from tests.numpy_backend import GlooNumpyBackend
        comm = world_comm()
        w, k = 8, 4
        dec = synth.synth_decomposition(4, w, levels=2, perm_kind="random", seed=77)
        n_blocks = np.array([2 * 4, 2 * 4])
        arrow = ArrowDecompositionMPI.initialize(comm, n_blocks, None, None, w, k, slim=True)
        plan = ShardPlan(dec, w, rank, world)
        eng = ShardedArrowEngine(plan, k, GlooNumpyBackend(comm, w, plan))
        arrow._engine = eng
        calls = []
        for name in ("fill", "h2d", "d2h", "alloc_shared_tiles", "spmm"):
            orig = getattr(eng.be, name)
            setattr(eng.be, name, lambda *a, _n=name, _o=orig, **kw: (calls.append(_n), _o(*a, **kw))[1])
        for d in (torch.bfloat16, "bfloat16"):
            try:
                arrow.B.zero_rhs(w, k, dtype=d)
                raise AssertionError("bf16 with two ranks was accepted")
            except NotImplementedError as e:
                assert "N-GPU" in str(e), e
        assert calls == [], calls                       # refused before any tile was touched
        arrow.B.zero_rhs(w, k, dtype=np.float32)         # float32 still works on the same world
        assert "fill" in calls
        dist.barrier()
        dist.destroy_process_group()
        q.put((rank, "ok"))
    except BaseException:     # noqa: BLE001
        import traceback
        q.put((rank, traceback.format_exc()))


def test_bf16_is_refused_with_two_ranks_before_any_device_call():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(30)
    bad = [f"rank {r}: {m}" for r, m in sorted(results) if m != "ok"]
    assert not bad, "\n".join(bad)


def test_new_symbols_are_declared_and_exported():
    hdr = open(os.path.join(ROOT, "include", "arrow_b200.h")).read()
    new = ["arrow_dense_alloc_dtype", "arrow_dense_dtype", "arrow_dense_put", "arrow_dense_get"]
    for name in new:
        assert re.search(rf"\b{name}\s*\(", hdr), name
        assert name in _lib.EXPORTS
    assert re.search(r"#define ARROW_DTYPE_F32\s+0\b", hdr) and re.search(r"#define ARROW_DTYPE_BF16\s+1\b", hdr)
    assert _lib.DTYPE_CODES == {"float32": 0, "bfloat16": 1}
    assert int(re.search(r"#define ARROW_ABI_VERSION (\d+)", hdr).group(1)) == _lib.ABI_VERSION == 3
    lib = _lib.load_library()
    for name in new:
        assert hasattr(lib, name)
    assert lib.arrow_b200_abi_version() == 3

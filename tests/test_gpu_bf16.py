"""bf16 feature tiles on one B200: exact rounding of every kernel path, the engine against the float64 protocol oracle,
the rank-1 property at full size, streaming, the reference-facing surface and the C-ABI refusals.

Numerics under test (DESIGN.md): kernels widen bf16 to fp32, accumulate in fp32 and round every stored row once to
nearest even.  With integer CSR values and integer features every fp32 partial sum is exact (< 2^24), so the device
result must EQUAL the round-to-nearest-even of the exact float64 result, bit for bit.
"""
import ctypes
from ctypes import byref, c_int, c_void_p

import numpy as np
import pytest
import torch
from scipy import sparse

pytestmark = pytest.mark.gpu

from oracle import oracle
from arrow_matrix_b200 import _lib, synth
from arrow_matrix_b200.engine import ArrowEngine

ERR_ARG = -2


def bits(t: torch.Tensor) -> np.ndarray:
    return t.view(torch.int16).numpy().view(np.uint16)


def rne(x64: np.ndarray) -> np.ndarray:
    """bits of round-to-nearest-even(x) for x exact in fp32"""
    x32 = np.asarray(x64, dtype=np.float32)
    assert np.array_equal(x32.astype(np.float64), x64)
    return bits(torch.from_numpy(np.ascontiguousarray(x32)).to(torch.bfloat16))


def bf16_of(x) -> torch.Tensor:
    return _lib.to_bf16(x)


def f64(t: torch.Tensor) -> np.ndarray:
    return t.float().numpy().astype(np.float64)


def int_csr(n_rows, n_cols, rng, nnz_per_row=10, hubs=(), hub_len=1500):
    """integer values in [-3, 3] \\ {0}; hub rows longer than the 512-entry long-row threshold"""
    rows, cols = [], []
    for r in range(n_rows):
        m = hub_len if r in hubs else int(rng.integers(0, 2 * nnz_per_row))
        c = np.unique(rng.integers(0, n_cols, m))
        rows.append(np.full(c.size, r))
        cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    vals = rng.integers(1, 4, rows.size) * rng.choice([-1, 1], rows.size)
    return sparse.csr_matrix((vals.astype(np.float32), (rows, cols)), shape=(n_rows, n_cols))


def int_features(n, k, rng, hi=256):
    """integers in [-hi, hi]: bf16-representable; products sum to values needing more than 8 significant bits"""
    return rng.integers(-hi, hi + 1, (n, k)).astype(np.float32)


@pytest.fixture(scope="module")
def ctx(cuda_device):
    c = _lib.Context(cuda_device)
    yield c
    c.close()


def _upload(ctx, X):
    d = ctx.dense_alloc(X.shape[0], X.shape[1], "bfloat16")
    d.h2d(bf16_of(X))
    return d


KS = [8, 16, 32, 64, 128, 256, 1, 5, 10, 300]          # tile kernel, paired rows (64), generic (1, 5, 10, 300)


@pytest.mark.parametrize("k", KS)
def test_spmm_rounds_once_exactly(ctx, k):
    rng = np.random.default_rng(k)
    n = 3000
    A = int_csr(n, n, rng, hubs=(7, 1500, 2999))
    X = int_features(n, k, rng)
    ref = A.astype(np.float64) @ X.astype(np.float64)
    assert np.abs(ref).max() < 2 ** 24 and np.any(np.abs(ref) > 512)       # exact in fp32, needs rounding in bf16
    Ad = ctx.csr_from_scipy(A)
    assert Ad.info()["n_long_rows"] == 3
    Xd = _upload(ctx, X)
    C = ctx.dense_alloc(n, k, "bfloat16")
    ctx.spmm(Ad, Xd, C)
    assert np.array_equal(bits(C.d2h()), rne(ref))
    # accumulate: C = RNE(C_old + A X), C_old read as bf16 and added in fp32
    C0 = int_features(n, k, rng, hi=200)
    C.h2d(bf16_of(C0))
    ctx.spmm(Ad, Xd, C, accumulate=True)
    assert np.array_equal(bits(C.d2h()), rne(C0.astype(np.float64) + ref))
    # row map: C[map[r]] (+)= (A X)[r], unmapped rows keep their bits
    perm = rng.permutation(n).astype(np.int64)
    perm[rng.random(n) < 0.2] = -1
    m = ctx.map_upload(perm, n)
    for acc in (False, True):
        C.h2d(bf16_of(C0))
        ctx.spmm(Ad, Xd, C, rowmap=m, accumulate=acc)
        exp = rne(C0.astype(np.float64))
        ok = perm >= 0
        exp[perm[ok]] = rne((C0[perm[ok]].astype(np.float64) if acc else 0.0) + ref[ok])
        assert np.array_equal(bits(C.d2h()), exp), f"rowmap acc={acc}"
    # gather-add epilogue: C[r] = RNE((A X)[r] + add[add_map[r]])
    S = int_features(n // 2, k, rng)
    Sd = _upload(ctx, S)
    amap = rng.integers(-1, n // 2, n).astype(np.int64)
    am = ctx.map_upload(amap, n // 2)
    ctx.spmm_add(Ad, Xd, C, Sd, am)
    addend = np.where((amap >= 0)[:, None], S[np.maximum(amap, 0)].astype(np.float64), 0.0)
    assert np.array_equal(bits(C.d2h()), rne(ref + addend))
    for h in (Ad, Xd, C, Sd, m, am):
        h.free()


@pytest.mark.parametrize("variant", [_lib.VARIANT_TILES | (1 << 8), _lib.VARIANT_TILES | (1 << 4)])
def test_forced_tile_shapes_round_exactly(ctx, variant):
    """k = 64 with one row per lane group (the default pairs rows) or one vector per lane; the generalised-kernel switch
    (ARROW_OPT_TILE_KERNEL = 0) is fp32-only and leaves bf16 launches on the round-1 kernel"""
    rng = np.random.default_rng(5)
    n, k = 2000, 64
    A = int_csr(n, n, rng)
    X = int_features(n, k, rng)
    exp = rne(A.astype(np.float64) @ X.astype(np.float64))
    Ad, Xd, C = ctx.csr_from_scipy(A), _upload(ctx, X), ctx.dense_alloc(n, k, "bfloat16")
    for tile_kernel in (1, 0):
        ctx.set_option(ctx.OPT_TILE_KERNEL, tile_kernel)
        C.fill(0.0)
        ctx.spmm(Ad, Xd, C, variant=variant)
        assert np.array_equal(bits(C.d2h()), exp)
    ctx.set_option(ctx.OPT_TILE_KERNEL, 1)
    for h in (Ad, Xd, C):
        h.free()


@pytest.mark.parametrize("k", [4, 8, 10, 128])
def test_gather_rows_copy_is_bit_exact_and_accumulate_rounds_once(ctx, k):
    rng = np.random.default_rng(11)
    n = 1500
    raw = torch.from_numpy(rng.integers(0, 2 ** 16, (n, k), dtype=np.uint16).view(np.int16)).view(torch.bfloat16)
    src = ctx.dense_alloc(n, k, "bfloat16")
    src.h2d(raw)                                            # any bit pattern, NaN payloads included
    dst = ctx.dense_alloc(n, k, "bfloat16")
    old = int_features(n, k, rng)
    dst.h2d(bf16_of(old))
    mp = rng.permutation(n).astype(np.int64)
    mp[rng.random(n) < 0.25] = -1
    m = ctx.map_upload(mp, n)
    ctx.gather_rows(dst, src, m)
    exp = rne(old.astype(np.float64))
    exp[mp >= 0] = bits(raw)[mp[mp >= 0]]
    assert np.array_equal(bits(dst.d2h()), exp)              # pure move; stale rows keep their bits
    a = int_features(n, k, rng)
    src.h2d(bf16_of(a))
    dst.h2d(bf16_of(old))
    ctx.gather_rows(dst, src, m, accumulate=True)
    exp = rne(old.astype(np.float64))
    exp[mp >= 0] = rne(old[mp >= 0].astype(np.float64) + a[mp[mp >= 0]])
    assert np.array_equal(bits(dst.d2h()), exp)
    for h in (src, dst, m):
        h.free()


# ---- the engine against the float64 protocol oracle -------------------------------------------------------------
def _step_and_bound(eng, po64):
    """One oracle step and the error bound of the device's step: one bf16 rounding (2^-8 relative) per store point.
    Fused mode stores each level's aggregated result tile once; exchange mode stores every level's product and, for the
    levels above the deepest, the backward accumulate as well."""
    po64.propagate_features()
    po64.spmm()
    products = [float(np.abs(C).max()) for C in po64.C]
    po64.aggregate()
    ref = po64.C[0]
    stores = [float(np.abs(C).max()) for C in po64.C]
    if eng.mode == "exchange":
        stores = products + stores[:-1]
    return ref, 2.0 ** -8 * sum(stores) + 1e-5 * float(np.abs(ref).max())


def _check_step(eng, po64):
    eng.step()
    ref, bound = _step_and_bound(eng, po64)
    got = f64(eng.result())
    err = float(np.abs(got - ref).max())
    assert err <= bound, (err, bound)
    po64.C[0][:] = got                                       # re-sync (X aliases C after the step)
    if eng.mode == "exchange":                               # stale rows of deeper levels carry device values too
        for j in range(1, eng.L):
            po64.C[j][:] = f64(eng.result(j))


def _check_chain(eng, po64, Xl0, iterations=3):
    eng.set_features(bf16_of(Xl0))
    po64.set_features(f64(bf16_of(Xl0)))
    for _ in range(iterations):
        _check_step(eng, po64)


@pytest.mark.parametrize("mode", ["fused", "exchange"])
@pytest.mark.parametrize("perm_kind", ["random", "local", "identity"])
@pytest.mark.parametrize("k,levels", [(16, 2), (128, 2), (4, 3), (10, 3)])
def test_engine_matches_float64_protocol_oracle(cuda_device, mode, perm_kind, k, levels):
    w, t0 = 64, 12
    dec = synth.synth_decomposition(t0, w, levels=levels, perm_kind=perm_kind, seed=21, hub_rows=2, hub_nnz=700)
    eng = ArrowEngine(dec, w, k, device=cuda_device, mode=mode, dtype="bfloat16")
    assert eng.mode == mode and eng.dtype == "bfloat16"
    po64 = oracle.ReferenceProtocolOracle(dec, w, k, dtype=np.float64)
    X = synth.generate_dense_matrix(t0 * w, k, np.float32, np.random.default_rng(42))
    _check_chain(eng, po64, X[po64.perms[0]])
    eng.close()


from tests.golden_util import GPU_CASES, GoldenCase          # noqa: E402


@pytest.mark.parametrize("name", [c for c in GPU_CASES if c.startswith(("slim_", "wide_"))])
def test_golden_fixtures_within_bf16_bound(cuda_device, name):
    g = GoldenCase(name)
    for mode in ("exchange", "fused"):
        eng = ArrowEngine(g.decomposition, g.width, g.k, block_diagonal=g.block_diagonal, device=cuda_device,
                          mode="exchange" if mode == "exchange" else "auto", dtype="bfloat16")
        if eng.mode != mode:
            eng.close()
            continue
        po64 = oracle.ReferenceProtocolOracle(g.decomposition, g.width, g.k, block_diagonal=g.block_diagonal,
                                              n_blocks=g.n_blocks, dtype=np.float64)
        for it in range(g.iterations):
            if g.X[it] is not None:
                eng.set_features(bf16_of(g.X[it]))
                po64.set_features(f64(bf16_of(g.X[it])))
            _check_step(eng, po64)
        eng.close()


def test_exchange_stale_rows_keep_their_bits(cuda_device):
    w, t0, k = 32, 8, 8
    dec = synth.synth_decomposition(t0, w, levels=3, perm_kind="random", seed=4, nested=False)
    eng = ArrowEngine(dec, w, k, device=cuda_device, dtype="bfloat16")
    assert eng.mode == "exchange"
    rng = np.random.default_rng(1)
    eng.set_features(bf16_of(synth.generate_dense_matrix(t0 * w, k, np.float32, rng)))
    eng.step()
    eng.set_features(bf16_of(synth.generate_dense_matrix(t0 * w, k, np.float32, rng)))
    before = [bits(eng.result(j)).copy() for j in range(eng.L)]
    eng.propagate_features()
    n_stale = 0
    for j in range(1, eng.L):
        st = eng.levels[j]
        stale = st.to_prev >= eng.levels[j - 1].rows
        n_stale += int(stale.sum())
        assert np.array_equal(bits(eng.features(j))[stale], before[j][stale])
    assert n_stale > 0
    eng.close()


# ---- full-size rank-1 property (BASELINE configs 1-3) -----------------------------------------------------------
def _rank1(eng, dec, w, k, seed):
    import bench
    n = eng.n_rows
    rng = np.random.default_rng(seed)
    u = f64(bf16_of((2.0 * rng.random(n) - 1.0).reshape(-1, 1))).ravel()          # bf16-representable
    v = 2.0 ** rng.integers(-2, 3, k)                                             # powers of two: X = u v^T exact in bf16
    X = torch.from_numpy(np.outer(u, v).astype(np.float32)).to(torch.bfloat16)
    assert np.array_equal(f64(X), np.outer(u, v))
    y, state_free = bench.expected_step_on_vector(dec, w, u)
    assert state_free
    eng.set_features(X)
    eng.step()
    got = f64(eng.result())
    ref = np.outer(y, v)
    levels = sum(float(np.abs(f64(eng.result(j))).max()) for j in range(1, eng.L))     # deeper levels' result tiles
    bound = 2.0 ** -8 * (float(np.abs(ref).max()) + levels) + 1e-5 * float(np.abs(ref).max())
    err = float(np.abs(got - ref).max())
    assert err <= bound, (err, bound)


def test_rank1_property_100k_rows_two_levels(cuda_device):
    w, k = 10000, 16
    dec = synth.synth_decomposition(10, w, levels=2, perm_kind="random", seed=503)
    for mode in ("fused", "exchange"):
        eng = ArrowEngine(dec, w, k, device=cuda_device, mode=mode, dtype="bfloat16")
        _rank1(eng, dec, w, k, seed=7)
        eng.close()


def test_rank1_property_1m_block_k_sweep(cuda_device):
    w = 10000
    dec = synth.synth_decomposition(100, w, levels=1, seed=503)
    eng = None
    for k in (16, 32, 64, 128, 256):
        eng = ArrowEngine(dec, w, k, device=cuda_device, dtype="bfloat16")
        assert eng.n_rows == 1_000_000
        _rank1(eng, dec, w, k, seed=k)
        eng.close()


# ---- streaming and the reference-facing surface ----------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fused", "exchange"])
def test_stream_step_bf16_matches_blocking_calls(cuda_device, mode):
    w, t0, k = 64, 10, 128
    dec = synth.synth_decomposition(t0, w, levels=2, perm_kind="random", seed=12)
    n = t0 * w
    rng = np.random.default_rng(3)
    Xs = [bf16_of(synth.generate_dense_matrix(n, k, np.float32, rng)) for _ in range(7)]
    eng = ArrowEngine(dec, w, k, device=cuda_device, mode=mode, dtype="bfloat16")
    ref = []
    for X in Xs:
        eng.set_features(X)
        eng.step()
        ref.append(bits(eng.result()).copy())
    eng.close()
    eng = ArrowEngine(dec, w, k, device=cuda_device, mode=mode, dtype="bfloat16")
    pairs = 3
    hx = [_lib.PinnedTensor((n, k)) for _ in range(pairs)]
    hc = [_lib.PinnedTensor((n, k)) for _ in range(pairs)]
    got = []
    for i, X in enumerate(Xs):
        if i >= pairs:
            eng.stream_drain()
            got.append(bits(hc[i % pairs].tensor).copy())
        hx[i % pairs].tensor.copy_(X)
        eng.stream_step(hx[i % pairs].tensor, hc[i % pairs].tensor)
    eng.stream_drain()
    for i in range(len(Xs) - pairs, len(Xs)):
        got.append(bits(hc[i % pairs].tensor).copy())
    for r, g in zip(ref, got):
        assert np.array_equal(r, g)
    eng.close()
    for p in hx + hc:
        p.close()


def test_reference_surface_bf16_and_back(cuda_device, tmp_path):
    from arrow_matrix_b200 import graphio
    from arrow_matrix_b200.arrow_dec_mpi import ArrowDecompositionMPI
    from arrow_matrix_b200.comm import SelfComm
    w, t0, k = 32, 8, 16
    dec = synth.synth_decomposition(t0, w, levels=2, perm_kind="random", seed=8)
    path = str(tmp_path / "dec")
    graphio.save_decomposition_new(dec, path, w, block_diagonal=True)
    comm = SelfComm()
    blocks, n_blocks, to_prev, to_next = ArrowDecompositionMPI.load_decomposition_new(comm, path, w, True)
    arrow = ArrowDecompositionMPI.initialize(comm, n_blocks, to_prev, to_next, w, k, slim=True)
    arrow.B.load_sparse_matrix_from_blocks(blocks)
    arrow.B.zero_rhs(w, k, dtype=torch.bfloat16)
    n = arrow._engine.n_rows
    X = synth.generate_dense_matrix(n, k, np.float32, np.random.default_rng(2))
    arrow.B.set_features(bf16_of(X))
    arrow.step()
    got = arrow.B.result_tile()
    assert got.dtype == torch.bfloat16 and arrow.B.C_i.dtype == torch.bfloat16
    eng = ArrowEngine(blocks.decomposition, w, k, device=cuda_device, n_blocks=list(n_blocks), dtype="bfloat16")
    eng.set_features(bf16_of(X))
    eng.step()
    assert np.array_equal(bits(got), bits(eng.result()))
    eng.set_dtype("float32")
    eng.set_features(X)
    eng.step()
    ref32 = eng.result()
    eng.close()
    arrow.B.zero_rhs(w, k, dtype=np.float32)
    arrow.B.set_features(X)
    arrow.step()
    got32 = arrow.B.result_tile()
    assert got32.dtype == np.float32 and np.array_equal(got32.view(np.uint32), ref32.view(np.uint32))
    with pytest.raises(ValueError):
        arrow.B.zero_rhs(w, k, dtype=np.float64)
    arrow._engine.close()


# ---- C-ABI refusals --------------------------------------------------------------------------------------------
def test_c_abi_refusals_leave_a_working_context(ctx):
    lib, h = ctx.lib, ctx._h
    rng = np.random.default_rng(0)
    n, k = 512, 16
    A = int_csr(n, n, rng)
    Ad = ctx.csr_from_scipy(A)
    X = int_features(n, k, rng)
    ref = rne(A.astype(np.float64) @ X.astype(np.float64))
    xb, cb = _upload(ctx, X), ctx.dense_alloc(n, k, "bfloat16")
    xf, cf = ctx.dense_alloc(n, k), ctx.dense_alloc(n, k)
    m = ctx.map_upload(np.arange(n), n)
    host = np.zeros((n, k), dtype=np.float32)
    hp = c_void_p(host.ctypes.data)

    def refused(rc):
        assert rc == ERR_ARG, rc
        assert lib.arrow_last_error(h)
        cb.fill(0.0)
        ctx.spmm(Ad, xb, cb)                                # the context still runs a correct launch
        assert np.array_equal(bits(cb.d2h()), ref)

    refused(lib.arrow_dense_h2d(h, xb.h, 0, n, hp))
    refused(lib.arrow_dense_d2h(h, xb.h, 0, n, hp))
    refused(lib.arrow_dense_h2d_lane(h, 1, xb.h, 0, n, hp))
    refused(lib.arrow_dense_d2h_lane(h, 2, xb.h, 0, n, hp))
    refused(lib.arrow_spmm(h, Ad.h, xb.h, cf.h, -1, 0, -1))                   # mixed dtypes
    refused(lib.arrow_spmm(h, Ad.h, xf.h, cb.h, -1, 0, -1))
    refused(lib.arrow_spmm_add(h, Ad.h, xb.h, cb.h, cf.h, m.h, -1))
    refused(lib.arrow_gather_rows(h, cb.h, xf.h, m.h, 0))
    refused(lib.arrow_dense_copy(h, cb.h, 0, xf.h, 0, n))
    refused(lib.arrow_spmm_ex(h, Ad.h, xb.h, -1, 0, cb.h, -1, -1, -1, -1))  # N-GPU entry points
    srcs = (c_int * 1)(xb.h)
    bounds = (ctypes.c_int64 * 2)(0, n)
    refused(lib.arrow_push_rows(h, (c_int * 1)(cb.h), bounds, 1, xb.h, m.h))
    refused(lib.arrow_reduce_rows(h, cb.h, -1, srcs, 1, n))
    refused(lib.arrow_gather_rows_multi(h, cb.h, srcs, bounds, 1, m.h, 0))
    refused(lib.arrow_ipc_export(h, xb.h, ctypes.create_string_buffer(_lib.IPC_HANDLE_BYTES)))
    assert lib.arrow_spmm(h, Ad.h, xb.h, cb.h, -1, 0, _lib.VARIANT_DIRECT) != 0     # bf16 runs the tile kernel only
    # wrapped tiles are fp32; dtype queries; fill rounds to nearest even
    d = c_int(-1)
    w = c_int(-1)
    assert lib.arrow_dense_wrap(h, c_void_p(xf.device_ptr()), n, k, byref(w)) == 0
    assert lib.arrow_dense_dtype(h, w.value, byref(d)) == 0 and d.value == 0
    assert lib.arrow_dense_dtype(h, xb.h, byref(d)) == 0 and d.value == 1
    assert lib.arrow_dense_free(h, w.value) == 0
    assert lib.arrow_dense_alloc_dtype(h, 4, 4, 7, byref(w)) == ERR_ARG
    for v in (1.0 / 3.0, -2.0 ** -130, 1e30, 257.0):
        cb.fill(v)
        assert np.all(bits(cb.d2h()) == bits(torch.tensor([v], dtype=torch.float32).to(torch.bfloat16))[0])
    for hd in (Ad, xb, cb, xf, cf, m):
        hd.free()

"""CPU tests: the oracle against the reference's known-answer vectors and against SciPy."""
import numpy as np
import pytest
from scipy import sparse

from oracle import oracle
from arrow_matrix_b200 import synth, graphio


# ---- routing-table KATs asserted by the reference's tests/test_arrowmpi.py:24-47 -----------------
def test_all_to_all_tables_reversed_kat():
    ranks, prev_ranks, rpr, cols = 2, 6, 4, 6
    perm = np.asarray(list(reversed(range(ranks * rpr))))
    for i in range(ranks):
        sl = perm[i * rpr:(i + 1) * rpr]
        counts, displs, p, out_p = oracle.all_to_all_tables(sl, rpr, cols, prev_ranks + ranks, prev_ranks)
        assert counts[ranks + prev_ranks - i - 1] == rpr * cols
        assert sum(counts) == rpr * cols
        assert displs[ranks + prev_ranks - i - 1] == 0
        counts, displs, p, out_p = oracle.all_to_all_tables(sl, rpr, cols, ranks + prev_ranks, 0)
        assert counts[ranks - i - 1] == rpr * cols
        assert sum(counts) == rpr * cols
        assert displs[ranks - i - 1] == 0


def test_all_to_all_tables_exact_values():
    # values listed in SURVEY.md 8c (computed from the reference source)
    c, d, sp, rp = oracle.all_to_all_tables(np.array([7, 6, 5, 4]), 4, 6, 8, 6)
    assert c == [0, 0, 0, 0, 0, 0, 0, 24] and d == [0] * 8
    assert list(sp) == [0, 1, 2, 3] and list(rp) == [3, 2, 1, 0]
    c, d, sp, rp = oracle.all_to_all_tables(np.array([7, 6, 5, 4]), 4, 6, 8, 0)
    assert c == [0, 24, 0, 0, 0, 0, 0, 0] and d == [0, 0, 24, 24, 24, 24, 24, 24]
    c, d, sp, rp = oracle.all_to_all_tables(np.array([3, 2, 1, 0]), 4, 6, 8, 6)
    assert c == [0, 0, 0, 0, 0, 0, 24, 0] and d == [0, 0, 0, 0, 0, 0, 0, 24]
    # sentinel handling
    c, d, sp, rp = oracle.all_to_all_tables(np.array([5, 999, 0, 6, 999, 1, 4, 2]), 8, 3, 3, 0)
    assert c == [18, 0, 0] and d == [0, 18, 18]
    assert list(sp) == [0, 2, 3, 5, 6, 7, 1, 4] and list(rp) == [2, 5, 7, 6, 0, 3]


def test_all_to_all_tables_random_like_reference_test():
    # the randomised half of tests/test_arrowmpi.py:50-94
    rng = np.random.default_rng(0)
    ranks, prev_ranks, rpr, cols = 2, 6, 4, 6
    perm = 2 * np.arange(ranks * rpr)
    rng.shuffle(perm)
    for i in range(ranks):
        sl = perm[i * rpr:(i + 1) * rpr]
        counts, displs, p, out_p = oracle.all_to_all_tables(sl, rpr, cols, ranks + prev_ranks, 0)
        after = sl[p] // rpr
        assert list(after) == sorted(sl // rpr)
        for j in range(ranks):
            assert counts[j] == np.count_nonzero(after == j) * cols


# ---- arithmetic: the C restatement against SciPy itself ------------------------------------------
@pytest.mark.parametrize("k", [1, 4, 10, 16, 128])
def test_c_kernel_matches_scipy_bitwise(k):
    rng = np.random.default_rng(42)
    A = synth.generate_sparse_matrix(500, 500, 5000, np.float32, rng)
    X = synth.generate_dense_matrix(500, k, np.float32, rng)
    got = oracle.csr_spmm_c(A, X)
    ref = A @ X
    assert got.dtype == np.float32
    assert np.array_equal(got, ref), np.abs(got - ref).max()


def test_c_kernel_int64_indices_and_empty_rows():
    rng = np.random.default_rng(1)
    A = sparse.random(64, 64, density=0.05, format="csr", dtype=np.float32, random_state=3)
    A.indices = A.indices.astype(np.int64)
    A.indptr = A.indptr.astype(np.int64)
    X = rng.random((64, 8), dtype=np.float32)
    assert np.array_equal(oracle.csr_spmm_c(A, X), A @ X)
    Z = sparse.csr_matrix((5, 5), dtype=np.float32)
    assert np.array_equal(oracle.csr_spmm_c(Z, np.ones((5, 3), np.float32)), np.zeros((5, 3), np.float32))


# ---- loader semantics -------------------------------------------------------------------------------
def test_number_of_blocks_and_masks():
    dec = synth.synth_decomposition(6, 8, levels=2, perm_kind="random", seed=1)
    assert oracle.number_of_blocks(dec[0][0], 8) == 6
    assert oracle.number_of_blocks(dec[1][0], 8) == 3
    M = oracle.arrow_mask(dec[0][0], 8, 6)
    assert M.nnz == dec[0][0].nnz       # the generator is exactly arrow shaped


def test_prepare_permutations_one_based_and_padding():
    p0 = np.arange(1, 11)          # one based, shorter than 2*8 rows
    p1 = np.array([3, 1, 2, 5, 4, 7, 6, 9, 8, 10])
    perms, to_prev, to_next, sent = oracle.prepare_permutations([p0, p1], [2, 1], 8)
    assert perms[0].tolist() == list(range(16))
    assert perms[1][:10].tolist() == [2, 0, 1, 4, 3, 6, 5, 8, 7, 9] and perms[1][10:].tolist() == list(range(10, 16))
    assert sent == 32
    assert to_prev[1].tolist() == perms[1].tolist()       # level 0 is the identity
    # to_next of level 0: rows of level 1 beyond n_blocks[1]*w = 8 are the sentinel
    inv1 = np.argsort(perms[1])
    exp = np.where(inv1 >= 8, 32, inv1)
    assert to_next[0].tolist() == exp.tolist()


# ---- protocol oracle vs the reference tests' own golden (compute_spmm) ------------------------------
@pytest.mark.parametrize("perm_kind", ["identity", "random", "local"])
@pytest.mark.parametrize("blockwise", [False, True])
def test_protocol_matches_compute_spmm(perm_kind, blockwise):
    w, t0, k = 8, 6, 4
    dec = synth.synth_decomposition(t0, w, levels=3, perm_kind=perm_kind, seed=11)
    n = t0 * w
    rng = np.random.default_rng(42)
    X = np.round(rng.random((n, k), dtype=np.float32), 0)    # integer valued -> exact (test_arrowmpi.py:259-260)
    po = oracle.ReferenceProtocolOracle(dec, w, k, blockwise=blockwise)
    assert po.dropped_nnz == [0, 0, 0]
    Xcur = X
    for _ in range(3):                                       # chained like test_arrowmpi.py:164-166
        po.set_features(Xcur[po.perms[0]])
        C0 = po.step()
        gold = oracle.compute_spmm(dec, Xcur)
        got = oracle.to_original_order(C0, po.perms[0], n)
        assert np.allclose(got, gold)
        Xcur = gold


def test_protocol_level_tiles_after_propagate():
    # after step() + _propagate_features(), level j holds golden_C[perm_j] (test_arrowmpi.py:306-309)
    w, t0, k = 8, 4, 3
    dec = synth.synth_decomposition(t0, w, levels=2, perm_kind="random", seed=5, shrink=1)
    n = t0 * w
    X = np.random.default_rng(3).random((n, k), dtype=np.float32)
    po = oracle.ReferenceProtocolOracle(dec, w, k)
    po.set_features(X[po.perms[0]])
    po.step()
    po.propagate_features()
    gold = oracle.compute_spmm(dec, X)
    assert np.allclose(po.C[1], gold[po.perms[1]][: po.rows[1]], rtol=1e-5, atol=1e-6)


def test_npy_layout_roundtrip(tmp_path):
    dec = synth.synth_decomposition(4, 8, levels=2, perm_kind="random", seed=2)
    base = str(tmp_path / "synth")
    graphio.save_decomposition_new(dec, base, 8, block_diagonal=True)
    assert (tmp_path / "synth_B_8_0_bd_indptr.npy").exists()
    back = graphio.load_decomposition_new(base, 8, True)
    assert len(back) == 2
    for (B, p), (B2, p2) in zip(dec, back):
        assert np.array_equal(B.indptr, B2.indptr) and np.array_equal(B.indices, B2.indices) and np.array_equal(B.data, B2.data) and np.array_equal(p, p2)
    mm = graphio.load_decomposition_new(base, 8, True, mem_map=True)
    assert np.array_equal(np.asarray(mm[1][0][1]), dec[1][0].indices)
    # Julia converter quirks: no data file, int64 indices, 1-based permutation
    base2 = str(tmp_path / "jl")
    graphio.save_decomposition_new(dec, base2, 8, True, write_data=False, index_dtype=np.int64, one_based_permutation=True)
    back2 = graphio.load_decomposition_new(base2, 8, True)
    assert np.all(back2[0][0].data == 1.0) and back2[0][0].data.dtype == np.float32
    raw = graphio.load_decomposition_new(base2, 8, True, mem_map=True)
    # value-less files: ones like the reference (graphio.py:292-298), as a zero-stride view on the memory-mapped route
    ones = raw[0][0][0]
    assert ones.dtype == np.float32 and ones.shape == raw[0][0][1].shape and ones.strides == (0,) and np.all(ones[:5] == 1.0)
    assert raw[0][0][1].dtype == np.int64 and raw[0][0][2].dtype == np.int64
    assert back2[0][1].min() == 1


@pytest.mark.parametrize("levels,k,threads", [(2, 16, 3), (3, 5, 8), (1, 4, 1)])
def test_cpu_baseline_steps_like_the_protocol(levels, k, threads):
    """the multi-threaded CPU baseline that bench.py times (cpu_baseline / --impl reference) computes what the pinned
    protocol oracle computes for a step on fresh features -- bit for bit (same kernel, same order inside a row)"""
    from oracle import cpu_parallel
    from arrow_matrix_b200 import synth
    w, t0 = 16, 9
    dec = synth.synth_decomposition(t0, w, levels=levels, perm_kind="random", seed=13, hub_rows=2, hub_nnz=60)
    ref = cpu_parallel.CpuArrowReference(dec, w, k, n_threads=threads)
    po = oracle.ReferenceProtocolOracle(dec, w, k)
    rng = np.random.default_rng(3)
    try:
        for _ in range(2):                                   # fresh features per step, like arrow_bench.py:113-116
            X = synth.generate_dense_matrix(t0 * w, k, np.float32, rng)
            ref.set_features(X)
            po.set_features(X.copy())
            got = ref.step()
            want = po.step()
            assert np.allclose(got, want, rtol=1e-6, atol=1e-6)
        assert ref.flops_per_step() == 2.0 * sum(M.nnz for M in po.mats) * k
    finally:
        ref.close()


@pytest.mark.parametrize("levels,nested", [(2, True), (3, True), (3, False), (1, True)])
def test_bench_full_size_property_matches_the_protocol(levels, nested, tmp_path):
    """bench.py checks every run at its own size with one step on all-ones features; its host-side expectation must be
    what the pinned protocol computes from a zeroed state (also from the memory-mapped level files bench.py uses)"""
    import bench
    from arrow_matrix_b200 import graphio, synth
    w, t0, k = 16, 9, 3
    dec = synth.synth_decomposition(t0, w, levels=levels, perm_kind="random", seed=29, nested=nested, hub_rows=2, hub_nnz=50)
    po = oracle.ReferenceProtocolOracle(dec, w, k)
    po.set_features(np.ones((po.rows[0], k), np.float32))
    want = po.step()
    got, state_free = bench.expected_ones_step(dec, w)
    assert state_free == nested or levels == 1
    if state_free:
        assert got.shape == (po.rows[0],)
        assert np.allclose(got[:, None], want, rtol=1e-5, atol=1e-5)
        base = str(tmp_path / "g")
        graphio.save_decomposition_new(dec, base, w, True)
        mm = graphio.load_decomposition_new(base, w, True, mem_map=True)
        got2, _ = bench.expected_ones_step(mm, w)
        assert np.array_equal(got, got2)

    class FakeEngine:                                    # drives verify_ones_step without a GPU
        def __init__(self, scale=1.0):
            self.scale = scale

        def set_features(self, X):
            po.set_features(X.copy())

        def step(self):
            self.out = po.step() * self.scale

        def result(self, level, out):
            out[:] = self.out
            return out

    class Host:
        def __init__(self):
            self.array = np.zeros((po.rows[0], k), np.float32)

    from arrow_matrix_b200.comm import SelfComm
    po = oracle.ReferenceProtocolOracle(dec, w, k)
    v = bench.verify_ones_step(FakeEngine(), dec, w, 0, Host(), Host(), SelfComm())
    if state_free:
        assert v["ok"] and v["max_rel_err"] <= 1e-5 and v["rows"] == po.rows[0]
        po = oracle.ReferenceProtocolOracle(dec, w, k)
        assert bench.verify_ones_step(FakeEngine(1.001), dec, w, 0, Host(), Host(), SelfComm())["ok"] is False
    else:
        assert "skipped" in v

    # the property the bench line carries since round 2: rank-1 random features.  Unlike all-ones features it must notice
    # a wrong exchange map / column index (every row of X differs)
    u, vv = bench.rank1_vectors(po.rows[0], k)
    y, sf = bench.expected_step_on_vector(dec, w, u)
    assert sf == state_free
    if state_free:
        po = oracle.ReferenceProtocolOracle(dec, w, k, dtype=np.float64)
        po.set_features(u[:, None] * vv[None, :])
        assert np.allclose(po.step(), y[:, None] * vv[None, :], rtol=1e-12, atol=1e-12)
    po = oracle.ReferenceProtocolOracle(dec, w, k)
    v = bench.verify_rank1_step(FakeEngine(), dec, w, 0, Host(), Host(), SelfComm())
    if state_free:
        assert v["ok"] and v["max_rel_err"] <= 1e-5 and v["rows"] == po.rows[0], v
        po = oracle.ReferenceProtocolOracle(dec, w, k)
        assert bench.verify_rank1_step(FakeEngine(1.001), dec, w, 0, Host(), Host(), SelfComm())["ok"] is False

        class WrongMap(FakeEngine):                      # an engine that routes two feature rows to the wrong place
            def set_features(self, X):
                X = X.copy()
                X[[1, w + 2]] = X[[w + 2, 1]]
                po.set_features(X)
        po = oracle.ReferenceProtocolOracle(dec, w, k)
        assert bench.verify_rank1_step(WrongMap(), dec, w, 0, Host(), Host(), SelfComm())["ok"] is False
        po = oracle.ReferenceProtocolOracle(dec, w, k)
        assert bench.verify_ones_step(WrongMap(), dec, w, 0, Host(), Host(), SelfComm())["ok"] is True      # blind: why it was replaced
        assert "error" in bench.verify_rank1_step(None, dec, w, 0, Host(), Host(), SelfComm())
    else:
        assert "skipped" in v


def test_bench_dump_outputs_fixed_sample_same_at_any_world_size(tmp_path):
    """bench.py --dump-outputs: the level-0 result, whole when small, else a seeded row sample of bounded size; a world of
    ranks writes the same file as one rank holding every row"""
    import threading
    import bench
    from arrow_matrix_b200.comm import SelfComm, ThreadWorld

    class Slice:                                         # a rank's engine: rows [r0, r1) of the level-0 result
        def __init__(self, full, r0, r1):
            self.tile = full[r0:r1]

        def result(self, level, out):
            out[:] = self.tile
            return out

    for n, k in ((300, 5), (100_000, 4), (70_000, 128)):
        full = np.random.default_rng(n).random((n, k), dtype=np.float32)
        rows = bench.dump_rows(n, k)
        assert np.array_equal(rows, bench.dump_rows(n, k)) and np.all(np.diff(rows) > 0)
        assert rows.size == n if n * k * 4 <= bench.DUMP_MAX_BYTES and n <= bench.DUMP_MAX_ROWS else rows.size < n
        assert rows.size * k * 4 <= bench.DUMP_MAX_BYTES
        one = tmp_path / f"one_{n}"
        bench.dump_result(str(one), "result", Slice(full, 0, n), np.empty((n, k), np.float32), 0, n, SelfComm())
        got = np.load(one / "result.npy")
        assert got.dtype == np.float32 and np.array_equal(got, full[rows])

        bounds = [0, n // 3, n // 3 + 7, n]
        world = ThreadWorld(3)
        three = tmp_path / f"three_{n}"

        def rank(r):
            r0, r1 = bounds[r], bounds[r + 1]
            bench.dump_result(str(three), "result", Slice(full, r0, r1), np.empty((r1 - r0, k), np.float32), r0, n,
                              world.comm(r))
        threads = [threading.Thread(target=rank, args=(r,)) for r in (2, 0, 1)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert np.array_equal(np.load(three / "result.npy"), got)

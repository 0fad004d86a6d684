"""CSR blocks with more than 2^31 - 1 non-zeros: every launch form across the 2^31 and 2^32 entry boundaries.

The device row pointer holds the low 32 bits of each row's 64-bit offset; tiles, long-row tasks and the anchors of the
per-row kernels carry the 64-bit bases.  Small blocks exercise the same code at small offsets (the rest of the suite);
this file builds blocks whose offsets cross 2^31 (sign bit of the low word) and 2^32 (the low word wraps).

Exactness: every CSR value is 1 and every row's columns are one contiguous run (start_r + t) mod n_cols, so a row's
sum is a difference of column prefix sums of X.  Features are integers of magnitude at most 64 and rows hold at most
2^17 entries: every partial sum is an integer below 2^24, exact in fp32 in any order, and the device must equal the host
result element for element (bf16: its round to nearest even, bit for bit).

Every large case checks free device memory and host RAM first and skips with the reason when there is too little;
device memory stays below about 60 GB.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from arrow_matrix_b200 import _lib
from arrow_matrix_b200.engine import ArrowEngine
from tests.test_gpu_bf16 import bits, rne

B31, B32 = 1 << 31, 1 << 32
THRESHOLD, SEGMENT = 512, 2048          # library default long-row tuning
XMAX = 64
GiB = 1 << 30


def host_available_bytes() -> int:
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def require(ctx, device_bytes: int, host_bytes: int):
    _, free, _ = ctx.device_info()
    if free < device_bytes:
        pytest.skip(f"needs {device_bytes / GiB:.0f} GiB of free device memory, {free / GiB:.0f} GiB free")
    have = host_available_bytes()
    if have < host_bytes:
        pytest.skip(f"needs {host_bytes / GiB:.0f} GiB of host RAM, {have / GiB:.0f} GiB available")


# ---- the contiguous-run recipe ------------------------------------------------------------------------------------
def fill(total, piece=200):
    """lengths of short rows covering `total` entries, `piece` at a time"""
    out = [piece] * (total // piece)
    if total % piece:
        out.append(total % piece)
    return out


def edge_rows(o, B, straddle_len_below):
    """Row lengths from offset `o` up to the row straddling B:
    a long row ending at E (E = 1 mod 4, a few thousand entries below B: the next tile starts unaligned), short rows,
    a run of 5 empty rows, then one row [B - straddle_len_below, B + 3).  Dropping a 3-entry first row shifts that row
    to end exactly at B."""
    E = B - straddle_len_below - 997 - 2
    E -= (E - 1) % 4                      # E = 1 mod 4
    long_len = 1500
    lens = fill(E - long_len - o)
    lens.append(long_len)
    lens += fill(B - straddle_len_below - E)
    lens += [0] * 5
    lens.append(straddle_len_below + 3)
    return lens, E


class WideBlock:
    """Host arrays of a block crossing 2^31 and 2^32 entries (module fixture)."""

    def __init__(self, n_rows, n_cols, mean_len, seed=7):
        rng = np.random.default_rng(seed)
        lens = rng.integers(0, 2 * mean_len + 1, n_rows).astype(np.int64)
        lens[0] = 3                                   # the shifted view drops this row
        self.events = {}
        for B, below in ((B31, 2), (B32, 5000)):      # a short row straddles 2^31, a long row (3 segments) 2^32
            ptr = np.cumsum(lens)
            j = int(np.searchsorted(ptr, B - 40000))  # row j ends at ptr[j] >= B - 40000
            o = int(ptr[j])
            edge, E = edge_rows(o, B, below)
            lens[j + 1: j + 1 + len(edge)] = edge
            self.events[B] = dict(first=j + 1, long_end=E, straddle=j + len(edge))
        self.lens = lens
        self.indptr = np.zeros(n_rows + 1, dtype=np.int64)
        np.cumsum(lens, out=self.indptr[1:])
        self.n_rows, self.n_cols, self.nnz = n_rows, n_cols, int(self.indptr[-1])
        assert self.nnz > B32 and int(lens.max()) <= 1 << 17
        self.start = (np.arange(n_rows, dtype=np.int64) * 2654435761) % n_cols
        self.indices = np.empty(self.nnz, dtype=np.int32)
        step = 1 << 19
        for r0 in range(0, n_rows, step):
            r1 = min(n_rows, r0 + step)
            a, b = int(self.indptr[r0]), int(self.indptr[r1])
            shift = np.repeat(self.start[r0:r1] - (self.indptr[r0:r1] - a), lens[r0:r1])
            self.indices[a:b] = (np.arange(b - a, dtype=np.int64) + shift) % n_cols

    def check_events(self):
        ip, lens = self.indptr, self.lens
        for B, ev in self.events.items():
            s = ev["straddle"]
            assert ip[s] < B < ip[s + 1] and ip[s + 1] == B + 3, "a row straddles B, and ends at B in the shifted view"
            assert np.all(lens[s - 5:s] == 0), "empty run before it"
            E = ev["long_end"]
            le = int(np.searchsorted(ip, E)) - 1      # the long row ending at E
            assert ip[le + 1] == E and lens[le] > THRESHOLD and E % 4 == 1 and B - 8192 < E < B
            assert lens[le + 1] > 0 and lens[le + 1] <= THRESHOLD, "a tile starts at E (after a long row): unaligned"
        s = self.events[B32]["straddle"]
        assert self.lens[s] > 2 * SEGMENT, "long row of several segments straddling 2^32"
        assert self.events[B31]["straddle"] < self.events[B32]["first"]

    def expected(self, X: np.ndarray) -> np.ndarray:
        """exact A X (float32) from column prefix sums"""
        n, k = X.shape
        P = np.zeros((n + 1, k), dtype=np.int64)
        np.cumsum(X.astype(np.int64), axis=0, out=P[1:])
        out = np.empty((self.n_rows, k), dtype=np.float32)
        step = 1 << 21
        for r0 in range(0, self.n_rows, step):
            r1 = min(self.n_rows, r0 + step)
            s, ln = self.start[r0:r1], self.lens[r0:r1]
            end = s + ln
            wrap = end > n
            y = P[np.minimum(end, n)] - P[s]
            y[wrap] += P[end[wrap] - n]
            out[r0:r1] = y
        return out

    def upload(self, ctx, row0: int = 0):
        """the block, or its view without the first `row0` rows (every offset shifted by -indptr[row0])"""
        a = int(self.indptr[row0])
        return ctx.csr_upload(self.n_rows - row0, self.n_cols, self.indptr[row0:], self.indices[a:], None)


N_ROWS, N_COLS, MEAN_LEN = 1 << 25, 1 << 24, 129       # 4.33e9 entries, 17 GB of indices on the host
DEV_BYTES = 60 * GiB


@pytest.fixture(scope="module")
def ctx(cuda_device):
    c = _lib.Context(cuda_device)
    yield c
    c.close()


class State:
    pass


@pytest.fixture(scope="module")
def wide(ctx):
    require(ctx, DEV_BYTES, 40 * GiB)
    st = State()
    st.block = WideBlock(N_ROWS, N_COLS, MEAN_LEN)
    rng = np.random.default_rng(11)
    st.X = rng.integers(-XMAX, XMAX + 1, (N_COLS, 16)).astype(np.float32)
    st.E = st.block.expected(st.X)
    st.A = st.block.upload(ctx)
    st.Xd = ctx.dense_from_host(st.X)
    st.C = ctx.dense_alloc(N_ROWS, 16)
    yield st
    for h in ("A", "Xd", "C"):
        if getattr(st, h, None) is not None:
            getattr(st, h).free()
    ctx.sync()


def test_layout_edges(wide):
    wide.block.check_events()
    assert wide.A.info()["nnz"] == wide.block.nnz


@pytest.mark.parametrize("k", [8, 16])
def test_plain_fp32(ctx, wide, k):
    if k == 16:
        X, C = wide.Xd, wide.C
    else:
        X, C = ctx.dense_from_host(wide.X[:, :k]), ctx.dense_alloc(N_ROWS, k)
    try:
        ctx.spmm(wide.A, X, C)
        assert np.array_equal(C.d2h(), wide.E[:, :k])
    finally:
        if k != 16:
            X.free()
            C.free()


def test_accumulate_rowmap_graph(ctx, wide):
    C = wide.C
    ctx.spmm(wide.A, wide.Xd, C)
    ctx.spmm(wide.A, wide.Xd, C, accumulate=True)
    assert np.array_equal(C.d2h(), 2 * wide.E)
    rev = np.arange(N_ROWS - 1, -1, -1, dtype=np.int64)
    rm = ctx.map_upload(rev, N_ROWS)
    C2 = ctx.dense_alloc(N_ROWS, 16)
    try:
        ctx.spmm(wide.A, wide.Xd, C2, rowmap=rm)
        assert np.array_equal(C2.d2h()[::-1], wide.E)
        # the tile kernel recorded in a CUDA graph and replayed (run once un-captured first)
        ctx.spmm(wide.A, wide.Xd, C2, rowmap=rm, accumulate=True)
        C2.fill(0.0)
        ctx.sync()
        ctx.graph_begin()
        ctx.spmm(wide.A, wide.Xd, C2, rowmap=rm, accumulate=True)
        g = ctx.graph_end()
        ctx.graph_launch(g)
        ctx.graph_launch(g)
        ctx.sync()
        ctx.graph_free(g)
        assert np.array_equal(C2.d2h()[::-1], 2 * wide.E)
    finally:
        rm.free()
        C2.free()


def test_gather_add_and_variants(ctx, wide):
    rng = np.random.default_rng(3)
    S = rng.integers(-XMAX, XMAX + 1, (4096, 16)).astype(np.float32)
    am = np.where(np.arange(N_ROWS) % 3 == 0, -1, np.arange(N_ROWS) % 4096).astype(np.int64)
    Sd, amd = ctx.dense_from_host(S), ctx.map_upload(am, 4096)
    try:
        ctx.spmm_add(wide.A, wide.Xd, wide.C, Sd, amd)
        want = wide.E.copy()
        want[am >= 0] += S[am[am >= 0]]
        assert np.array_equal(wide.C.d2h(), want)
        del want
    finally:
        Sd.free()
        amd.free()
    # the A/B variants: generalised tile kernel, direct and shuffle per-row kernels
    for opt, variant in ((0, _lib.VARIANT_AUTO), (1, 0), (1, 1)):
        ctx.set_option(ctx.OPT_TILE_KERNEL, opt)
        try:
            wide.C.fill(0.0)
            ctx.spmm(wide.A, wide.Xd, wide.C, variant=variant)
            assert np.array_equal(wide.C.d2h(), wide.E), (opt, variant)
        finally:
            ctx.set_option(ctx.OPT_TILE_KERNEL, 1)


def test_generic_k(ctx, wide):
    X, C = ctx.dense_from_host(wide.X[:, :5]), ctx.dense_alloc(N_ROWS, 5)
    try:
        ctx.spmm(wide.A, X, C)
        assert np.array_equal(C.d2h(), wide.E[:, :5])
    finally:
        X.free()
        C.free()


def test_spmm_ex_split_pointer_table(ctx, wide):
    split = N_COLS // 2 + 5
    X1, X2 = ctx.dense_from_host(wide.X[:split]), ctx.dense_from_host(wide.X[split:])
    rows = np.arange(N_ROWS, dtype=np.int64)
    which = np.where(rows % 7 == 3, -1, 0).astype(np.int32)         # some rows are dropped
    dest = N_ROWS - 1 - rows
    C2 = ctx.dense_alloc(N_ROWS, 16)
    table = ctx.ptrtable_upload([C2], which, dest)
    try:
        C2.fill(-1.0)
        ctx.spmm_ex(wide.A, X1, None, X2=X2, x_split=split, out_table=table)
        got = C2.d2h()[::-1]
        keep = which >= 0
        assert np.array_equal(got[keep], wide.E[keep])
        assert np.all(got[~keep] == -1.0)
    finally:
        table.free()
        C2.free()
        X1.free()
        X2.free()


def test_bf16_plain(ctx, wide):
    X = ctx.dense_alloc(N_COLS, 16, "bfloat16")
    C = ctx.dense_alloc(N_ROWS, 16, "bfloat16")
    try:
        X.h2d(wide.X)                                 # integers of magnitude <= 64: exact in bf16
        ctx.spmm(wide.A, X, C)
        got = bits(C.d2h())
        step = 1 << 22
        for r0 in range(0, N_ROWS, step):
            assert np.array_equal(got[r0:r0 + step], rne(wide.E[r0:r0 + step].astype(np.float64))), r0
    finally:
        X.free()
        C.free()


def test_remapped_copy(ctx, wide):
    shift = np.roll(np.arange(N_COLS, dtype=np.int64), -1)          # column c -> c + 1 (mod n_cols)
    m = ctx.map_upload(shift, N_COLS)
    R = wide.A.remap_columns(m, N_COLS)
    Xs = ctx.dense_from_host(np.roll(wide.X, 1, axis=0))            # Xs[c + 1] = X[c]
    try:
        wide.C.fill(0.0)
        ctx.spmm(R, Xs, wide.C)
        assert np.array_equal(wide.C.d2h(), wide.E)
    finally:
        Xs.free()
        R.free()
        m.free()


def test_shifted_view(ctx, wide):
    """The same rows without the first one: the straddling rows now end exactly at 2^31 and 2^32."""
    wide.A.free()
    wide.A = None
    ctx.sync()
    A = wide.block.upload(ctx, row0=1)
    C = ctx.dense_alloc(N_ROWS - 1, 16)
    try:
        ip = wide.block.indptr - wide.block.indptr[1]
        for B in (B31, B32):
            assert ip[wide.block.events[B]["straddle"] + 1] == B
        ctx.spmm(A, wide.Xd, C)
        assert np.array_equal(C.d2h(), wide.E[1:])
        for variant in (0, 1):                        # per-row kernels: anchors cross both boundaries
            C.fill(0.0)
            ctx.spmm(A, wide.Xd, C, variant=variant)
            assert np.array_equal(C.d2h(), wide.E[1:]), variant
        Xg, Cg = ctx.dense_from_host(wide.X[:, :5]), ctx.dense_alloc(N_ROWS - 1, 5)
        ctx.spmm(A, Xg, Cg)
        assert np.array_equal(Cg.d2h(), wide.E[1:, :5])
        Xg.free()
        Cg.free()
    finally:
        C.free()
        A.free()
        ctx.sync()
    # case 1 is done: release its host arrays for the engine case
    wide.block.indices = None
    wide.E = None


# ---- engine level: level 0 of just over 2^31 arrow-pattern entries ------------------------------------------------
def test_engine_level0_over_2g(ctx, wide):
    for h in ("Xd", "C"):
        getattr(wide, h).free()
        setattr(wide, h, None)
    require(ctx, 30 * GiB, 30 * GiB)
    width, nb, k = 4096, 1 << 13, 8
    rows = width * nb
    rng = np.random.default_rng(5)
    lens = rng.integers(0, 131, rows).astype(np.int64)
    indptr = np.zeros(rows + 1, dtype=np.int64)
    np.cumsum(lens, out=indptr[1:])
    nnz = int(indptr[-1])
    assert nnz > B31
    start = rng.integers(0, width, rows)                 # run inside the row's diagonal block
    base = (np.arange(rows, dtype=np.int64) // width) * width
    indices = np.empty(nnz, dtype=np.int32)
    step = 1 << 20
    for r0 in range(0, rows, step):
        r1 = min(rows, r0 + step)
        a, b = int(indptr[r0]), int(indptr[r1])
        t = np.arange(b - a, dtype=np.int64) - np.repeat(indptr[r0:r1] - a, lens[r0:r1])
        indices[a:b] = np.repeat(base[r0:r1], lens[r0:r1]) + (np.repeat(start[r0:r1], lens[r0:r1]) + t) % width
    # level 1: one block-row of `width` rows, a random sparse block (values 1..3)
    from scipy import sparse
    l1 = sparse.random(width, width, density=0.01, random_state=1, format="csr")
    l1.data = rng.integers(1, 4, l1.nnz).astype(np.float32)
    perm0 = np.arange(rows, dtype=np.int64)
    perm1 = rows - 1 - perm0                             # level-1 row r is level-0 row rows-1-r
    X = rng.integers(-XMAX, XMAX + 1, (rows, k)).astype(np.float32)
    eng = ArrowEngine([((None, indices, indptr), perm0), (l1, perm1)], width, k, mode="fused", ctx=ctx,
                      n_blocks=[nb, 1])
    try:
        assert eng.mode == "fused" and eng.levels[0].nnz == nnz
        del indices
        eng.set_features(X)
        eng.step()
        got = eng.result()
    finally:
        eng._release_buffers()
        for st in eng.levels:
            for h in (st.csr, st.to_prev_dev, st.to_next_dev, st.cmap_dev):
                if h is not None:
                    h.free()
        ctx.sync()
    P = np.zeros((rows + 1, k), dtype=np.int64)
    np.cumsum(X.astype(np.int64), axis=0, out=P[1:])
    want = np.empty((rows, k), dtype=np.float64)
    for r0 in range(0, rows, 1 << 21):
        r1 = min(rows, r0 + (1 << 21))
        s, ln, b0 = start[r0:r1], lens[r0:r1], base[r0:r1]
        end = s + ln
        wrap = end > width
        y = P[b0 + np.minimum(end, width)] - P[b0 + s]
        y[wrap] += P[b0[wrap] + end[wrap] - width] - P[b0[wrap]]
        want[r0:r1] = y
    # routed level-1 rows: C0[rows-1-r] += (A1 X1)[r], X1[r] = X[rows-1-r]
    X1 = X[rows - 1 - np.arange(width)].astype(np.float64)
    want[rows - 1 - np.arange(width)] += l1.astype(np.float64) @ X1
    assert np.array_equal(got, want.astype(np.float32))
    assert np.array_equal(got.astype(np.float64), want)


# ---- limits that stay ---------------------------------------------------------------------------------------------
def test_limits_refused(ctx):
    ip = np.zeros(2, dtype=np.int64)
    idx = np.zeros(0, dtype=np.int32)
    for n_rows, n_cols in ((1 << 31, 10), (10, 1 << 31)):
        with pytest.raises(_lib.ArrowError) as e:
            ctx.csr_upload(n_rows, n_cols, ip, idx, None)
        assert e.value.code == -4, str(e.value)
    # 64 consecutive rows spanning 2^32 entries: refused from the row pointer alone, before any index is read
    ip = np.array([0, B32 - 1, B32], dtype=np.int64)
    h = ctypes.c_int()
    rc = ctx.lib.arrow_csr_upload(ctx._h, 2, 10, B32, ip.ctypes.data_as(ctypes.c_void_p), 8,
                                  idx.ctypes.data_as(ctypes.c_void_p), 4, None, ctypes.byref(h))
    assert rc == -4
    # the context still runs a correct launch
    from scipy import sparse
    A = sparse.random(300, 200, density=0.05, random_state=2, format="csr")
    A.data = np.ones_like(A.data)
    X = np.random.default_rng(0).integers(-8, 9, (200, 8)).astype(np.float32)
    Ad, Xd, Cd = ctx.csr_from_scipy(A), ctx.dense_from_host(X), ctx.dense_alloc(300, 8)
    try:
        ctx.spmm(Ad, Xd, Cd)
        assert np.array_equal(Cd.d2h(), (A @ X.astype(np.float64)).astype(np.float32))
    finally:
        Ad.free()
        Xd.free()
        Cd.free()

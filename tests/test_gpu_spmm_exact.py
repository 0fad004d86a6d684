"""Bit-exact SpMM tests for the launch paths and tile schedules a tolerance test cannot pin down.

Exactness contract: CSR values are integers in {+-1, +-2, +-3} and features (and the old C rows and addends a launch
reads) are integers of at most 256 in magnitude.  The host asserts that every row's sum_p |v_p| * max|x|, plus the old
row and the addend, stays below 2^24: every fp32 product, FMA and add is then exact whatever the order of summation, so
the device result must EQUAL the float64 result element for element (bf16: its round-to-nearest-even, bit for bit).
No tolerance is used anywhere in this file.

The float64 reference is built from explicit COO triplets (duplicate (row, col) entries and unsorted columns inside a
row each count).  One matrix builder supplies the row patterns where kernels go wrong: empty rows (a run of 200 at the
start, the first and the last row), 1-entry rows, every length 0..17 (each remainder of the 8 / 4 / 2 unroll and the
predicated tail batches), rows at the long-row threshold and one above, long rows of exactly 1, 2, 3 segments and of
m * segment + 1 entries, a tile filled to exactly nnz_cap - 4 entries followed by one more entry (64-row and 128-row
tiles), tiles whose first row and first non-zero are not multiples of 4, duplicate and unsorted columns.

Each test restores every option and the tuning to the library defaults afterwards (options are per context, the
context is shared by the module).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from arrow_matrix_b200 import _lib
from tests.test_gpu_bf16 import bits, rne

Ctx = _lib.Context
EXACT_LIMIT = 2 ** 24
TILE_NNZ, TILE_ROWS, TILE_NNZ_BIG, TILE_ROWS_BIG = 1024, 64, 2048, 128     # arrow_b200.cu

DEFAULT_OPTIONS = {
    Ctx.OPT_L2_HINTS_PLAIN: 3, Ctx.OPT_L2_HINTS_FUSED: 0, Ctx.OPT_BIG_TILES: 1, Ctx.OPT_SPMM_CTAS_PER_SM: 0,
    Ctx.OPT_ROWS_PER_GROUP: 0, Ctx.OPT_SPMM_SM_LIMIT: 0, Ctx.OPT_TILE_KERNEL: 1, Ctx.OPT_FORCE_PREDICATED: 0,
    Ctx.OPT_PUSH_CTAS: 0, Ctx.OPT_PUSH_INTERLEAVE: 1,
}
DEFAULT_TUNING = (512, 2048)

# tile schedules: the default grid (one tile per CTA at these sizes), one CTA walking every tile (ticket, next-tile
# prefetch into the other stage, mbarrier parity flips, stage reuse), three CTAs competing for the ticket
SCHEDULES = {
    "grid": {},
    "one_cta": {Ctx.OPT_SPMM_SM_LIMIT: 1, Ctx.OPT_SPMM_CTAS_PER_SM: 1},
    "three_ctas": {Ctx.OPT_SPMM_SM_LIMIT: 3, Ctx.OPT_SPMM_CTAS_PER_SM: 1},
}


@pytest.fixture(scope="module")
def ctx(cuda_device):
    c = _lib.Context(cuda_device)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def _library_defaults(ctx):
    yield
    ctx.set_lane(0)
    for opt, val in DEFAULT_OPTIONS.items():
        ctx.set_option(opt, val)
    ctx.set_tuning(*DEFAULT_TUNING)


def _apply(ctx, options):
    for opt, val in options.items():
        ctx.set_option(opt, val)


# ---- data contract ------------------------------------------------------------------------------------------------
def int_values(rng, n):
    return (rng.integers(1, 4, n) * rng.choice([-1, 1], n)).astype(np.float32)


def int_features(rng, n, k, hi=256):
    return rng.integers(-hi, hi + 1, (n, k)).astype(np.float32)


class Block:
    """CSR block as explicit triplets (CSR order: rows non-decreasing, columns as generated)"""

    def __init__(self, lens, n_cols, rng):
        self.n_rows, self.n_cols = len(lens), n_cols
        self.lens = np.asarray(lens, dtype=np.int64)
        self.indptr = np.concatenate([[0], np.cumsum(self.lens)]).astype(np.int64)
        self.rows = np.repeat(np.arange(self.n_rows), self.lens)
        self.cols = rng.integers(0, n_cols, self.rows.size).astype(np.int64)      # with replacement, unsorted
        self.vals = int_values(rng, self.rows.size)
        self.row_abs = np.bincount(self.rows, weights=np.abs(self.vals), minlength=self.n_rows)

    def upload(self, ctx):
        return ctx.csr_upload(self.n_rows, self.n_cols, self.indptr, self.cols, self.vals)

    def check_exact(self, xmax, *extra_max):
        """host side of the contract: every partial sum of every row is an integer below 2^24"""
        bound = float(self.row_abs.max(initial=0.0)) * xmax + sum(extra_max)
        assert bound < EXACT_LIMIT, f"test data leaves the exact fp32 range: {bound}"

    def product(self, X, col_map=None):
        """float64 sum_p v_p X[col_p] per row from the triplets (col_map: columns sent through it, -1 entries skipped)"""
        cols = self.cols if col_map is None else col_map[self.cols]
        keep = cols >= 0
        X64 = np.asarray(X, dtype=np.float64)
        out = np.zeros((self.n_rows, X64.shape[1]))
        r, c, v = self.rows[keep], cols[keep], self.vals[keep].astype(np.float64)
        for j in range(X64.shape[1]):
            out[:, j] = np.bincount(r, weights=v * X64[c, j], minlength=self.n_rows)
        return out


def pattern_lens(thr, seg, n_rows, rng):
    """row lengths with every pattern of the module docstring, padded with random 0..17-entry rows to n_rows"""
    L = []
    L += [0] * 200                                          # a block whose first 200 rows are empty
    L += [1] * 20                                           # 1-entry rows
    L += list(range(18))                                    # every length 0..17
    L += [thr, thr + 1, thr, 0, thr + 1]                    # at the threshold (short) and one above (long)
    m0 = thr // seg + 1                                     # fewest whole segments that make a long row
    long_lens = sorted({n for n in (seg, 2 * seg, 3 * seg, 3 * seg + 1, m0 * seg, m0 * seg + 1, (m0 + 1) * seg) if n > thr})
    for n in long_lens:
        L += [n, 3, 5]
    if thr >= 17:
        # directly after a long row a tile starts: fill it to exactly nnz_cap - 4 entries, then one more entry
        L += [long_lens[0]] + [17] * 60 + [1, 2]            # 64-row tiles: 60 x 17 = 1020 = TILE_NNZ - 4
        L += [long_lens[0]] + [17] * 120 + [4, 1, 2]        # 128-row tiles: 120 x 17 + 4 = 2044 = TILE_NNZ_BIG - 4
    L += [7, 0, 9, 3]                                       # odd offsets before the random rows
    rest = n_rows - len(L) - 1
    assert rest >= 0
    L += list(rng.integers(0, 18, rest))
    L += [0]                                                # the last row is empty
    return L


def tiles_of(indptr, thr, rows_cap, nnz_cap):
    """the row tiles build_long_rows makes at upload: (row_begin, row_end, nnz_begin, nnz_end)"""
    lens = np.diff(indptr)
    out, r, n = [], 0, len(lens)
    while r < n:
        if lens[r] > thr:
            r += 1
            continue
        e = r
        while e < n and e - r < rows_cap:
            if lens[e] > thr or (indptr[e + 1] - indptr[r] > nnz_cap - 4 and e > r):
                break
            e += 1
        e = max(e, r + 1)
        out.append((r, e, int(indptr[r]), int(indptr[e])))
        r = e
    return out


def make_block(thr, seg, n_rows, seed, n_cols=None):
    rng = np.random.default_rng(seed)
    lens = pattern_lens(thr, seg, n_rows, rng)
    blk = Block(lens, n_cols or n_rows, rng)
    # a row with one column repeated and the others in descending order
    r = int(np.flatnonzero(blk.lens == 9)[0])
    p = blk.indptr[r]
    blk.cols[p:p + 9] = [5, 5, 5, 40, 30, 20, 10, 5, 0]
    if thr >= 17:
        for cap, rows_cap in ((TILE_NNZ, TILE_ROWS), (TILE_NNZ_BIG, TILE_ROWS_BIG)):
            t = tiles_of(blk.indptr, thr, rows_cap, cap)
            assert any(d[3] - d[2] == cap - 4 for d in t), "no tile filled to nnz_cap - 4"
            assert any(d[0] % 4 and d[2] % 4 for d in t), "no tile with unaligned first row and first non-zero"
    return blk


def assert_exact(got, exp, blk, thr, what, src_row=None):
    """element-wise equality; the first mismatch is reported with its row, the row's length and whether it is long"""
    got, exp = np.asarray(got), np.asarray(exp)
    assert got.shape == exp.shape, (what, got.shape, exp.shape)
    if np.array_equal(got, exp):
        return
    bad = np.argwhere(got != exp)
    r, c = (int(x) for x in bad[0])
    sr = r if src_row is None else int(src_row[r])
    length = int(blk.lens[sr]) if 0 <= sr < blk.n_rows else -1
    raise AssertionError(f"{what}: {len(bad)} mismatches; first at (row {r}, col {c}), CSR row {sr} of length {length} "
                         f"({'long' if length > thr else 'short'} under threshold {thr}): got {got[r, c]!r}, "
                         f"expected {exp[r, c]!r}")


# ---- the forms of a tile launch -----------------------------------------------------------------------------------
_CASES = {}


def _case(thr, seg, n_rows, k, seed=0):
    """matrix, operands and float64 references, shared by the configurations of one (tuning, k)"""
    key = (thr, seg, n_rows, k, seed)
    if key not in _CASES:
        if len(_CASES) > 8:
            _CASES.clear()
        blk = make_block(thr, seg, n_rows, seed=1000 + seed)
        rng = np.random.default_rng(k + seed)
        n = blk.n_rows
        X = int_features(rng, blk.n_cols, k)
        C0 = int_features(rng, n, k, hi=200)
        S = int_features(rng, n // 2, k, hi=200)
        amap = rng.integers(-1, n // 2, n)
        perm = rng.permutation(n)
        perm[rng.random(n) < 0.2] = -1
        n0 = blk.n_cols + 100
        cmap = rng.permutation(n0)[:blk.n_cols]
        cmap[rng.random(blk.n_cols) < 0.1] = 2 * n0             # invalid image: the remapped copy skips the entry
        X0 = int_features(rng, n0, k)
        blk.check_exact(256.0, 200.0, 200.0)
        valid = np.where(cmap < n0, cmap, -1)
        _CASES[key] = dict(blk=blk, X=X, C0=C0, S=S, amap=amap, perm=perm, cmap=cmap, n0=n0, X0=X0,
                           ref=blk.product(X), ref_remap=blk.product(X0, valid))
    return _CASES[key]


FORMS = ("plain", "accumulate", "rowmap", "rowmap_accumulate", "gather_add", "remapped_skip")


def expected_forms(cs):
    """float64 expected tile per form, with the CSR row that produced each output row (for the failure report)"""
    n = cs["blk"].n_rows
    ref, C0, perm, amap, S = cs["ref"], cs["C0"].astype(np.float64), cs["perm"], cs["amap"], cs["S"]
    ok = perm >= 0
    src = np.full(n, -1)
    src[perm[ok]] = np.flatnonzero(ok)
    out = {"plain": (ref, None), "accumulate": (C0 + ref, None)}
    e = C0.copy()
    e[perm[ok]] = ref[ok]
    out["rowmap"] = (e, src)
    e = C0.copy()
    e[perm[ok]] += ref[ok]
    out["rowmap_accumulate"] = (e, src)
    out["gather_add"] = (ref + np.where((amap >= 0)[:, None], S[np.maximum(amap, 0)].astype(np.float64), 0.0), None)
    out["remapped_skip"] = (cs["ref_remap"], None)
    return out


def run_forms(ctx, cs, k, variant=_lib.VARIANT_AUTO, dtype="float32", thr=DEFAULT_TUNING[0]):
    blk = cs["blk"]
    n = blk.n_rows
    bf = dtype == "bfloat16"

    def tile(a):
        d = ctx.dense_alloc(a.shape[0], k, dtype)
        d.h2d(a)
        return d

    def down(d):
        return bits(d.d2h()) if bf else d.d2h()

    def want(e64):
        return rne(e64) if bf else e64.astype(np.float32)

    A = blk.upload(ctx)
    cm = ctx.map_upload(cs["cmap"], cs["n0"])
    Ar = A.remap_columns(cm, cs["n0"])
    X, X0, S, C = tile(cs["X"]), tile(cs["X0"]), tile(cs["S"]), ctx.dense_alloc(n, k, dtype)
    pm, am = ctx.map_upload(cs["perm"], n), ctx.map_upload(cs["amap"], n // 2)
    exp = expected_forms(cs)
    for form in FORMS:
        if form in ("accumulate", "rowmap", "rowmap_accumulate"):
            C.h2d(cs["C0"])
        else:
            C.fill(7.0)                                     # plain launches overwrite every row, empty ones too
        if form == "plain":
            ctx.spmm(A, X, C, variant=variant)
        elif form == "accumulate":
            ctx.spmm(A, X, C, accumulate=True, variant=variant)
        elif form == "rowmap":
            ctx.spmm(A, X, C, rowmap=pm, variant=variant)
        elif form == "rowmap_accumulate":
            ctx.spmm(A, X, C, rowmap=pm, accumulate=True, variant=variant)
        elif form == "gather_add":
            ctx.spmm_add(A, X, C, S, am, variant=variant)
        else:
            ctx.spmm(Ar, X0, C, variant=variant)
        e64, src = exp[form]
        assert_exact(down(C), want(e64), blk, thr, f"{dtype} k={k} {form}", src)
    for h in (Ar, A, cm, X, X0, S, C, pm, am):
        h.free()


# ---- 1. tile-kernel forms x configuration x schedule --------------------------------------------------------------
def tile_shape(k, vpl_req=0, rpg_req=0, big_tiles=1, bf=False):
    """(G, VPL, big tiles, RPG) that launch_tiles picks (arrow_b200.cu), to prune configurations that run the same
    instantiation as one already in the matrix"""
    k4 = k // (8 if bf else 4)
    vpl = vpl_req if vpl_req in (1, 2, 4) else (4 if k4 >= 32 else (2 if k4 >= 8 else 1))
    if bf and vpl > 2:
        vpl = 2
    while vpl > 1 and k4 < vpl:
        vpl >>= 1
    lanes = (k4 + vpl - 1) // vpl
    if lanes > 32:
        vpl = 2 if (k4 + 31) // 32 <= 2 else 4
        lanes = (k4 + vpl - 1) // vpl
    g = 1
    while g < lanes:
        g <<= 1
    big = k4 <= 8 and bool(big_tiles)
    rpg = rpg_req or (2 if vpl == 2 else 1)
    if not big or rpg != 2:
        rpg = 1
    paired = {(4, 2)} if bf else {(4, 1), (8, 1), (2, 2), (4, 2)}
    if rpg == 2 and (g, vpl) not in paired:
        rpg = 1
    return g, vpl, big, rpg


TILE_KS = [4, 8, 16, 32, 48, 64, 128, 256]
TILE_CONFIGS = {                                    # name: (options, variant bits)
    "default": ({}, 0),
    "tile_kernel_0": ({Ctx.OPT_TILE_KERNEL: 0}, 0),
    "big_tiles_0": ({Ctx.OPT_BIG_TILES: 0}, 0),
    "force_predicated": ({Ctx.OPT_FORCE_PREDICATED: 1}, 0),
    "vpl1": ({}, 1 << 4), "vpl2": ({}, 2 << 4), "vpl4": ({}, 4 << 4),
    "rpg1": ({}, 1 << 8), "rpg2": ({}, 2 << 8),
}


def tile_matrix():
    """Configurations x k, pruned: a forced vpl / rpg or BIG_TILES = 0 that launch_tiles maps onto the (G, VPL, tile
    size, RPG) of the default -- or of a forced shape already kept at that k -- runs the same kernels and is left out
    (BIG_TILES = 0 above k = 32, vpl / rpg forcing where k4 clamps them, rpg above k = 32).  TILE_KERNEL = 0 and
    FORCE_PREDICATED = 1 select other code at every k and are always kept."""
    out = []
    for k in TILE_KS:
        seen = set()
        for name, (opts, bits_) in TILE_CONFIGS.items():
            shape = tile_shape(k, (bits_ >> 4) & 0xF, (bits_ >> 8) & 3, opts.get(Ctx.OPT_BIG_TILES, 1))
            if name in ("default", "tile_kernel_0", "force_predicated"):
                if name == "default":
                    seen.add(shape)
                out.append((k, name))
            elif shape not in seen:
                seen.add(shape)
                out.append((k, name))
    return out


@pytest.mark.parametrize("schedule", list(SCHEDULES))
@pytest.mark.parametrize("k,config", tile_matrix())
def test_tile_forms_exact(ctx, k, config, schedule):
    """plain, accumulate, row map with -1 entries (with and without accumulate), gather-add and a remapped-column copy
    with invalid columns, on 3 000+ rows, in every configuration and schedule"""
    opts, vbits = TILE_CONFIGS[config]
    _apply(ctx, opts)
    _apply(ctx, SCHEDULES[schedule])
    run_forms(ctx, _case(*DEFAULT_TUNING, 3200, k), k, variant=_lib.VARIANT_TILES | vbits)


# ---- 2. bf16 under the same schedules -----------------------------------------------------------------------------
@pytest.mark.parametrize("big_tiles", [1, 0])
@pytest.mark.parametrize("k", [16, 64, 128, 256])
def test_bf16_tile_forms_one_cta(ctx, k, big_tiles):
    _apply(ctx, SCHEDULES["one_cta"])
    ctx.set_option(ctx.OPT_BIG_TILES, big_tiles)
    run_forms(ctx, _case(*DEFAULT_TUNING, 3200, k), k, dtype="bfloat16")


@pytest.mark.parametrize("k", [12, 264])
def test_bf16_generic_forms(ctx, k):
    """k = 12: a multiple of 4 but not of 8 (no bf16 vector); k = 264: above 256"""
    run_forms(ctx, _case(*DEFAULT_TUNING, 3200, k), k, dtype="bfloat16")


# ---- 3. generic / direct / shuffle / TMA, over more rows than one pass of their grid-stride loops ---------------------
def _resident_rows_max(ctx, rows_per_cta):
    sm = ctx.device_info()[0]
    return 8 * sm * rows_per_cta             # at most 8 CTAs of 256 threads per SM (2048 threads)


def _vec_rows_per_cta(k):
    k4 = k // 4
    g = next(g for g in (1, 2, 4, 8, 16, 32) if k4 <= g or g == 32)
    return 8 * (32 // g)


@pytest.mark.parametrize("kind,k", [("generic", k) for k in (1, 3, 5, 10, 130, 260, 300)]
                         + [(v, k) for v in ("direct", "shfl") for k in (4, 48, 128, 200, 256)]
                         + [("tma", k) for k in (32, 100, 128)])
def test_grid_stride_kernels_exact(ctx, kind, k):
    variant = {"generic": _lib.VARIANT_AUTO, "direct": _lib.VARIANT_DIRECT, "shfl": _lib.VARIANT_SHFL,
               "tma": _lib.VARIANT_TMA}[kind]
    per_cta = {"generic": 8, "tma": 8}.get(kind) or _vec_rows_per_cta(k)
    n = max(20000, _resident_rows_max(ctx, per_cta) + 1000)
    rng = np.random.default_rng(k)
    blk = Block(pattern_lens(512, 2048, n, rng), n, rng)
    X = int_features(rng, n, k)
    C0 = int_features(rng, n, k, hi=200)
    perm = rng.permutation(n)
    perm[::7] = -1
    blk.check_exact(256.0, 200.0)
    ref = blk.product(X)
    A, dX, C = blk.upload(ctx), ctx.dense_from_host(X), ctx.dense_alloc(n, k)
    pm = ctx.map_upload(perm, n)
    C.fill(7.0)
    ctx.spmm(A, dX, C, variant=variant)
    assert_exact(C.d2h(), ref.astype(np.float32), blk, 512, f"{kind} k={k} plain")
    C.h2d(C0)
    ctx.spmm(A, dX, C, accumulate=True, variant=variant)
    assert_exact(C.d2h(), (C0 + ref).astype(np.float32), blk, 512, f"{kind} k={k} accumulate")
    C.h2d(C0)
    ctx.spmm(A, dX, C, rowmap=pm, accumulate=True, variant=variant)
    exp = C0.astype(np.float64)
    exp[perm[perm >= 0]] += ref[perm >= 0]
    src = np.full(n, -1)
    src[perm[perm >= 0]] = np.flatnonzero(perm >= 0)
    assert_exact(C.d2h(), exp.astype(np.float32), blk, 512, f"{kind} k={k} rowmap accumulate", src)
    for h in (A, dX, C, pm):
        h.free()


# ---- 4. long-row tuning -------------------------------------------------------------------------------------------
TUNINGS = [(1, 32), (31, 32), (512, 2048), (1016, 64)]


@pytest.mark.parametrize("k", [16, 128, 10])
@pytest.mark.parametrize("thr,seg", TUNINGS)
def test_long_row_tuning_exact(ctx, thr, seg, k):
    """t = 1: every row of two or more entries takes the long path; t = 1016 (the largest accepted): single-row tiles
    that fill the bulk-copy stage.  Plain, row map, accumulate, gather-add, remapped copy, then spmm_ex with a pointer
    table and a dual X base"""
    ctx.set_tuning(thr, seg)
    cs = _case(thr, seg, 3200, k, seed=thr)
    blk = cs["blk"]
    n_long = int(np.count_nonzero(blk.lens > thr))
    A = blk.upload(ctx)
    assert A.info()["n_long_rows"] == n_long
    A.free()
    run_forms(ctx, cs, k, thr=thr)
    _spmm_ex_exact(ctx, cs, k, thr)


def _spmm_ex_exact(ctx, cs, k, thr):
    """two-part X (columns >= split read X2), pointer table with dropped rows into two tiles, gather-add"""
    blk = cs["blk"]
    n = blk.n_rows
    rng = np.random.default_rng(k)
    split = blk.n_cols // 3
    X1 = cs["X"][:split + 17]                                # X may be longer than the split
    X2 = np.ascontiguousarray(cs["X"][split:])
    which = rng.integers(-1, 2, n).astype(np.int32)
    row = np.zeros(n, dtype=np.int64)
    for t in (0, 1):
        sel = np.flatnonzero(which == t)
        row[sel] = rng.permutation(n)[:sel.size]
    ref = cs["ref"] + np.where((cs["amap"] >= 0)[:, None], cs["S"][np.maximum(cs["amap"], 0)].astype(np.float64), 0.0)
    A = blk.upload(ctx)
    d1, d2, dS = ctx.dense_from_host(X1), ctx.dense_from_host(X2), ctx.dense_from_host(cs["S"])
    am = ctx.map_upload(cs["amap"], n // 2)
    t0, t1 = ctx.dense_alloc(n, k), ctx.dense_alloc(n, k)
    t0.fill(7.0)
    t1.fill(7.0)
    tab = ctx.ptrtable_upload([t0, t1], which, row)
    ctx.spmm_ex(A, d1, X2=d2, x_split=split, out_table=tab, add=dS, add_map=am)
    for t, tile in enumerate((t0, t1)):
        sel = np.flatnonzero(which == t)
        exp = np.full((n, k), 7.0)
        exp[row[sel]] = ref[sel]
        src = np.full(n, -1)
        src[row[sel]] = sel
        assert_exact(tile.d2h(), exp.astype(np.float32), blk, thr, f"spmm_ex k={k} table tile {t}", src)
    C = ctx.dense_alloc(n, k)
    C.fill(7.0)
    ctx.spmm_ex(A, d1, C=C, X2=d2, x_split=split, add=dS, add_map=am)
    assert_exact(C.d2h(), ref.astype(np.float32), blk, thr, f"spmm_ex k={k} dual X into C")
    dX = ctx.dense_from_host(cs["X"])                        # one X base into C: the launch ARROW_OPT_TILE_KERNEL switches
    C.fill(7.0)
    ctx.spmm_ex(A, dX, C=C, add=dS, add_map=am)
    assert_exact(C.d2h(), ref.astype(np.float32), blk, thr, f"spmm_ex k={k} gather-add into C")
    for h in (tab, A, d1, d2, dS, am, t0, t1, C, dX):
        h.free()


def test_block_keeps_its_upload_threshold(ctx):
    """a block (and a remapped copy made later, which shares its long-row task list) keeps the threshold it was
    uploaded with when set_tuning changes afterwards"""
    k = 16
    ctx.set_tuning(31, 32)
    cs = _case(31, 32, 3200, k, seed=31)
    blk = cs["blk"]
    A = blk.upload(ctx)
    ctx.set_tuning(512, 2048)
    assert A.info()["n_long_rows"] == int(np.count_nonzero(blk.lens > 31))
    cm = ctx.map_upload(cs["cmap"], cs["n0"])
    Ar = A.remap_columns(cm, cs["n0"])
    X, X0, C = ctx.dense_from_host(cs["X"]), ctx.dense_from_host(cs["X0"]), ctx.dense_alloc(blk.n_rows, k)
    for schedule in ("grid", "one_cta"):
        _apply(ctx, SCHEDULES[schedule])
        C.fill(7.0)
        ctx.spmm(A, X, C)
        assert_exact(C.d2h(), cs["ref"].astype(np.float32), blk, 31, f"block after set_tuning ({schedule})")
        C.fill(7.0)
        ctx.spmm(Ar, X0, C)
        assert_exact(C.d2h(), cs["ref_remap"].astype(np.float32), blk, 31, f"remapped copy after set_tuning ({schedule})")
    for h in (Ar, A, cm, X, X0, C):
        h.free()


def test_out_of_range_tuning_is_refused(ctx):
    for thr, seg in ((0, 32), (TILE_NNZ - 7, 64), (512, 31)):
        with pytest.raises(_lib.ArrowError):
            ctx.set_tuning(thr, seg)
    run_forms(ctx, _case(*DEFAULT_TUNING, 3200, 32), 32)       # the refused calls left the context's tuning alone


# ---- 5. the N-GPU building blocks on one GPU ----------------------------------------------------------------------
@pytest.mark.parametrize("config", ["one_cta", "tile_kernel_0"])
@pytest.mark.parametrize("k", [16, 32, 128, 6])
def test_spmm_ex_exact(ctx, k, config):
    _apply(ctx, SCHEDULES["one_cta"] if config == "one_cta" else {Ctx.OPT_TILE_KERNEL: 0})
    _spmm_ex_exact(ctx, _case(*DEFAULT_TUNING, 3200, k), k, DEFAULT_TUNING[0])


@pytest.mark.parametrize("push_ctas", [0, 1])
@pytest.mark.parametrize("interleave", [1, 0])
@pytest.mark.parametrize("k", [4, 6, 128, 256])
def test_push_rows_exact(ctx, k, interleave, push_ctas):
    """item i of destination d lands in slot i - bound[d]; an empty destination in the middle; unrouted items (-1)
    leave their slot alone; block-after-block and interleaved walks, a one-CTA push grid"""
    ctx.set_option(ctx.OPT_PUSH_INTERLEAVE, interleave)
    ctx.set_option(ctx.OPT_PUSH_CTAS, push_ctas)
    rng = np.random.default_rng(k)
    src = int_features(rng, 3000, k)
    counts = [1700, 0, 333, 1]
    bounds = np.concatenate([[0], np.cumsum(counts)])
    m = rng.integers(0, 3000, bounds[-1])
    m[::11] = -1
    dsrc, dm = ctx.dense_from_host(src), ctx.map_upload(m, 3000)
    dsts = [ctx.dense_alloc(c + 5, k) if c else None for c in counts]
    for d in dsts:
        if d is not None:
            d.fill(7.0)
    ctx.push_rows(dsts, bounds, dsrc, dm)
    for d, c in enumerate(counts):
        if c:
            exp = np.full((c + 5, k), 7.0, np.float32)
            mm = m[bounds[d]:bounds[d + 1]]
            exp[:c][mm >= 0] = src[mm[mm >= 0]]
            assert np.array_equal(dsts[d].d2h(), exp), f"destination {d}"
    for h in [dsrc, dm] + [d for d in dsts if d is not None]:
        h.free()


@pytest.mark.parametrize("k", [6, 130])
def test_reduce_rows_non_vector_k(ctx, k):
    rng = np.random.default_rng(k)
    parts = [int_features(rng, 700, k) for _ in range(5)]
    dparts = [ctx.dense_from_host(p) for p in parts]
    out = ctx.dense_alloc(700, k)
    ctx.reduce_rows(dparts, 700, dst=out)
    assert np.array_equal(out.d2h(), np.sum(np.stack(parts).astype(np.float64), axis=0).astype(np.float32))
    for h in dparts + [out]:
        h.free()


# ---- 6. scheduler words across launches ---------------------------------------------------------------------------
@pytest.mark.parametrize("first", ["round1", "generalised"])
def test_ticket_is_reset_between_tile_kernels(ctx, first):
    """a round-1 launch (which leaves its ticket behind) and a generalised launch (which re-arms it) back to back on one
    lane with no sync in between, three CTAs competing for the ticket"""
    k = 64
    _apply(ctx, SCHEDULES["three_ctas"])
    cs = _case(*DEFAULT_TUNING, 3200, k)
    blk = cs["blk"]
    split = blk.n_cols // 2
    A = blk.upload(ctx)
    X = ctx.dense_from_host(cs["X"])
    X1, X2 = ctx.dense_from_host(cs["X"][:split]), ctx.dense_from_host(np.ascontiguousarray(cs["X"][split:]))
    C1, C2 = ctx.dense_alloc(blk.n_rows, k), ctx.dense_alloc(blk.n_rows, k)
    launches = {"round1": lambda: ctx.spmm(A, X, C1),                                 # k_spmm_tiles_v1
                "generalised": lambda: ctx.spmm_ex(A, X1, C=C2, X2=X2, x_split=split)}  # k_spmm_tiles, dual X
    out = {"round1": C1, "generalised": C2}
    order = [first] + [f for f in launches if f != first]
    for _ in range(2):
        for f in order:
            out[f].fill(7.0)            # stream-ordered: the last launch alone decides what the tile holds
            launches[f]()
    exp = cs["ref"].astype(np.float32)
    assert_exact(C1.d2h(), exp, blk, 512, "round-1 kernel")
    assert_exact(C2.d2h(), exp, blk, 512, "generalised kernel")
    for h in (A, X, X1, X2, C1, C2):
        h.free()


# ---- empty blocks -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tile_kernel", [1, 0])
@pytest.mark.parametrize("k", [4, 32, 10])
def test_empty_blocks(ctx, k, tile_kernel):
    """nnz = 0 with rows: plain launches overwrite C (pre-filled with 7) with zeros, accumulate launches leave it alone;
    n_rows = 0: nothing is written"""
    ctx.set_option(ctx.OPT_TILE_KERNEL, tile_kernel)
    n = 300
    X = ctx.dense_from_host(np.ones((n, k), np.float32))
    A = ctx.csr_upload(n, n, np.zeros(n + 1, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32))
    C = ctx.dense_alloc(n, k)
    rm = ctx.map_upload(np.arange(n)[::-1].copy(), n)
    for acc in (False, True):
        for m in (None, rm):
            C.fill(7.0)
            ctx.spmm(A, X, C, rowmap=m, accumulate=acc)
            exp = np.full((n, k), 7.0 if acc else 0.0, np.float32)
            assert np.array_equal(C.d2h(), exp), (acc, m is not None)
    E = ctx.csr_upload(0, n, np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32))
    C.fill(7.0)
    ctx.spmm(E, X, C)
    ctx.spmm(E, X, C, accumulate=True)
    assert np.array_equal(C.d2h(), np.full((n, k), 7.0, np.float32))
    for h in (X, A, C, rm, E):
        h.free()


# ---- long-row scratch growth after a graph was recorded -----------------------------------------------------------
def test_graph_replay_after_long_row_scratch_grows(cuda_device):
    """record a graph whose SpMM has long rows, then run (eagerly, same lane) a block that needs more long-row tasks
    -- the per-lane scratch grows -- and replay the graph: the replay must still compute the exact product.  A context
    of its own: the module's context already holds a large scratch"""
    ctx = _lib.Context(cuda_device)
    k = 32
    rng = np.random.default_rng(99)
    small = Block([0, 600, 3, 700, 5] + [4] * 300, 2000, rng)          # 2 long rows, one segment each
    big = Block([2048 * 3 + 1] * 6 + [2] * 100, 2000, rng)            # 6 long rows of 4 segments
    for b in (small, big):
        b.check_exact(256.0)
    X = int_features(rng, 2000, k)
    dX = ctx.dense_from_host(X)
    As, Ab = small.upload(ctx), big.upload(ctx)
    Cs, Cb = ctx.dense_alloc(small.n_rows, k), ctx.dense_alloc(big.n_rows, k)
    ctx.spmm(As, dX, Cs)                                              # un-captured run first: scratch for 2 tasks
    ctx.sync()
    ctx.graph_begin()
    ctx.spmm(As, dX, Cs)
    g = ctx.graph_end()
    ctx.spmm(Ab, dX, Cb)                                              # 24 tasks: the scratch grows
    Cs.fill(7.0)
    ctx.graph_launch(g)
    assert_exact(Cs.d2h(), small.product(X).astype(np.float32), small, 512, "graph replay after the scratch grew")
    assert_exact(Cb.d2h(), big.product(X).astype(np.float32), big, 512, "the block that grew the scratch")
    ctx.graph_free(g)                                                 # releases the retired buffer
    Cs.fill(7.0)
    ctx.spmm(As, dX, Cs)
    assert_exact(Cs.d2h(), small.product(X).astype(np.float32), small, 512, "eager run after the graph was freed")
    for h in (dX, As, Ab, Cs, Cb):
        h.free()
    ctx.close()

/*
 * arrow_b200.h -- C ABI of libarrow_b200.so: B200 (sm_100a) arrow-decomposed SpMM hot path.
 *
 * The reference (spcl/arrow-matrix) is pure Python and has no FFI of its own; this is the
 * boundary a maintainer binds with ctypes (see INTEGRATION.md) to replace the arithmetic and the
 * data movement of
 *     arrow/arrow_slim_mpi.py:78-244   (_ad_spmm / _ad_spmm_gpu: three CSR x dense products)
 *     arrow/arrow_mpi.py:177-336       (wide layout: row-tile / column-tile products)
 *     arrow/common/sp2cp.py:6-16       (_sp2cp: per-iteration CSR upload -> upload once)
 *     arrow/arrow_dec_mpi.py:404-440   (backward exchange: C_{j-1}[to_prev[r]] += C_j[r])
 *     arrow/arrow_dec_mpi.py:507-550   (forward exchange:  X_j[r] = X_{j-1}[to_prev[r]])
 *
 * Conventions: extern "C", opaque context, int return codes (0 = ok, negative = error, text via
 * arrow_last_error), no exceptions cross the boundary.  The caller owns host memory; the library
 * owns device memory (handles are small non-negative ints, valid for one context).  All work is
 * stream-ordered on the context's stream; arrow_sync() waits for it.  One host thread per context.
 * Dense tiles are row-major [rows x k] of fp32 (default) or bf16 (ARROW_DTYPE_BF16, one-GPU launches only); CSR is fp32
 * values with int32 column indices on the device and 64-bit non-zero offsets (rows and columns < 2^31, non-zeros bounded
 * by device memory).  Arithmetic is fp32 in both: a kernel widens bf16 inputs to fp32, accumulates
 * in fp32 and rounds every stored bf16 row once, to nearest even.
 */
#ifndef ARROW_B200_H
#define ARROW_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct arrow_ctx arrow_ctx;

#define ARROW_ABI_VERSION 3

/* error codes */
#define ARROW_OK              0
#define ARROW_ERR_CUDA       -1
#define ARROW_ERR_ARG        -2
#define ARROW_ERR_HANDLE     -3
#define ARROW_ERR_RANGE      -4   /* index / size exceeds the device layout (rows, columns, map entries < 2^31) */
#define ARROW_ERR_NOMEM      -5
#define ARROW_ERR_UNSUPPORTED -6

/* flags for arrow_spmm / arrow_gather_rows */
#define ARROW_ACCUMULATE      1   /* C += ... instead of C = ...  (reference: `C_i += A_i0 @ X_0`,
                                     arrow_slim_mpi.py:142-144; scatter-add, arrow_dec_mpi.py:437) */

/* SpMM kernel variants (arrow_spmm `variant`); ARROW_VARIANT_AUTO picks per k. */
#define ARROW_VARIANT_AUTO    -1
#define ARROW_VARIANT_DIRECT   0  /* sub-warp per row, broadcast index loads, float4 X gathers          */
#define ARROW_VARIANT_SHFL     1  /* sub-warp per row, coalesced index/value chunk + shuffle broadcast  */
#define ARROW_VARIANT_TMA      2  /* X rows staged into shared memory with cp.async.bulk + mbarrier     */
#define ARROW_VARIANT_TILES    3  /* default: CSR row tiles streamed by cp.async.bulk (TMA) + mbarrier,
                                     two stages; warps only issue X gathers.  Bits 4..7 of `variant`
                                     optionally force the float4-per-lane count (1, 2 or 4), bits 8..9 the
                                     rows a lane group works on at once (1 or 2; 2 needs k <= 32).     */

int  arrow_b200_abi_version(void);

/* ---- context ------------------------------------------------------------------------------- */
/* `stream` is a cudaStream_t to run on (e.g. torch's current stream) or NULL: the context then
 * creates its own non-blocking stream. */
int  arrow_ctx_create(int device, void *stream, arrow_ctx **out);
void arrow_ctx_destroy(arrow_ctx *ctx);
const char *arrow_last_error(const arrow_ctx *ctx);      /* ctx may be NULL: last creation error */
int  arrow_sync(arrow_ctx *ctx);
int  arrow_device_info(arrow_ctx *ctx, int *sm_count, int64_t *free_bytes, int64_t *total_bytes);
int  arrow_set_tuning(arrow_ctx *ctx, int long_row_threshold, int long_row_segment);
/* Tuning knobs.  L2 hint masks of the tile kernel: bit 0 = X gathers evict_last, bit 1 = CSR and C streams
 * evict_first; PLAIN applies to C = A X launches, FUSED to launches with a row map or ARROW_ACCUMULATE. */
#define ARROW_OPT_L2_HINTS_PLAIN 1
#define ARROW_OPT_L2_HINTS_FUSED 2
#define ARROW_OPT_BIG_TILES      3   /* 1 (default): 128-row / 2048-entry CSR tiles when k <= 32 */
#define ARROW_OPT_PREFETCH        5   /* bulk L2 prefetch (cp.async.bulk.prefetch.L2, one request per X row) of a CSR tile's X rows
                                        before its math: bit 0 = plain launches, bit 4 = fused launches (row map / accumulate /
                                        gather-add / dual X / row pointers).  Measured as a loss (profiles/r02_kernel_sweep.md);
                                        off by default, kept as the A/B switch */
#define ARROW_OPT_SPMM_CTAS_PER_SM 4 /* cap on resident SpMM CTAs per SM (0 = no cap): leaves SM resources to exchange
                                        kernels running on the side lane */
#define ARROW_OPT_ROWS_PER_GROUP  6   /* rows a lane group gathers for at once when k <= 32: 0 (default) = auto (2 at k = 32, else 1), 1, 2 */
#define ARROW_OPT_SPMM_SM_LIMIT   7   /* cap on the SMs a SpMM grid covers (0 = all): concurrent launches on two lanes share the GPU */
#define ARROW_OPT_PUSH_CTAS       8   /* grid of arrow_push_rows (0 = 2 per SM) */
#define ARROW_OPT_SMEM_CARVEOUT  10   /* preferred shared-memory carve-out (percent, -1 = driver default) of the tile kernel: the rest of
                                        the SM's 228 KB is L1, the landing buffer of the gathers in flight (measurement switch) */
#define ARROW_OPT_FORCE_PREDICATED 11  /* 1: the tile kernel takes its predicated gather path even when every column is valid (measurement switch) */
#define ARROW_OPT_TILE_KERNEL     12   /* 1 (default): plain / row-map / accumulate launches with one row per lane group run the round-1 tile
                                        kernel, 0: the generalised kernel everywhere (A/B switch, profiles/r02_kernel_sweep.md).  fp32
                                        only: bf16 launches always run the round-1 kernel */
#define ARROW_OPT_PUSH_INTERLEAVE 13   /* 1 (default): arrow_push_rows walks its destination blocks interleaved (every peer is written to at
                                        every instant); 0: block after block */
#define ARROW_OPT_BARRIER_TIMEOUT_MS 9 /* arrow_peer_barrier gives up after this long (default 30000) and poisons the context */
int  arrow_set_option(arrow_ctx *ctx, int option, int value);

/* ---- sparse blocks (replaces _sp2cp, sp2cp.py:6-16: uploaded once, resident) ----------------- */
/* indptr has n_rows+1 entries of indptr_bytes (4 or 8) each and may start at any base value
 * (a row slice of a bigger file); indices/data point at the entry indptr[0] refers to.
 * data == NULL means all ones (missing _data.npy, graphio.py:292-298).
 * nnz may exceed 2^31 - 1 (any size that fits in device memory).
 * Rejected with ARROW_ERR_ARG / ARROW_ERR_RANGE (nothing stays allocated): a row pointer that is not a
 * non-decreasing sequence spanning exactly nnz entries, a column index outside [0, n_cols), n_rows >= 2^31 - 1 or
 * n_cols >= 2^31 (ARROW_ERR_RANGE before any host array is read), 64 consecutive rows spanning 2^32 or more entries
 * (ARROW_ERR_RANGE). */
int  arrow_csr_upload(arrow_ctx *ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                      const void *indptr, int indptr_bytes,
                      const void *indices, int indices_bytes,
                      const float *data, int *csr_out);
/* Refused (ARROW_ERR_ARG) while remapped copies made by arrow_csr_remap_columns still share the block's arrays. */
int  arrow_csr_free(arrow_ctx *ctx, int csr);
int  arrow_csr_info(arrow_ctx *ctx, int csr, int64_t *n_rows, int64_t *n_cols, int64_t *nnz,
                    int64_t *max_row_nnz, int64_t *n_long_rows);
/* New CSR sharing indptr/values with `csr`, columns sent through `map` (col' = map[col]; entries
 * whose image is invalid are skipped by the kernels).  This folds the forward permutation gather
 * (arrow_dec_mpi.py:526, 544) into the SpMM's X read.  `map`'s limit must not exceed new_n_cols; the copy must be
 * freed before its source. */
int  arrow_csr_remap_columns(arrow_ctx *ctx, int csr, int map, int64_t new_n_cols, int *csr_out);

/* ---- row maps (to_prev / to_next slices, arrow_dec_mpi.py:737-749) ---------------------------- */
/* int64 host map -> int32 device map; entries < 0 or >= limit (the reference's sentinel
 * 2*width*n_blocks[0] lands here) become -1 = "not routed". */
int  arrow_map_upload(arrow_ctx *ctx, const int64_t *map, int64_t n, int64_t limit, int *map_out);
int  arrow_map_free(arrow_ctx *ctx, int map);
/* out[r] = outer[inner[r]] (invalid if either step is); chains level maps for the fused path. */
int  arrow_map_compose(arrow_ctx *ctx, int inner, int outer, int *map_out);
/* out[q] = r where map[r] == q (injective maps only), size n_out, -1 elsewhere. */
int  arrow_map_invert(arrow_ctx *ctx, int map, int64_t n_out, int *map_out);
int  arrow_map_d2h(arrow_ctx *ctx, int map, int32_t *host, int64_t n);

/* ---- dense tiles (X_i / C_i / X_0 / C_0 of arrow_slim_mpi.py:354-394, concatenated) ----------- */
/* Element types of a dense tile.  Every launch needs all its tiles in one dtype (ARROW_ERR_ARG otherwise).  bf16 tiles
 * serve the one-GPU launches (arrow_spmm, arrow_spmm_add, arrow_gather_rows, arrow_dense_*); the N-GPU entry points
 * (arrow_spmm_ex, arrow_push_rows, arrow_reduce_rows, arrow_gather_rows_multi, arrow_ipc_export) refuse them, and
 * arrow_dense_wrap / arrow_ipc_import make fp32 tiles. */
#define ARROW_DTYPE_F32  0
#define ARROW_DTYPE_BF16 1
int  arrow_dense_alloc(arrow_ctx *ctx, int64_t rows, int k, int *buf_out);      /* zero filled, fp32 */
int  arrow_dense_alloc_dtype(arrow_ctx *ctx, int64_t rows, int k, int dtype, int *buf_out);   /* zero filled */
int  arrow_dense_dtype(arrow_ctx *ctx, int buf, int *dtype);
int  arrow_dense_free(arrow_ctx *ctx, int buf);
int  arrow_dense_fill(arrow_ctx *ctx, int buf, float value);      /* bf16 tiles: value rounded to nearest even */
/* fp32 tiles only (a bf16 tile is refused): */
int  arrow_dense_h2d(arrow_ctx *ctx, int buf, int64_t row0, int64_t rows, const float *host);
int  arrow_dense_d2h(arrow_ctx *ctx, int buf, int64_t row0, int64_t rows, float *host);
/* Rows in the tile's own dtype (rows x k x 4 or 2 bytes), on copy lane `lane` (ARROW_LANE_*, below; ARROW_LANE_MAIN =
 * the context's stream).  Stream-ordered like arrow_dense_h2d / d2h: the host memory must stay valid until the lane
 * has been synchronised. */
int  arrow_dense_put(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, const void *host);
int  arrow_dense_get(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, void *host);
int  arrow_dense_copy(arrow_ctx *ctx, int dst, int64_t dst_row0, int src, int64_t src_row0, int64_t rows);   /* equal dtypes */
int  arrow_dense_ptr(arrow_ctx *ctx, int buf, void **device_ptr, int64_t *rows, int *k);
/* Wrap device memory owned by someone else (a torch tensor, an IPC-imported peer tile). */
int  arrow_dense_wrap(arrow_ctx *ctx, void *device_ptr, int64_t rows, int k, int *buf_out);
/* Copy lanes: host<->device staging on side streams so that step i's download, step i+1's upload and the
 * compute in between overlap (PCIe is full duplex).  Lane 0 is the context's main stream.  arrow_lane_wait
 * makes `waiting_lane` wait for everything submitted so far on `signalling_lane` (event, no host sync).
 * Replaces the blocking cp.asarray / cp.asnumpy round trips of arrow_slim_mpi.py:186-191, 228-232. */
#define ARROW_LANE_MAIN 0
#define ARROW_LANE_H2D  1
#define ARROW_LANE_D2H  2
#define ARROW_LANE_SIDE 3   /* compute-side lane: exchange kernels overlapping the main lane's SpMM */
#define ARROW_N_LANES   4
int  arrow_dense_h2d_lane(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, const float *host);
int  arrow_dense_d2h_lane(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, float *host);
int  arrow_lane_wait(arrow_ctx *ctx, int waiting_lane, int signalling_lane);
int  arrow_lane_sync(arrow_ctx *ctx, int lane);
/* Select the lane on which the following arrow_spmm* / arrow_gather_rows[_multi] / arrow_push_rows / arrow_reduce_rows /
 * arrow_peer_barrier / arrow_dense_copy calls are launched (every lane has its own tile scheduler state).  Used to run
 * the exchange chain of the deeper levels beside the level-0 SpMM; a barrier issued on lane L must use flag tiles
 * reserved for lane L. */
int  arrow_set_lane(arrow_ctx *ctx, int lane);
/* Named events for finer ordering between lanes (waiting on a never-recorded event is a no-op). */
#define ARROW_MAX_EVENTS 16
int  arrow_event_record(arrow_ctx *ctx, int event, int lane);
int  arrow_event_wait(arrow_ctx *ctx, int event, int lane);
/* pinned host staging */
int  arrow_host_alloc(size_t bytes, void **ptr);
int  arrow_host_free(void *ptr);
/* Pinned staging memory placed on the NUMA node of `device` (mmap + mbind + first touch + cudaHostRegister); freed with
 * arrow_host_free.  arrow_bind_thread_to_device_numa pins the calling thread to that node's CPUs (node_out = -1 when
 * the topology is unknown: nothing is changed); device < 0 undoes it (every CPU, default memory policy). */
int  arrow_host_alloc_numa(size_t bytes, int device, void **ptr);
int  arrow_bind_thread_to_device_numa(int device, int *node_out, int *n_cpus_out);

/* ---- the hot path ------------------------------------------------------------------------------ */
/* C[out(r), :] (+)= sum_p A[r, col_p] * X[col_p, :]   for every row r of `csr`
 *   out(r) = r, or rowmap[r] when rowmap >= 0 (rows with rowmap[r] == -1 are dropped): the backward
 *   scatter-add of arrow_dec_mpi.py:421-437 folded into the SpMM epilogue.
 * X must have >= n_cols rows; C must cover every out(r); X and C must not alias. */
int  arrow_spmm(arrow_ctx *ctx, int csr, int x_buf, int c_buf, int rowmap, int flags, int variant);

/* C[r, :] = sum_p A[r, col_p] * X[col_p, :] + add[add_map[r], :]   (rows with add_map[r] == -1 get the product only).
 * The backward exchange C_{j-1}[to_prev[r]] += C_j[r] (arrow_dec_mpi.py:437) folded into the RECEIVING level's SpMM as
 * a gather-add: levels are multiplied deepest first, each writes its tile once, nothing is read-modify-written. */
int  arrow_spmm_add(arrow_ctx *ctx, int csr, int x_buf, int c_buf, int add_buf, int add_map, int variant);

/* dst[r, :] (+)= src[map[r], :] for r in [0, map length); rows with map[r] == -1 are left alone
 * (the reference's stale-row behaviour, arrow_dec_mpi.py:544).  Forward exchange with to_prev,
 * backward exchange (as a gather-add) with to_next. */
int  arrow_gather_rows(arrow_ctx *ctx, int dst_buf, int src_buf, int map, int flags);

/* Multi-source gather over NVLink peer memory: `map` holds GLOBAL source rows; source s owns global
 * rows [row_bounds[s], row_bounds[s+1]) and src_bufs[s] is its (wrapped / IPC-imported) tile. */
int  arrow_gather_rows_multi(arrow_ctx *ctx, int dst_buf, const int *src_bufs,
                             const int64_t *row_bounds, int n_src, int map, int flags);

/* ---- the fused multi-GPU step ------------------------------------------------------------------- */
/* A pointer table holds one destination per row: tile bufs[which[i]], row row[i] (which[i] < 0: the row is dropped).
 * The tiles may be peer GPUs' memory (arrow_ipc_import): a SpMM with a pointer table delivers every result row
 * straight to the GPU that needs it -- the backward exchange (pack + Alltoallv + scatter-add,
 * arrow_dec_mpi.py:421, 442-475, 437) folded into the epilogue as NVLink stores. */
int  arrow_ptrtable_upload(arrow_ctx *ctx, const int *bufs, int n_bufs, const int32_t *which, const int64_t *row,
                           int64_t n, int *table_out);
int  arrow_ptrtable_free(arrow_ctx *ctx, int table);
/* Generalised product.  Columns < x_split read X[col], columns >= x_split read X2[col - x_split] (x2_buf < 0: X only):
 * the feature operand of a level > 0 is [this GPU's level-0 tile | receive region filled by its peers], never
 * materialised as a tile of its own (forward exchange, arrow_dec_mpi.py:507-550, folded into the column indices).
 * out_table >= 0: row r is written to table[r] (c_buf may be -1); else to C[r].  add_buf / add_map as arrow_spmm_add. */
int  arrow_spmm_ex(arrow_ctx *ctx, int csr, int x_buf, int x2_buf, int64_t x_split, int c_buf, int out_table,
                   int add_buf, int add_map, int variant);
/* Push: for item i in [item_bounds[d], item_bounds[d+1]):  dst_bufs[d][i - item_bounds[d]] = src[map[i]].
 * The forward exchange in one pass: local gather, sequential posted stores into each peer's receive region. */
int  arrow_push_rows(arrow_ctx *ctx, const int *dst_bufs, const int64_t *item_bounds, int n_dst, int src_buf, int map);
/* out(r) = sum_s src_bufs[s][r] (source order, deterministic) for r < rows; out(r) = table[r] when out_table >= 0 and the
 * entry is non-null, else dst_buf[r] (dst_buf may be -1: rows without a table entry are skipped).  The reduction of
 * the partial head tiles (Reduce, arrow_slim_mpi.py:116) in one launch, reading the peers over NVLink. */
int  arrow_reduce_rows(arrow_ctx *ctx, int dst_buf, int out_table, const int *src_bufs, int n_src, int64_t rows);

/* ---- CUDA graphs: record a whole step once, replay it with one call ------------------------------ */
/* Between begin and end every launch on the main lane (and on lanes forked from / joined back into it with
 * arrow_lane_wait) is recorded, not executed.  Run the step once un-captured first (lazy allocations). */
int  arrow_graph_begin(arrow_ctx *ctx);
int  arrow_graph_end(arrow_ctx *ctx, int *graph_out);
int  arrow_graph_launch(arrow_ctx *ctx, int graph);
int  arrow_graph_free(arrow_ctx *ctx, int graph);

/* ---- cross-process peer memory (one process per GPU; NVLink P2P through CUDA IPC) -------------- */
/* handle = 64-byte cudaIpcMemHandle_t + 8-byte offset of the tile inside the exported allocation + padding */
#define ARROW_IPC_HANDLE_BYTES 80
int  arrow_ipc_export(arrow_ctx *ctx, int buf, void *handle);
int  arrow_ipc_import(arrow_ctx *ctx, const void *handle, int64_t rows, int k, int *buf_out);
/* Device-side barrier across `world` ranks over peer-mapped flag words (no host sync, no NCCL):
 * flags_buf[s] is rank s's flag tile (>= world words), my slot = rank.  The epoch counter is device resident (one per
 * lane), so the launch can be part of a captured graph.  A barrier that waits longer than ARROW_OPT_BARRIER_TIMEOUT_MS
 * sets a device flag; arrow_sync / arrow_lane_sync then fail and the context refuses further launches. */
int  arrow_peer_barrier(arrow_ctx *ctx, const int *flag_bufs, int rank, int world);

/* ---- timing (CUDA events on the context's stream) ----------------------------------------------- */
#define ARROW_MAX_TIMERS 32
int  arrow_timer_start(arrow_ctx *ctx, int slot);
int  arrow_timer_stop(arrow_ctx *ctx, int slot);
int  arrow_timer_elapsed_ms(arrow_ctx *ctx, int slot, float *ms);   /* synchronises on the stop event */
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int  arrow_launch_count(arrow_ctx *ctx, int64_t *count);

/* Run every kernel a step with `k` feature columns can launch once, on tiny operands.  CUDA loads a kernel lazily at
 * its first launch and loading synchronises the context: if that happens while arrow_peer_barrier spins on another lane
 * (or, with several rank threads in one process, in another rank) the step hangs until the barrier times out.  Call it
 * after arrow_ctx_create, before the first barrier -- or start the process with CUDA_MODULE_LOADING=EAGER. */
int  arrow_preload_kernels(arrow_ctx *ctx, int k);

/* measurement helpers used by bench.py: write `bytes` of scratch (L2 flush) */
int  arrow_l2_flush(arrow_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* ARROW_B200_H */

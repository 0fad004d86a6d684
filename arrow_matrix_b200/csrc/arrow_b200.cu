// libarrow_b200.so -- hand-written sm_100a kernels + C ABI for the arrow-decomposed SpMM hot path.
//
// What each piece replaces in the reference (spcl/arrow-matrix, paths relative to /root/reference):
//   k_spmm_*            scipy `csr @ dense` / cupy->cuSPARSE SpMM at arrow_slim_mpi.py:109-111,125-127,
//                       142-144,190,211,231 and arrow_mpi.py:198-219,250-269,289-291,323
//   csr upload (once)   common/sp2cp.py:6-16 (_sp2cp, redone every iteration by the reference)
//   rowmap epilogue     arrow_dec_mpi.py:421,437  (pack + alltoallv + `C_i[perm] += recvbuf`)
//   remapped columns    arrow_dec_mpi.py:526,544  (`feature_tile()[perm]` + `C_i[perm] = recvbuf`)
//   k_gather_rows*      the same two exchanges as standalone (un-fused / cross-GPU) steps
//
// Layout: CSR = 4-byte row pointer holding the low 32 bits of 64-bit offsets (rebased to 0; tiles, long-row tasks and
// 64-row anchors carry the 64-bit bases) / int32 indices / fp32 values; dense tiles row-major fp32 or bf16 (one-GPU
// launches; fp32 arithmetic, each stored bf16 row rounded once to nearest even).
// All kernels are HBM/L2-bandwidth bound gathers (about 2 FLOP/B): no tensor cores on purpose.
#include "../../include/arrow_b200.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <ctype.h>
#include <dlfcn.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <type_traits>
#include <string>
#include <vector>

// ------------------------------------------------------------------------------------------------
// context + handle tables
// ------------------------------------------------------------------------------------------------
namespace {

struct DenseBuf {
    float *p = nullptr;               // ARROW_DTYPE_BF16: the bits of bf16 elements (use esize(), never p + i for an offset)
    int64_t rows = 0;
    int k = 0;
    int dtype = ARROW_DTYPE_F32;
    bool owned = false;
    bool ipc = false;
    void *ipc_base = nullptr;
    bool live = false;
    size_t esize() const { return dtype == ARROW_DTYPE_BF16 ? 2 : 4; }
    char *row(int64_t r) const { return reinterpret_cast<char *>(p) + (size_t)r * k * esize(); }
};

struct LongTask {      // one segment of a long row
    long long begin;   // nnz offsets (rebased, 64-bit)
    long long end;
    int row;
    int slot;          // partial-sum slot
};

// Rows per anchor of the per-row kernels: the 64-bit offset of row r is anchors[r / ROW_GROUP] plus the 32-bit wrapping
// difference of the row pointer's low words, exact while one group spans fewer than 2^32 entries (checked at upload).
constexpr int ROW_GROUP_SHIFT = 6;
constexpr int ROW_GROUP = 1 << ROW_GROUP_SHIFT;

struct Csr {
    int64_t n_rows = 0, n_cols = 0, nnz = 0;
    int *indptr = nullptr;            // low 32 bits of each row's 64-bit first entry
    int *indices = nullptr;
    float *vals = nullptr;
    bool owns_indptr = false, owns_indices = false, owns_vals = false;
    bool may_skip = false;            // indices may contain -1 (remapped through a partial map)
    int64_t max_row_nnz = 0;
    // long rows (nnz > threshold) are processed by whole CTAs in segments, then reduced in order
    int n_long_rows = 0;
    int n_long_tasks = 0;
    LongTask *long_tasks = nullptr;   // device
    int *long_rows = nullptr;         // device: row ids
    int *long_first = nullptr;        // device: first slot of each long row (n_long_rows+1)
    bool owns_long = false;
    int long_threshold = 0;
    long long *anchors = nullptr;     // device: 64-bit first entry of every ROW_GROUP-th row (owned with the long rows)
    // row tiles for the CSR-streaming kernel: {row_begin, row_end, low 32 bits of nnz_begin, of nnz_end}, and the
    // tile's 64-bit nnz_begin in a parallel array
    int4 *tiles = nullptr;
    long long *tile_base = nullptr;
    int n_tiles = 0;
    int4 *tiles_big = nullptr;        // TILE_ROWS_BIG / TILE_NNZ_BIG variant for narrow feature tiles
    long long *tile_base_big = nullptr;
    int n_tiles_big = 0;
    int parent = -1;                  // handle of the block whose indptr / values / tiles this one shares (remapped copy)
    int children = 0;                 // live remapped copies that share this block's arrays
    bool live = false;
};

struct IdxMap {
    int *p = nullptr;
    int64_t n = 0;
    int64_t limit = 0;
    bool live = false;
};

struct Timer {
    cudaEvent_t a = nullptr, b = nullptr;
};

struct PtrTable {                     // one device pointer per row: where a SpMM / reduction writes that row
    float **p = nullptr;
    int64_t n = 0;
    int k = 0;
    bool live = false;
};

thread_local std::string g_create_error;
std::mutex g_numa_mu;                         // arrow_host_alloc_numa bookkeeping (pointer -> mapped length)
std::map<void *, size_t> g_numa_allocs;

}  // namespace

struct arrow_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    std::string err;
    std::vector<DenseBuf> dense;
    std::vector<Csr> csrs;
    std::vector<IdxMap> maps;
    Timer timers[ARROW_MAX_TIMERS];
    int64_t launches = 0;
    int long_threshold = 512;
    int long_segment = 2048;
    int l2_hints_plain = 3;           // arrow_set_option(ARROW_OPT_L2_HINTS_PLAIN)
    int l2_hints_fused = 0;           // arrow_set_option(ARROW_OPT_L2_HINTS_FUSED)
    int big_tiles = 1;                // arrow_set_option(ARROW_OPT_BIG_TILES): 128-row tiles when k <= 32
    int spmm_ctas_per_sm = 0;         // arrow_set_option(ARROW_OPT_SPMM_CTAS_PER_SM): 0 = as many as fit
    int prefetch_plain = 0;           // arrow_set_option(ARROW_OPT_PREFETCH): low nibble = plain launches, high nibble = fused launches;
    int prefetch_fused = 0;           //   0 none, 1 bulk L2 prefetch of the current tile's X rows, 2 of the next tile's (look-ahead)
    int rows_per_group = 0;           // arrow_set_option(ARROW_OPT_ROWS_PER_GROUP): 0 = auto (pairs at k = 32), 1 / 2 forced
    int spmm_sm_limit = 0;            // arrow_set_option(ARROW_OPT_SPMM_SM_LIMIT): cap on the SMs a SpMM grid covers (0 = all)
    int clock_khz = 2000000;          // SM clock (kHz) for the barrier time-out
    int tile_kernel = 1;              // arrow_set_option(ARROW_OPT_TILE_KERNEL): 1 = round-1 kernel for the launches it covers, 0 = generalised kernel everywhere
    int force_skip_path = 0;          // arrow_set_option(ARROW_OPT_FORCE_PREDICATED): measurement switch
    int smem_carveout = -1;           // arrow_set_option(ARROW_OPT_SMEM_CARVEOUT): preferred shared-memory carve-out (percent) of the tile kernel
    int push_interleave = 1;          // arrow_set_option(ARROW_OPT_PUSH_INTERLEAVE): 1 = the push grid serves all destinations at once
    int push_ctas = 0;                // arrow_set_option(ARROW_OPT_PUSH_CTAS): grid of the NVLink push kernel (0 = default)
    long long barrier_timeout_ms = 30000;   // arrow_set_option(ARROW_OPT_BARRIER_TIMEOUT_MS)
    bool poisoned = false;            // a peer barrier timed out: later launches are refused (results would be racy)
    float *long_scratch[ARROW_N_LANES] = {};    // [slots][k] partial sums of long-row segments, per lane
    size_t long_scratch_bytes[ARROW_N_LANES] = {};
    std::vector<float *> retired_scratch;       // replaced long-row scratch a recorded graph may still address: freed
                                                // with the last graph (arrow_graph_free) or the context
    void *flush_buf = nullptr;
    size_t flush_bytes = 0;
    unsigned int *barrier_epoch = nullptr;        // device: one epoch counter per lane (each lane has its own flag set);
                                                  // device-resident so that a captured CUDA graph can be replayed
    int cur_lane = 0;                             // lane used by the launches that follow (arrow_set_lane)
    int *dev_status = nullptr;        // device-side status word (barrier timeout)
    int *tile_ticket = nullptr;       // device: per lane {next tile, finished CTAs} of the dynamic tile scheduler
    std::vector<PtrTable> ptrtabs;
    std::vector<cudaGraphExec_t> graphs;
    std::vector<int64_t> graph_kernels;           // kernels recorded in each graph (arrow_launch_count stays truthful under replay)
    int64_t capture_launches0 = 0;
    bool capturing = false;
    cudaStream_t lanes[ARROW_N_LANES] = {};   // lane 0 = main stream
    cudaEvent_t lane_events[ARROW_N_LANES] = {};
    cudaEvent_t user_events[ARROW_MAX_EVENTS] = {};
};

namespace {

int fail(arrow_ctx *ctx, int code, const char *fmt, ...) __attribute__((format(printf, 3, 4)));
int fail(arrow_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

cudaStream_t cur_stream(arrow_ctx *ctx) {
    return (ctx->cur_lane > 0 && ctx->lanes[ctx->cur_lane]) ? ctx->lanes[ctx->cur_lane] : ctx->stream;
}

#define CUDA_TRY(ctx, expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail((ctx), ARROW_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                \
                        cudaGetErrorString(_e), __FILE__, __LINE__);                          \
    } while (0)

#define CHECK_CTX(ctx)                                                                        \
    do {                                                                                      \
        if (!(ctx)) return fail(nullptr, ARROW_ERR_ARG, "null context");                      \
        cudaError_t _e = cudaSetDevice((ctx)->device);                                        \
        if (_e != cudaSuccess)                                                                \
            return fail((ctx), ARROW_ERR_CUDA, "cudaSetDevice(%d): %s", (ctx)->device,        \
                        cudaGetErrorString(_e));                                              \
    } while (0)

cudaStream_t cur_stream(arrow_ctx *ctx);

template <class T>
int new_slot(std::vector<T> &v) {
    for (size_t i = 0; i < v.size(); ++i)
        if (!v[i].live) return (int)i;
    v.emplace_back();
    return (int)v.size() - 1;
}

DenseBuf *get_dense(arrow_ctx *ctx, int h) {
    if (h < 0 || h >= (int)ctx->dense.size() || !ctx->dense[h].live) return nullptr;
    return &ctx->dense[h];
}
Csr *get_csr(arrow_ctx *ctx, int h) {
    if (h < 0 || h >= (int)ctx->csrs.size() || !ctx->csrs[h].live) return nullptr;
    return &ctx->csrs[h];
}
IdxMap *get_map(arrow_ctx *ctx, int h) {
    if (h < 0 || h >= (int)ctx->maps.size() || !ctx->maps[h].live) return nullptr;
    return &ctx->maps[h];
}

// the entry points of the N-GPU path and the float * copies take fp32 tiles only
#define REQUIRE_F32(ctx, d, what)                                                                              \
    do {                                                                                                       \
        if ((d)->dtype != ARROW_DTYPE_F32) return fail((ctx), ARROW_ERR_ARG, "%s needs an fp32 tile (this one is bf16)", (what)); \
    } while (0)

inline int ceil_div_i64(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

bool graphs_live(const arrow_ctx *ctx) {
    for (auto g : ctx->graphs)
        if (g) return true;
    return false;
}

// frees whatever device arrays the block owns (cudaFree waits for the device, so no launch can still read them)
void csr_release(Csr &c) {
    if (c.owns_indptr) cudaFree(c.indptr);
    if (c.owns_indices) cudaFree(c.indices);
    if (c.owns_vals) cudaFree(c.vals);
    if (c.owns_long) {
        cudaFree(c.long_tasks);
        cudaFree(c.long_rows);
        cudaFree(c.long_first);
        cudaFree(c.tiles);
        cudaFree(c.tiles_big);
        cudaFree(c.tile_base);
        cudaFree(c.tile_base_big);
        cudaFree(c.anchors);
    }
    c = Csr();
}

struct DevTmp {                       // scratch allocation released on every exit path
    void *p = nullptr;
    ~DevTmp() { if (p) cudaFree(p); }
};

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void f4_fma(float4 &acc, float a, const float4 &x) {
    acc.x = fmaf(a, x.x, acc.x);
    acc.y = fmaf(a, x.y, acc.y);
    acc.z = fmaf(a, x.z, acc.z);
    acc.w = fmaf(a, x.w, acc.w);
}
__device__ __forceinline__ void f4_add(float4 &acc, const float4 &x) {
    acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
}

typedef __nv_bfloat16 bf16;

// Element type of the dense tiles of a launch.  The vector kernels move rows as 16-byte vectors held in float4
// registers as raw bits (4 fp32 or 8 bf16 values) and accumulate one vector in an `Acc` of fp32; `pack` is the one
// rounding of a stored row.  Scalar kernels use to_f / from_f.
template <typename T>
struct Elt;
template <>
struct Elt<float> {
    static constexpr int PER_VEC = 4;
    using Acc = float4;
    static __device__ __forceinline__ Acc zero() { return f4_zero(); }
    static __device__ __forceinline__ Acc widen(const float4 &x) { return x; }
    static __device__ __forceinline__ void fma(Acc &acc, float a, const float4 &x) { f4_fma(acc, a, x); }
    static __device__ __forceinline__ void add(Acc &acc, const float4 &x) { f4_add(acc, x); }
    static __device__ __forceinline__ float4 pack(const Acc &acc) { return acc; }
    static __device__ __forceinline__ float to_f(float x) { return x; }
    static __device__ __forceinline__ float from_f(float x) { return x; }
};
template <>
struct Elt<bf16> {
    static constexpr int PER_VEC = 8;
    struct Acc { float4 lo, hi; };                  // elements 0..3, 4..7 of the vector
    // bf16 -> fp32 is exact: the element becomes the upper half of an fp32 word (a shift or a mask, no F2F).  Element
    // 2i is the low half of word i (little endian), element 2i+1 the high half.
    static __device__ __forceinline__ float lo(float w) { return __uint_as_float(__float_as_uint(w) << 16); }
    static __device__ __forceinline__ float hi(float w) { return __uint_as_float(__float_as_uint(w) & 0xffff0000u); }
    static __device__ __forceinline__ Acc zero() { return Acc{f4_zero(), f4_zero()}; }
    static __device__ __forceinline__ Acc widen(const float4 &x) {
        return Acc{make_float4(lo(x.x), hi(x.x), lo(x.y), hi(x.y)), make_float4(lo(x.z), hi(x.z), lo(x.w), hi(x.w))};
    }
    static __device__ __forceinline__ void fma(Acc &acc, float a, const float4 &x) {
        acc.lo.x = fmaf(a, lo(x.x), acc.lo.x);
        acc.lo.y = fmaf(a, hi(x.x), acc.lo.y);
        acc.lo.z = fmaf(a, lo(x.y), acc.lo.z);
        acc.lo.w = fmaf(a, hi(x.y), acc.lo.w);
        acc.hi.x = fmaf(a, lo(x.z), acc.hi.x);
        acc.hi.y = fmaf(a, hi(x.z), acc.hi.y);
        acc.hi.z = fmaf(a, lo(x.w), acc.hi.z);
        acc.hi.w = fmaf(a, hi(x.w), acc.hi.w);
    }
    static __device__ __forceinline__ void add(Acc &acc, const float4 &x) {
        const Acc w = widen(x);
        f4_add(acc.lo, w.lo);
        f4_add(acc.hi, w.hi);
    }
    static __device__ __forceinline__ float pack2(float e0, float e1) {      // round-to-nearest-even, e0 in the low half
        uint32_t r;
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));
        return __uint_as_float(r);
    }
    static __device__ __forceinline__ float4 pack(const Acc &a) {
        return make_float4(pack2(a.lo.x, a.lo.y), pack2(a.lo.z, a.lo.w), pack2(a.hi.x, a.hi.y), pack2(a.hi.z, a.hi.w));
    }
    static __device__ __forceinline__ float to_f(bf16 x) { return __bfloat162float(x); }
    static __device__ __forceinline__ bf16 from_f(float x) { return __float2bfloat16_rn(x); }
};
template <typename T>
constexpr bool is_bf16() { return std::is_same<T, bf16>::value; }

struct SpmmArgs {
    const int *__restrict__ indptr;   // low 32 bits of the 64-bit row offsets
    const long long *__restrict__ anchors;   // 64-bit offset of every ROW_GROUP-th row (per-row kernels)
    const int *__restrict__ indices;
    const float *__restrict__ vals;
    const float *__restrict__ X;      // dense tiles (X, C, X2, add_src) hold the launch's element type T (Elt<T>)
    float *__restrict__ C;
    const int *__restrict__ rowmap;   // nullptr: identity
    long long n_rows;
    int k;                            // feature columns
    int k4;                           // 16-byte vectors per row: k / Elt<T>::PER_VEC (vector kernels)
    int long_threshold;               // rows with more entries are left to the long-row kernels
    const float *__restrict__ add_src;   // optional addend: C[r] = sum + add_src[add_map[r]] (add_map[r] >= 0), else nullptr
    const int *__restrict__ add_map;
    const float *__restrict__ X2;        // optional second X base: columns >= x_split address X2[col - x_split] (else nullptr)
    int x_split;
    float *const *__restrict__ out_ptr;  // optional destination pointer per row (nullptr entry = row dropped); overrides C / rowmap
};

// a - b of two row-pointer low words: exact for any two offsets less than 2^32 apart (no signed overflow)
__device__ __forceinline__ int wdiff(int a, int b) { return (int)((unsigned)a - (unsigned)b); }

// 64-bit first entry and length of `row` (per-row kernels)
__device__ __forceinline__ long long row_begin(const SpmmArgs &a, long long row, long long &len) {
    const long long anchor = __ldg(a.anchors + (row >> ROW_GROUP_SHIFT));
    const int lo = __ldg(a.indptr + row);
    len = (unsigned)wdiff(__ldg(a.indptr + row + 1), lo);
    return anchor + (unsigned)wdiff(lo, (int)anchor);
}

// ------------------------------------------------------------------------------------------------
// variant 0: a group of G lanes owns one row; every lane of the group reads the same index/value
// (hardware broadcast) and its own float4 slice of the X row.  UNROLL independent X gathers in flight.
// ------------------------------------------------------------------------------------------------
// __launch_bounds__(256, 4): without the min-blocks bound ptxas aims at full occupancy (<= 40 registers)
// and serialises every gather behind the FFMAs of the previous one; with it all UNROLL gathers of a
// batch are issued back to back (checked in SASS), which is what hides the L2 / HBM latency.
template <int G, int VPL, bool ROWMAP, bool ACC>
__global__ void __launch_bounds__(256, 4) k_spmm_direct(SpmmArgs a) {
    constexpr int RPW = 32 / G;
    constexpr int UNROLL = (VPL == 1) ? 8 : 4;
    const int lane = threadIdx.x & 31;
    const int gl = lane % G;                      // lane inside the group
    const int gi = lane / G;                      // group inside the warp
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const float4 *__restrict__ X4 = reinterpret_cast<const float4 *>(a.X);
    float4 *__restrict__ C4 = reinterpret_cast<float4 *>(a.C);
    const int k4 = a.k4;

    for (long long row = warp_id * RPW + gi; row < a.n_rows; row += warps_total * RPW) {
        long long len;
        const long long s = row_begin(a, row, len);
        if (len > a.long_threshold) continue;
        const long long e = s + len;
        long long orow = row;
        if (ROWMAP) {
            orow = __ldg(a.rowmap + row);
            if (orow < 0) continue;
        }
        float4 acc[VPL];
#pragma unroll
        for (int i = 0; i < VPL; ++i) acc[i] = f4_zero();

        for (long long p = s; p < e; p += UNROLL) {
            int c[UNROLL];
            float v[UNROLL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                const bool ok = p + u < e;
                c[u] = ok ? __ldcs(a.indices + p + u) : -1;
                v[u] = ok ? __ldcs(a.vals + p + u) : 0.f;
            }
            float4 x[UNROLL][VPL];
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                for (int i = 0; i < VPL; ++i) {
                    const int vec = gl + i * G;
                    x[u][i] = (c[u] >= 0 && vec < k4) ? __ldg(X4 + (long long)c[u] * k4 + vec) : f4_zero();
                }
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                for (int i = 0; i < VPL; ++i) f4_fma(acc[i], v[u], x[u][i]);
        }
#pragma unroll
        for (int i = 0; i < VPL; ++i) {
            const int vec = gl + i * G;
            if (vec < k4) {
                float4 *dst = C4 + orow * k4 + vec;
                if (ACC) {
                    float4 old = *dst;
                    f4_add(acc[i], old);
                    *dst = acc[i];
                } else {
                    __stcs(dst, acc[i]);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// variant 1: the group loads G consecutive (index, value) pairs of its row with ONE coalesced request
// each and broadcasts them with width-G shuffles; the X gathers are issued UNROLL at a time.
// ------------------------------------------------------------------------------------------------
template <int G, int VPL, bool ROWMAP, bool ACC>
__global__ void __launch_bounds__(256, 4) k_spmm_shfl(SpmmArgs a) {
    constexpr int RPW = 32 / G;
    constexpr int UWANT = (VPL == 1) ? 8 : 4;
    constexpr int UNROLL = (G >= UWANT) ? UWANT : G;
    const int lane = threadIdx.x & 31;
    const int gl = lane % G;
    const int gi = lane / G;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const float4 *__restrict__ X4 = reinterpret_cast<const float4 *>(a.X);
    float4 *__restrict__ C4 = reinterpret_cast<float4 *>(a.C);
    const int k4 = a.k4;

    // warp-uniform trip count: every lane of the warp runs the same number of row iterations
    for (long long row0 = warp_id * RPW; row0 < a.n_rows; row0 += warps_total * RPW) {
        const long long row = row0 + gi;
        long long s = 0;
        int len = 0;
        long long orow = -1;
        if (row < a.n_rows) {
            long long n;
            s = row_begin(a, row, n);
            orow = row;
            if (ROWMAP) orow = __ldg(a.rowmap + row);
            if (n > a.long_threshold || orow < 0) orow = -1;
            else len = (int)n;
        }
        const int maxlen = __reduce_max_sync(0xffffffffu, len);
        float4 acc[VPL];
#pragma unroll
        for (int i = 0; i < VPL; ++i) acc[i] = f4_zero();

        for (int base = 0; base < maxlen; base += G) {
            int myc = -1;
            float myv = 0.f;
            if (base + gl < len) {
                myc = __ldcs(a.indices + s + base + gl);
                myv = __ldcs(a.vals + s + base + gl);
            }
            const int cnt = min(G, maxlen - base);               // warp-uniform
            for (int u0 = 0; u0 < cnt; u0 += UNROLL) {
                int c[UNROLL];
                float v[UNROLL];
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) {
                    c[u] = __shfl_sync(0xffffffffu, myc, (u0 + u) % G, G);
                    v[u] = __shfl_sync(0xffffffffu, myv, (u0 + u) % G, G);
                    if (u0 + u >= G) c[u] = -1;
                }
                float4 x[UNROLL][VPL];
#pragma unroll
                for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                    for (int i = 0; i < VPL; ++i) {
                        const int vec = gl + i * G;
                        x[u][i] = (c[u] >= 0 && vec < k4) ? __ldg(X4 + (long long)c[u] * k4 + vec) : f4_zero();
                    }
#pragma unroll
                for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                    for (int i = 0; i < VPL; ++i) f4_fma(acc[i], v[u], x[u][i]);
            }
        }
        if (orow >= 0) {
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
                const int vec = gl + i * G;
                if (vec < k4) {
                    float4 *dst = C4 + orow * k4 + vec;
                    if (ACC) {
                        float4 old = *dst;
                        f4_add(acc[i], old);
                        *dst = acc[i];
                    } else {
                        __stcs(dst, acc[i]);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// variant 2: TMA-style staging.  Each warp stages the X rows its rows reference into shared memory
// with one cp.async.bulk (UBLKCP) per non-zero, completion tracked by a per-warp mbarrier, two stages
// deep, and accumulates out of shared memory.  No registers are spent on in-flight gathers.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- L2 eviction policies (createpolicy + .L2::cache_hint) ---------------------------------------------
// The X rows are the only data with reuse (each row of a block's panel is hit ~nnz/row times from L2);
// CSR streams and the C tile are touched once.  Marking the gathers evict_last and everything else
// evict_first keeps the streams from pushing the panels out of L2 (fused level > 0: DRAM traffic was
// 13.9 GB vs 8.1 GB algorithmic before the hints).
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p;
    asm("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ float4 ldg_f4_hint(const float4 *ptr, uint64_t pol) {
    float4 r;
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
        : "l"(ptr), "l"(pol));
    return r;
}
__device__ __forceinline__ float4 ld_f4_hint(const float4 *ptr, uint64_t pol) {      // coherent load (C tile RMW)
    float4 r;
    asm("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
        : "l"(ptr), "l"(pol));
    return r;
}
__device__ __forceinline__ void st_f4_hint(float4 *ptr, const float4 &v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1,%2,%3,%4}, %5;" ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar,
                                              uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
        : "memory");
}

constexpr int TMA_WARPS = 8;      // warps per CTA
constexpr int TMA_SLOTS = 16;     // X rows staged per stage per warp
constexpr int TMA_STAGES = 2;

// One warp per row (VPL float4 per lane).  The warp walks a stream of work items -- (row, chunk of up
// to TMA_SLOTS non-zeros) -- and keeps the NEXT item's X rows in flight while it accumulates the
// current one out of shared memory, so the pipeline spans row boundaries.
struct TmaItem {
    long long row;     // -1: end of stream
    long long orow;
    long long p0;      // first nnz of this chunk
    int cnt;           // nnz in this chunk
    int last;          // chunk closes its row
    int myc;           // this lane's column (lane < cnt), -1 otherwise
    float myv;
};

template <int VPL, bool ROWMAP, bool ACC>
__global__ void __launch_bounds__(TMA_WARPS * 32) k_spmm_tma(SpmmArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int k4 = a.k4;
    const uint32_t row_bytes = (uint32_t)a.k * 4u;
    float *wbase = reinterpret_cast<float *>(smem_raw) + (size_t)warp * TMA_STAGES * TMA_SLOTS * a.k;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)TMA_WARPS * TMA_STAGES * TMA_SLOTS * row_bytes) +
                     warp * TMA_STAGES;
    if (lane == 0) {
        for (int st = 0; st < TMA_STAGES; ++st) mbar_init(&bars[st], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    uint32_t parity0 = 0u, parity1 = 0u;

    const long long warps_total = (long long)gridDim.x * TMA_WARPS;
    const long long warp_id = (long long)blockIdx.x * TMA_WARPS + warp;
    float4 *__restrict__ C4 = reinterpret_cast<float4 *>(a.C);

    // work-item iterator (all lanes hold identical copies)
    long long it_row = warp_id - warps_total;
    long long it_p = 0, it_e = 0;
    long long it_orow = -1;
    auto next_item = [&](TmaItem &t) {
        while (it_p >= it_e) {                       // advance to the next non-empty, non-long, routed row
            it_row += warps_total;
            if (it_row >= a.n_rows) { t.row = -1; t.cnt = 0; t.myc = -1; t.myv = 0.f; t.last = 0; return; }
            long long len;
            const long long s = row_begin(a, it_row, len);
            long long orow = it_row;
            if (ROWMAP) orow = __ldg(a.rowmap + it_row);
            if (orow < 0 || len > a.long_threshold) continue;
            it_orow = orow;
            it_p = s;
            it_e = s + len;
            if (len == 0) {                          // empty row still has to store zeros / keep C
                t.row = it_row; t.orow = orow; t.p0 = s; t.cnt = 0; t.last = 1; t.myc = -1; t.myv = 0.f;
                return;
            }
        }
        t.row = it_row;
        t.orow = it_orow;
        t.p0 = it_p;
        t.cnt = (int)min((long long)TMA_SLOTS, it_e - it_p);
        it_p += t.cnt;
        t.last = (it_p >= it_e);
        t.myc = -1;
        t.myv = 0.f;
        if (lane < t.cnt) {
            t.myc = __ldcs(a.indices + t.p0 + lane);
            t.myv = __ldcs(a.vals + t.p0 + lane);
        }
    };
    auto issue = [&](const TmaItem &t, int st) {
        const unsigned valid = __ballot_sync(0xffffffffu, t.myc >= 0);
        if (lane == 0) mbar_expect_tx(&bars[st], (uint32_t)__popc(valid) * row_bytes);
        __syncwarp();
        if (t.myc >= 0)
            bulk_g2s(wbase + ((size_t)st * TMA_SLOTS + lane) * a.k, a.X + (long long)t.myc * a.k, row_bytes, &bars[st]);
    };

    float4 acc[VPL];
#pragma unroll
    for (int i = 0; i < VPL; ++i) acc[i] = f4_zero();

    TmaItem cur, nxt;
    int stage = 0;
    next_item(cur);
    if (cur.row >= 0) issue(cur, stage);
    while (cur.row >= 0) {
        next_item(nxt);
        if (nxt.row >= 0) issue(nxt, stage ^ 1);
        if (stage == 0) { mbar_wait(&bars[0], parity0); parity0 ^= 1u; }
        else            { mbar_wait(&bars[1], parity1); parity1 ^= 1u; }
        const float4 *sm4 = reinterpret_cast<const float4 *>(wbase + (size_t)stage * TMA_SLOTS * a.k);
        for (int u = 0; u < cur.cnt; ++u) {
            const int c = __shfl_sync(0xffffffffu, cur.myc, u);
            const float v = __shfl_sync(0xffffffffu, cur.myv, u);
            if (c >= 0) {
#pragma unroll
                for (int i = 0; i < VPL; ++i) {
                    const int vec = lane + i * 32;
                    if (vec < k4) f4_fma(acc[i], v, sm4[(size_t)u * k4 + vec]);
                }
            }
        }
        if (cur.last) {
#pragma unroll
            for (int i = 0; i < VPL; ++i) {
                const int vec = lane + i * 32;
                if (vec < k4) {
                    float4 *dst = C4 + cur.orow * k4 + vec;
                    if (ACC) {
                        float4 old = *dst;
                        f4_add(acc[i], old);
                        *dst = acc[i];
                    } else {
                        __stcs(dst, acc[i]);
                    }
                }
                acc[i] = f4_zero();
            }
        }
        __syncwarp();           // every lane is done with this stage before it is refilled
        cur = nxt;
        stage ^= 1;
    }
}

// ------------------------------------------------------------------------------------------------
// variant 3 (default): CSR streamed by TMA.  A persistent CTA walks row tiles (<= TILE_ROWS rows,
// <= TILE_NNZ non-zeros, built at upload).  One elected thread brings the tile's slice of indptr /
// indices / values into shared memory with three cp.async.bulk copies (UBLKCP) that complete on an
// mbarrier, one tile ahead of the math (two stages).  Warps then only issue the X gathers: a group of
// G lanes owns a row, reads (col, val) from shared memory (broadcast) and VPL float4 of the X row.
// ------------------------------------------------------------------------------------------------
constexpr int TILE_ROWS = 64;       // small tiles keep the rows in flight (grid x TILE_ROWS) inside ~4 blocks => L2 hits
constexpr int TILE_NNZ = 1024;
constexpr int TILE_ROWS_BIG = 128;  // k <= 32: the panels are small, bigger tiles amortise the per-tile fixed cost
constexpr int TILE_NNZ_BIG = 2048;
constexpr int TILE_THREADS = 256;
constexpr int TILE_STAGES = 2;      // CSR slices in shared memory: tile t (math), t+1 (in flight).  A third stage (tried in round 2 for a
                                    // look-ahead prefetch) cost more L1 than it bought: the L1 data array is the landing buffer of the gathers in flight
template <int TR, int TN>
struct TileCfg {
    static constexpr int PTR_WORDS = TR + 8;           // row pointer slice (+ alignment slack)
    static constexpr int NNZ_WORDS = TN + 8;
    static constexpr int STAGE_WORDS = PTR_WORDS + 2 * NNZ_WORDS;
    static constexpr size_t SMEM_BYTES = (size_t)TILE_STAGES * STAGE_WORDS * 4 + 64;
};

// where a result row goes
constexpr int OUT_IDENTITY = 0;     // C[r]
constexpr int OUT_ROWMAP = 1;       // C[rowmap[r]]           (rows with rowmap[r] < 0 are dropped)
constexpr int OUT_ROWPTR = 2;       // *(out_ptr[r])          (device pointer per row: a local tile or a peer GPU's staging slot)

struct TileArgs {
    SpmmArgs a;
    const int4 *__restrict__ tiles;
    const long long *__restrict__ tile_base;   // 64-bit nnz_begin of each tile: the source of its bulk copies
    int n_tiles;
    int skip;            // indices may hold -1
    int *ticket;         // dynamic tile scheduler: [0] next tile, [1] CTAs that finished (the last one re-arms both)
    int l2_hints;        // bit 0: X gathers evict_last, bit 1: CSR / C streams evict_first
    int prefetch;        // 1: bulk L2 prefetch of the tile's X rows before the math (A/B switch, off by default)
};

__device__ __forceinline__ void bulk_prefetch_l2(const void *gptr, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
// ------------------------------------------------------------------------------------------------
// The round-1 tile kernel, verbatim (one row per lane group, identity / row-map output, no dual operand): kept as the
// production path of those launches.  The generalised kernel below produces the same numbers but its fused level-1
// launch (scattered first-touch gathers, latency bound) measured 2.2-2.6 ms against 1.8 ms for this code on the same GPU
// (profiles/r02_kernel_sweep.md, section 5); ARROW_OPT_TILE_KERNEL switches between the two.
// ------------------------------------------------------------------------------------------------
template <typename T, int G, int VPL, bool ROWMAP, bool ACC, int TR, int TN>
__global__ void __launch_bounds__(TILE_THREADS, 4) k_spmm_tiles_v1(TileArgs t) {
    using E = Elt<T>;
    constexpr int TILE_PTR_WORDS = TileCfg<TR, TN>::PTR_WORDS;
    constexpr int TILE_NNZ_WORDS = TileCfg<TR, TN>::NNZ_WORDS;
    constexpr int TILE_STAGE_WORDS = TileCfg<TR, TN>::STAGE_WORDS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    int *stage_base = reinterpret_cast<int *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)2 * TILE_STAGE_WORDS * 4);
    const SpmmArgs &a = t.a;
    constexpr int RPW = 32 / G;
    constexpr int UNROLL = (VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8);
    constexpr int TAIL = (UNROLL >= 4) ? UNROLL / 2 : UNROLL;     // predicated tail batches
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const bool EXACT = (t.a.k4 == G * VPL);                       // every lane owns valid columns
    const int gl = lane % G;
    const int gi = lane / G;
    const int k4 = a.k4;
    const float4 *__restrict__ Xl = reinterpret_cast<const float4 *>(a.X) + gl;
    float4 *__restrict__ Cl = reinterpret_cast<float4 *>(a.C) + gl;
    const uint64_t pol_keep = (t.l2_hints & 1) ? l2_policy_evict_last() : l2_policy_evict_normal();
    const uint64_t pol_stream = (t.l2_hints & 2) ? l2_policy_evict_first() : l2_policy_evict_normal();

    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto prefetch = [&](int tile, int st) {
        const int4 d = __ldg(t.tiles + tile);
        const int rb4 = d.x & ~3;
        const long long a0 = __ldg(t.tile_base + tile) & ~3LL;
        const uint32_t ptr_bytes = (uint32_t)(((d.y - rb4 + 1) + 3) & ~3) * 4u;
        const uint32_t nnz_bytes = (uint32_t)((wdiff(d.w, d.z & ~3) + 3) & ~3) * 4u;
        int *sp = stage_base + (size_t)st * TILE_STAGE_WORDS;
        mbar_expect_tx(&bars[st], ptr_bytes + 2u * nnz_bytes);
        bulk_g2s_hint(sp, a.indptr + rb4, ptr_bytes, &bars[st], pol_stream);
        if (nnz_bytes) {
            bulk_g2s_hint(sp + TILE_PTR_WORDS, a.indices + a0, nnz_bytes, &bars[st], pol_stream);
            bulk_g2s_hint(sp + TILE_PTR_WORDS + TILE_NNZ_WORDS, a.vals + a0, nnz_bytes, &bars[st], pol_stream);
        }
    };

    // Dynamic scheduling: the first tile is blockIdx.x, every further tile comes from an atomic ticket.  All CTAs
    // therefore work on one compact, moving window of ~gridDim.x consecutive tiles; a static round-robin lets
    // CTAs drift apart over the ~260 tiles each one processes at 10M rows and the live X panels fall out of L2
    // (measured: 62 % L2 hit rate, DRAM traffic 1.30x algorithmic before this change).
    __shared__ int s_next[2];
    uint32_t parity0 = 0u, parity1 = 0u;
    int tile = blockIdx.x;
    int st = 0;
    if (tile < t.n_tiles && threadIdx.x == 0) prefetch(tile, 0);
    for (; tile < t.n_tiles; st ^= 1) {
        if (threadIdx.x == 0) {
            const int next = atomicAdd(t.ticket, 1) + (int)gridDim.x;
            s_next[st] = next;
            if (next < t.n_tiles) prefetch(next, st ^ 1);
        }
        const int4 d = __ldg(t.tiles + tile);
        if (st == 0) { mbar_wait(&bars[0], parity0); parity0 ^= 1u; }
        else         { mbar_wait(&bars[1], parity1); parity1 ^= 1u; }
        const int *sp = stage_base + (size_t)st * TILE_STAGE_WORDS;
        const int *s_ptr = sp + (d.x - (d.x & ~3));
        const int a0 = d.z & ~3;                                        // low word of the slice's first entry
        const int *s_idx = sp + TILE_PTR_WORDS;                         // index with tile-local offsets
        const float *s_val = reinterpret_cast<const float *>(sp + TILE_PTR_WORDS + TILE_NNZ_WORDS);
        const int n_rows_tile = d.y - d.x;

        for (int lr = warp * RPW + gi; lr < n_rows_tile; lr += (TILE_THREADS / 32) * RPW) {
            const int s = wdiff(s_ptr[lr], a0);
            const int e = wdiff(s_ptr[lr + 1], a0);
            if (e - s > a.long_threshold) continue;
            const long long row = (long long)d.x + lr;
            long long orow = row;
            if (ROWMAP) {
                orow = __ldg(a.rowmap + row);
                if (orow < 0) continue;
            }
            if (false && t.prefetch) {
                // software prefetch into L2: the X rows the group's NEXT row of this tile will gather (their column
                // indices are already in shared memory); hides DRAM latency of first-touch / scattered rows
                const int nlr = lr + (TILE_THREADS / 32) * RPW;
                if (nlr < n_rows_tile) {
                    const int ns = wdiff(s_ptr[nlr], a0), ne = wdiff(s_ptr[nlr + 1], a0);
                    if (ne - ns <= a.long_threshold) {
                        const int lines = (a.k * 4 + 127) >> 7;
                        for (int q = ns + gl; q < ne; q += G) {
                            const int cq = s_idx[q];
                            if (cq >= 0) {
                                const char *xr = reinterpret_cast<const char *>(a.X) + (long long)cq * a.k * 4;
                                for (int l = 0; l < lines; ++l)
                                    asm volatile("prefetch.global.L2 [%0];" ::"l"(xr + l * 128));
                            }
                        }
                    }
                }
            }
            // accumulate mode: the old C row is read FIRST so that its latency hides behind the gathers (only this
            // group ever touches the row: the row maps are injective)
            typename E::Acc acc[VPL];
            float4 *cr = Cl + orow * k4;
#pragma unroll
            for (int i = 0; i < VPL; ++i)
                acc[i] = (ACC && gl + i * G < k4) ? E::widen(ld_f4_hint(cr + i * G, pol_stream)) : E::zero();
            if (a.add_map != nullptr) {
                // epilogue gather-add, issued first so its latency hides behind the gathers: the backward exchange
                // C_{j-1}[to_prev[r]] += C_j[r] (arrow_dec_mpi.py:437) seen from the receiving row
                const int am = __ldg(a.add_map + row);
                if (am >= 0) {
                    const float4 *ar = reinterpret_cast<const float4 *>(a.add_src) + (long long)am * k4 + gl;
#pragma unroll
                    for (int i = 0; i < VPL; ++i)
                        if (gl + i * G < k4) E::add(acc[i], ld_f4_hint(ar + i * G, pol_stream));
                }
            }
            int p = s;
            if (EXACT && !t.skip) {
                // unpredicated batches: full UNROLL batches, then the remainder as 4 / 2 / 1 (binary decomposition) --
                // a predicated tail batch costs as many instructions as a full one
                auto batch = [&](auto n_tag) {
                    constexpr int N = decltype(n_tag)::value;
                    int c[N];
                    float v[N];
#pragma unroll
                    for (int u = 0; u < N; ++u) {
                        c[u] = s_idx[p + u];
                        v[u] = s_val[p + u];
                    }
                    float4 x[N][VPL];
#pragma unroll
                    for (int u = 0; u < N; ++u) {
                        const float4 *xr = Xl + (long long)c[u] * k4;
#pragma unroll
                        for (int i = 0; i < VPL; ++i) x[u][i] = ldg_f4_hint(xr + i * G, pol_keep);
                    }
#pragma unroll
                    for (int u = 0; u < N; ++u)
#pragma unroll
                        for (int i = 0; i < VPL; ++i) E::fma(acc[i], v[u], x[u][i]);
                    p += N;
                };
                while (p + UNROLL <= e) batch(std::integral_constant<int, UNROLL>{});
                if constexpr (UNROLL >= 8) { if (e - p >= 4) batch(std::integral_constant<int, 4>{}); }
                if constexpr (UNROLL >= 4) { if (e - p >= 2) batch(std::integral_constant<int, 2>{}); }
                if (e - p >= 1) batch(std::integral_constant<int, 1>{});
            }
            // tail (and the general case): predicated batches of TAIL
            for (; p < e; p += TAIL) {
                int c[TAIL];
                float v[TAIL];
#pragma unroll
                for (int u = 0; u < TAIL; ++u) {
                    const bool ok = p + u < e;
                    c[u] = ok ? s_idx[p + u] : -1;
                    v[u] = ok ? s_val[p + u] : 0.f;
                }
                float4 x[TAIL][VPL];
#pragma unroll
                for (int u = 0; u < TAIL; ++u) {
                    const float4 *xr = Xl + (long long)c[u] * k4;
#pragma unroll
                    for (int i = 0; i < VPL; ++i)
                        x[u][i] = (c[u] >= 0 && gl + i * G < k4) ? ldg_f4_hint(xr + i * G, pol_keep) : f4_zero();
                }
#pragma unroll
                for (int u = 0; u < TAIL; ++u)
#pragma unroll
                    for (int i = 0; i < VPL; ++i) E::fma(acc[i], v[u], x[u][i]);
            }
#pragma unroll
            for (int i = 0; i < VPL; ++i)
                if (gl + i * G < k4) st_f4_hint(cr + i * G, E::pack(acc[i]), pol_stream);
        }
        __syncthreads();            // stage `st` may be refilled by the next iteration's prefetch
        tile = s_next[st];
    }
}

// G lanes own a row (VPL float4 each).  RPG = 2: a group works on two rows at once (rows lr and lr + rows-per-pass) with
// half the batch size per row: the gathers of both rows are issued before either row's FMAs.  Same registers, but the
// short tail batch of one row (a 10-entry row is 8 + 2 gathers: the second round trip keeps 2 of 8 slots busy) overlaps
// the other row's -- narrow feature tiles (k <= 32) are bound by gathers in flight, not by bandwidth.
template <typename T, int G, int VPL, int OUT, bool ACC, int TR, int TN, int RPG, int MINB, bool DUALX>
__global__ void __launch_bounds__(TILE_THREADS, 4) k_spmm_tiles(TileArgs t) {
    using E = Elt<T>;
    constexpr int TILE_PTR_WORDS = TileCfg<TR, TN>::PTR_WORDS;
    constexpr int TILE_NNZ_WORDS = TileCfg<TR, TN>::NNZ_WORDS;
    constexpr int TILE_STAGE_WORDS = TileCfg<TR, TN>::STAGE_WORDS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    int *stage_base = reinterpret_cast<int *>(smem_raw);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + (size_t)TILE_STAGES * TILE_STAGE_WORDS * 4);
    const SpmmArgs &a = t.a;
    constexpr int RPW = 32 / G;
    constexpr int ROWS_PER_PASS = (TILE_THREADS / 32) * RPW;
    // gathers a group keeps in flight: UNROLL per row x RPG rows = the same 32 registers of X data per lane in every shape
    constexpr int UNROLL = ((VPL >= 4) ? 2 : (VPL == 2 ? 4 : 8)) / RPG;
    constexpr int TAIL = (UNROLL >= 4) ? UNROLL / 2 : UNROLL;     // predicated tail batches
    static_assert(MINB == 4 && UNROLL >= 1, "tile kernel shape");
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const bool EXACT = (t.a.k4 == G * VPL);                       // every lane owns valid columns
    const int gl = lane % G;
    const int gi = lane / G;
    const int k4 = a.k4;
    const float4 *__restrict__ Xl = reinterpret_cast<const float4 *>(a.X) + gl;
    const float4 *__restrict__ X2l = reinterpret_cast<const float4 *>(a.X2) + gl;
    float4 *__restrict__ Cl = reinterpret_cast<float4 *>(a.C) + gl;
    const uint64_t pol_keep = (t.l2_hints & 1) ? l2_policy_evict_last() : l2_policy_evict_normal();
    const uint64_t pol_stream = (t.l2_hints & 2) ? l2_policy_evict_first() : l2_policy_evict_normal();

    auto xrow = [&](int c) -> const float4 * {
        if constexpr (DUALX) {
            return (c < a.x_split) ? Xl + (long long)c * k4 : X2l + (long long)(c - a.x_split) * k4;
        } else {
            return Xl + (long long)c * k4;
        }
    };

    __shared__ int s_tile[TILE_STAGES];
    auto issue_csr = [&](int tile, int st) {
        const int4 d = __ldg(t.tiles + tile);
        const int rb4 = d.x & ~3;
        const long long a0 = __ldg(t.tile_base + tile) & ~3LL;
        const uint32_t ptr_bytes = (uint32_t)(((d.y - rb4 + 1) + 3) & ~3) * 4u;
        const uint32_t nnz_bytes = (uint32_t)((wdiff(d.w, d.z & ~3) + 3) & ~3) * 4u;
        int *sp = stage_base + (size_t)st * TILE_STAGE_WORDS;
        mbar_expect_tx(&bars[st], ptr_bytes + 2u * nnz_bytes);
        bulk_g2s_hint(sp, a.indptr + rb4, ptr_bytes, &bars[st], pol_stream);
        if (nnz_bytes) {
            bulk_g2s_hint(sp + TILE_PTR_WORDS, a.indices + a0, nnz_bytes, &bars[st], pol_stream);
            bulk_g2s_hint(sp + TILE_PTR_WORDS + TILE_NNZ_WORDS, a.vals + a0, nnz_bytes, &bars[st], pol_stream);
        }
    };

    // Dynamic scheduling: the first tile is blockIdx.x, every further tile comes from an atomic ticket.  All CTAs
    // therefore work on one compact, moving window of ~gridDim.x consecutive tiles; a static round-robin lets
    // CTAs drift apart over the ~260 tiles each one processes at 10M rows and the live X panels fall out of L2
    // (measured: 62 % L2 hit rate, DRAM traffic 1.30x algorithmic before this change).
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < TILE_STAGES; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if ((int)blockIdx.x < t.n_tiles) issue_csr(blockIdx.x, 0);
    }
    __syncthreads();

    uint32_t phase = 0u;                  // bit s = parity the next wait on stage s expects
    int tile = blockIdx.x;
    for (int st = 0; tile < t.n_tiles; st ^= 1) {
        if (threadIdx.x == 0) {
            const int nn = atomicAdd(t.ticket, 1) + (int)gridDim.x;
            s_tile[st] = nn;
            if (nn < t.n_tiles) issue_csr(nn, st ^ 1);
        }
        const int4 d = __ldg(t.tiles + tile);
        mbar_wait(&bars[st], (phase >> st) & 1u);
        phase ^= (1u << st);
        const int *sp = stage_base + (size_t)st * TILE_STAGE_WORDS;
        const int *s_ptr = sp + (d.x - (d.x & ~3));
        const int a0 = d.z & ~3;                                        // low word of the slice's first entry
        const int *s_idx = sp + TILE_PTR_WORDS;                         // index with tile-local offsets
        const float *s_val = reinterpret_cast<const float *>(sp + TILE_PTR_WORDS + TILE_NNZ_WORDS);
        const int n_rows_tile = d.y - d.x;

        if (t.prefetch) {
            // Bulk L2 prefetch of this tile's X rows (one cp.async.bulk.prefetch.L2 per row, issued by the TMA unit: no
            // registers, no LSU wavefronts).  Measured in round 2 (profiles/r02_kernel_sweep.md): a LOSS at every k -- the
            // request rate of the unit, not DRAM latency, becomes the bound.  Off by default; kept as the A/B switch.
            const uint32_t row_bytes = (uint32_t)a.k * (uint32_t)sizeof(T);
            for (int q = wdiff(d.z, a0) + (int)threadIdx.x; q < wdiff(d.w, a0); q += TILE_THREADS) {
                const int cq = s_idx[q];
                if (cq >= 0) bulk_prefetch_l2(xrow(cq) - gl, row_bytes);
            }
        }

        // one or RPG rows of this lane group: setup, joint batches, store
        auto do_rows = [&](auto nr_tag, int lr0) {
            constexpr int NR = decltype(nr_tag)::value;
            int p[NR], e[NR];
            bool live[NR];
            float4 *cr[NR];
            typename E::Acc acc[NR][VPL];
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int lr = lr0 + r * ROWS_PER_PASS;
                live[r] = lr < n_rows_tile;
                p[r] = e[r] = 0;
                cr[r] = nullptr;
                if (live[r]) {
                    p[r] = wdiff(s_ptr[lr], a0);
                    e[r] = wdiff(s_ptr[lr + 1], a0);
                    if (e[r] - p[r] > a.long_threshold) { live[r] = false; e[r] = p[r]; }
                }
                const long long row = (long long)d.x + lr;
                if (live[r]) {
                    if constexpr (OUT == OUT_ROWMAP) {
                        const long long orow = __ldg(a.rowmap + row);
                        if (orow < 0) { live[r] = false; e[r] = p[r]; } else cr[r] = Cl + orow * k4;
                    } else if constexpr (OUT == OUT_ROWPTR) {
                        float *dst = reinterpret_cast<float *>(__ldg(reinterpret_cast<const unsigned long long *>(a.out_ptr) + row));
                        if (dst == nullptr) { live[r] = false; e[r] = p[r]; } else cr[r] = reinterpret_cast<float4 *>(dst) + gl;
                    } else {
                        cr[r] = Cl + row * k4;
                    }
                }
                if constexpr (NR == 1) {
                    if (!live[0]) return;               // one row per group: nothing to keep predicated past this point
                    live[0] = true;
                }
                // accumulate mode: the old C row is read FIRST so that its latency hides behind the gathers (only this
                // group ever touches the row: the row maps are injective)
#pragma unroll
                for (int i = 0; i < VPL; ++i)
                    acc[r][i] = (ACC && live[r] && gl + i * G < k4) ? E::widen(ld_f4_hint(cr[r] + i * G, pol_stream)) : E::zero();
                if (a.add_map != nullptr && live[r]) {
                    // epilogue gather-add, issued first so its latency hides behind the gathers: the backward exchange
                    // C_{j-1}[to_prev[r]] += C_j[r] (arrow_dec_mpi.py:437) seen from the receiving row
                    const int am = __ldg(a.add_map + row);
                    if (am >= 0) {
                        const float4 *ar = reinterpret_cast<const float4 *>(a.add_src) + (long long)am * k4 + gl;
#pragma unroll
                        for (int i = 0; i < VPL; ++i)
                            if (gl + i * G < k4) E::add(acc[r][i], ld_f4_hint(ar + i * G, pol_stream));
                    }
                }
            }
            if (EXACT && !t.skip) {
                if constexpr (NR == 1) {
                    // unpredicated batches: full UNROLL batches, then the remainder as 4 / 2 / 1 (binary decomposition) --
                    // a predicated tail batch costs as many instructions as a full one
                    auto batch = [&](auto n_tag) {
                        constexpr int N = decltype(n_tag)::value;
                        float v[N];
                        float4 x[N][VPL];
#pragma unroll
                        for (int u = 0; u < N; ++u) {
                            const int c = s_idx[p[0] + u];
                            v[u] = s_val[p[0] + u];
                            const float4 *xr = xrow(c);
#pragma unroll
                            for (int i = 0; i < VPL; ++i) x[u][i] = ldg_f4_hint(xr + i * G, pol_keep);
                        }
#pragma unroll
                        for (int u = 0; u < N; ++u)
#pragma unroll
                            for (int i = 0; i < VPL; ++i) E::fma(acc[0][i], v[u], x[u][i]);
                        p[0] += N;
                    };
                    while (p[0] + UNROLL <= e[0]) batch(std::integral_constant<int, UNROLL>{});
                    if constexpr (UNROLL >= 8) { if (e[0] - p[0] >= 4) batch(std::integral_constant<int, 4>{}); }
                    if constexpr (UNROLL >= 4) { if (e[0] - p[0] >= 2) batch(std::integral_constant<int, 2>{}); }
                    if (e[0] - p[0] >= 1) batch(std::integral_constant<int, 1>{});
                } else {
                    // paired rows: while both have a full batch left, 2 x UNROLL unpredicated gathers go out back to back;
                    // the values are read from shared memory when the gathers are back (registers)
                    while (e[0] - p[0] >= UNROLL && e[1] - p[1] >= UNROLL) {
                        float4 x[NR][UNROLL][VPL];
#pragma unroll
                        for (int r = 0; r < NR; ++r)
#pragma unroll
                            for (int u = 0; u < UNROLL; ++u) {
                                const float4 *xr = xrow(s_idx[p[r] + u]);
#pragma unroll
                                for (int i = 0; i < VPL; ++i) x[r][u][i] = __ldg(xr + i * G);
                            }
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
#pragma unroll
                            for (int u = 0; u < UNROLL; ++u) {
                                const float v = s_val[p[r] + u];
#pragma unroll
                                for (int i = 0; i < VPL; ++i) E::fma(acc[r][i], v, x[r][u][i]);
                            }
                            p[r] += UNROLL;
                        }
                    }
                    // remainders of both rows share predicated batches (one round trip for two short tails)
                    while (p[0] < e[0] || p[1] < e[1]) {
                        float4 x[NR][UNROLL][VPL];
#pragma unroll
                        for (int r = 0; r < NR; ++r)
#pragma unroll
                            for (int u = 0; u < UNROLL; ++u) {
                                const bool ok = p[r] + u < e[r];
                                const float4 *xr = xrow(ok ? s_idx[p[r] + u] : 0);
#pragma unroll
                                for (int i = 0; i < VPL; ++i) x[r][u][i] = ok ? __ldg(xr + i * G) : f4_zero();
                            }
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
#pragma unroll
                            for (int u = 0; u < UNROLL; ++u) {
                                const float v = (p[r] + u < e[r]) ? s_val[p[r] + u] : 0.f;
#pragma unroll
                                for (int i = 0; i < VPL; ++i) E::fma(acc[r][i], v, x[r][u][i]);
                            }
                            p[r] = min(p[r] + UNROLL, e[r]);
                        }
                    }
                }
            }
            // tail (and the general case): predicated batches of TAIL, one row at a time
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                for (; p[r] < e[r]; p[r] += TAIL) {
                    int c[TAIL];
                    float v[TAIL];
#pragma unroll
                    for (int u = 0; u < TAIL; ++u) {
                        const bool ok = p[r] + u < e[r];
                        c[u] = ok ? s_idx[p[r] + u] : -1;
                        v[u] = ok ? s_val[p[r] + u] : 0.f;
                    }
                    float4 x[TAIL][VPL];
#pragma unroll
                    for (int u = 0; u < TAIL; ++u) {
                        const float4 *xr = xrow(c[u]);                    // c = -1: address arithmetic only, never dereferenced
#pragma unroll
                        for (int i = 0; i < VPL; ++i)
                            x[u][i] = (c[u] >= 0 && gl + i * G < k4) ? ldg_f4_hint(xr + i * G, pol_keep) : f4_zero();
                    }
#pragma unroll
                    for (int u = 0; u < TAIL; ++u)
#pragma unroll
                        for (int i = 0; i < VPL; ++i) E::fma(acc[r][i], v[u], x[u][i]);
                }
                if (live[r]) {
#pragma unroll
                    for (int i = 0; i < VPL; ++i) {
                        if (gl + i * G < k4) {
                            if constexpr (OUT == OUT_ROWPTR) {
                                *(cr[r] + i * G) = E::pack(acc[r][i]);       // may be a peer GPU's memory (NVLink store): no L2 policy
                            } else {
                                st_f4_hint(cr[r] + i * G, E::pack(acc[r][i]), pol_stream);
                            }
                        }
                    }
                }
            }
        };

        if constexpr (RPG == 2) {
            for (int lr = warp * RPW + gi; lr < n_rows_tile; lr += 2 * ROWS_PER_PASS) do_rows(std::integral_constant<int, 2>{}, lr);
        } else {
            for (int lr = warp * RPW + gi; lr < n_rows_tile; lr += ROWS_PER_PASS) do_rows(std::integral_constant<int, 1>{}, lr);
        }
        __syncthreads();            // stage `st` may be refilled by the next iteration's CSR copy
        tile = s_tile[st];
    }
    // the last CTA to leave re-arms the scheduler for the next launch on this lane (no memset between launches)
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(t.ticket + 1, 1) == (int)gridDim.x - 1) {
            t.ticket[0] = 0;
            t.ticket[1] = 0;
            __threadfence();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// generic k (not a multiple of one 16-byte vector: 4 fp32 / 8 bf16): warp per row, lanes over columns, scalar accesses.
// ------------------------------------------------------------------------------------------------
template <typename T, bool ROWMAP, bool ACC>
__global__ void __launch_bounds__(256) k_spmm_generic(SpmmArgs a) {
    using E = Elt<T>;
    const T *__restrict__ X = reinterpret_cast<const T *>(a.X);
    const T *__restrict__ X2 = reinterpret_cast<const T *>(a.X2);
    const T *__restrict__ add_src = reinterpret_cast<const T *>(a.add_src);
    const int lane = threadIdx.x & 31;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (long long row = warp_id; row < a.n_rows; row += warps_total) {
        long long len;
        const long long s = row_begin(a, row, len);
        if (len > a.long_threshold) continue;
        const long long e = s + len;
        long long orow = row;
        if (ROWMAP) {
            orow = __ldg(a.rowmap + row);
            if (orow < 0) continue;
        }
        T *crow = reinterpret_cast<T *>(a.C) + orow * a.k;
        if (a.out_ptr != nullptr) {
            crow = reinterpret_cast<T *>(a.out_ptr[row]);
            if (crow == nullptr) continue;
        }
        for (int c0 = 0; c0 < a.k; c0 += 128) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            for (long long p = s; p < e; ++p) {
                const int c = __ldg(a.indices + p);
                const float v = __ldg(a.vals + p);
                if (c < 0) continue;
                const T *xr = (X2 != nullptr && c >= a.x_split) ? X2 + (long long)(c - a.x_split) * a.k : X + (long long)c * a.k;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int col = c0 + lane + 32 * i;
                    if (col < a.k) acc[i] = fmaf(v, E::to_f(__ldg(xr + col)), acc[i]);
                }
            }
            const int am = (a.add_map != nullptr) ? __ldg(a.add_map + row) : -1;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int col = c0 + lane + 32 * i;
                if (col < a.k) {
                    T *dst = crow + col;
                    float r = ACC ? (E::to_f(*dst) + acc[i]) : acc[i];
                    if (am >= 0) r += E::to_f(add_src[(long long)am * a.k + col]);
                    *dst = E::from_f(r);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// long rows (hubs of the arrow head): one CTA per segment of `segment` non-zeros, partial sums to
// scratch, then an in-order reduction per row -- deterministic, no atomics.
// ------------------------------------------------------------------------------------------------
struct LongArgs {
    const LongTask *__restrict__ tasks;
    const int *__restrict__ indices;
    const float *__restrict__ vals;
    const float *__restrict__ X;      // element type T of k_spmm_long_partial<T>
    float *__restrict__ scratch;      // [slot][k], fp32 whatever T
    int k;
    const float *__restrict__ X2;     // second X base (see SpmmArgs)
    int x_split;
};

template <typename T>
__global__ void __launch_bounds__(256) k_spmm_long_partial(LongArgs a) {
    const T *__restrict__ X = reinterpret_cast<const T *>(a.X);
    const T *__restrict__ X2 = reinterpret_cast<const T *>(a.X2);
    extern __shared__ float red[];    // [warps][k]
    const LongTask t = a.tasks[blockIdx.x];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int c0 = 0; c0 < a.k; c0 += 128) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (long long p = t.begin + warp; p < t.end; p += nwarps) {
            const int c = __ldg(a.indices + p);
            const float v = __ldg(a.vals + p);
            if (c < 0) continue;
            const T *xr = (X2 != nullptr && c >= a.x_split) ? X2 + (long long)(c - a.x_split) * a.k : X + (long long)c * a.k;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int col = c0 + lane + 32 * i;
                if (col < a.k) acc[i] = fmaf(v, Elt<T>::to_f(__ldg(xr + col)), acc[i]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int col = c0 + lane + 32 * i;
            if (col < a.k) red[warp * a.k + col] = acc[i];
        }
    }
    __syncthreads();
    for (int col = threadIdx.x; col < a.k; col += blockDim.x) {
        float sum = 0.f;
        for (int w = 0; w < nwarps; ++w) sum += red[w * a.k + col];
        a.scratch[(long long)t.slot * a.k + col] = sum;
    }
}

template <typename T, bool ROWMAP, bool ACC>
__global__ void __launch_bounds__(128) k_spmm_long_reduce(const int *__restrict__ long_rows,
                                                          const int *__restrict__ long_first,
                                                          const float *__restrict__ scratch,
                                                          T *__restrict__ C, const int *__restrict__ rowmap, int k,
                                                          const T *__restrict__ add_src, const int *__restrict__ add_map,
                                                          float *const *__restrict__ out_ptr) {
    using E = Elt<T>;
    const int r = long_rows[blockIdx.x];
    long long orow = r;
    if (ROWMAP) {
        orow = rowmap[r];
        if (orow < 0) return;
    }
    T *crow = C + orow * k;
    if (out_ptr != nullptr) {
        crow = reinterpret_cast<T *>(out_ptr[r]);
        if (crow == nullptr) return;
    }
    const int s0 = long_first[blockIdx.x], s1 = long_first[blockIdx.x + 1];
    for (int col = threadIdx.x; col < k; col += blockDim.x) {
        float sum = 0.f;
        for (int s = s0; s < s1; ++s) sum += scratch[(long long)s * k + col];
        if (add_map != nullptr) {
            const int am = add_map[r];
            if (am >= 0) sum += E::to_f(add_src[(long long)am * k + col]);
        }
        T *dst = crow + col;
        *dst = E::from_f(ACC ? (E::to_f(*dst) + sum) : sum);
    }
}

// ------------------------------------------------------------------------------------------------
// exchange kernels: dst[r] (+)= src[map[r]]
// ------------------------------------------------------------------------------------------------
constexpr int MAX_SRC = 16;
struct MultiSrc {
    const float *p[MAX_SRC];
    long long bound[MAX_SRC + 1];
    int n;
};

// A group of G lanes moves one row (VPR vectors of VT); rows are taken warp-strided so that a warp's
// destination rows are consecutive (coalesced stores) while the sources are wherever the map points --
// local HBM, or a peer GPU's memory over NVLink when MULTI.
// dst row (+)= src row for one vector (4 fp32 / 8 bf16 values in a float4) or one element: added in fp32, rounded once
template <typename T>
__device__ __forceinline__ void add_rows(float4 &v, const float4 &old) {
    typename Elt<T>::Acc acc = Elt<T>::widen(v);
    Elt<T>::add(acc, old);
    v = Elt<T>::pack(acc);
}
template <typename T>
__device__ __forceinline__ void add_rows(T &v, const T &old) {
    v = Elt<T>::from_f(Elt<T>::to_f(v) + Elt<T>::to_f(old));
}

// T: element type of the tiles; VT: what one lane moves at once (float4, or a single T when k is not a multiple of a vector)
template <typename T, typename VT, int G, bool ACC, bool MULTI>
__global__ void __launch_bounds__(256) k_gather_rows(VT *__restrict__ dst, const VT *__restrict__ src, MultiSrc ms,
                                                     const int *__restrict__ map, long long n_rows, int vec_per_row) {
    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31;
    const int gl = lane % G, gi = lane / G;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    for (long long r = warp_id * RPW + gi; r < n_rows; r += warps_total * RPW) {
        const int m = __ldg(map + r);
        if (m < 0) continue;
        const VT *sp;
        if (MULTI) {
            int s = 0;
#pragma unroll 1
            while (s + 1 < ms.n && (long long)m >= ms.bound[s + 1]) ++s;
            sp = reinterpret_cast<const VT *>(ms.p[s]) + ((long long)m - ms.bound[s]) * vec_per_row;
        } else {
            sp = src + (long long)m * vec_per_row;
        }
        VT *dp = dst + r * vec_per_row;
        for (int v0 = gl; v0 < vec_per_row; v0 += 4 * G) {
            VT val[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (v0 + j * G < vec_per_row) val[j] = sp[v0 + j * G];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (v0 + j * G < vec_per_row) {
                    if (ACC) add_rows<T>(val[j], dp[v0 + j * G]);
                    dp[v0 + j * G] = val[j];
                }
            }
        }
    }
}

// Push: dst_d[i - bound[d]] = src[map[i]] for item i in [bound[d], bound[d+1]) -- the forward exchange of the fused
// multi-GPU step.  The items are sorted by destination GPU and, inside one destination, by the slot of its receive
// region, so every destination sees ONE sequential stream of 512-byte rows arriving over NVLink (posted stores: the
// sender never waits for the link) while the reads are local HBM gathers.  Replaces pack kernel + all-to-all + unpack
// kernel (arrow_dec_mpi.py:526, 584-610, 544) by a single pass.
struct MultiDst {
    float *p[MAX_SRC];
    long long bound[MAX_SRC + 1];
    int n;
    long long max_len;        // longest block; > 0: the grid walks the blocks interleaved (item q -> block q % n, position q / n)
};

// `md.max_len > 0`: consecutive lane groups serve DIFFERENT destinations, so at every instant a GPU sends to all its peers
// at once and every receiver hears from all senders at once -- the uniform all-to-all an NVSwitch serves at full rate
// whatever the relative timing of the GPUs.  Block after block (max_len == 0) depends on the GPUs staying in lockstep:
// 4 B200 reached 508 GB/s per GPU that way against 700 GB/s for a single destination.
template <typename VT, int G>
__global__ void __launch_bounds__(256) k_push_rows(MultiDst md, const VT *__restrict__ src, const int *__restrict__ map,
                                                   long long n_items, int vec_per_row) {
    constexpr int RPW = 32 / G;
    const int lane = threadIdx.x & 31;
    const int gl = lane % G, gi = lane / G;
    const long long warps_total = (long long)gridDim.x * (blockDim.x >> 5);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long n_walk = md.max_len > 0 ? md.max_len * md.n : n_items;
    for (long long q = warp_id * RPW + gi; q < n_walk; q += warps_total * RPW) {
        long long i = q;
        int d = 0;
        if (md.max_len > 0) {
            d = (int)(q % md.n);
            const long long pos = q / md.n;
            if (pos >= md.bound[d + 1] - md.bound[d]) continue;
            i = md.bound[d] + pos;
        }
        const int m = __ldg(map + i);
        if (m < 0) continue;
        if (md.max_len == 0) {
#pragma unroll 1
            while (d + 1 < md.n && i >= md.bound[d + 1]) ++d;
        }
        const VT *sp = src + (long long)m * vec_per_row;
        VT *dp = reinterpret_cast<VT *>(md.p[d]) + (i - md.bound[d]) * vec_per_row;
        for (int v0 = gl; v0 < vec_per_row; v0 += 4 * G) {
            VT val[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (v0 + j * G < vec_per_row) val[j] = sp[v0 + j * G];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (v0 + j * G < vec_per_row) dp[v0 + j * G] = val[j];
        }
    }
}

// out(r) = sum_s src_s[r] in source order (deterministic): the reduction of the partial head tiles
// (C_0 = sum_i A_0i X_i, arrow_slim_mpi.py:116) in one launch; the sources are peer tiles read over NVLink.  With a
// pointer table the sum goes wherever the row is routed (a peer's staging slot: head rows of a level > 0 on their way
// to the level below), else into dst.
template <typename VT>
__global__ void __launch_bounds__(256) k_reduce_rows(VT *__restrict__ dst, float *const *__restrict__ out_ptr, MultiSrc ms,
                                                     long long n_rows, int vec_per_row) {
    const long long total = n_rows * vec_per_row;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long r = i / vec_per_row;
        const int v = (int)(i - r * vec_per_row);
        VT *o = dst ? dst + i : nullptr;
        if (out_ptr != nullptr) {
            float *q = out_ptr[r];
            if (q != nullptr) o = reinterpret_cast<VT *>(q) + v;
        }
        if (o == nullptr) continue;
        VT sum = reinterpret_cast<const VT *>(ms.p[0])[i];
        for (int s = 1; s < ms.n; ++s) {
            const VT x = reinterpret_cast<const VT *>(ms.p[s])[i];
            if constexpr (sizeof(VT) == 16) {
                f4_add(sum, x);
            } else {
                sum += x;
            }
        }
        *o = sum;
    }
}

__global__ void k_fill_ptr_table(float **table, const int *__restrict__ which, const long long *__restrict__ row,
                                 const unsigned long long *__restrict__ bases, long long n, int k) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int w = which[i];
        table[i] = (w < 0) ? nullptr : reinterpret_cast<float *>(bases[w]) + row[i] * k;
    }
}

// ------------------------------------------------------------------------------------------------
// small utility kernels
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_fill(T *p, T v, long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}

template <typename SrcT>
__global__ void k_to_i32(const SrcT *__restrict__ in, int *__restrict__ out, long long n, long long base, int *bad) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const long long v = (long long)in[i] - base;
        if (v < 0 || v > 2147483647LL) atomicExch(bad, 1);
        out[i] = (int)v;
    }
}

__global__ void k_check_cols(const int *__restrict__ idx, long long n, long long n_cols, int *bad) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = idx[i];
        if (c < 0 || c >= n_cols) atomicExch(bad, 1);
    }
}

__global__ void k_map_from_i64(const long long *__restrict__ in, int *__restrict__ out, long long n, long long limit) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const long long v = in[i];
        out[i] = (v < 0 || v >= limit) ? -1 : (int)v;
    }
}

__global__ void k_remap(const int *__restrict__ idx, const int *__restrict__ map, long long map_n, int *__restrict__ out,
                        long long n, int *any_invalid) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    bool bad = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = idx[i];
        const int m = (c < 0 || c >= map_n) ? -1 : map[c];
        out[i] = m;
        bad = bad || m < 0;
    }
    if (bad && any_invalid != nullptr) atomicExch(any_invalid, 1);
}

__global__ void k_map_invert(const int *__restrict__ map, long long n, int *__restrict__ out, long long n_out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int q = map[i];
        if (q >= 0 && q < n_out) out[q] = (int)i;
    }
}

// Cross-GPU barrier over peer-mapped flag words: rank r writes the lane's next epoch into slot r of every peer's
// flag array, then waits until every slot of its own array reached that epoch.  The epoch counter lives in device
// memory (one per lane) so the launch carries no per-call state: a captured CUDA graph replays it unchanged.
struct PeerFlags {
    unsigned int *p[MAX_SRC];
};
__global__ void k_peer_barrier(PeerFlags flags, int rank, int world, unsigned int *epoch_ctr, int *status, long long timeout_clocks) {
    __shared__ unsigned int s_epoch;
    __threadfence_system();
    if (threadIdx.x == 0) {
        s_epoch = *epoch_ctr + 1u;
        *epoch_ctr = s_epoch;
    }
    __syncthreads();
    const unsigned int epoch = s_epoch;
    const int s = threadIdx.x;
    if (s < world) {
        volatile unsigned int *remote = flags.p[s] + rank;
        *remote = epoch;
        __threadfence_system();
        volatile unsigned int *mine = flags.p[rank] + s;
        const long long t0 = clock64();
        while ((int)(*mine - epoch) < 0) {
            if (clock64() - t0 > timeout_clocks) {    // give up instead of hanging the box; the context is poisoned
                atomicExch(status, 1);
                break;
            }
        }
    }
    __syncthreads();
    __threadfence_system();
}

// ------------------------------------------------------------------------------------------------
// launch helpers
// ------------------------------------------------------------------------------------------------
int grid_for(arrow_ctx *ctx, const void *fn, int threads, size_t smem, long long work_ctas) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, threads, smem) != cudaSuccess || occ < 1) occ = 1;
    long long resident = (long long)occ * ctx->sm_count;
    long long g = std::min<long long>(std::max<long long>(work_ctas, 1), resident);
    return (int)g;
}

template <int G, int VPL>
int launch_vec(arrow_ctx *ctx, const SpmmArgs &a, bool rowmap, bool acc, int variant) {
    constexpr int RPW = 32 / G;
    const int threads = 256;
    const long long rows_per_cta = (long long)(threads / 32) * RPW;
    const long long ctas = (a.n_rows + rows_per_cta - 1) / rows_per_cta;
#define LAUNCH_K(KERNEL)                                                                              \
    do {                                                                                              \
        auto fn = KERNEL;                                                                             \
        int grid = grid_for(ctx, (const void *)fn, threads, 0, ctas);                                 \
        fn<<<grid, threads, 0, cur_stream(ctx)>>>(a);                                                     \
    } while (0)
    if (variant == ARROW_VARIANT_SHFL) {
        if (rowmap && acc) LAUNCH_K((k_spmm_shfl<G, VPL, true, true>));
        else if (rowmap) LAUNCH_K((k_spmm_shfl<G, VPL, true, false>));
        else if (acc) LAUNCH_K((k_spmm_shfl<G, VPL, false, true>));
        else LAUNCH_K((k_spmm_shfl<G, VPL, false, false>));
    } else {
        if (rowmap && acc) LAUNCH_K((k_spmm_direct<G, VPL, true, true>));
        else if (rowmap) LAUNCH_K((k_spmm_direct<G, VPL, true, false>));
        else if (acc) LAUNCH_K((k_spmm_direct<G, VPL, false, true>));
        else LAUNCH_K((k_spmm_direct<G, VPL, false, false>));
    }
#undef LAUNCH_K
    ctx->launches++;
    return ARROW_OK;
}

template <int VPL>
int launch_tma(arrow_ctx *ctx, const SpmmArgs &a, bool rowmap, bool acc) {
    const int threads = TMA_WARPS * 32;
    const size_t smem = (size_t)TMA_WARPS * TMA_STAGES * TMA_SLOTS * a.k * 4 + TMA_WARPS * TMA_STAGES * 8;
    const long long ctas = (a.n_rows + TMA_WARPS - 1) / TMA_WARPS;
#define LAUNCH_T(KERNEL)                                                                              \
    do {                                                                                              \
        auto fn = KERNEL;                                                                             \
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);             \
        int grid = grid_for(ctx, (const void *)fn, threads, smem, ctas);                              \
        fn<<<grid, threads, smem, cur_stream(ctx)>>>(a);                                                  \
    } while (0)
    if (rowmap && acc) LAUNCH_T((k_spmm_tma<VPL, true, true>));
    else if (rowmap) LAUNCH_T((k_spmm_tma<VPL, true, false>));
    else if (acc) LAUNCH_T((k_spmm_tma<VPL, false, true>));
    else LAUNCH_T((k_spmm_tma<VPL, false, false>));
#undef LAUNCH_T
    ctx->launches++;
    return ARROW_OK;
}

// what a tile launch needs beyond the template parameters
struct TileLaunch {
    int out_mode = OUT_IDENTITY;     // OUT_*
    bool acc = false;
    bool dualx = false;
    int vpl_req = 0;                 // 0 = default float4-per-lane count
    int rpg_req = 0;                 // 0 = default rows per lane group, 1 / 2 forced
};

template <typename T, int G, int VPL, int OUT, bool ACC, int TR, int TN, int RPG, int MINB, bool DUALX>
int launch_tiles_one(arrow_ctx *ctx, const TileArgs &t) {
    constexpr size_t SMEM = TileCfg<TR, TN>::SMEM_BYTES;
    auto fn = k_spmm_tiles<T, G, VPL, OUT, ACC, TR, TN, RPG, MINB, DUALX>;
    static bool attr_set[64] = {};            /* function attributes are per device */
    static int occ_dev[64] = {};
    const int dv = ctx->device & 63;
    if (!attr_set[dv]) {
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_dev[dv], fn, TILE_THREADS, SMEM) != cudaSuccess || occ_dev[dv] < 1) occ_dev[dv] = 1;
        attr_set[dv] = true;
    }
    static int carve_dev[64];
    if (ctx->smem_carveout != carve_dev[dv] - 1000) {       // measurement switch: how much of the 228 KB is L1
        cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, ctx->smem_carveout);
        carve_dev[dv] = ctx->smem_carveout + 1000;
    }
    const int occ = occ_dev[dv];
    const int per_sm = (ctx->spmm_ctas_per_sm > 0) ? std::min(occ, ctx->spmm_ctas_per_sm) : occ;
    int sms = ctx->sm_count;
    if (ctx->spmm_sm_limit > 0) sms = std::min(sms, ctx->spmm_sm_limit);
    int grid = (int)std::min<long long>((long long)per_sm * sms, t.n_tiles);
    // the scheduler words are zeroed before every launch: the round-1 kernel (which shares them) leaves its ticket behind,
    // and a launch must never depend on how the previous one on this lane ended
    cudaMemsetAsync(t.ticket, 0, 2 * sizeof(int), cur_stream(ctx));
    fn<<<grid, TILE_THREADS, SMEM, cur_stream(ctx)>>>(t);
    ctx->launches++;
    return ARROW_OK;
}

template <typename T, int G, int VPL, bool ROWMAP, bool ACC, int TR, int TN>
int launch_tiles_v1(arrow_ctx *ctx, const TileArgs &t) {
    constexpr size_t SMEM = TileCfg<TR, TN>::SMEM_BYTES;
    auto fn = k_spmm_tiles_v1<T, G, VPL, ROWMAP, ACC, TR, TN>;
    static bool attr_set[64] = {};
    static int occ_dev[64] = {};
    const int dv = ctx->device & 63;
    if (!attr_set[dv]) {
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_dev[dv], fn, TILE_THREADS, SMEM) != cudaSuccess || occ_dev[dv] < 1) occ_dev[dv] = 1;
        attr_set[dv] = true;
    }
    const int occ = occ_dev[dv];
    const int per_sm = (ctx->spmm_ctas_per_sm > 0) ? std::min(occ, ctx->spmm_ctas_per_sm) : occ;
    int sms = ctx->sm_count;
    if (ctx->spmm_sm_limit > 0) sms = std::min(sms, ctx->spmm_sm_limit);
    int grid = (int)std::min<long long>((long long)per_sm * sms, t.n_tiles);
    cudaMemsetAsync(t.ticket, 0, 2 * sizeof(int), cur_stream(ctx));
    fn<<<grid, TILE_THREADS, SMEM, cur_stream(ctx)>>>(t);
    ctx->launches++;
    return ARROW_OK;
}

template <typename T, int G, int VPL, int TR, int TN, int RPG, int MINB>
int launch_tiles_gv(arrow_ctx *ctx, const TileArgs &t, const TileLaunch &L) {
    if constexpr (is_bf16<T>()) {
        // bf16 launches are one-GPU launches (no row pointers, no dual X base; refused before this point) and always run
        // the round-1 kernel, except the paired-row shape
        if constexpr (RPG == 2) {
            if (L.out_mode == OUT_IDENTITY && !L.acc) return launch_tiles_one<T, G, VPL, OUT_IDENTITY, false, TR, TN, 2, MINB, false>(ctx, t);
        }
        const bool rowmap = L.out_mode == OUT_ROWMAP;
        if (rowmap && L.acc) return launch_tiles_v1<T, G, VPL, true, true, TR, TN>(ctx, t);
        if (rowmap) return launch_tiles_v1<T, G, VPL, true, false, TR, TN>(ctx, t);
        if (L.acc) return launch_tiles_v1<T, G, VPL, false, true, TR, TN>(ctx, t);
        return launch_tiles_v1<T, G, VPL, false, false, TR, TN>(ctx, t);
    } else {
        if (L.out_mode == OUT_ROWPTR) {
            // the multi-GPU fused path: row-pointer epilogue, optionally the [recv region | local tile] dual X base
            if (L.acc) return fail(ctx, ARROW_ERR_UNSUPPORTED, "row-pointer epilogue does not accumulate");
            if (L.dualx) return launch_tiles_one<T, G, VPL, OUT_ROWPTR, false, TR, TN, RPG, MINB, true>(ctx, t);
            return launch_tiles_one<T, G, VPL, OUT_ROWPTR, false, TR, TN, RPG, MINB, false>(ctx, t);
        }
        if (L.dualx) {
            if (L.out_mode != OUT_IDENTITY || L.acc) return fail(ctx, ARROW_ERR_UNSUPPORTED, "dual X base needs a plain or row-pointer epilogue");
            return launch_tiles_one<T, G, VPL, OUT_IDENTITY, false, TR, TN, RPG, MINB, true>(ctx, t);
        }
        if constexpr (RPG == 2) {
            // the two-rows-per-group family exists for plain and row-pointer launches (the narrow-k fast path)
            if (L.out_mode == OUT_IDENTITY && !L.acc) return launch_tiles_one<T, G, VPL, OUT_IDENTITY, false, TR, TN, 2, MINB, false>(ctx, t);
            return launch_tiles_gv<T, G, VPL, TR, TN, 1, 4>(ctx, t, L);
        } else {
            const bool rowmap = L.out_mode == OUT_ROWMAP;
            if (ctx->tile_kernel == 1) {
                if (rowmap && L.acc) return launch_tiles_v1<T, G, VPL, true, true, TR, TN>(ctx, t);
                if (rowmap) return launch_tiles_v1<T, G, VPL, true, false, TR, TN>(ctx, t);
                if (L.acc) return launch_tiles_v1<T, G, VPL, false, true, TR, TN>(ctx, t);
                return launch_tiles_v1<T, G, VPL, false, false, TR, TN>(ctx, t);
            }
            if (rowmap && L.acc) return launch_tiles_one<T, G, VPL, OUT_ROWMAP, true, TR, TN, 1, MINB, false>(ctx, t);
            if (rowmap) return launch_tiles_one<T, G, VPL, OUT_ROWMAP, false, TR, TN, 1, MINB, false>(ctx, t);
            if (L.acc) return launch_tiles_one<T, G, VPL, OUT_IDENTITY, true, TR, TN, 1, MINB, false>(ctx, t);
            return launch_tiles_one<T, G, VPL, OUT_IDENTITY, false, TR, TN, 1, MINB, false>(ctx, t);
        }
    }
}

// (lanes per row, 16-byte vectors per lane) for k4 vectors per row; vpl_req = 0 picks the default.  The shape follows the row's
// bytes, so a bf16 row of k columns is served like an fp32 row of k/2 -- except that a bf16 vector needs 8 fp32 accumulators
// where fp32 needs 4: VPL <= 2 keeps accumulators plus the gathers in flight (32 registers of X data per lane in every
// shape) within the 64 registers of __launch_bounds__(256, 4).
template <typename T>
int launch_tiles(arrow_ctx *ctx, TileArgs &t, const Csr *A, const TileLaunch &L) {
    const int k4 = t.a.k4;
    int vpl = L.vpl_req;
    // measured on B200 (profiles/r01_kernel_sweep.md): ~8 lanes per row is the sweet spot
    if (vpl != 1 && vpl != 2 && vpl != 4) vpl = (k4 >= 32) ? 4 : (k4 >= 8 ? 2 : 1);
    if (is_bf16<T>() && vpl > 2) vpl = 2;
    while (vpl > 1 && k4 < vpl) vpl >>= 1;
    int lanes = (k4 + vpl - 1) / vpl;                 // lanes needed per row
    if (lanes > 32) { vpl = (k4 + 31) / 32 <= 2 ? 2 : 4; lanes = (k4 + vpl - 1) / vpl; }
    int g = 1;
    while (g < lanes) g <<= 1;
    const bool big = (k4 <= 8) && ctx->big_tiles && A->n_tiles_big > 0;     // rows of <= 128 bytes (fp32 k <= 32, bf16 k <= 64)
    if (big) { t.tiles = A->tiles_big; t.tile_base = A->tile_base_big; t.n_tiles = A->n_tiles_big; }
    // measured at 10M rows (profiles/r02_kernel_sweep.md): pairs win at k = 32 (+3.5 %), lose at k = 16 (-10 %)
    int rpg = L.rpg_req ? L.rpg_req : (ctx->rows_per_group ? ctx->rows_per_group : (vpl == 2 ? 2 : 1));
    if (!big || rpg != 2) rpg = 1;                                           // pairs need >= 2 passes per tile
#define TL(GG, VV)                                                                                       \
    if (g == GG && vpl == VV) return launch_tiles_gv<T, GG, VV, TILE_ROWS, TILE_NNZ, 1, 4>(ctx, t, L)
#define TLB(GG, VV)                                                                                      \
    if (big && rpg == 1 && g == GG && vpl == VV) return launch_tiles_gv<T, GG, VV, TILE_ROWS_BIG, TILE_NNZ_BIG, 1, 4>(ctx, t, L)
#define TLP(GG, VV)                                                                                      \
    if (big && rpg == 2 && g == GG && vpl == VV) return launch_tiles_gv<T, GG, VV, TILE_ROWS_BIG, TILE_NNZ_BIG, 2, 4>(ctx, t, L)
    if constexpr (is_bf16<T>()) {
        // the shapes the defaults reach for k <= 256 (k = 16: 2 x 1, 32: 4 x 1, 64: 4 x 2 paired, 128: 8 x 2, 256: 16 x 2),
        // plus those of big tiles off / one row per group; other forced shapes are refused below
        TLP(4, 2);
        if (rpg == 2) rpg = 1;
        TLB(1, 1); TLB(2, 1); TLB(4, 1); TLB(8, 1); TLB(4, 2);
        TL(1, 1); TL(2, 1); TL(4, 1); TL(8, 1); TL(4, 2); TL(8, 2); TL(16, 2);
    } else {
        TLP(4, 1); TLP(8, 1); TLP(2, 2); TLP(4, 2);
        if (rpg == 2) rpg = 1;                                                   // no paired kernel for this shape
        TLB(1, 1); TLB(2, 1); TLB(4, 1); TLB(8, 1); TLB(1, 2); TLB(2, 2); TLB(4, 2); TLB(1, 4); TLB(2, 4);
        TL(1, 1); TL(2, 1); TL(4, 1); TL(8, 1); TL(16, 1); TL(32, 1);
        TL(1, 2); TL(2, 2); TL(4, 2); TL(8, 2); TL(16, 2); TL(32, 2);
        TL(1, 4); TL(2, 4); TL(4, 4); TL(8, 4); TL(16, 4);
    }
#undef TL
#undef TLB
#undef TLP
    return fail(ctx, ARROW_ERR_UNSUPPORTED, "no tile kernel for k4=%d vpl=%d", k4, vpl);
}

int pick_variant(int k) {
    (void)k;
    return 3;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int arrow_b200_abi_version(void) { return ARROW_ABI_VERSION; }

const char *arrow_last_error(const arrow_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int arrow_ctx_create(int device, void *stream, arrow_ctx **out) {
    if (!out) return fail(nullptr, ARROW_ERR_ARG, "out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, ARROW_ERR_CUDA, "no CUDA device available (%s); libarrow_b200 has no CPU fallback",
                    cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, ARROW_ERR_ARG, "device %d out of range [0,%d)", device, n);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, ARROW_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    arrow_ctx *ctx = new arrow_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        delete ctx;
        return fail(nullptr, ARROW_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    }
    ctx->sm_count = prop.multiProcessorCount;
    if (stream) {
        ctx->stream = (cudaStream_t)stream;
    } else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete ctx;
            return fail(nullptr, ARROW_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
        }
        ctx->own_stream = true;
    }
    e = cudaMalloc(&ctx->dev_status, sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(ctx->dev_status, 0, sizeof(int));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->barrier_epoch, ARROW_N_LANES * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemset(ctx->barrier_epoch, 0, ARROW_N_LANES * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMalloc(&ctx->tile_ticket, 2 * ARROW_N_LANES * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(ctx->tile_ticket, 0, 2 * ARROW_N_LANES * sizeof(int));
    if (e != cudaSuccess) {
        if (ctx->dev_status) cudaFree(ctx->dev_status);
        if (ctx->barrier_epoch) cudaFree(ctx->barrier_epoch);
        if (ctx->tile_ticket) cudaFree(ctx->tile_ticket);
        delete ctx;
        return fail(nullptr, ARROW_ERR_CUDA, "context state alloc: %s", cudaGetErrorString(e));
    }
    ctx->clock_khz = prop.clockRate > 0 ? prop.clockRate : 2000000;
    *out = ctx;
    return ARROW_OK;
}

void arrow_ctx_destroy(arrow_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &d : ctx->dense)
        if (d.live) {
            if (d.owned) cudaFree(d.p);
            else if (d.ipc) cudaIpcCloseMemHandle(d.ipc_base);
        }
    for (auto &c : ctx->csrs)
        if (c.live) csr_release(c);
    for (auto &m : ctx->maps)
        if (m.live) cudaFree(m.p);
    for (auto &t : ctx->timers) {
        if (t.a) cudaEventDestroy(t.a);
        if (t.b) cudaEventDestroy(t.b);
    }
    for (int l = 0; l < ARROW_N_LANES; ++l)
        if (ctx->long_scratch[l]) cudaFree(ctx->long_scratch[l]);
    for (float *p : ctx->retired_scratch) cudaFree(p);
    for (auto &pt : ctx->ptrtabs)
        if (pt.live) cudaFree(pt.p);
    for (auto g : ctx->graphs)
        if (g) cudaGraphExecDestroy(g);
    if (ctx->flush_buf) cudaFree(ctx->flush_buf);
    if (ctx->dev_status) cudaFree(ctx->dev_status);
    if (ctx->barrier_epoch) cudaFree(ctx->barrier_epoch);
    if (ctx->tile_ticket) cudaFree(ctx->tile_ticket);
    for (int l = 1; l < ARROW_N_LANES; ++l)
        if (ctx->lanes[l]) { cudaStreamSynchronize(ctx->lanes[l]); cudaStreamDestroy(ctx->lanes[l]); }
    for (int l = 0; l < ARROW_N_LANES; ++l)
        if (ctx->lane_events[l]) cudaEventDestroy(ctx->lane_events[l]);
    for (int e = 0; e < ARROW_MAX_EVENTS; ++e)
        if (ctx->user_events[e]) cudaEventDestroy(ctx->user_events[e]);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int arrow_sync(arrow_ctx *ctx) {
    CHECK_CTX(ctx);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    int st = 0;
    CUDA_TRY(ctx, cudaMemcpy(&st, ctx->dev_status, sizeof(int), cudaMemcpyDeviceToHost));
    if (st != 0) {
        ctx->poisoned = true;
        return fail(ctx, ARROW_ERR_CUDA, "device-side failure flag %d: a peer barrier timed out after %lld ms; the context is "
                    "poisoned (results after the time-out are racy) -- destroy it", st, ctx->barrier_timeout_ms);
    }
    return ARROW_OK;
}

int arrow_device_info(arrow_ctx *ctx, int *sm_count, int64_t *free_bytes, int64_t *total_bytes) {
    CHECK_CTX(ctx);
    size_t f = 0, t = 0;
    CUDA_TRY(ctx, cudaMemGetInfo(&f, &t));
    if (sm_count) *sm_count = ctx->sm_count;
    if (free_bytes) *free_bytes = (int64_t)f;
    if (total_bytes) *total_bytes = (int64_t)t;
    return ARROW_OK;
}

int arrow_set_tuning(arrow_ctx *ctx, int long_row_threshold, int long_row_segment) {
    CHECK_CTX(ctx);
    if (long_row_threshold < 1 || long_row_segment < 32 || long_row_threshold > TILE_NNZ - 8)
        return fail(ctx, ARROW_ERR_ARG, "bad tuning values (threshold must be in [1, %d])", TILE_NNZ - 8);
    ctx->long_threshold = long_row_threshold;
    ctx->long_segment = long_row_segment;
    return ARROW_OK;
}

int arrow_set_option(arrow_ctx *ctx, int option, int value) {
    CHECK_CTX(ctx);
    switch (option) {
        case ARROW_OPT_L2_HINTS_PLAIN: ctx->l2_hints_plain = value & 3; return ARROW_OK;
        case ARROW_OPT_L2_HINTS_FUSED: ctx->l2_hints_fused = value & 3; return ARROW_OK;
        case ARROW_OPT_BIG_TILES: ctx->big_tiles = value ? 1 : 0; return ARROW_OK;
        case ARROW_OPT_SPMM_CTAS_PER_SM: ctx->spmm_ctas_per_sm = value < 0 ? 0 : value; return ARROW_OK;
        case ARROW_OPT_PREFETCH: ctx->prefetch_plain = value & 0xF; ctx->prefetch_fused = (value >> 4) & 0xF;
            if (ctx->prefetch_plain > 1 || ctx->prefetch_fused > 1) { ctx->prefetch_plain = ctx->prefetch_fused = 0; return fail(ctx, ARROW_ERR_ARG, "prefetch modes are 0..1 per nibble"); }
            return ARROW_OK;
        case ARROW_OPT_ROWS_PER_GROUP: ctx->rows_per_group = (value == 1 || value == 2) ? value : 0; return ARROW_OK;
        case ARROW_OPT_SMEM_CARVEOUT: ctx->smem_carveout = value; return ARROW_OK;
        case ARROW_OPT_FORCE_PREDICATED: ctx->force_skip_path = value ? 1 : 0; return ARROW_OK;
        case ARROW_OPT_TILE_KERNEL: ctx->tile_kernel = value ? 1 : 0; return ARROW_OK;
        case ARROW_OPT_SPMM_SM_LIMIT: ctx->spmm_sm_limit = value < 0 ? 0 : value; return ARROW_OK;
        case ARROW_OPT_PUSH_CTAS: ctx->push_ctas = value < 0 ? 0 : value; return ARROW_OK;
        case ARROW_OPT_PUSH_INTERLEAVE: ctx->push_interleave = value ? 1 : 0; return ARROW_OK;
        case ARROW_OPT_BARRIER_TIMEOUT_MS: ctx->barrier_timeout_ms = value < 1 ? 1 : value; return ARROW_OK;
        default: return fail(ctx, ARROW_ERR_ARG, "unknown option %d", option);
    }
}

// ---- sparse -------------------------------------------------------------------------------------
inline int low_word(int64_t v) { return (int)(uint32_t)(uint64_t)v; }

static int build_long_rows(arrow_ctx *ctx, Csr &c, const std::vector<int64_t> &h_indptr) {
    // host pass over the (rebased) row pointer: rows above the threshold become segment tasks
    std::vector<LongTask> tasks;
    std::vector<int> rows, first;
    int64_t mx = 0;
    const int thr = ctx->long_threshold, seg = ctx->long_segment;
    for (int64_t r = 0; r < c.n_rows; ++r) {
        const int64_t len = h_indptr[r + 1] - h_indptr[r];
        mx = std::max<int64_t>(mx, len);
        if (len > thr) {
            rows.push_back((int)r);
            first.push_back((int)tasks.size());
            for (int64_t b = h_indptr[r]; b < h_indptr[r + 1]; b += seg)
                tasks.push_back(LongTask{b, std::min<int64_t>(b + seg, h_indptr[r + 1]), (int)r, (int)tasks.size()});
        }
    }
    first.push_back((int)tasks.size());
    // row tiles for k_spmm_tiles: contiguous rows, <= rows_cap rows and <= nnz_cap entries, cut around long rows
    auto build_tiles = [&](int rows_cap, int nnz_cap, int4 **out, long long **base_out, int *n_out) -> int {
        std::vector<int4> tiles;
        std::vector<long long> base;
        int64_t r = 0;
        while (r < c.n_rows) {
            const int64_t len0 = h_indptr[r + 1] - h_indptr[r];
            if (len0 > thr) { ++r; continue; }                     // long rows are not tiled
            int64_t e = r;
            while (e < c.n_rows && e - r < rows_cap) {
                const int64_t len = h_indptr[e + 1] - h_indptr[e];
                if (len > thr) break;
                if (h_indptr[e + 1] - h_indptr[r] > nnz_cap - 4 && e > r) break;
                ++e;
            }
            if (e == r) ++e;                                       // a single row always fits: thr <= TILE_NNZ - 8
            tiles.push_back(make_int4((int)r, (int)e, low_word(h_indptr[r]), low_word(h_indptr[e])));
            base.push_back(h_indptr[r]);
            r = e;
        }
        *n_out = (int)tiles.size();
        if (!tiles.empty()) {
            CUDA_TRY(ctx, cudaMalloc(out, tiles.size() * sizeof(int4)));
            CUDA_TRY(ctx, cudaMemcpy(*out, tiles.data(), tiles.size() * sizeof(int4), cudaMemcpyHostToDevice));
            CUDA_TRY(ctx, cudaMalloc(base_out, base.size() * sizeof(long long)));
            CUDA_TRY(ctx, cudaMemcpy(*base_out, base.data(), base.size() * sizeof(long long), cudaMemcpyHostToDevice));
        }
        return ARROW_OK;
    };
    {
        int rc = build_tiles(TILE_ROWS, TILE_NNZ, &c.tiles, &c.tile_base, &c.n_tiles);
        if (rc != ARROW_OK) return rc;
        rc = build_tiles(TILE_ROWS_BIG, TILE_NNZ_BIG, &c.tiles_big, &c.tile_base_big, &c.n_tiles_big);
        if (rc != ARROW_OK) return rc;
    }
    {
        std::vector<long long> anchors((size_t)((c.n_rows + ROW_GROUP - 1) >> ROW_GROUP_SHIFT) + 1);
        for (size_t g = 0; g < anchors.size(); ++g)
            anchors[g] = h_indptr[std::min<int64_t>((int64_t)g << ROW_GROUP_SHIFT, c.n_rows)];
        CUDA_TRY(ctx, cudaMalloc(&c.anchors, anchors.size() * sizeof(long long)));
        CUDA_TRY(ctx, cudaMemcpy(c.anchors, anchors.data(), anchors.size() * sizeof(long long), cudaMemcpyHostToDevice));
    }
    c.max_row_nnz = mx;
    c.long_threshold = thr;
    c.n_long_rows = (int)rows.size();
    c.n_long_tasks = (int)tasks.size();
    c.owns_long = true;
    if (!rows.empty()) {
        CUDA_TRY(ctx, cudaMalloc(&c.long_tasks, tasks.size() * sizeof(LongTask)));
        CUDA_TRY(ctx, cudaMalloc(&c.long_rows, rows.size() * sizeof(int)));
        CUDA_TRY(ctx, cudaMalloc(&c.long_first, first.size() * sizeof(int)));
        CUDA_TRY(ctx, cudaMemcpy(c.long_tasks, tasks.data(), tasks.size() * sizeof(LongTask), cudaMemcpyHostToDevice));
        CUDA_TRY(ctx, cudaMemcpy(c.long_rows, rows.data(), rows.size() * sizeof(int), cudaMemcpyHostToDevice));
        CUDA_TRY(ctx, cudaMemcpy(c.long_first, first.data(), first.size() * sizeof(int), cudaMemcpyHostToDevice));
    }
    return ARROW_OK;
}

// device side of arrow_csr_upload; on failure the caller releases whatever `c` already owns
static int csr_fill(arrow_ctx *ctx, Csr &c, int64_t n_rows, int64_t n_cols, int64_t nnz, const std::vector<int64_t> &h_indptr,
                    const void *indices, int indices_bytes, const float *data) {
    c.n_rows = n_rows;
    c.n_cols = n_cols;
    c.nnz = nnz;
    c.owns_indptr = c.owns_indices = c.owns_vals = c.owns_long = true;     // every array below belongs to this block
    std::vector<int> h_low((size_t)n_rows + 1);              // the device row pointer: low 32 bits of every offset
    for (size_t r = 0; r < h_low.size(); ++r) h_low[r] = low_word(h_indptr[r]);
    CUDA_TRY(ctx, cudaMalloc(&c.indptr, ((size_t)n_rows + 1 + 8) * sizeof(int)));
    CUDA_TRY(ctx, cudaMemsetAsync(c.indptr, 0, ((size_t)n_rows + 1 + 8) * sizeof(int), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(c.indptr, h_low.data(), ((size_t)n_rows + 1) * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    const size_t nz = (size_t)nnz + 8;                       // slack: bulk copies round up to 16 bytes
    CUDA_TRY(ctx, cudaMalloc(&c.indices, nz * sizeof(int)));
    CUDA_TRY(ctx, cudaMalloc(&c.vals, nz * sizeof(float)));
    CUDA_TRY(ctx, cudaMemsetAsync(c.indices, 0, nz * sizeof(int), ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(c.vals, 0, nz * sizeof(float), ctx->stream));
    DevTmp wide, bad;
    int hbad = 0;
    if (nnz > 0) {
        CUDA_TRY(ctx, cudaMalloc(&bad.p, sizeof(int)));
        CUDA_TRY(ctx, cudaMemsetAsync(bad.p, 0, sizeof(int), ctx->stream));
        if (indices_bytes == 4) {
            CUDA_TRY(ctx, cudaMemcpyAsync(c.indices, indices, (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
        } else {
            // 64-bit columns are narrowed through a bounded staging buffer: a block of billions of entries needs no
            // second copy of its index stream at twice the width
            const int64_t chunk = std::min<int64_t>(nnz, (int64_t)1 << 26);
            CUDA_TRY(ctx, cudaMalloc(&wide.p, (size_t)chunk * 8));
            for (int64_t o = 0; o < nnz; o += chunk) {
                const int64_t n = std::min(chunk, nnz - o);
                CUDA_TRY(ctx, cudaMemcpyAsync(wide.p, (const int64_t *)indices + o, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
                k_to_i32<long long><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((const long long *)wide.p, c.indices + o, n, 0, (int *)bad.p);
                ctx->launches++;
            }
        }
        // a column outside [0, n_cols) would read outside the X tile: reject the block instead
        k_check_cols<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(c.indices, nnz, n_cols, (int *)bad.p);
        ctx->launches++;
        CUDA_TRY(ctx, cudaMemcpyAsync(&hbad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        if (data) {
            CUDA_TRY(ctx, cudaMemcpyAsync(c.vals, data, (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
        } else {
            k_fill<float><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(c.vals, 1.0f, nnz);
            ctx->launches++;
        }
    }
    const int rc = build_long_rows(ctx, c, h_indptr);
    if (rc != ARROW_OK) return rc;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));      // the host staging arrays may go out of scope now
    CUDA_TRY(ctx, cudaGetLastError());
    if (hbad) return fail(ctx, ARROW_ERR_RANGE, "a column index lies outside [0, %lld)", (long long)n_cols);
    return ARROW_OK;
}

int arrow_csr_upload(arrow_ctx *ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const void *indptr, int indptr_bytes,
                     const void *indices, int indices_bytes, const float *data, int *csr_out) {
    CHECK_CTX(ctx);
    if (!csr_out || !indptr || (nnz > 0 && !indices)) return fail(ctx, ARROW_ERR_ARG, "null pointer argument");
    if (n_rows < 0 || n_cols < 0 || nnz < 0) return fail(ctx, ARROW_ERR_ARG, "negative size");
    if ((indptr_bytes != 4 && indptr_bytes != 8) || (indices_bytes != 4 && indices_bytes != 8))
        return fail(ctx, ARROW_ERR_ARG, "index width must be 4 or 8 bytes");
    if (n_rows >= 2147483647LL || n_cols > 2147483647LL)
        return fail(ctx, ARROW_ERR_RANGE, "rows / columns exceed the int32 device layout (rows=%lld cols=%lld); shard it",
                    (long long)n_rows, (long long)n_cols);
    // host view of the row pointer, rebased
    std::vector<int64_t> h_indptr((size_t)n_rows + 1);
    int64_t base = 0;
    if (indptr_bytes == 8) {
        const int64_t *ip = (const int64_t *)indptr;
        base = ip[0];
        for (int64_t r = 0; r <= n_rows; ++r) {
            const int64_t v = ip[r] - base;
            if (v < 0 || v > nnz || (r > 0 && v < h_indptr[r - 1]))
                return fail(ctx, ARROW_ERR_ARG, "indptr is not a non-decreasing sequence inside [0, nnz] at row %lld", (long long)r);
            h_indptr[r] = v;
        }
    } else {
        const int32_t *ip = (const int32_t *)indptr;
        base = ip[0];
        for (int64_t r = 0; r <= n_rows; ++r) {
            const int64_t v = (int64_t)ip[r] - base;
            if (v < 0 || v > nnz || (r > 0 && v < h_indptr[r - 1]))
                return fail(ctx, ARROW_ERR_ARG, "indptr is not a non-decreasing sequence inside [0, nnz] at row %lld", (long long)r);
            h_indptr[r] = v;
        }
    }
    if (h_indptr[n_rows] != nnz)
        return fail(ctx, ARROW_ERR_ARG, "indptr[n_rows]-indptr[0] = %lld but nnz = %lld", (long long)h_indptr[n_rows], (long long)nnz);
    // the per-row kernels find a row's 64-bit offset from the first row of its group of ROW_GROUP rows and a 32-bit
    // difference: no group may span 2^32 entries (rows averaging 2^26 entries)
    for (int64_t g = 0; g < n_rows; g += ROW_GROUP) {
        const int64_t span = h_indptr[std::min<int64_t>(g + ROW_GROUP, n_rows)] - h_indptr[g];
        if (span > 0xffffffffLL)
            return fail(ctx, ARROW_ERR_RANGE, "rows %lld..%lld hold %lld entries; a group of %d rows must hold fewer than 2^32",
                        (long long)g, (long long)std::min<int64_t>(g + ROW_GROUP, n_rows) - 1, (long long)span, ROW_GROUP);
    }

    Csr c;
    const int rc = csr_fill(ctx, c, n_rows, n_cols, nnz, h_indptr, indices, indices_bytes, data);
    if (rc != ARROW_OK) {
        cudaStreamSynchronize(ctx->stream);                  // nothing may still write into what is released next
        cudaGetLastError();
        csr_release(c);
        return rc;
    }
    c.live = true;
    const int h = new_slot(ctx->csrs);
    ctx->csrs[h] = c;
    *csr_out = h;
    return ARROW_OK;
}

int arrow_csr_free(arrow_ctx *ctx, int csr) {
    CHECK_CTX(ctx);
    Csr *c = get_csr(ctx, csr);
    if (!c) return fail(ctx, ARROW_ERR_HANDLE, "bad csr handle %d", csr);
    if (c->children > 0)
        return fail(ctx, ARROW_ERR_ARG, "csr %d still backs %d remapped block(s); free those first", csr, c->children);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (Csr *parent = get_csr(ctx, c->parent)) parent->children--;
    csr_release(*c);
    return ARROW_OK;
}

int arrow_csr_info(arrow_ctx *ctx, int csr, int64_t *n_rows, int64_t *n_cols, int64_t *nnz, int64_t *max_row_nnz,
                   int64_t *n_long_rows) {
    CHECK_CTX(ctx);
    Csr *c = get_csr(ctx, csr);
    if (!c) return fail(ctx, ARROW_ERR_HANDLE, "bad csr handle %d", csr);
    if (n_rows) *n_rows = c->n_rows;
    if (n_cols) *n_cols = c->n_cols;
    if (nnz) *nnz = c->nnz;
    if (max_row_nnz) *max_row_nnz = c->max_row_nnz;
    if (n_long_rows) *n_long_rows = c->n_long_rows;
    return ARROW_OK;
}

int arrow_csr_remap_columns(arrow_ctx *ctx, int csr, int map, int64_t new_n_cols, int *csr_out) {
    CHECK_CTX(ctx);
    Csr *c = get_csr(ctx, csr);
    IdxMap *m = get_map(ctx, map);
    if (!c) return fail(ctx, ARROW_ERR_HANDLE, "bad csr handle %d", csr);
    if (!m) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (!csr_out) return fail(ctx, ARROW_ERR_ARG, "csr_out is null");
    if (new_n_cols < 0 || new_n_cols > 2147483647LL || m->limit > new_n_cols)
        return fail(ctx, ARROW_ERR_ARG, "map reaches column %lld but the remapped block has %lld columns", (long long)m->limit, (long long)new_n_cols);
    if (c->parent >= 0) return fail(ctx, ARROW_ERR_ARG, "csr %d is itself a remapped copy; remap its source", csr);
    Csr d = *c;
    d.owns_indptr = d.owns_vals = d.owns_long = false;      // shared with the source block
    d.owns_indices = true;
    d.indices = nullptr;
    d.n_cols = new_n_cols;
    d.parent = csr;
    d.children = 0;
    CUDA_TRY(ctx, cudaMalloc(&d.indices, ((size_t)c->nnz + 8) * sizeof(int)));
    cudaError_t e = cudaMemsetAsync(d.indices, 0, ((size_t)c->nnz + 8) * sizeof(int), ctx->stream);
    int h_invalid = 0;
    if (e == cudaSuccess && c->nnz > 0) {
        DevTmp flag;
        e = cudaMalloc(&flag.p, sizeof(int));
        if (e == cudaSuccess) e = cudaMemsetAsync(flag.p, 0, sizeof(int), ctx->stream);
        if (e == cudaSuccess) {
            k_remap<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(c->indices, m->p, m->n, d.indices, c->nnz, (int *)flag.p);
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(&h_invalid, flag.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    if (e != cudaSuccess) {
        cudaFree(d.indices);
        return fail(ctx, ARROW_ERR_CUDA, "column remap failed: %s", cudaGetErrorString(e));
    }
    // entries whose image is invalid are skipped by the kernels (predicated gathers); when every entry maps to a valid
    // column -- always the case on the fused path -- the copy runs the unpredicated batches like its source
    d.may_skip = c->may_skip || h_invalid != 0;
    const int h = new_slot(ctx->csrs);       // may grow the table: `c` is not used past this point
    ctx->csrs[h] = d;
    ctx->csrs[csr].children++;
    *csr_out = h;
    return ARROW_OK;
}

// ---- maps ---------------------------------------------------------------------------------------
int arrow_map_upload(arrow_ctx *ctx, const int64_t *map, int64_t n, int64_t limit, int *map_out) {
    CHECK_CTX(ctx);
    if (!map_out || (n > 0 && !map)) return fail(ctx, ARROW_ERR_ARG, "null pointer argument");
    if (n < 0 || limit < 0 || limit > 2147483647LL || n > 2147483647LL)
        return fail(ctx, ARROW_ERR_RANGE, "map size/limit exceed the int32 device layout");
    IdxMap m;
    m.n = n;
    m.limit = limit;
    CUDA_TRY(ctx, cudaMalloc(&m.p, (size_t)std::max<int64_t>(n, 1) * sizeof(int)));
    cudaError_t e = cudaSuccess;
    if (n > 0) {
        DevTmp wide;
        e = cudaMalloc(&wide.p, (size_t)n * 8);
        if (e == cudaSuccess) e = cudaMemcpyAsync(wide.p, map, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            k_map_from_i64<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((const long long *)wide.p, m.p, n, limit);
            ctx->launches++;
            e = cudaStreamSynchronize(ctx->stream);
        }
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(m.p);
        return fail(ctx, ARROW_ERR_CUDA, "map upload failed: %s", cudaGetErrorString(e));
    }
    m.live = true;
    const int h = new_slot(ctx->maps);
    ctx->maps[h] = m;
    *map_out = h;
    return ARROW_OK;
}

int arrow_map_free(arrow_ctx *ctx, int map) {
    CHECK_CTX(ctx);
    IdxMap *m = get_map(ctx, map);
    if (!m) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(m->p);
    *m = IdxMap();
    return ARROW_OK;
}

int arrow_map_compose(arrow_ctx *ctx, int inner, int outer, int *map_out) {
    CHECK_CTX(ctx);
    IdxMap *a = get_map(ctx, inner), *b = get_map(ctx, outer);
    if (!a || !b) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle");
    if (!map_out) return fail(ctx, ARROW_ERR_ARG, "map_out is null");
    IdxMap m;
    m.n = a->n;
    m.limit = b->limit;
    CUDA_TRY(ctx, cudaMalloc(&m.p, (size_t)std::max<int64_t>(m.n, 1) * sizeof(int)));
    if (m.n > 0) {
        k_remap<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(a->p, b->p, b->n, m.p, m.n, nullptr);
        ctx->launches++;
    }
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) {
        cudaFree(m.p);
        return fail(ctx, ARROW_ERR_CUDA, "map compose failed: %s", cudaGetErrorString(e));
    }
    m.live = true;
    const int h = new_slot(ctx->maps);
    ctx->maps[h] = m;
    *map_out = h;
    return ARROW_OK;
}

int arrow_map_invert(arrow_ctx *ctx, int map, int64_t n_out, int *map_out) {
    CHECK_CTX(ctx);
    IdxMap *a = get_map(ctx, map);
    if (!a) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (!map_out || n_out < 0 || n_out > 2147483647LL) return fail(ctx, ARROW_ERR_ARG, "bad argument");
    IdxMap m;
    m.n = n_out;
    m.limit = a->n;
    CUDA_TRY(ctx, cudaMalloc(&m.p, (size_t)std::max<int64_t>(n_out, 1) * sizeof(int)));
    if (n_out > 0) {
        k_fill<int><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(m.p, -1, n_out);
        ctx->launches++;
    }
    if (a->n > 0) {
        k_map_invert<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(a->p, a->n, m.p, n_out);
        ctx->launches++;
    }
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) {
        cudaFree(m.p);
        return fail(ctx, ARROW_ERR_CUDA, "map invert failed: %s", cudaGetErrorString(e));
    }
    m.live = true;
    const int h = new_slot(ctx->maps);
    ctx->maps[h] = m;
    *map_out = h;
    return ARROW_OK;
}

int arrow_map_d2h(arrow_ctx *ctx, int map, int32_t *host, int64_t n) {
    CHECK_CTX(ctx);
    IdxMap *a = get_map(ctx, map);
    if (!a) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (!host || n < 0 || n > a->n) return fail(ctx, ARROW_ERR_ARG, "bad host buffer / length");
    CUDA_TRY(ctx, cudaMemcpyAsync(host, a->p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return ARROW_OK;
}

// ---- dense --------------------------------------------------------------------------------------
int arrow_dense_alloc(arrow_ctx *ctx, int64_t rows, int k, int *buf_out) {
    return arrow_dense_alloc_dtype(ctx, rows, k, ARROW_DTYPE_F32, buf_out);
}

int arrow_dense_alloc_dtype(arrow_ctx *ctx, int64_t rows, int k, int dtype, int *buf_out) {
    CHECK_CTX(ctx);
    if (!buf_out || rows < 0 || k < 1) return fail(ctx, ARROW_ERR_ARG, "bad dense shape %lld x %d", (long long)rows, k);
    if (dtype != ARROW_DTYPE_F32 && dtype != ARROW_DTYPE_BF16) return fail(ctx, ARROW_ERR_ARG, "unknown dtype %d", dtype);
    DenseBuf d;
    d.rows = rows;
    d.k = k;
    d.dtype = dtype;
    const size_t bytes = std::max<size_t>((size_t)rows * (size_t)k * d.esize(), 16);
    cudaError_t e = cudaMalloc(&d.p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, ARROW_ERR_NOMEM, "cudaMalloc(%zu bytes) for a %lld x %d tile: %s", bytes, (long long)rows, k,
                    cudaGetErrorString(e));
    }
    CUDA_TRY(ctx, cudaMemsetAsync(d.p, 0, bytes, ctx->stream));
    d.owned = true;
    d.live = true;
    const int h = new_slot(ctx->dense);
    ctx->dense[h] = d;
    *buf_out = h;
    return ARROW_OK;
}

int arrow_dense_dtype(arrow_ctx *ctx, int buf, int *dtype) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!dtype) return fail(ctx, ARROW_ERR_ARG, "dtype is null");
    *dtype = d->dtype;
    return ARROW_OK;
}

int arrow_dense_free(arrow_ctx *ctx, int buf) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (d->owned) cudaFree(d->p);
    else if (d->ipc) cudaIpcCloseMemHandle(d->ipc_base);
    *d = DenseBuf();
    return ARROW_OK;
}

int arrow_dense_fill(arrow_ctx *ctx, int buf, float value) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    const long long n = (long long)d->rows * d->k;
    if (n == 0) return ARROW_OK;
    if (value == 0.f) {
        CUDA_TRY(ctx, cudaMemsetAsync(d->p, 0, (size_t)n * d->esize(), ctx->stream));
    } else if (d->dtype == ARROW_DTYPE_BF16) {
        k_fill<bf16><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(reinterpret_cast<bf16 *>(d->p), __float2bfloat16_rn(value), n);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
    } else {
        k_fill<float><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d->p, value, n);
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
    }
    return ARROW_OK;
}

int arrow_dense_h2d(arrow_ctx *ctx, int buf, int64_t row0, int64_t rows, const float *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows)
        return fail(ctx, ARROW_ERR_ARG, "h2d rows [%lld,%lld) outside tile of %lld rows", (long long)row0, (long long)(row0 + rows), (long long)d->rows);
    REQUIRE_F32(ctx, d, "arrow_dense_h2d (float rows; arrow_dense_put copies any dtype)");
    if (rows == 0) return ARROW_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(d->p + (size_t)row0 * d->k, host, (size_t)rows * d->k * 4, cudaMemcpyHostToDevice, ctx->stream));
    return ARROW_OK;
}

int arrow_dense_d2h(arrow_ctx *ctx, int buf, int64_t row0, int64_t rows, float *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows)
        return fail(ctx, ARROW_ERR_ARG, "d2h rows [%lld,%lld) outside tile of %lld rows", (long long)row0, (long long)(row0 + rows), (long long)d->rows);
    REQUIRE_F32(ctx, d, "arrow_dense_d2h (float rows; arrow_dense_get copies any dtype)");
    if (rows == 0) return ARROW_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(host, d->p + (size_t)row0 * d->k, (size_t)rows * d->k * 4, cudaMemcpyDeviceToHost, ctx->stream));
    return ARROW_OK;
}

int arrow_dense_copy(arrow_ctx *ctx, int dst, int64_t dst_row0, int src, int64_t src_row0, int64_t rows) {
    CHECK_CTX(ctx);
    DenseBuf *a = get_dense(ctx, dst), *b = get_dense(ctx, src);
    if (!a || !b) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle");
    if (a->k != b->k) return fail(ctx, ARROW_ERR_ARG, "feature width mismatch %d vs %d", a->k, b->k);
    if (a->dtype != b->dtype) return fail(ctx, ARROW_ERR_ARG, "copy between tiles of different dtype (%d vs %d)", b->dtype, a->dtype);
    if (rows < 0 || dst_row0 < 0 || src_row0 < 0 || dst_row0 + rows > a->rows || src_row0 + rows > b->rows)
        return fail(ctx, ARROW_ERR_ARG, "copy range outside tiles");
    if (rows == 0) return ARROW_OK;
    CUDA_TRY(ctx, cudaMemcpyAsync(a->row(dst_row0), b->row(src_row0), (size_t)rows * a->k * a->esize(),
                                  cudaMemcpyDeviceToDevice, cur_stream(ctx)));
    return ARROW_OK;
}

int arrow_dense_ptr(arrow_ctx *ctx, int buf, void **device_ptr, int64_t *rows, int *k) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (device_ptr) *device_ptr = d->p;
    if (rows) *rows = d->rows;
    if (k) *k = d->k;
    return ARROW_OK;
}

int arrow_dense_wrap(arrow_ctx *ctx, void *device_ptr, int64_t rows, int k, int *buf_out) {
    CHECK_CTX(ctx);
    if (!device_ptr || !buf_out || rows < 0 || k < 1) return fail(ctx, ARROW_ERR_ARG, "bad wrap arguments");
    DenseBuf d;
    d.p = (float *)device_ptr;
    d.rows = rows;
    d.k = k;
    d.live = true;
    const int h = new_slot(ctx->dense);
    ctx->dense[h] = d;
    *buf_out = h;
    return ARROW_OK;
}

int arrow_host_alloc(size_t bytes, void **ptr) {
    if (!ptr) return ARROW_ERR_ARG;
    cudaError_t e = cudaMallocHost(ptr, std::max<size_t>(bytes, 16));
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, ARROW_ERR_NOMEM, "cudaMallocHost(%zu): %s", bytes, cudaGetErrorString(e));
    }
    return ARROW_OK;
}

int arrow_host_free(void *ptr) {
    if (!ptr) return ARROW_OK;
    size_t len = 0;
    {
        std::lock_guard<std::mutex> lk(g_numa_mu);
        auto it = g_numa_allocs.find(ptr);
        if (it != g_numa_allocs.end()) { len = it->second; g_numa_allocs.erase(it); }
    }
    if (len) {
        const bool ok = cudaHostUnregister(ptr) == cudaSuccess;
        munmap(ptr, len);
        return ok ? ARROW_OK : ARROW_ERR_CUDA;
    }
    return cudaFreeHost(ptr) == cudaSuccess ? ARROW_OK : ARROW_ERR_CUDA;
}

// ---- hot path -----------------------------------------------------------------------------------
struct SpmmCall {
    int csr = -1, x_buf = -1, c_buf = -1;
    int rowmap = -1, flags = 0, variant = ARROW_VARIANT_AUTO;
    int add_buf = -1, add_map = -1;
    int x2_buf = -1;
    int64_t x_split = 0;
    int out_table = -1;
};
static int spmm_impl(arrow_ctx *ctx, const SpmmCall &q);

#define CHECK_POISON(ctx)                                                                                     \
    do {                                                                                                      \
        if ((ctx)->poisoned) return fail((ctx), ARROW_ERR_CUDA, "context is poisoned by a peer-barrier time-out"); \
    } while (0)

int arrow_spmm(arrow_ctx *ctx, int csr, int x_buf, int c_buf, int rowmap, int flags, int variant) {
    SpmmCall q;
    q.csr = csr; q.x_buf = x_buf; q.c_buf = c_buf; q.rowmap = rowmap; q.flags = flags; q.variant = variant;
    return spmm_impl(ctx, q);
}

int arrow_spmm_add(arrow_ctx *ctx, int csr, int x_buf, int c_buf, int add_buf, int add_map, int variant) {
    SpmmCall q;
    q.csr = csr; q.x_buf = x_buf; q.c_buf = c_buf; q.variant = variant; q.add_buf = add_buf; q.add_map = add_map;
    return spmm_impl(ctx, q);
}

int arrow_spmm_ex(arrow_ctx *ctx, int csr, int x_buf, int x2_buf, int64_t x_split, int c_buf, int out_table,
                  int add_buf, int add_map, int variant) {
    CHECK_CTX(ctx);
    for (int h : {x_buf, x2_buf, c_buf, add_buf}) {
        const DenseBuf *d = get_dense(ctx, h);
        if (d && d->dtype != ARROW_DTYPE_F32) return fail(ctx, ARROW_ERR_ARG, "arrow_spmm_ex (N-GPU path) needs fp32 tiles; buffer %d is bf16", h);
    }
    SpmmCall q;
    q.csr = csr; q.x_buf = x_buf; q.x2_buf = x2_buf; q.x_split = x_split; q.c_buf = c_buf; q.out_table = out_table;
    q.add_buf = add_buf; q.add_map = add_map; q.variant = variant;
    return spmm_impl(ctx, q);
}

static int spmm_impl(arrow_ctx *ctx, const SpmmCall &q) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    Csr *A = get_csr(ctx, q.csr);
    DenseBuf *X = get_dense(ctx, q.x_buf);
    DenseBuf *C = q.c_buf >= 0 ? get_dense(ctx, q.c_buf) : nullptr;
    if (!A) return fail(ctx, ARROW_ERR_HANDLE, "bad csr handle %d", q.csr);
    if (!X) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle (x=%d)", q.x_buf);
    PtrTable *OT = nullptr;
    if (q.out_table >= 0) {
        if (q.out_table >= (int)ctx->ptrtabs.size() || !ctx->ptrtabs[q.out_table].live)
            return fail(ctx, ARROW_ERR_HANDLE, "bad pointer table handle %d", q.out_table);
        OT = &ctx->ptrtabs[q.out_table];
        if (OT->n < A->n_rows) return fail(ctx, ARROW_ERR_ARG, "pointer table has %lld entries, block has %lld rows", (long long)OT->n, (long long)A->n_rows);
        if (OT->k != X->k) return fail(ctx, ARROW_ERR_ARG, "pointer table was built for %d feature columns, X has %d", OT->k, X->k);
        if (q.rowmap >= 0 || (q.flags & ARROW_ACCUMULATE)) return fail(ctx, ARROW_ERR_ARG, "a pointer table excludes rowmap / accumulate");
    } else if (!C) {
        return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle (c=%d)", q.c_buf);
    }
    const bool bf = X->dtype == ARROW_DTYPE_BF16;
    if (C) {
        if (X->k != C->k) return fail(ctx, ARROW_ERR_ARG, "X has %d feature columns, C has %d", X->k, C->k);
        if (X->p == C->p) return fail(ctx, ARROW_ERR_ARG, "X and C must not alias");
        if (X->dtype != C->dtype) return fail(ctx, ARROW_ERR_ARG, "X and C differ in dtype (%d vs %d)", X->dtype, C->dtype);
    }
    DenseBuf *X2 = nullptr;
    if (q.x2_buf >= 0) {
        X2 = get_dense(ctx, q.x2_buf);
        if (!X2) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle (x2=%d)", q.x2_buf);
        if (X2->k != X->k) return fail(ctx, ARROW_ERR_ARG, "X2 has %d feature columns, X has %d", X2->k, X->k);
        if (q.x_split < 0 || q.x_split > X->rows || q.x_split > A->n_cols)
            return fail(ctx, ARROW_ERR_ARG, "x_split %lld outside X (%lld rows) / the block's %lld columns", (long long)q.x_split, (long long)X->rows, (long long)A->n_cols);
        if (X2->rows < A->n_cols - q.x_split)
            return fail(ctx, ARROW_ERR_ARG, "X2 has %lld rows, columns beyond the split need %lld", (long long)X2->rows, (long long)(A->n_cols - q.x_split));
        if (C && X2->p == C->p) return fail(ctx, ARROW_ERR_ARG, "X2 and C must not alias");
    } else if (X->rows < A->n_cols) {
        return fail(ctx, ARROW_ERR_ARG, "X has %lld rows, block has %lld columns", (long long)X->rows, (long long)A->n_cols);
    }
    IdxMap *rm = nullptr;
    if (q.rowmap >= 0) {
        rm = get_map(ctx, q.rowmap);
        if (!rm) return fail(ctx, ARROW_ERR_HANDLE, "bad rowmap handle %d", q.rowmap);
        if (rm->n < A->n_rows) return fail(ctx, ARROW_ERR_ARG, "rowmap has %lld entries, block has %lld rows", (long long)rm->n, (long long)A->n_rows);
        if (rm->limit > C->rows) return fail(ctx, ARROW_ERR_ARG, "rowmap reaches row %lld, C has %lld rows", (long long)rm->limit, (long long)C->rows);
    } else if (C && !OT && C->rows < A->n_rows) {
        return fail(ctx, ARROW_ERR_ARG, "C has %lld rows, block has %lld rows", (long long)C->rows, (long long)A->n_rows);
    }
    if (A->n_rows == 0) return ARROW_OK;
    const bool acc = (q.flags & ARROW_ACCUMULATE) != 0;
    const int k = X->k;
    const int lane = ctx->cur_lane;
    cudaStream_t stream = cur_stream(ctx);
    SpmmArgs a;
    a.indptr = A->indptr;
    a.anchors = A->anchors;
    a.indices = A->indices;
    a.vals = A->vals;
    a.X = X->p;
    a.C = C ? C->p : nullptr;
    a.rowmap = rm ? rm->p : nullptr;
    a.n_rows = A->n_rows;
    a.k = k;
    a.k4 = k / (bf ? Elt<bf16>::PER_VEC : Elt<float>::PER_VEC);
    a.long_threshold = A->long_threshold;
    a.add_src = nullptr;
    a.add_map = nullptr;
    a.X2 = X2 ? X2->p : nullptr;
    a.x_split = X2 ? (int)q.x_split : 0;
    a.out_ptr = OT ? OT->p : nullptr;
    if (q.add_buf >= 0 || q.add_map >= 0) {
        DenseBuf *S = get_dense(ctx, q.add_buf);
        IdxMap *am = get_map(ctx, q.add_map);
        if (!S || !am) return fail(ctx, ARROW_ERR_HANDLE, "bad addend handles (buf=%d map=%d)", q.add_buf, q.add_map);
        if (S->k != k) return fail(ctx, ARROW_ERR_ARG, "addend has %d feature columns, expected %d", S->k, k);
        if (S->dtype != X->dtype) return fail(ctx, ARROW_ERR_ARG, "addend and X differ in dtype (%d vs %d)", S->dtype, X->dtype);
        if (am->n < A->n_rows) return fail(ctx, ARROW_ERR_ARG, "addend map has %lld entries, block has %lld rows", (long long)am->n, (long long)A->n_rows);
        if (am->limit > S->rows) return fail(ctx, ARROW_ERR_ARG, "addend map reaches row %lld, addend tile has %lld rows", (long long)am->limit, (long long)S->rows);
        if (C && S->p == C->p) return fail(ctx, ARROW_ERR_ARG, "addend and C must not alias");
        a.add_src = S->p;
        a.add_map = am->p;
    }
    int variant = q.variant;
    if (variant == ARROW_VARIANT_AUTO) variant = pick_variant(k);
    const int vpl_req = (variant >> 4) & 0xF;          // optional float4-per-lane override (tile kernel)
    const int rpg_req = (variant >> 8) & 0x3;          // optional rows-per-group override (tile kernel, k <= 32)
    variant &= 0xF;
    // the epilogue gather-add, the dual X base and the row-pointer epilogue live in the tile / generic / long kernels
    if ((a.add_map != nullptr || X2 || OT) && variant != 3) variant = 3;
    if (variant < 0 || variant > 3) return fail(ctx, ARROW_ERR_ARG, "unknown variant %d", variant);
    if (bf && variant != ARROW_VARIANT_TILES) return fail(ctx, ARROW_ERR_UNSUPPORTED, "bf16 tiles run the tile kernel only (variant %d)", variant);
    const bool fused_launch = rm != nullptr || acc || OT != nullptr || X2 != nullptr || a.add_map != nullptr;

    const bool vec_ok = (k % (bf ? 8 : 4) == 0) && k <= 256;
    if (!vec_ok) {
        const long long ctas = (A->n_rows + 7) / 8;
#define LAUNCH_G(KERNEL)                                                                              \
    do {                                                                                              \
        auto fn = KERNEL;                                                                             \
        int grid = grid_for(ctx, (const void *)fn, 256, 0, ctas);                                     \
        fn<<<grid, 256, 0, stream>>>(a);                                                              \
    } while (0)
        if (bf) {
            if (rm && acc) LAUNCH_G((k_spmm_generic<bf16, true, true>));
            else if (rm) LAUNCH_G((k_spmm_generic<bf16, true, false>));
            else if (acc) LAUNCH_G((k_spmm_generic<bf16, false, true>));
            else LAUNCH_G((k_spmm_generic<bf16, false, false>));
        } else {
            if (rm && acc) LAUNCH_G((k_spmm_generic<float, true, true>));
            else if (rm) LAUNCH_G((k_spmm_generic<float, true, false>));
            else if (acc) LAUNCH_G((k_spmm_generic<float, false, true>));
            else LAUNCH_G((k_spmm_generic<float, false, false>));
        }
#undef LAUNCH_G
        ctx->launches++;
    } else if (variant == 3) {
        if (A->n_tiles > 0) {
            TileArgs t;
            t.a = a;
            t.tiles = A->tiles;
            t.tile_base = A->tile_base;
            t.n_tiles = A->n_tiles;
            t.skip = (A->may_skip || ctx->force_skip_path) ? 1 : 0;
            t.ticket = ctx->tile_ticket + 2 * lane;
            t.l2_hints = (rm != nullptr || acc) ? ctx->l2_hints_fused : ctx->l2_hints_plain;
            t.prefetch = fused_launch ? ctx->prefetch_fused : ctx->prefetch_plain;
            TileLaunch L;
            L.out_mode = OT ? OUT_ROWPTR : (rm ? OUT_ROWMAP : OUT_IDENTITY);
            L.acc = acc;
            L.dualx = X2 != nullptr;
            L.vpl_req = vpl_req;
            L.rpg_req = rpg_req;
            int rc = bf ? launch_tiles<bf16>(ctx, t, A, L) : launch_tiles<float>(ctx, t, A, L);
            if (rc != ARROW_OK) return rc;
        }
    } else if (variant == ARROW_VARIANT_TMA && k >= 32 && k <= 128) {
        if (a.k4 <= 32) launch_tma<1>(ctx, a, rm != nullptr, acc);
        else launch_tma<2>(ctx, a, rm != nullptr, acc);
    } else {
        if (variant == ARROW_VARIANT_TMA) variant = ARROW_VARIANT_SHFL;
        const int k4 = a.k4;
        if (k4 <= 1) launch_vec<1, 1>(ctx, a, rm != nullptr, acc, variant);
        else if (k4 <= 2) launch_vec<2, 1>(ctx, a, rm != nullptr, acc, variant);
        else if (k4 <= 4) launch_vec<4, 1>(ctx, a, rm != nullptr, acc, variant);
        else if (k4 <= 8) launch_vec<8, 1>(ctx, a, rm != nullptr, acc, variant);
        else if (k4 <= 16) launch_vec<16, 1>(ctx, a, rm != nullptr, acc, variant);
        else if (k4 <= 32) launch_vec<32, 1>(ctx, a, rm != nullptr, acc, variant);
        else launch_vec<32, 2>(ctx, a, rm != nullptr, acc, variant);
    }
    CUDA_TRY(ctx, cudaGetLastError());

    if (A->n_long_tasks > 0) {
        const size_t need = (size_t)A->n_long_tasks * k * 4;
        if (need > ctx->long_scratch_bytes[lane]) {
            if (ctx->capturing) return fail(ctx, ARROW_ERR_UNSUPPORTED, "long-row scratch would grow during graph capture: run the step once first");
            CUDA_TRY(ctx, cudaStreamSynchronize(stream));
            // a graph recorded earlier replays with the pointer it captured: while one is live the old buffer is retired,
            // not freed, so that a replay after this growth still reads and writes memory it owns
            if (ctx->long_scratch[lane]) {
                if (graphs_live(ctx)) ctx->retired_scratch.push_back(ctx->long_scratch[lane]);
                else cudaFree(ctx->long_scratch[lane]);
            }
            ctx->long_scratch[lane] = nullptr;
            ctx->long_scratch_bytes[lane] = 0;
            CUDA_TRY(ctx, cudaMalloc(&ctx->long_scratch[lane], need));
            ctx->long_scratch_bytes[lane] = need;
        }
        LongArgs la;
        la.tasks = A->long_tasks;
        la.indices = A->indices;
        la.vals = A->vals;
        la.X = X->p;
        la.scratch = ctx->long_scratch[lane];
        la.k = k;
        la.X2 = a.X2;
        la.x_split = a.x_split;
        const size_t smem = (size_t)8 * k * 4;
        auto partial = bf ? k_spmm_long_partial<bf16> : k_spmm_long_partial<float>;
        if (smem > 48 * 1024)
            CUDA_TRY(ctx, cudaFuncSetAttribute(partial, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        partial<<<A->n_long_tasks, 256, smem, stream>>>(la);
        ctx->launches++;
        const int *rmp = rm ? rm->p : nullptr;
        float *cp = C ? C->p : nullptr;
        float *scr = ctx->long_scratch[lane];
#define LAUNCH_R(TT, RM, AC)                                                                                        \
    k_spmm_long_reduce<TT, RM, AC><<<A->n_long_rows, 128, 0, stream>>>(A->long_rows, A->long_first, scr,            \
                                                                      reinterpret_cast<TT *>(cp), rmp, k,           \
                                                                      reinterpret_cast<const TT *>(a.add_src), a.add_map, a.out_ptr)
        if (bf) {
            if (rm && acc) LAUNCH_R(bf16, true, true);
            else if (rm) LAUNCH_R(bf16, true, false);
            else if (acc) LAUNCH_R(bf16, false, true);
            else LAUNCH_R(bf16, false, false);
        } else {
            if (rm && acc) LAUNCH_R(float, true, true);
            else if (rm) LAUNCH_R(float, true, false);
            else if (acc) LAUNCH_R(float, false, true);
            else LAUNCH_R(float, false, false);
        }
#undef LAUNCH_R
        ctx->launches++;
        CUDA_TRY(ctx, cudaGetLastError());
    }
    return ARROW_OK;
}

// ---- pointer tables -------------------------------------------------------------------------------
int arrow_ptrtable_upload(arrow_ctx *ctx, const int *bufs, int n_bufs, const int32_t *which, const int64_t *row, int64_t n,
                          int *table_out) {
    CHECK_CTX(ctx);
    if (!table_out || n < 0 || n_bufs < 1 || n_bufs > 64 || !bufs || (n > 0 && (!which || !row)))
        return fail(ctx, ARROW_ERR_ARG, "bad pointer table arguments");
    unsigned long long bases[64];
    int64_t rows_of[64];
    int k = 0;
    for (int b = 0; b < n_bufs; ++b) {
        DenseBuf *d = get_dense(ctx, bufs[b]);
        if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", bufs[b]);
        REQUIRE_F32(ctx, d, "arrow_ptrtable_upload (N-GPU path)");
        if (b == 0) k = d->k;
        else if (d->k != k) return fail(ctx, ARROW_ERR_ARG, "tiles of a pointer table must share the feature width");
        bases[b] = (unsigned long long)d->p;
        rows_of[b] = d->rows;
    }
    for (int64_t i = 0; i < n; ++i) {
        const int w = which[i];
        if (w >= n_bufs) return fail(ctx, ARROW_ERR_ARG, "row %lld refers to tile %d of %d", (long long)i, w, n_bufs);
        if (w >= 0 && (row[i] < 0 || row[i] >= rows_of[w]))
            return fail(ctx, ARROW_ERR_ARG, "row %lld points at row %lld of a %lld-row tile", (long long)i, (long long)row[i], (long long)rows_of[w]);
    }
    PtrTable t;
    t.n = n;
    t.k = k;
    CUDA_TRY(ctx, cudaMalloc(&t.p, (size_t)std::max<int64_t>(n, 1) * sizeof(float *)));
    cudaError_t e = cudaSuccess;
    if (n > 0) {
        DevTmp dw, dr, db;
        e = cudaMalloc(&dw.p, (size_t)n * 4);
        if (e == cudaSuccess) e = cudaMalloc(&dr.p, (size_t)n * 8);
        if (e == cudaSuccess) e = cudaMalloc(&db.p, sizeof bases);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dw.p, which, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dr.p, row, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(db.p, bases, sizeof bases, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) {
            k_fill_ptr_table<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(t.p, (const int *)dw.p, (const long long *)dr.p,
                                                                         (const unsigned long long *)db.p, n, k);
            ctx->launches++;
            e = cudaStreamSynchronize(ctx->stream);
        }
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        cudaFree(t.p);
        return fail(ctx, ARROW_ERR_CUDA, "pointer table upload failed: %s", cudaGetErrorString(e));
    }
    t.live = true;
    int h = -1;
    for (size_t i = 0; i < ctx->ptrtabs.size(); ++i)
        if (!ctx->ptrtabs[i].live) { h = (int)i; break; }
    if (h < 0) { ctx->ptrtabs.emplace_back(); h = (int)ctx->ptrtabs.size() - 1; }
    ctx->ptrtabs[h] = t;
    *table_out = h;
    return ARROW_OK;
}

int arrow_ptrtable_free(arrow_ctx *ctx, int table) {
    CHECK_CTX(ctx);
    if (table < 0 || table >= (int)ctx->ptrtabs.size() || !ctx->ptrtabs[table].live)
        return fail(ctx, ARROW_ERR_HANDLE, "bad pointer table handle %d", table);
    CUDA_TRY(ctx, cudaDeviceSynchronize());
    cudaFree(ctx->ptrtabs[table].p);
    ctx->ptrtabs[table] = PtrTable();
    return ARROW_OK;
}

static int gather_common(arrow_ctx *ctx, DenseBuf *D, const float *src, const MultiSrc &ms, bool multi, IdxMap *m, bool acc) {
    CHECK_POISON(ctx);
    const long long n_rows = m->n;
    if (n_rows == 0) return ARROW_OK;
    const int k = D->k;
    const bool bf = D->dtype == ARROW_DTYPE_BF16;
    const int per_vec = bf ? Elt<bf16>::PER_VEC : Elt<float>::PER_VEC;
    const bool vec = (k % per_vec == 0);
    const int vpr = vec ? k / per_vec : k;
    int g = 1;
    while (g < vpr && g < 32) g <<= 1;                       // lanes per row
    if (g > 8 && vpr <= 32) g = 8;                           // 8 lanes x 4 vectors cover k <= 128 in one pass
    const int threads = 256;
    const long long rows_per_cta = (threads / 32) * (32 / g);
    int grid = (int)std::min<long long>((n_rows + rows_per_cta - 1) / rows_per_cta, (long long)ctx->sm_count * 8);
    grid = std::max(grid, 1);
#define LAUNCH_GA(T, VT, GG, ACCV, MULTIV)                                                                       \
    k_gather_rows<T, VT, GG, ACCV, MULTIV><<<grid, threads, 0, cur_stream(ctx)>>>(reinterpret_cast<VT *>(D->p),  \
                                                                           reinterpret_cast<const VT *>(src), ms, m->p, n_rows, vpr)
#define DISPATCH_G(T, VT, ACCV, MULTIV)                                                                          \
    do {                                                                                                         \
        switch (g) {                                                                                             \
            case 1: LAUNCH_GA(T, VT, 1, ACCV, MULTIV); break;                                                    \
            case 2: LAUNCH_GA(T, VT, 2, ACCV, MULTIV); break;                                                    \
            case 4: LAUNCH_GA(T, VT, 4, ACCV, MULTIV); break;                                                    \
            case 8: LAUNCH_GA(T, VT, 8, ACCV, MULTIV); break;                                                    \
            case 16: LAUNCH_GA(T, VT, 16, ACCV, MULTIV); break;                                                  \
            default: LAUNCH_GA(T, VT, 32, ACCV, MULTIV); break;                                                  \
        }                                                                                                        \
    } while (0)
    if (bf) {                           // one-GPU exchanges only (arrow_gather_rows_multi refuses bf16)
        if (vec) { if (acc) DISPATCH_G(bf16, float4, true, false); else DISPATCH_G(bf16, float4, false, false); }
        else     { if (acc) DISPATCH_G(bf16, bf16, true, false); else DISPATCH_G(bf16, bf16, false, false); }
    } else if (vec) {
        if (multi) { if (acc) DISPATCH_G(float, float4, true, true); else DISPATCH_G(float, float4, false, true); }
        else       { if (acc) DISPATCH_G(float, float4, true, false); else DISPATCH_G(float, float4, false, false); }
    } else {
        if (multi) { if (acc) DISPATCH_G(float, float, true, true); else DISPATCH_G(float, float, false, true); }
        else       { if (acc) DISPATCH_G(float, float, true, false); else DISPATCH_G(float, float, false, false); }
    }
#undef DISPATCH_G
#undef LAUNCH_GA
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return ARROW_OK;
}

int arrow_gather_rows(arrow_ctx *ctx, int dst_buf, int src_buf, int map, int flags) {
    CHECK_CTX(ctx);
    DenseBuf *D = get_dense(ctx, dst_buf), *S = get_dense(ctx, src_buf);
    IdxMap *m = get_map(ctx, map);
    if (!D || !S) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle (dst=%d src=%d)", dst_buf, src_buf);
    if (!m) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (D->k != S->k) return fail(ctx, ARROW_ERR_ARG, "feature width mismatch %d vs %d", D->k, S->k);
    if (D->dtype != S->dtype) return fail(ctx, ARROW_ERR_ARG, "gather source and destination differ in dtype (%d vs %d)", S->dtype, D->dtype);
    if (D->p == S->p) return fail(ctx, ARROW_ERR_ARG, "gather source and destination must not alias");
    if (m->n > D->rows) return fail(ctx, ARROW_ERR_ARG, "map has %lld entries, destination has %lld rows", (long long)m->n, (long long)D->rows);
    if (m->limit > S->rows) return fail(ctx, ARROW_ERR_ARG, "map reaches row %lld, source has %lld rows", (long long)m->limit, (long long)S->rows);
    MultiSrc ms;
    memset(&ms, 0, sizeof ms);
    return gather_common(ctx, D, S->p, ms, false, m, (flags & ARROW_ACCUMULATE) != 0);
}

int arrow_gather_rows_multi(arrow_ctx *ctx, int dst_buf, const int *src_bufs, const int64_t *row_bounds, int n_src, int map, int flags) {
    CHECK_CTX(ctx);
    DenseBuf *D = get_dense(ctx, dst_buf);
    IdxMap *m = get_map(ctx, map);
    if (!D) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", dst_buf);
    if (!m) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (!src_bufs || !row_bounds || n_src < 1 || n_src > MAX_SRC) return fail(ctx, ARROW_ERR_ARG, "need 1..%d sources", MAX_SRC);
    REQUIRE_F32(ctx, D, "arrow_gather_rows_multi (N-GPU path)");
    if (m->n > D->rows) return fail(ctx, ARROW_ERR_ARG, "map has %lld entries, destination has %lld rows", (long long)m->n, (long long)D->rows);
    MultiSrc ms;
    memset(&ms, 0, sizeof ms);
    ms.n = n_src;
    for (int s = 0; s < n_src; ++s) {
        DenseBuf *S = get_dense(ctx, src_bufs[s]);
        if (!S) return fail(ctx, ARROW_ERR_HANDLE, "bad source handle %d", src_bufs[s]);
        if (S->k != D->k) return fail(ctx, ARROW_ERR_ARG, "feature width mismatch in source %d", s);
        REQUIRE_F32(ctx, S, "arrow_gather_rows_multi (N-GPU path)");
        if (row_bounds[s + 1] < row_bounds[s] || row_bounds[s + 1] - row_bounds[s] > S->rows)
            return fail(ctx, ARROW_ERR_ARG, "source %d owns %lld rows but its tile has %lld", s, (long long)(row_bounds[s + 1] - row_bounds[s]), (long long)S->rows);
        if (S->p == D->p) return fail(ctx, ARROW_ERR_ARG, "gather source and destination must not alias");
        ms.p[s] = S->p;
        ms.bound[s] = row_bounds[s];
    }
    ms.bound[n_src] = row_bounds[n_src];
    if (m->limit > row_bounds[n_src]) return fail(ctx, ARROW_ERR_ARG, "map reaches row %lld beyond the last source bound %lld", (long long)m->limit, (long long)row_bounds[n_src]);
    return gather_common(ctx, D, nullptr, ms, true, m, (flags & ARROW_ACCUMULATE) != 0);
}

int arrow_push_rows(arrow_ctx *ctx, const int *dst_bufs, const int64_t *item_bounds, int n_dst, int src_buf, int map) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    DenseBuf *S = get_dense(ctx, src_buf);
    IdxMap *m = get_map(ctx, map);
    if (!S) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", src_buf);
    if (!m) return fail(ctx, ARROW_ERR_HANDLE, "bad map handle %d", map);
    if (!dst_bufs || !item_bounds || n_dst < 1 || n_dst > MAX_SRC) return fail(ctx, ARROW_ERR_ARG, "need 1..%d destinations", MAX_SRC);
    REQUIRE_F32(ctx, S, "arrow_push_rows (N-GPU path)");
    if (m->limit > S->rows) return fail(ctx, ARROW_ERR_ARG, "map reaches row %lld, source has %lld rows", (long long)m->limit, (long long)S->rows);
    if (item_bounds[0] != 0 || item_bounds[n_dst] != m->n) return fail(ctx, ARROW_ERR_ARG, "item bounds must span [0, %lld]", (long long)m->n);
    MultiDst md;
    memset(&md, 0, sizeof md);
    md.n = n_dst;
    for (int d = 0; d < n_dst; ++d) {
        const int64_t cnt = item_bounds[d + 1] - item_bounds[d];
        if (cnt < 0) return fail(ctx, ARROW_ERR_ARG, "item bounds must not decrease");
        md.bound[d] = item_bounds[d];
        if (cnt == 0) { md.p[d] = nullptr; continue; }
        DenseBuf *D = get_dense(ctx, dst_bufs[d]);
        if (!D) return fail(ctx, ARROW_ERR_HANDLE, "bad destination handle %d", dst_bufs[d]);
        if (D->k != S->k) return fail(ctx, ARROW_ERR_ARG, "feature width mismatch in destination %d", d);
        REQUIRE_F32(ctx, D, "arrow_push_rows (N-GPU path)");
        if (cnt > D->rows) return fail(ctx, ARROW_ERR_ARG, "destination %d receives %lld rows but its region has %lld", d, (long long)cnt, (long long)D->rows);
        if (D->p == S->p) return fail(ctx, ARROW_ERR_ARG, "push source and destination must not alias");
        md.p[d] = D->p;
    }
    md.bound[n_dst] = item_bounds[n_dst];
    md.max_len = 0;
    if (ctx->push_interleave && n_dst > 1)
        for (int d = 0; d < n_dst; ++d) md.max_len = std::max<long long>(md.max_len, md.bound[d + 1] - md.bound[d]);
    const long long n_items = m->n;
    if (n_items == 0) return ARROW_OK;
    const int k = S->k;
    const bool vec = (k % 4 == 0);
    const int vpr = vec ? k / 4 : k;
    int g = 1;
    while (g < vpr && g < 32) g <<= 1;
    if (g > 8 && vpr <= 32) g = 8;
    const int threads = 256;
    const long long rows_per_cta = (threads / 32) * (32 / g);
    const long long want = ctx->push_ctas > 0 ? ctx->push_ctas : (long long)ctx->sm_count * 2;
    int grid = (int)std::max<long long>(1, std::min<long long>((n_items + rows_per_cta - 1) / rows_per_cta, want));
#define LAUNCH_PU(VT, GG) k_push_rows<VT, GG><<<grid, threads, 0, cur_stream(ctx)>>>(md, reinterpret_cast<const VT *>(S->p), m->p, n_items, vpr)
#define DISPATCH_PU(VT)                                                                                          \
    do {                                                                                                         \
        switch (g) {                                                                                             \
            case 1: LAUNCH_PU(VT, 1); break;                                                                     \
            case 2: LAUNCH_PU(VT, 2); break;                                                                     \
            case 4: LAUNCH_PU(VT, 4); break;                                                                     \
            case 8: LAUNCH_PU(VT, 8); break;                                                                     \
            case 16: LAUNCH_PU(VT, 16); break;                                                                   \
            default: LAUNCH_PU(VT, 32); break;                                                                   \
        }                                                                                                        \
    } while (0)
    if (vec) DISPATCH_PU(float4); else DISPATCH_PU(float);
#undef DISPATCH_PU
#undef LAUNCH_PU
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return ARROW_OK;
}

int arrow_reduce_rows(arrow_ctx *ctx, int dst_buf, int out_table, const int *src_bufs, int n_src, int64_t rows) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    if (!src_bufs || n_src < 1 || n_src > MAX_SRC || rows < 0) return fail(ctx, ARROW_ERR_ARG, "need 1..%d sources", MAX_SRC);
    DenseBuf *D = dst_buf >= 0 ? get_dense(ctx, dst_buf) : nullptr;
    if (dst_buf >= 0 && !D) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", dst_buf);
    if (D) REQUIRE_F32(ctx, D, "arrow_reduce_rows (N-GPU path)");
    PtrTable *OT = nullptr;
    if (out_table >= 0) {
        if (out_table >= (int)ctx->ptrtabs.size() || !ctx->ptrtabs[out_table].live)
            return fail(ctx, ARROW_ERR_HANDLE, "bad pointer table handle %d", out_table);
        OT = &ctx->ptrtabs[out_table];
        if (OT->n < rows) return fail(ctx, ARROW_ERR_ARG, "pointer table has %lld entries, %lld rows are reduced", (long long)OT->n, (long long)rows);
    }
    if (!D && !OT) return fail(ctx, ARROW_ERR_ARG, "no destination");
    if (D && D->rows < rows) return fail(ctx, ARROW_ERR_ARG, "destination has %lld rows, %lld are reduced", (long long)D->rows, (long long)rows);
    MultiSrc ms;
    memset(&ms, 0, sizeof ms);
    ms.n = n_src;
    int k = 0;
    for (int s2 = 0; s2 < n_src; ++s2) {
        DenseBuf *S = get_dense(ctx, src_bufs[s2]);
        if (!S) return fail(ctx, ARROW_ERR_HANDLE, "bad source handle %d", src_bufs[s2]);
        if (s2 == 0) k = S->k;
        REQUIRE_F32(ctx, S, "arrow_reduce_rows (N-GPU path)");
        if (S->k != k || (D && D->k != k) || (OT && OT->k != k)) return fail(ctx, ARROW_ERR_ARG, "feature width mismatch in source %d", s2);
        if (S->rows < rows) return fail(ctx, ARROW_ERR_ARG, "source %d has %lld rows, %lld are reduced", s2, (long long)S->rows, (long long)rows);
        ms.p[s2] = S->p;
    }
    if (rows == 0) return ARROW_OK;
    const bool vec = (k % 4 == 0);
    const int vpr = vec ? k / 4 : k;
    const long long total = rows * vpr;
    const int grid = (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 4));
    float *const *tab = OT ? OT->p : nullptr;
    if (vec) k_reduce_rows<float4><<<grid, 256, 0, cur_stream(ctx)>>>(D ? reinterpret_cast<float4 *>(D->p) : nullptr, tab, ms, rows, vpr);
    else k_reduce_rows<float><<<grid, 256, 0, cur_stream(ctx)>>>(D ? D->p : nullptr, tab, ms, rows, vpr);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return ARROW_OK;
}

// ---- IPC / peer barrier -------------------------------------------------------------------------
// cudaIpcGetMemHandle names the whole underlying allocation; a pointer that was sub-allocated inside a larger
// driver block must be re-based on the importing side.  The base comes from the driver (cuMemGetAddressRange),
// resolved at run time so the library does not link libcuda.
static long long ipc_base_offset(void *ptr) {
    typedef int (*range_fn)(unsigned long long *, size_t *, unsigned long long);
    static range_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *h = dlopen("libcuda.so.1", RTLD_LAZY | RTLD_GLOBAL);
        if (h) fn = (range_fn)dlsym(h, "cuMemGetAddressRange_v2");
    }
    if (!fn) return 0;
    unsigned long long base = 0;
    size_t size = 0;
    if (fn(&base, &size, (unsigned long long)ptr) != 0) return 0;
    return (long long)((unsigned long long)ptr - base);
}

int arrow_ipc_export(arrow_ctx *ctx, int buf, void *handle) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d || !d->owned) return fail(ctx, ARROW_ERR_HANDLE, "ipc export needs a tile this context allocated (handle %d)", buf);
    if (!handle) return fail(ctx, ARROW_ERR_ARG, "handle is null");
    REQUIRE_F32(ctx, d, "arrow_ipc_export (N-GPU path)");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
    cudaIpcMemHandle_t h;
    CUDA_TRY(ctx, cudaIpcGetMemHandle(&h, d->p));
    memset(handle, 0, ARROW_IPC_HANDLE_BYTES);
    memcpy(handle, &h, sizeof h);
    const long long off = ipc_base_offset(d->p);
    memcpy((char *)handle + 64, &off, sizeof off);
    return ARROW_OK;
}

int arrow_ipc_import(arrow_ctx *ctx, const void *handle, int64_t rows, int k, int *buf_out) {
    CHECK_CTX(ctx);
    if (!handle || !buf_out || rows < 0 || k < 1) return fail(ctx, ARROW_ERR_ARG, "bad ipc import arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    long long off = 0;
    memcpy(&off, (const char *)handle + 64, sizeof off);
    void *p = nullptr;
    CUDA_TRY(ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    DenseBuf d;
    d.p = (float *)((char *)p + off);
    d.ipc_base = p;
    d.rows = rows;
    d.k = k;
    d.ipc = true;
    d.live = true;
    const int hh = new_slot(ctx->dense);
    ctx->dense[hh] = d;
    *buf_out = hh;
    return ARROW_OK;
}

int arrow_peer_barrier(arrow_ctx *ctx, const int *flag_bufs, int rank, int world) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    if (!flag_bufs || world < 1 || world > MAX_SRC || rank < 0 || rank >= world) return fail(ctx, ARROW_ERR_ARG, "bad barrier arguments");
    PeerFlags pf;
    memset(&pf, 0, sizeof pf);
    for (int s = 0; s < world; ++s) {
        DenseBuf *d = get_dense(ctx, flag_bufs[s]);
        if (!d || (long long)d->rows * d->k < world) return fail(ctx, ARROW_ERR_HANDLE, "bad flag tile for rank %d", s);
        pf.p[s] = reinterpret_cast<unsigned int *>(d->p);
    }
    const long long timeout_clocks = ctx->barrier_timeout_ms * (long long)ctx->clock_khz;
    k_peer_barrier<<<1, 32, 0, cur_stream(ctx)>>>(pf, rank, world, ctx->barrier_epoch + ctx->cur_lane, ctx->dev_status, timeout_clocks);
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return ARROW_OK;
}

// ---- lanes: side streams ordered against the main stream with events ---------------------------------
static int lane_stream(arrow_ctx *ctx, int lane, cudaStream_t *out);

int arrow_set_lane(arrow_ctx *ctx, int lane) {
    CHECK_CTX(ctx);
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);          // creates the stream on first use
    if (rc != ARROW_OK) return rc;
    ctx->cur_lane = lane;
    return ARROW_OK;
}

static int lane_stream(arrow_ctx *ctx, int lane, cudaStream_t *out) {
    if (lane < 0 || lane >= ARROW_N_LANES) return fail(ctx, ARROW_ERR_ARG, "lane %d out of range", lane);
    if (lane == ARROW_LANE_MAIN) { *out = ctx->stream; return ARROW_OK; }
    if (!ctx->lanes[lane]) CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->lanes[lane], cudaStreamNonBlocking));
    *out = ctx->lanes[lane];
    return ARROW_OK;
}

int arrow_dense_h2d_lane(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, const float *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows) return fail(ctx, ARROW_ERR_ARG, "h2d range outside tile");
    REQUIRE_F32(ctx, d, "arrow_dense_h2d_lane (float rows; arrow_dense_put copies any dtype)");
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    if (rows) CUDA_TRY(ctx, cudaMemcpyAsync(d->p + (size_t)row0 * d->k, host, (size_t)rows * d->k * 4, cudaMemcpyHostToDevice, st));
    return ARROW_OK;
}

int arrow_dense_d2h_lane(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, float *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows) return fail(ctx, ARROW_ERR_ARG, "d2h range outside tile");
    REQUIRE_F32(ctx, d, "arrow_dense_d2h_lane (float rows; arrow_dense_get copies any dtype)");
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    if (rows) CUDA_TRY(ctx, cudaMemcpyAsync(host, d->p + (size_t)row0 * d->k, (size_t)rows * d->k * 4, cudaMemcpyDeviceToHost, st));
    return ARROW_OK;
}

int arrow_dense_put(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, const void *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows)
        return fail(ctx, ARROW_ERR_ARG, "put rows [%lld,%lld) outside tile of %lld rows", (long long)row0, (long long)(row0 + rows), (long long)d->rows);
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    if (rows) CUDA_TRY(ctx, cudaMemcpyAsync(d->row(row0), host, (size_t)rows * d->k * d->esize(), cudaMemcpyHostToDevice, st));
    return ARROW_OK;
}

int arrow_dense_get(arrow_ctx *ctx, int lane, int buf, int64_t row0, int64_t rows, void *host) {
    CHECK_CTX(ctx);
    DenseBuf *d = get_dense(ctx, buf);
    if (!d) return fail(ctx, ARROW_ERR_HANDLE, "bad dense handle %d", buf);
    if (!host || row0 < 0 || rows < 0 || row0 + rows > d->rows)
        return fail(ctx, ARROW_ERR_ARG, "get rows [%lld,%lld) outside tile of %lld rows", (long long)row0, (long long)(row0 + rows), (long long)d->rows);
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    if (rows) CUDA_TRY(ctx, cudaMemcpyAsync(host, d->row(row0), (size_t)rows * d->k * d->esize(), cudaMemcpyDeviceToHost, st));
    return ARROW_OK;
}

int arrow_lane_wait(arrow_ctx *ctx, int waiting_lane, int signalling_lane) {
    CHECK_CTX(ctx);
    cudaStream_t w, sgn;
    int rc = lane_stream(ctx, waiting_lane, &w);
    if (rc != ARROW_OK) return rc;
    rc = lane_stream(ctx, signalling_lane, &sgn);
    if (rc != ARROW_OK) return rc;
    if (w == sgn) return ARROW_OK;
    cudaEvent_t &ev = ctx->lane_events[signalling_lane];
    if (!ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CUDA_TRY(ctx, cudaEventRecord(ev, sgn));
    CUDA_TRY(ctx, cudaStreamWaitEvent(w, ev, 0));
    return ARROW_OK;
}

int arrow_event_record(arrow_ctx *ctx, int event, int lane) {
    CHECK_CTX(ctx);
    if (event < 0 || event >= ARROW_MAX_EVENTS) return fail(ctx, ARROW_ERR_ARG, "event %d out of range", event);
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    if (!ctx->user_events[event]) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->user_events[event], cudaEventDisableTiming));
    CUDA_TRY(ctx, cudaEventRecord(ctx->user_events[event], st));
    return ARROW_OK;
}

int arrow_event_wait(arrow_ctx *ctx, int event, int lane) {
    CHECK_CTX(ctx);
    if (event < 0 || event >= ARROW_MAX_EVENTS) return fail(ctx, ARROW_ERR_ARG, "event %d out of range", event);
    if (!ctx->user_events[event]) return ARROW_OK;            // never recorded: nothing to wait for
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->user_events[event], 0));
    return ARROW_OK;
}

int arrow_lane_sync(arrow_ctx *ctx, int lane) {
    CHECK_CTX(ctx);
    cudaStream_t st;
    int rc = lane_stream(ctx, lane, &st);
    if (rc != ARROW_OK) return rc;
    CUDA_TRY(ctx, cudaStreamSynchronize(st));
    int flag = 0;
    CUDA_TRY(ctx, cudaMemcpy(&flag, ctx->dev_status, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag != 0) {
        ctx->poisoned = true;
        return fail(ctx, ARROW_ERR_CUDA, "device-side failure flag %d: a peer barrier timed out after %lld ms; the context is "
                    "poisoned (results after the time-out are racy) -- destroy it", flag, ctx->barrier_timeout_ms);
    }
    return ARROW_OK;
}

// ---- CUDA graphs: one host call per step ---------------------------------------------------------------
// Everything between begin and end is recorded instead of executed: launches on the main lane and on every lane that
// joined through arrow_lane_wait / arrow_event_wait (fork) and was joined back before the end.  Device-side state
// (tile tickets, barrier epochs) lives in device memory, so the recorded step can be replayed any number of times.
int arrow_graph_begin(arrow_ctx *ctx) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    if (ctx->capturing) return fail(ctx, ARROW_ERR_ARG, "a capture is already in progress");
    CUDA_TRY(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
    ctx->capturing = true;
    ctx->capture_launches0 = ctx->launches;
    ctx->cur_lane = 0;
    return ARROW_OK;
}

int arrow_graph_end(arrow_ctx *ctx, int *graph_out) {
    CHECK_CTX(ctx);
    if (!ctx->capturing) return fail(ctx, ARROW_ERR_ARG, "no capture in progress");
    ctx->capturing = false;
    const int64_t recorded = ctx->launches - ctx->capture_launches0;
    ctx->launches = ctx->capture_launches0;                  // recorded, not executed
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
    if (e != cudaSuccess || !g) {
        cudaGetLastError();
        return fail(ctx, ARROW_ERR_CUDA, "cudaStreamEndCapture: %s (was every side lane joined back into the main lane?)", cudaGetErrorString(e));
    }
    cudaGraphExec_t ex = nullptr;
    e = cudaGraphInstantiate(&ex, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, ARROW_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
    }
    if (!graph_out) { cudaGraphExecDestroy(ex); return fail(ctx, ARROW_ERR_ARG, "graph_out is null"); }
    int h = -1;
    for (size_t i = 0; i < ctx->graphs.size(); ++i)
        if (!ctx->graphs[i]) { h = (int)i; break; }
    if (h < 0) { ctx->graphs.push_back(nullptr); ctx->graph_kernels.push_back(0); h = (int)ctx->graphs.size() - 1; }
    ctx->graphs[h] = ex;
    ctx->graph_kernels[h] = recorded;
    *graph_out = h;
    return ARROW_OK;
}

int arrow_graph_launch(arrow_ctx *ctx, int graph) {
    CHECK_CTX(ctx);
    CHECK_POISON(ctx);
    if (graph < 0 || graph >= (int)ctx->graphs.size() || !ctx->graphs[graph]) return fail(ctx, ARROW_ERR_HANDLE, "bad graph handle %d", graph);
    if (ctx->capturing) return fail(ctx, ARROW_ERR_ARG, "cannot launch a graph while capturing");
    CUDA_TRY(ctx, cudaGraphLaunch(ctx->graphs[graph], ctx->stream));
    ctx->launches += ctx->graph_kernels[graph];
    return ARROW_OK;
}

int arrow_graph_free(arrow_ctx *ctx, int graph) {
    CHECK_CTX(ctx);
    if (graph < 0 || graph >= (int)ctx->graphs.size() || !ctx->graphs[graph]) return fail(ctx, ARROW_ERR_HANDLE, "bad graph handle %d", graph);
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    cudaGraphExecDestroy(ctx->graphs[graph]);
    ctx->graphs[graph] = nullptr;
    if (!graphs_live(ctx)) {                                  // no replay can address a retired scratch buffer any more
        for (float *p : ctx->retired_scratch) cudaFree(p);
        ctx->retired_scratch.clear();
    }
    return ARROW_OK;
}

// ---- host memory next to the GPU --------------------------------------------------------------------------
// On a two-socket HGX box GPUs 0-3 hang off socket 0 and 4-7 off socket 1: staging buffers that live on the other
// socket cross the inter-socket link on every copy (round 1: 33 GB/s per GPU at N=4 vs 84 GB/s at N=1).  These calls
// pin the calling thread to the CPUs of the GPU's NUMA node and place the pinned buffer there.
static int numa_node_of_device(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char *c = bus; *c; ++c) *c = (char)tolower(*c);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE *f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

int arrow_bind_thread_to_device_numa(int device, int *node_out, int *n_cpus_out) {
    if (device < 0) {                                    // undo: every CPU, default memory policy
        cpu_set_t all;
        CPU_ZERO(&all);
        for (int c = 0; c < CPU_SETSIZE; ++c) CPU_SET(c, &all);
        sched_setaffinity(0, sizeof all, &all);
        syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0);
        if (node_out) *node_out = -1;
        if (n_cpus_out) *n_cpus_out = 0;
        return ARROW_OK;
    }
    int node = numa_node_of_device(device);
    if (node_out) *node_out = node;
    if (n_cpus_out) *n_cpus_out = 0;
    if (node < 0) return ARROW_OK;                       // single-node machine or unknown topology: nothing to do
    char path[128];
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    FILE *f = fopen(path, "r");
    if (!f) return ARROW_OK;
    char buf[4096] = {0};
    const size_t got = fread(buf, 1, sizeof buf - 1, f);
    fclose(f);
    buf[got] = 0;
    cpu_set_t set;
    CPU_ZERO(&set);
    int n = 0;
    for (char *tok = strtok(buf, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int a = 0, b = 0;
        if (sscanf(tok, "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, &set); ++n; } }
        else if (sscanf(tok, "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, &set); ++n; }
    }
    if (n > 0 && sched_setaffinity(0, sizeof set, &set) == 0) {
        if (n_cpus_out) *n_cpus_out = n;
        unsigned long mask[16] = {0};
        if (node < (int)(sizeof mask * 8)) {
            mask[node / (8 * sizeof(unsigned long))] |= 1UL << (node % (8 * sizeof(unsigned long)));
            syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, sizeof mask * 8);
        }
    }
    return ARROW_OK;
}

int arrow_host_alloc_numa(size_t bytes, int device, void **ptr) {
    if (!ptr) return ARROW_ERR_ARG;
    *ptr = nullptr;
    const size_t page = 2u << 20;
    const size_t len = ((std::max<size_t>(bytes, 16) + page - 1) / page) * page;
    void *p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return fail(nullptr, ARROW_ERR_NOMEM, "mmap(%zu) failed", len);
    madvise(p, len, MADV_HUGEPAGE);
    const int node = numa_node_of_device(device);
    if (node >= 0) {
        unsigned long mask[16] = {0};
        if (node < (int)(sizeof mask * 8)) {
            mask[node / (8 * sizeof(unsigned long))] |= 1UL << (node % (8 * sizeof(unsigned long)));
            syscall(SYS_mbind, p, len, 2 /* MPOL_BIND */, mask, sizeof mask * 8, 0);      // best effort
        }
    }
    memset(p, 0, len);                                   // first touch: pages materialise on the bound node
    cudaError_t e = cudaHostRegister(p, len, cudaHostRegisterPortable);
    if (e != cudaSuccess) {
        cudaGetLastError();
        munmap(p, len);
        return fail(nullptr, ARROW_ERR_NOMEM, "cudaHostRegister(%zu): %s", len, cudaGetErrorString(e));
    }
    {
        std::lock_guard<std::mutex> lk(g_numa_mu);
        g_numa_allocs[p] = len;
    }
    *ptr = p;
    return ARROW_OK;
}

// ---- timing -------------------------------------------------------------------------------------
int arrow_timer_start(arrow_ctx *ctx, int slot) {
    CHECK_CTX(ctx);
    if (slot < 0 || slot >= ARROW_MAX_TIMERS) return fail(ctx, ARROW_ERR_ARG, "timer slot %d", slot);
    Timer &t = ctx->timers[slot];
    if (!t.a) CUDA_TRY(ctx, cudaEventCreate(&t.a));
    if (!t.b) CUDA_TRY(ctx, cudaEventCreate(&t.b));
    CUDA_TRY(ctx, cudaEventRecord(t.a, ctx->stream));
    return ARROW_OK;
}

int arrow_timer_stop(arrow_ctx *ctx, int slot) {
    CHECK_CTX(ctx);
    if (slot < 0 || slot >= ARROW_MAX_TIMERS || !ctx->timers[slot].b) return fail(ctx, ARROW_ERR_ARG, "timer slot %d not started", slot);
    CUDA_TRY(ctx, cudaEventRecord(ctx->timers[slot].b, ctx->stream));
    return ARROW_OK;
}

int arrow_timer_elapsed_ms(arrow_ctx *ctx, int slot, float *ms) {
    CHECK_CTX(ctx);
    if (slot < 0 || slot >= ARROW_MAX_TIMERS || !ctx->timers[slot].b || !ms) return fail(ctx, ARROW_ERR_ARG, "timer slot %d not started", slot);
    CUDA_TRY(ctx, cudaEventSynchronize(ctx->timers[slot].b));
    CUDA_TRY(ctx, cudaEventElapsedTime(ms, ctx->timers[slot].a, ctx->timers[slot].b));
    return ARROW_OK;
}

int arrow_launch_count(arrow_ctx *ctx, int64_t *count) {
    if (!ctx || !count) return ARROW_ERR_ARG;
    *count = ctx->launches;
    return ARROW_OK;
}

// Lazy module loading (the CUDA default) loads a kernel at its first launch, and loading synchronises the context.  A
// kernel that spin-waits -- arrow_peer_barrier on one lane -- while another lane (or, with rank threads, another
// rank) launches a kernel for the first time therefore deadlocks until the barrier times out.  This runs every kernel
// the step of a given feature width can launch once, on tiny operands, before any barrier is in flight.
int arrow_preload_kernels(arrow_ctx *ctx, int k) {
    CHECK_CTX(ctx);
    if (k < 1) return fail(ctx, ARROW_ERR_ARG, "k must be positive");
    const int64_t n = 700;
    std::vector<int32_t> ip(n + 1), ix;
    std::vector<float> val;
    for (int64_t r = 0; r < n; ++r) {
        ip[r] = (int32_t)ix.size();
        const int len = (r == 3) ? 600 : 3;                       // one long row: the segmented kernels load too
        for (int j = 0; j < len; ++j) { ix.push_back((int32_t)((r * 7 + j) % n)); val.push_back(1.0f); }
        std::sort(ix.begin() + ip[r], ix.end());
        ix.erase(std::unique(ix.begin() + ip[r], ix.end()), ix.end());
        val.resize(ix.size());
    }
    ip[n] = (int32_t)ix.size();
    int csr = -1, x = -1, x2 = -1, c = -1, c2 = -1, map = -1, tab = -1, rc = ARROW_OK;
    std::vector<int64_t> ident(n);
    for (int64_t i = 0; i < n; ++i) ident[i] = i;
    std::vector<int32_t> which(n, 0);
    const int saved_kernel = ctx->tile_kernel, saved_lane = ctx->cur_lane;
    ctx->cur_lane = 0;
#define PRE(expr) do { if (rc == ARROW_OK) rc = (expr); } while (0)
    PRE(arrow_csr_upload(ctx, n, n, (int64_t)ix.size(), ip.data(), 4, ix.data(), 4, val.data(), &csr));
    PRE(arrow_dense_alloc(ctx, n, k, &x));
    PRE(arrow_dense_alloc(ctx, n, k, &x2));
    PRE(arrow_dense_alloc(ctx, n, k, &c));
    PRE(arrow_dense_alloc(ctx, n, k, &c2));
    PRE(arrow_map_upload(ctx, ident.data(), n, n, &map));
    if (rc == ARROW_OK) { const int tiles[1] = {c2}; rc = arrow_ptrtable_upload(ctx, tiles, 1, which.data(), ident.data(), n, &tab); }
    for (int tk = 0; tk < 2 && rc == ARROW_OK; ++tk) {
        ctx->tile_kernel = tk;
        for (int rpg = 1; rpg <= 2; ++rpg) {
            const int variant = ARROW_VARIANT_TILES | (rpg << 8);
            PRE(arrow_spmm(ctx, csr, x, c, -1, 0, variant));
            PRE(arrow_spmm(ctx, csr, x, c, -1, ARROW_ACCUMULATE, variant));
            PRE(arrow_spmm(ctx, csr, x, c, map, 0, variant));
            PRE(arrow_spmm(ctx, csr, x, c, map, ARROW_ACCUMULATE, variant));
            PRE(arrow_spmm_add(ctx, csr, x, c, c2, map, variant));
            PRE(arrow_spmm_ex(ctx, csr, x, x2, n / 2, c, -1, -1, -1, variant));
            PRE(arrow_spmm_ex(ctx, csr, x, x2, n / 2, -1, tab, -1, -1, variant));
            PRE(arrow_spmm_ex(ctx, csr, x, -1, 0, -1, tab, c, map, variant));
        }
    }
    ctx->tile_kernel = saved_kernel;
    PRE(arrow_gather_rows(ctx, c, x, map, 0));
    PRE(arrow_gather_rows(ctx, c, x, map, ARROW_ACCUMULATE));
    if (rc == ARROW_OK) {
        const int srcs[1] = {x};
        const int64_t bounds[2] = {0, n};
        PRE(arrow_gather_rows_multi(ctx, c, srcs, bounds, 1, map, 0));
        PRE(arrow_gather_rows_multi(ctx, c, srcs, bounds, 1, map, ARROW_ACCUMULATE));
        const int dsts[1] = {c};
        PRE(arrow_push_rows(ctx, dsts, bounds, 1, x, map));
        PRE(arrow_reduce_rows(ctx, c, -1, srcs, 1, n));
        PRE(arrow_reduce_rows(ctx, -1, tab, srcs, 1, n));
        PRE(arrow_dense_fill(ctx, c, 1.0f));
        // the barrier kernel against this context's own flag word (world of one): loads it, never waits
        const int flags[1] = {c};
        for (int lane = 0; lane < ARROW_N_LANES && rc == ARROW_OK; lane += ARROW_LANE_SIDE) {
            cudaStream_t st;
            rc = lane_stream(ctx, lane, &st);
            ctx->cur_lane = lane;
            if (lane) PRE(arrow_lane_wait(ctx, lane, 0));
            PRE(arrow_dense_fill(ctx, c, 0.0f));
            PRE(arrow_peer_barrier(ctx, flags, 0, 1));
            if (lane) PRE(arrow_lane_wait(ctx, 0, lane));
        }
    }
#undef PRE
    ctx->cur_lane = saved_lane;
    cudaStreamSynchronize(ctx->stream);
    for (int l = 1; l < ARROW_N_LANES; ++l)
        if (ctx->lanes[l]) cudaStreamSynchronize(ctx->lanes[l]);
    if (tab >= 0) arrow_ptrtable_free(ctx, tab);
    if (map >= 0) arrow_map_free(ctx, map);
    for (int h : {x, x2, c, c2}) if (h >= 0) arrow_dense_free(ctx, h);
    if (csr >= 0) arrow_csr_free(ctx, csr);
    // the barrier test bumped the epoch counters of a flag word that no longer exists: start clean
    cudaMemset(ctx->barrier_epoch, 0, ARROW_N_LANES * sizeof(unsigned int));
    return rc;
}

int arrow_l2_flush(arrow_ctx *ctx) {
    CHECK_CTX(ctx);
    const size_t bytes = (size_t)256 << 20;      // 256 MiB > 126 MB of L2
    if (!ctx->flush_buf) {
        CUDA_TRY(ctx, cudaMalloc(&ctx->flush_buf, bytes));
        ctx->flush_bytes = bytes;
    }
    k_fill<float><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((float *)ctx->flush_buf, 0.f, (long long)(ctx->flush_bytes / 4));
    ctx->launches++;
    CUDA_TRY(ctx, cudaGetLastError());
    return ARROW_OK;
}

}  // extern "C"

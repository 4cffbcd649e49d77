// bwts_b200.cu -- C ABI of libbwts_b200.so and the host-side drivers of the two hot paths.
//
// forward  (replaces /root/reference/mk_bwts_sa.c:47-52):  Lyndon boundaries -> packed
//          initial keys -> onesweep sort -> prefix-doubling rounds -> emit
// inverse  (replaces /root/reference/unbwts.c:31-86):      tile counts -> LF map -> splitter
//          walks -> reduced-list ranking -> offsets scan -> placement
// There is no CPU fallback anywhere in this file: without a device every call fails.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/bwts_b200.h"
#include "common.cuh"
#include "fm.cuh"
#include "forward.cuh"
#include "inverse.cuh"
#include "lcp.cuh"
#include "lz.cuh"
#include "lzd.cuh"
#include "lyndon.cuh"
#include "radix.cuh"
#include "scan.cuh"

#define BWTS_VERSION "bwts-b200 0.2 (sm_100a)"

enum KClass {
    KC_LYNDON = 0, KC_FACTORS, KC_INIT_KEYS, KC_RADIX_HIST, KC_ONESWEEP, KC_BUILD_KEYS, KC_RERANK, KC_EMIT,
    KC_INV_HIST, KC_INV_LF, KC_INV_WALK, KC_INV_JUMP, KC_INV_SCAN, KC_INV_PLACE, KC_LOCAL_SORT, KC_TUPLE
};
static const char *kclass_names[BWTS_B200_NCLASS] = {
    "lyndon", "factor_table", "init_keys", "radix_hist", "onesweep_pass", "build_keys", "rerank", "emit",
    "inv_tile_hist", "inv_lf_rank", "inv_walk", "inv_jump", "inv_scan", "inv_place", "local_sort", "tuple_round"};

static std::atomic<u32> g_epoch{0};  // onesweep status epoch, unique per pass across all contexts
static long g_tune_chunk = 0;      // Lyndon chunk bytes (0 = auto)
static long g_tune_spl_shift = 0;  // splitter shift   (0 = 26)
static long g_tune_onesweep = 0;   // onesweep tile configuration (see radix_sort)
static long g_tune_local = 0;      // 1 = never use the warp-local sort path
static long g_tune_lyndon = 0;     // 1 = always take the suffix-sort fallback for the Lyndon boundaries
static long g_tune_keybits = 0;    // cap on the bits of the initial packed key (0 = 64)
static long g_tune_emit = 0;       // emit: 0 = packed-binned from 512 Mi bytes, 1 = always rank windows, 2 = always packed-binned, 3 = always binned as (rank, byte) pairs
static long g_tune_nocta = 0;      // 1 = never use the CTA-local sort for the L set
static long g_tune_scatterbin = 0;  // first re-rank: 0 = bin the rank scatter when n >= 4 Mi, 1 = never, 2 = always
static long g_tune_l2gran = 0;     // cudaLimitMaxL2FetchGranularity applied when a transform starts (0 = leave the device's setting)
static long g_tune_hist = 0;       // 1 = digit histograms of the initial sort by k_radix_hist (eight shared atomics per key)
static long g_tune_partial = 0;    // 1 = initial keys of whole symbols only (no partial symbol in the spare bits)
static long g_tune_emitwin = 0;    // MiB of output per emit window (16..1024; 0 = 64)
static long g_tune_ctasort = 0;    // CTA-local sort: 0 = radix in shared memory, 1 = bitonic network (round 1)
static long g_tune_lyscan = 0;     // Lyndon chunk-minimum scan: 0 = Hillis-Steele levels under a probe budget, else CTA-wide; 1 / 2 = force either
static long g_tune_tmode = 0;      // tuple set: 0 = one thread per member (up to 8 members), 1 = one thread per group (up to 32)
static long g_tune_tmax = 0;       // tuple set: largest group it takes (0 = 8, 1 = set switched off, 2..32)
static long g_tune_invpath = 0;    // inverse: 0 = staged single walk (default), 1 = two read-only walks (round 1)
static long g_tune_invq = 0;       // inverse staged walk: sublists per warp (0 = auto: one full wave of warps)
static long g_tune_invmark = 0;    // inverse staged walk marks: 0 = by size (counts per 128 above 256 MiB), 1 = one bit per element, 2 = counts
static long g_tune_invbudget = 0;  // inverse fallback walks: step budget per attempt (0 = 32 n)
static long g_tune_nomark = 0;     // TIMING EXPERIMENT ONLY: inverse first walk without visited marks (wrong output when a cycle has no splitter)
static long g_tune_lcp = 0;        // LCP pairs: 0 = by length through the three tiers, 1 = all from the warp tier on, 2 = all through the multi-CTA tier
static long g_tune_lz = 0;         // LPF / LZ77 / LZ77 decoding: log2 of the tile and chunk width (5..12; 0 = 12)

static void apply_device_limits()
{
    if (g_tune_l2gran == 32 || g_tune_l2gran == 64 || g_tune_l2gran == 128)
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)g_tune_l2gran);
    if (getenv("BWTS_B200_TRACE")) {
        size_t g = 0;
        cudaDeviceGetLimit(&g, cudaLimitMaxL2FetchGranularity);
        fprintf(stderr, "[trace] cudaLimitMaxL2FetchGranularity = %zu\n", g);
    }
}

static bool use_binned_scatter(unsigned n, unsigned kb)
{
    if (g_tune_scatterbin == 1 || kb < 8) return false;
    return g_tune_scatterbin == 2 || g_tune_scatterbin == 4 || n >= (1u << 22);
}

struct LaunchRec { int cls; double bytes; cudaEvent_t e0, e1; const char *name; int phase; };

struct bwts_b200_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    u8 *arena = nullptr;
    size_t arena_bytes = 0, arena_used = 0;
    size_t io_end = 0;       // bytes at the bottom of the arena that hold the running call's I/O region (0: none)
    u32 *h_small = nullptr;  // pinned + mapped, 4 KiB, for counter read-backs
    u32 *h_small_dev = nullptr;  // its device-side address
    int last_cuda = 0;
    int phase = 0;           // phase the next launches are booked under (stats.phase_ms)
    bool profile = true;
    std::vector<LaunchRec> recs;
    std::vector<cudaEvent_t> pool;
    size_t pool_used = 0;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr, ev_io0 = nullptr, ev_io1 = nullptr;
    bwts_b200_stats stats;
    u32 epoch = 0;
    // block pipeline state, created on first use and kept: cudaMalloc / cudaFree of the GiB-sized
    // I/O slots cost 100-700 ms per call when something polls the driver (nvidia-smi -lms)
    u8 *pipe_io = nullptr;
    size_t pipe_io_bytes = 0;
    cudaStream_t pipe_s_in = nullptr, pipe_s_out = nullptr;
    cudaEvent_t pipe_ev_loaded[2] = {nullptr, nullptr};
    struct PinnedRing *pipe_ring_in = nullptr, *pipe_ring_out = nullptr;
};
static void pipe_state_destroy(bwts_b200_ctx *ctx);

#define CK(call)                                                                  \
    do {                                                                          \
        cudaError_t e__ = (call);                                                 \
        if (e__ != cudaSuccess) {                                                 \
            ctx->last_cuda = (int)e__;                                            \
            return (e__ == cudaErrorMemoryAllocation) ? BWTS_B200_ENOMEM : BWTS_B200_ECUDA; \
        }                                                                         \
    } while (0)

static cudaEvent_t ctx_event(bwts_b200_ctx *ctx)
{
    if (ctx->pool_used == ctx->pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ctx->pool.push_back(e);
    }
    return ctx->pool[ctx->pool_used++];
}

// BWTS_B200_SYNC=1 (debugging): wait for every kernel and name the one that failed
static cudaError_t launch_check(const char *name, cudaStream_t st)
{
    static const bool sync = getenv("BWTS_B200_SYNC") != nullptr;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && sync) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess && sync) fprintf(stderr, "[bwts_b200] kernel %s failed: %s\n", name, cudaGetErrorString(e));
    return e;
}

// LAUNCH_REC(class, algorithmic bytes, name, launch): books the launch statement under the current phase, between
// two events when profiling
#define LAUNCH_REC(KCLS_, NBYTES_, NAME_, ...)                                       \
    do {                                                                             \
        LaunchRec r__{(KCLS_), (double)(NBYTES_), nullptr, nullptr, (NAME_), ctx->phase}; \
        if (ctx->profile) { r__.e0 = ctx_event(ctx); if (r__.e0) cudaEventRecord(r__.e0, st); } \
        __VA_ARGS__;                                                                 \
        if (r__.e0) { r__.e1 = ctx_event(ctx); if (r__.e1) cudaEventRecord(r__.e1, st); } \
        ctx->recs.push_back(r__);                                                    \
        CK(launch_check((NAME_), st));                                               \
    } while (0)

// LAUNCH(class, algorithmic bytes, kernel, grid, block, args...)
#define LAUNCH(KCLS_, NBYTES_, kern, grid, block, ...) \
    LAUNCH_REC(KCLS_, NBYTES_, #kern, kern<<<(grid), (block), 0, st>>>(__VA_ARGS__))
#define LAUNCH_SMEM(KCLS_, NBYTES_, kern, grid, block, smem_, ...) \
    LAUNCH_REC(KCLS_, NBYTES_, #kern, kern<<<(grid), (block), (smem_), st>>>(__VA_ARGS__))

static void stats_begin(bwts_b200_ctx *ctx, long len, int direction, cudaStream_t st)
{
    memset(&ctx->stats, 0, sizeof ctx->stats);
    ctx->stats.len = len;
    ctx->stats.direction = direction;
    ctx->recs.clear();
    ctx->pool_used = 0;
    ctx->phase = 0;
    cudaEventRecord(ctx->ev_begin, st);
}
static void stats_end(bwts_b200_ctx *ctx, cudaStream_t st)
{
    cudaEventRecord(ctx->ev_end, st);
    cudaEventSynchronize(ctx->ev_end);
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end);
    ctx->stats.total_ms = ms;
    ctx->stats.arena_bytes = (long)ctx->arena_bytes;
    ctx->stats.launches = (long)ctx->recs.size();
    static const bool trace = getenv("BWTS_B200_TRACE") != nullptr;  // one line per launch to stderr
    int seq = 0;
    for (const LaunchRec &r : ctx->recs) {
        ctx->stats.class_launches[r.cls]++;
        ctx->stats.class_bytes[r.cls] += r.bytes;
        float t = 0;
        if (r.e0 && r.e1) {
            if (cudaEventElapsedTime(&t, r.e0, r.e1) == cudaSuccess) {
                ctx->stats.class_ms[r.cls] += t;
                if (r.phase >= 0 && r.phase < BWTS_B200_NPHASE) ctx->stats.phase_ms[r.phase] += t;
            }
        }
        if (trace)
            fprintf(stderr, "[trace %s n=%ld] %3d %-14s %-24s %9.4f ms %12.0f B %8.1f GB/s\n", ctx->stats.direction ? "inv" : "fwd",
                    ctx->stats.len, seq, kclass_names[r.cls], r.name, t, r.bytes, t > 0 ? r.bytes / t * 1e-6 : 0.0);
        seq++;
    }
}

// ---- arena ---------------------------------------------------------------------------------
static int arena_reserve(bwts_b200_ctx *ctx, size_t bytes)
{
    if (bytes <= ctx->arena_bytes) return 0;
    if (ctx->arena) { cudaFree(ctx->arena); ctx->arena = nullptr; ctx->arena_bytes = 0; }
    CK(cudaMalloc((void **)&ctx->arena, bytes));
    // no clearing: every array is written (or memset on the transform's stream) before it is read; the one
    // consumer of stale bytes, the look-back status region, is cleared per transform
    ctx->arena_bytes = bytes;
    return 0;
}
template <typename T>
static T *arena_take(bwts_b200_ctx *ctx, size_t count)
{
    size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
    if (ctx->arena_used + bytes > ctx->arena_bytes) return nullptr;
    T *p = (T *)(ctx->arena + ctx->arena_used);
    ctx->arena_used += bytes;
    return p;
}
static size_t workspace_bytes(size_t n)
{
    // forward is the larger of the two (bytes per input byte): L set keys 2 x 8 and idx 2 x 4 (radix
    // ping-pong), grp / gst / gid 4 each (compacted in place), S set key2 / idx / grp / gst 4 each,
    // tuple set ring links 2 x 4 and rank increments 1, rank 4, FS 4 (worst case: n factors), flags 1,
    // onesweep status 0.5, tile tables ~0.03 = 70.5; the inverse needs ~34 (prev 4, cycle tables 16,
    // staged bytes 4, fallback records 8, ...)
    return n * 71 + (64u << 20);
}

static inline u32 cdiv(u64 a, u64 b) { return (u32)((a + b - 1) / b); }
static size_t r256(size_t b) { return (b + 255) & ~(size_t)255; }
// look-back status of a re-rank over m slots: one word per tile + one per block of 32 tiles (forward.cuh)
static inline size_t rr_status_bytes(u32 m)
{
    const size_t tiles = cdiv(m, RR_TILE);
    return (tiles + tiles / 32 + 2) * 8;
}
static inline int bit_length(u64 v) { int b = 0; while (v) { b++; v >>= 1; } return b; }

// Counter read-backs go through a kernel that stores into mapped pinned memory, not through a
// D2H memcpy: a memcpy would queue on the copy engine behind the block pipeline's bulk
// transfers (up to 5 ms per read-back with 256 MiB blocks in flight).
__global__ void k_readback(const u32 *__restrict__ src, u32 *__restrict__ host_dst, u32 words)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < words) host_dst[i] = src[i];
}
static int readback(bwts_b200_ctx *ctx, cudaStream_t st, const void *dptr, size_t bytes)
{
    const u32 words = (u32)((bytes + 3) / 4);
    k_readback<<<cdiv(words, 128), 128, 0, st>>>((const u32 *)dptr, ctx->h_small_dev, words);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(st));
    return 0;
}

// ---- radix sort driver ------------------------------------------------------------------------
struct SortBufs {
    u64 *k[2];
    u32 *v[2];
    int cur;        // index of the buffers holding the data
    u32 *hist;      // [8][256] (+ 8 spare words)
    u64 *status;    // tiles * 256
};

static int radix_prepare(bwts_b200_ctx *ctx, cudaStream_t st, SortBufs &sb)
{
    CK(cudaMemsetAsync(sb.hist, 0, (RADIX_MAX_PASSES * RADIX_BINS + RADIX_MAX_PASSES) * sizeof(u32), st));
    return 0;
}

// have_hist: the digit histograms are already in sb.hist (radix_prepare + the key-building kernel)
static int radix_sort(bwts_b200_ctx *ctx, cudaStream_t st, SortBufs &sb, u32 m, int passes, bool identity_vals,
                      bool have_hist)
{
    if (passes < 1 || passes > RADIX_MAX_PASSES) return BWTS_B200_EINTERNAL;
    if (!have_hist) {
        int rc0 = radix_prepare(ctx, st, sb);
        if (rc0) return rc0;
        const u32 hgrid = min(cdiv(m, 256), 148u * 8u);
        LAUNCH(KC_RADIX_HIST, 8.0 * m, k_radix_hist, hgrid, 256, sb.k[sb.cur], m, passes, sb.hist);
    }
    LAUNCH(KC_RADIX_HIST, 0, k_radix_hist_scan, passes, 256, sb.hist);
    for (int p = 0; p < passes; p++) {
        const int a = sb.cur, b = sb.cur ^ 1;
        const bool ident = identity_vals && p == 0;
        do { ctx->epoch = (g_epoch.fetch_add(1) + 1) & 0x3fffffffu; } while (ctx->epoch == 0);
        const u32 *vin = ident ? (const u32 *)nullptr : sb.v[a];
        const double bytes = (ident ? 20.0 : 24.0) * m;
#define OS_LAUNCH(NT_, IPT_, MINB_, LB_)                                                                           \
    LAUNCH_REC(KC_ONESWEEP, bytes, "k_onesweep_pass<u64>",                                                          \
               k_onesweep_pass<u64, NT_, IPT_, MINB_, LB_><<<cdiv(m, (NT_) * (IPT_)), NT_, OsSmem<u64, NT_, IPT_>::bytes, st>>>( \
                   sb.k[a], vin, sb.k[b], sb.v[b], m, (u32)(p * RADIX_BITS), sb.hist + p * RADIX_BINS, sb.status, ctx->epoch))
        switch (g_tune_onesweep) {
        case 1: OS_LAUNCH(512, 8, 3, 8); break;
        case 2: OS_LAUNCH(256, 16, 3, 8); break;
        case 3: OS_LAUNCH(384, 12, 3, 8); break;
        case 4: OS_LAUNCH(384, 12, 3, 4); break;
        default: OS_LAUNCH(384, 12, 3, 2); break;
        }
#undef OS_LAUNCH
        sb.cur = b;
        ctx->stats.radix_passes++;
    }
    return 0;
}

// ---- LCP array (lcp.cuh) ------------------------------------------------------------------------
// After the FWD_SA emit: d_lcp[r] = lcp of the suffixes d_sa[r-1] and d_sa[r].  Scratch, all dead after
// the sort: P n words (the text-order PLCP array), tiles n / LCP_TILE words, res and the two pair lists
// n entries each, cnt 10 words: [0..2] open-pair counts, [4..9] three u64 counters of compared bytes
// (rows, warp tier, the current round), read back with the counts and added to the launches' byte
// figures.  Booked to kernel class emit and the forward's phase 3 by the caller.
static int lcp_stage(bwts_b200_ctx *ctx, cudaStream_t st, const u8 *dT, u32 n, const i32 *d_sa, i32 *d_lcp, u32 *P,
                     u32 *tiles, u32 *res, u64 *listA, u64 *listB, u32 *cnt)
{
    const u32 mode = (g_tune_lcp == 1 || g_tune_lcp == 2) ? (u32)g_tune_lcp : 0u;
    unsigned long long *cmp = (unsigned long long *)(cnt + 4);
    const auto compared = [&](int k) { return (double)((u64)ctx->h_small[4 + 2 * k] | ((u64)ctx->h_small[5 + 2 * k] << 32)); };
    CK(cudaMemsetAsync(P, 0, (size_t)n * 4, st));
    CK(cudaMemsetAsync(cnt, 0, 10 * sizeof(u32), st));
    // SA 4, B 1 (gather), P 4 (scatter, irreducible rows only: an upper bound), plus the bytes compared
    LAUNCH(KC_EMIT, 9.0 * n, k_lcp_rows, cdiv(n, 256), 256, dT, n, d_sa, P, listA, cnt, mode, cmp);
    const size_t rec_rows = ctx->recs.size() - 1;
    int rc = readback(ctx, st, cnt, 40);
    if (rc) return rc;
    ctx->recs[rec_rows].bytes += compared(0);
    const u32 m2 = ctx->h_small[0];
    if (m2) {
        LAUNCH(KC_EMIT, 8.0 * m2, k_lcp_warp, cdiv(m2, 8), 256, dT, n, listA, m2, mode == 0 ? LCP_T1 : 0u,
               mode == 2 ? 0u : LCP_T2, P, listB, cnt + 1, cmp + 1);
        const size_t rec_warp = ctx->recs.size() - 1;
        rc = readback(ctx, st, cnt, 40);
        if (rc) return rc;
        ctx->recs[rec_warp].bytes += compared(1);
        u32 m = ctx->h_small[1];
        u64 off = mode == 2 ? 0 : LCP_T2;
        u64 *cur = listB, *nxt = listA;
        while (m) {
            // each round covers [off, off + W) of every open pair, W at least 4 x what is behind it, so an
            // a^n pair of 2^31 bytes takes seven rounds; segments past a pair's mismatch or end return at once
            const u64 W = max((u64)LCP_SEG * 16, 4 * off);
            const u32 S = (u32)(W / LCP_SEG);
            const u64 items = (u64)m * S;
            const u32 gx = (u32)min(items, (u64)1 << 30), gy = (u32)((items + gx - 1) / gx);
            CK(cudaMemsetAsync(res, 0xff, (size_t)m * 4, st));
            CK(cudaMemsetAsync(cnt + 2, 0, 4, st));
            CK(cudaMemsetAsync(cmp + 2, 0, 8, st));
            LAUNCH(KC_EMIT, 8.0 * m, k_lcp_span, dim3(gx, gy), 256, dT, n, cur, m, S, (u32)off, res, cmp + 2);
            const size_t rec_span = ctx->recs.size() - 1;
            LAUNCH(KC_EMIT, 16.0 * m, k_lcp_span_close, cdiv(m, 256), 256, n, cur, m, off + W, res, P, nxt, cnt + 2);
            rc = readback(ctx, st, cnt, 40);
            if (rc) return rc;
            ctx->recs[rec_span].bytes += compared(2);
            m = ctx->h_small[2];
            off += W;
            u64 *t = cur; cur = nxt; nxt = t;
        }
    }
    const u32 nt = cdiv(n, LCP_TILE);
    LAUNCH(KC_EMIT, 4.0 * n, k_lcp_tile_max, nt, 256, P, n, tiles);
    LAUNCH(KC_EMIT, 8.0 * nt, k_lcp_tile_scan, 1, 1024, tiles, nt);
    LAUNCH(KC_EMIT, 8.0 * n, k_lcp_plcp, nt, 256, P, n, tiles);
    LAUNCH(KC_EMIT, 12.0 * n, k_lcp_emit, cdiv(n, 256), 256, d_sa, n, P, d_lcp);
    return 0;
}

// ---- LPF array and greedy LZ77 parse (lz.cuh) ----------------------------------------------------
// lpf != nullptr: LPF and PREV into lpf / prev (text order).  Otherwise the parse: LPF / PREV into scratch,
// z = the number of factors, and the pairs into factors when z <= cap (else BWTS_B200_EINVAL).
struct LzOut {
    i32 *lpf = nullptr, *prev = nullptr;
    i32 *factors = nullptr;
    long cap = 0;
    long z = -1;
};
// scratch, all dead after the LCP stage: lpf / prev n words each (the parse only), w[0..5] n words each, e n
// words, d[0..1] 2n words each, cnt 2 words
struct LzScratch {
    i32 *lpf, *prev;
    u32 *w[6], *e;
    u64 *d[2];
    u32 *cnt;
};
// log2 of the tile / chunk width: bwts_b200_tune key 25, and no wider than the next power of two of n
static u32 lz_tile_bits(u32 n)
{
    u32 tb = (g_tune_lz >= LZ_TB_MIN && g_tune_lz <= LZ_TB_MAX) ? (u32)g_tune_lz : (u32)LZ_TB_MAX;
    while (tb > LZ_TB_MIN && (1u << (tb - 1)) >= n) tb--;
    return tb;
}
// After the LCP stage, SA and LCP in rank order.  Booked to kernel class emit and the forward's phase 3.
//   LPF: gtree n / 2 bytes at most (w[5]), top 16 P <= n + 32 bytes (e), the listed rows (w[4], d[0]).
//   parse: X_1 .. X_L in w[0..5] (L <= 6: ceil(n / 32^6) <= 32), the entries of every level in e, chunk
//   counts in d[0], offsets and tile sums in d[1].
static int lz_stage(bwts_b200_ctx *ctx, cudaStream_t st, const u8 *dT, u32 n, const i32 *SA, const i32 *LCP, LzOut *lz,
                    const LzScratch &s)
{
    const u32 tb = lz_tile_bits(n), W = 1u << tb, nt = cdiv(n, W);
    u32 P = 1;
    while (P < nt) P <<= 1;
    uint2 *gtree = (uint2 *)s.w[5], *top = (uint2 *)s.e, *listP = (uint2 *)s.d[0];
    u32 *listR = s.w[4];
    i32 *lpf = lz->lpf ? lz->lpf : s.lpf, *prev = lz->lpf ? lz->prev : s.prev;
    CK(cudaMemsetAsync(top, 0xff, (size_t)16 * P, st));
    CK(cudaMemsetAsync(s.cnt, 0, 8, st));
    // SA 4, LCP 4 (rank order), LPF 4 and PREV 4 (text order), the tree nodes over 32 rows 0.5
    LAUNCH_SMEM(KC_EMIT, 16.5 * n, k_lpf_tile, nt, 1024, (size_t)16 * W, SA, LCP, n, tb, gtree, top, P, lpf, prev, listR,
                listP, s.cnt);
    for (u32 half = P / 2; half >= 1; half >>= 1) {
        if (half <= 1024) {
            LAUNCH(KC_EMIT, 48.0 * half, k_lpf_top, 1, 1024, top, half, 1u);
            break;
        }
        LAUNCH(KC_EMIT, 24.0 * half, k_lpf_top, cdiv(half, 1024), 1024, top, half, 0u);
    }
    int rc = readback(ctx, st, s.cnt, 4);
    if (rc) return rc;
    const u32 m = ctx->h_small[0];
    // per listed row: the list 12, SA 4, LPF / PREV 16, the tree walks and one group of 32 rows (~ 2 x 256)
    if (m) LAUNCH(KC_EMIT, 540.0 * m, k_lpf_cross, cdiv(m, 256), 256, SA, LCP, n, tb, gtree, top, P, lpf, prev, listR, listP, m);
    if (lz->lpf) return 0;

    int L = 1;
    while ((u64)cdiv(n, (u64)1 << (L * tb)) > W) L++;
    if (L > 6) return BWTS_B200_EINTERNAL;
    u32 *ent[7];
    ent[1] = s.e;
    for (int l = 1; l < L; l++) ent[l + 1] = ent[l] + cdiv(n, (u64)1 << (l * tb));
    CK(cudaMemsetAsync(s.e, 0xff, (size_t)(ent[L] + cdiv(n, (u64)1 << (L * tb)) - s.e) * 4, st));
    LAUNCH_SMEM(KC_EMIT, 8.0 * n, k_lz_exit1, nt, 256, (size_t)4 * W, lpf, n, tb, s.w[0]);
    for (int l = 2; l <= L; l++)
        for (u32 r = 0; r < tb; r++)
            LAUNCH(KC_EMIT, 12.0 * n, k_lz_jump, cdiv(n, 256), 256, r == 0 ? s.w[l - 2] : s.w[l - 1], s.w[l - 1], n,
                   (u32)(l * tb));
    LAUNCH(KC_EMIT, 0, k_lz_top, 1, 1, s.w[L - 1], n, (u32)(L * tb), ent[L]);
    for (int l = L; l >= 2; l--) {
        const u32 nb = cdiv(n, (u64)1 << (l * tb));
        LAUNCH(KC_EMIT, 8.0 * nb, k_lz_down, cdiv(nb, 256), 256, s.w[l - 2], n, (u32)(l * tb), (u32)((l - 1) * tb), ent[l],
               nb, ent[l - 1]);
    }
    u32 *cnt = (u32 *)s.d[0], *off = (u32 *)s.d[1];
    u32 *tiles = off + (((size_t)nt + 63) & ~(size_t)63);
    const u32 ntl = cdiv(nt, SC_TILE);
    LAUNCH_SMEM(KC_EMIT, 4.0 * n, k_lz_chunk<false>, nt, 256, (size_t)8 * W, dT, lpf, prev, n, tb, ent[1], cnt,
                (const u32 *)nullptr, (i32 *)nullptr);
    LAUNCH(KC_EMIT, 4.0 * nt, k_tile_sum_u32, ntl, 256, cnt, nt, tiles, nullptr);
    LAUNCH(KC_EMIT, 8.0 * ntl, k_scan_excl_u32_block, 1, 1024, tiles, tiles, ntl, s.cnt + 1);
    LAUNCH(KC_EMIT, 8.0 * nt, k_tile_scan_apply_u32, ntl, 256, cnt, off, nt, tiles);
    rc = readback(ctx, st, s.cnt + 1, 4);
    if (rc) return rc;
    const u32 z = ctx->h_small[0];
    lz->z = z;
    if ((long)z > lz->cap) return BWTS_B200_EINVAL;
    // LPF 4 per position, and per factor PREV or the byte, and the pair 8
    LAUNCH_SMEM(KC_EMIT, 4.0 * n + 12.0 * z, k_lz_chunk<true>, nt, 256, (size_t)8 * W, dT, lpf, prev, n, tb, ent[1],
                (u32 *)nullptr, off, lz->factors);
    return 0;
}

// ---- forward ---------------------------------------------------------------------------------
enum FwdMode {
    FWD_BWTS = 0,        // forward BWTS into d_out
    FWD_SA = 1,          // suffix array into d_sa (successor i+1, end of text smallest), then the LCP array into d_lcp if given
    FWD_LYNDON = 2,      // suffix sort, then factor-start flags (prefix minima of the ISA) into d_out
    FWD_BWTS_FLAGS = 3,  // forward BWTS, factor-start flags already in d_out (after FWD_LYNDON)
    FWD_BWT = 4,         // classic BWT into d_out: rotations of the one factor [0, n), *primary = rank[0]
    FWD_DIVBWT = 5,      // libdivsufsort's divbwt into d_out: the FWD_SA sort, bytes at shifted rows, *primary = rank[0] + 1
    FWD_FM = 6,          // FM-index build: the FWD_DIVBWT emit into d_out, then the suffix array into d_sa (fm_build)
    FWD_LZ = 7           // the FWD_SA sort and LCP stage into scratch, then LPF / PREV or the LZ77 parse into *lz
};
static int forward_core(bwts_b200_ctx *ctx, const u8 *dT, u32 n, u8 *d_out, i32 *d_sa, int mode, cudaStream_t st,
                        long *primary = nullptr, i32 *d_lcp = nullptr, LzOut *lz = nullptr)
{
    const int linear = (mode == FWD_SA || mode == FWD_LYNDON || mode == FWD_DIVBWT || mode == FWD_FM || mode == FWD_LZ);
    int rc = arena_reserve(ctx, workspace_bytes(n));
    if (rc) return rc;
    ctx->arena_used = ctx->io_end;

    const u32 ntl = cdiv(n, FL_TILE);
    const u32 nblk = cdiv(n, 1u << COARSE_BITS);
    const u32 os_tiles = cdiv(n, OS_TILE_MIN), rr_tiles = cdiv(n, RR_TILE);

    SortBufs sb;
    sb.k[0] = arena_take<u64>(ctx, n);
    sb.k[1] = arena_take<u64>(ctx, n);
    sb.v[0] = arena_take<u32>(ctx, n);
    sb.v[1] = arena_take<u32>(ctx, n);
    sb.cur = 0;
    sb.hist = arena_take<u32>(ctx, RADIX_MAX_PASSES * RADIX_BINS + RADIX_MAX_PASSES);
    sb.status = arena_take<u64>(ctx, (size_t)os_tiles * RADIX_BINS);
    // one array each: the re-rank compacts in place (k_rerank, "IN PLACE")
    u32 *grp = arena_take<u32>(ctx, n), *gst = arena_take<u32>(ctx, n);
    u32 *gid = arena_take<u32>(ctx, n);  // dense group index of the L set (written by the re-rank, read by k_build_keys)
    u32 *rank = arena_take<u32>(ctx, n);
    u32 *FS = arena_take<u32>(ctx, (size_t)n + 1);
    u32 *cidx = arena_take<u32>(ctx, (size_t)nblk + 2);
    u8 *flags = arena_take<u8>(ctx, n);
    u32 *tilecnt = arena_take<u32>(ctx, ntl + 1);
    u64 *rr_statusA = arena_take<u64>(ctx, rr_tiles + rr_tiles / 32 + 4);
    u64 *rr_statusB = arena_take<u64>(ctx, rr_tiles + rr_tiles / 32 + 4);
    u32 *kS = arena_take<u32>(ctx, n);   // S set: key2 of the last warp-local sort
    u32 *vS = arena_take<u32>(ctx, n), *grpS = arena_take<u32>(ctx, n), *gstS = arena_take<u32>(ctx, n);
    // tuple set T (k_tuple_round): ring links by text position, double-buffered, + the rank increments
    // tune 14: 0 = groups of up to 8, switched on by what the first small-group round finds (below); 1 = off;
    // 2..32 = that size, on from the first re-rank (tests)
    // tune 20: 0 = one thread per member (groups of up to 8), 1 = one thread per group (k_tuple_round_heads, up to
    // 32; measured slower: C4 forward 287.8 ms against 276.9 -- half the lanes idle, the head's loads are serial)
    const bool theads = g_tune_tmode == 1;
    const u32 thead = theads ? TUPLE_HEAD : 0u;
    const u32 tmax = g_tune_local ? 1u : (g_tune_tmax == 0 ? (theads ? 32u : 8u) : (u32)g_tune_tmax);
    bool t_on = !g_tune_local && g_tune_tmax >= 2, t_decided = t_on || tmax < 2;
    u32 *nxtT[2] = {nullptr, nullptr};
    u8 *drT = nullptr;
    if (tmax >= 2) {
        nxtT[0] = arena_take<u32>(ctx, n);
        nxtT[1] = arena_take<u32>(ctx, n);
        drT = arena_take<u8>(ctx, n);
        if (!nxtT[0] || !nxtT[1] || !drT) return BWTS_B200_EINTERNAL;
    }
    u32 *whist = arena_take<u32>(ctx, 16384);  // histogram of the leading symbols of the initial keys (k_init_keys)
    u32 *small = arena_take<u32>(ctx, 1024);  // [0] F, [1] lmax, [2] sigma, [8..15] presence, [16..] rerank counters
    u8 *code = (u8 *)arena_take<u32>(ctx, 64);
    if (!sb.k[0] || !sb.k[1] || !sb.v[0] || !sb.v[1] || !sb.hist || !sb.status || !grp || !gst || !gid || !rank || !FS ||
        !cidx || !flags || !tilecnt || !rr_statusA || !rr_statusB || !small || !whist || !code || !kS || !vS || !grpS || !gstS)
        return BWTS_B200_EINTERNAL;
    RerankCounters *rrc = (RerankCounters *)(small + 16);
    u32 *tcnt = (u32 *)(rrc + 2);  // tuple round: [0] still in the set, [1] saw a split, [2] processed; read back with rrc

    CK(cudaMemsetAsync(small, 0, 1024 * sizeof(u32), st));
    // The arena is re-laid-out per call, so the look-back status region may hold stale keys
    // whose high bits look like a live epoch: clear it once per transform (0.5 B / element);
    // from here on the per-pass epoch keeps the passes apart without further clearing.
    CK(cudaMemsetAsync(sb.status, 0, (size_t)os_tiles * RADIX_BINS * sizeof(u64), st));
    u32 F = 1, lmax = n;

    if (mode == FWD_BWTS_FLAGS) {
        CK(cudaMemcpyAsync(flags, d_out, n, cudaMemcpyDeviceToDevice, st));
    } else if (mode == FWD_BWT) {
        // no Lyndon boundaries: the factor table is {0, n}; nothing below assumes a factor is Lyndon or primitive
        // (the cyclic successor is taken mod the factor length, ties that survive are equal rotations)
        CK(cudaMemsetAsync(flags, 0, n, st));
        LAUNCH(KC_FACTORS, 0, k_one_factor, 1, 1, n, FS, flags, small);
    } else if (!linear) {
        // -- Lyndon boundaries
        u32 chunk = g_tune_chunk > 0 ? (u32)g_tune_chunk : max(512u, cdiv(n, 1u << 21));
        const u32 nch = cdiv(n, chunk), ngroups = cdiv(nch, LY_GROUP);
        u32 *chunk_last = arena_take<u32>(ctx, nch);
        u32 *group_min = arena_take<u32>(ctx, ngroups);
        u32 *group_alt = arena_take<u32>(ctx, (size_t)ngroups + ngroups / 8 + 512);
        u32 *group_alt2 = arena_take<u32>(ctx, ngroups);
        if (!chunk_last || !group_min || !group_alt || !group_alt2) return BWTS_B200_EINTERNAL;
        CK(cudaMemsetAsync(flags, 0, n, st));
        // work budgets: all Duval threads together may run n bytes (at least 32 MiB) past their
        // chunks, a warp may compare 16 MiB; beyond that the text is periodic enough for the
        // suffix-sort route to be cheaper
        LyBudget bud_thread = {small + 3, g_tune_lyndon ? 0u : max(1u << 22, n >> 3), small + 4};
        LyBudget bud_warp = {small + 3, g_tune_lyndon ? 0u : (16u << 10), small + 4};
        if (g_tune_lyndon) CK(cudaMemsetAsync(small + 3, 0xff, 4, st));
        LAUNCH(KC_LYNDON, 2.0 * n, k_duval_chunks, cdiv(nch, 128), 128, dT, n, chunk, nch, flags, chunk_last,
               bud_thread);
        if (nch > 1) {
            LAUNCH(KC_LYNDON, 0, k_chunkmin_reduce, cdiv((u64)ngroups * 32, 128), 128, dT, n, chunk_last, nch,
                   group_min, ngroups, bud_warp);
            // Which scan over the groups?  The log-depth Hillis-Steele levels (one warp per comparison) are
            // cheapest where a few bytes decide a comparison (text, DNA: 0.65 ms at 1 GiB); on tiled / periodic
            // text the minima of different tile copies agree for up to 1 MiB and the work-efficient CTA-wide
            // levels are 6x faster.  So the Hillis-Steele levels run first under a small budget of their own
            // (256 KiB per comparison, flag small[7]); if a comparison exceeds it they stop at once and the
            // CTA-wide levels take over from the untouched group minima.
            bool hs_done = false;
            if (g_tune_lyscan != 2) {
                const bool probe = g_tune_lyscan == 0;
                LyBudget bud_hs = probe ? LyBudget{small + 7, 256u, small + 4} : bud_warp;
                u32 *gin = group_min, *gout = group_alt;
                for (u32 stride = 1; stride < ngroups; stride <<= 1) {
                    LAUNCH(KC_LYNDON, 0, k_chunkmin_level, cdiv((u64)ngroups * 32, 128), 128, dT, n, gin, gout, ngroups,
                           stride, bud_hs);
                    gin = gout;
                    gout = (gout == group_alt) ? group_alt2 : group_alt;
                }
                hs_done = true;
                if (probe && ngroups > 1) {
                    rc = readback(ctx, st, small + 7, 4);
                    if (rc) return rc;
                    hs_done = ctx->h_small[0] == 0;
                }
                if (hs_done)
                    LAUNCH(KC_LYNDON, 0, k_chunk_threshold, cdiv((u64)ngroups * 32, 128), 128, dT, n, chunk, nch, flags,
                           chunk_last, gin, 0, ngroups, bud_warp);
            }
            if (!hs_done) {
                // reduce 32 -> 1 until one CTA can scan the top, then hand the exclusive prefixes back down
                LyBudget bud_cta = {small + 3, g_tune_lyndon ? 0u : (64u << 10), small + 4};  // KiB per CTA
                u32 *val[8], *pre[8], cnt[8];
                int top = 0;
                val[0] = group_min; cnt[0] = ngroups;
                u32 *pool = group_alt;  // ngroups + ngroups / 8 + 512 words: prefixes of level 0, then the upper levels
                pre[0] = pool; pool += ngroups;
                while (cnt[top] > LY_GROUP && top < 6) {
                    cnt[top + 1] = cdiv(cnt[top], LY_GROUP);
                    val[top + 1] = pool; pool += cnt[top + 1];
                    pre[top + 1] = pool; pool += cnt[top + 1];
                    LAUNCH(KC_LYNDON, 0, k_sufmin_reduce_cta, cnt[top + 1], LY_CTA, dT, n, val[top], cnt[top], val[top + 1], bud_cta);
                    top++;
                }
                for (int l = top; l >= 0; l--)
                    LAUNCH(KC_LYNDON, 0, k_sufmin_down_cta, cdiv(cnt[l], LY_GROUP), LY_CTA, dT, n, val[l], cnt[l],
                           l == top ? (const u32 *)nullptr : pre[l + 1], pre[l], bud_cta);
                LAUNCH(KC_LYNDON, 0, k_chunk_threshold, cdiv((u64)ngroups * 32, 128), 128, dT, n, chunk, nch, flags,
                       chunk_last, pre[0], 1, ngroups, bud_warp);
            }
        }
    }
    if (!linear && mode != FWD_BWT) {
        // -- factor table
        LAUNCH(KC_FACTORS, 1.0 * n, k_flag_count, ntl, 256, flags, n, tilecnt);
        LAUNCH(KC_FACTORS, 8.0 * ntl, k_scan_excl_u32_block, 1, 1024, tilecnt, tilecnt, ntl, small + 0);
        LAUNCH(KC_FACTORS, 1.0 * n, k_flag_write, ntl, 256, flags, n, tilecnt, FS);
        LAUNCH(KC_FACTORS, 0, k_set_u32, 1, 1, FS, small + 0, n);
    }
    // -- alphabet
    LAUNCH(KC_INIT_KEYS, 1.0 * n, k_byte_presence, min(cdiv(n, 16 * 256) + 1, 148u * 8u), 256, dT, n, small + 8);
    LAUNCH(KC_INIT_KEYS, 0, k_code_table, 1, 256, small + 8, code, small + 2);
    rc = readback(ctx, st, small, 16);
    if (rc) return rc;
    const u32 sigma = ctx->h_small[2];
    if (mode == FWD_BWTS && ctx->h_small[3]) {
        // the chunk kernels ran over budget, their marks are unusable: take the factor starts
        // from a suffix sort (prefix minima of the ISA) and start again with them
        ctx->stats.lyndon_fallback = 1;
        rc = forward_core(ctx, dT, n, d_out, nullptr, FWD_LYNDON, st);
        if (rc) return rc;
        return forward_core(ctx, dT, n, d_out, nullptr, FWD_BWTS_FLAGS, st);
    }
    if (!linear) {
        F = ctx->h_small[0];
        if (F < 1 || F > n) return BWTS_B200_EINTERNAL;
        LAUNCH(KC_FACTORS, 4.0 * F, k_factor_lmax, min(cdiv(F, 256), 148u * 4u), 256, FS, F, small + 1);
        LAUNCH(KC_FACTORS, 4.0 * nblk, k_coarse_index, cdiv(nblk + 1, 256), 256, FS, F, cidx, nblk);
    }
    const u32 syms = linear ? sigma + 1 : sigma;  // linear mode reserves code 0 for "past the end"
    const u32 bits = max(1, bit_length(syms - 1));
    const u32 keybits = (g_tune_keybits >= 8 && g_tune_keybits <= 64) ? (u32)g_tune_keybits : 64u;
    const u32 k0 = max(1u, keybits / bits);
    // bits the whole symbols leave free take the top of the next symbol (k_init_keys; tune 22 = 1: off)
    const u32 extra = (linear || g_tune_partial == 1 || keybits <= k0 * bits) ? 0u : min(bits - 1, keybits - k0 * bits);
    const int P0 = (int)cdiv((u64)k0 * bits + extra, 8);
    ctx->stats.alphabet_bits = (int)bits;
    ctx->stats.initial_depth = (int)k0;

    // digit histograms of the initial sort from one histogram of the leading symbols (k_init_keys): possible when the
    // widest digit spans symbols worth at most 14 bits (alphabets of 1-4 and 6-8 bits per symbol; 5 bits: 15)
    u32 wsyms = 0;
    {
        const u32 k0p = k0 + (extra ? 1u : 0u), d = extra ? bits - extra : 0u;
        for (int p = 0; p < P0; p++) {
            const u32 lo_bit = 8u * p + d, hi_bit = min(8u * p + 7u + d, k0p * bits - 1u);
            wsyms = max(wsyms, hi_bit / bits - lo_bit / bits + 1u);
        }
    }
    const bool use_wh = !linear && g_tune_hist != 1 && wsyms * bits <= 14 && k0 >= wsyms;
    const u32 wbins = use_wh ? 1u << (wsyms * bits) : 0u;
    if (!linear) {
        if (use_wh) CK(cudaMemsetAsync(whist, 0, wbins * sizeof(u32), st));
        // shared memory per CTA: 18.7 KB of staging + the histogram (4 bytes per bin, 2 above 4096 bins)
        const size_t whb = wbins > 4096 ? wbins * 2 : wbins * sizeof(u32);
        LAUNCH_SMEM(KC_INIT_KEYS, 9.0 * n, k_init_keys, min(cdiv(n, 2048), (u32)ctx->sm_count * (wbins > 4096 ? 4u : 6u)), 256, whb, dT, n,
                    FS, cidx, code, bits, k0, extra, sb.k[0], use_wh ? whist : (u32 *)nullptr,
                    extra + bits * (k0 - min(k0, wsyms)), wbins);
    } else {
        LAUNCH(KC_INIT_KEYS, 9.0 * n, k_init_keys_linear, cdiv(cdiv(n, 8), 256), 256, dT, n, code, bits, k0, sb.k[0]);
    }
    if (use_wh) LAUNCH(KC_RADIX_HIST, 4.0 * wbins * P0, k_digit_hists, P0, 256, whist, wbins, wsyms, bits, k0, extra, sb.hist);
    rc = radix_sort(ctx, st, sb, n, P0, true, use_wh);
    if (rc) return rc;

    CK(cudaMemsetAsync(rank, 0, (size_t)n * 4, st));
    if (!t_decided && n >= (1u << 20)) {
        // vote on the tuple set before the first re-rank: 64 Ki sorted neighbours; if most of the tied ones
        // still agree 32 bytes further on, the ties come from long repeats (see k_sample_lcp).  Where the
        // vote says no, the first small-group round gets a second look (survival of its ties, below).
        const u32 samples = 1u << 16;
        CK(cudaMemsetAsync(tcnt + 4, 0, 8, st));
        LAUNCH(KC_TUPLE, 24.0 * samples, k_sample_lcp, samples / 256, 256, sb.k[sb.cur], sb.v[sb.cur], dT, n, samples, k0, 32u,
               tcnt + 4);
        rc = readback(ctx, st, tcnt + 4, 8);
        if (rc) return rc;
        if (ctx->h_small[0] >= samples / 16 && 2 * ctx->h_small[1] >= ctx->h_small[0]) { t_on = true; t_decided = true; }
    }
    if (t_on) {  // every position starts outside the tuple set, in both buffers
        CK(cudaMemsetAsync(nxtT[0], 0xff, (size_t)n * 4, st));
        CK(cudaMemsetAsync(nxtT[1], 0xff, (size_t)n * 4, st));
    }
    const int PH_SORT0 = 0, PH_ISA = 1, PH_FIX = 2, PH_EMIT = 3;  // bwts_b200_phase_name(0, .)

    // Two live sets.  L: groups of any size, sorted by the global radix path (sb, grp, gst).
    // S: groups of at most 32 members, sorted warp-locally (kS, vS, grpS, gstS).
    // T: groups of at most tmax members, refined in text order (nxtT, drT); they never come back.
    u32 mL = n, mS = 0, mT = 0, groups_before = 1, groupsL = 0;
    int tc = 0;  // nxtT[tc] holds the rings
    const u32 tgrid = min(cdiv(n, 256), (u32)ctx->sm_count * 16u);
    u64 k = k0;
    const u32 kb = linear ? bit_length(n) : max(1, bit_length((u64)n - 1));
    bool first = true, sortedL = true;  // the L set enters the loop freshly sorted (initial sort)
    bool binned_now = false;
    u64 changedL = 0;  // estimate of the ranks the last L re-rank moved
    u64 changedS = ~0ull >> 4;  // the same for the S set; before its first re-rank: assume all of them
    bool sortedS = false;
    const LiveOut none = {nullptr, nullptr, nullptr, nullptr};
    // rank[pos[j]] = nr[j] for j < m through one u32 onesweep pass that bins the pairs by the top 8 bits of the position
    // and a streaming scatter, region by region (§4.2 "Where the ranks go")
    auto scatter_binned = [&](const u32 *pos, const u32 *nr, u32 m, u32 *bin_pos, u32 *bin_val) -> int {
        const u32 shift = kb - 8;
        if (m == n) {
            LAUNCH(KC_RERANK, 0, k_bin_bases, 1, 256, n, shift, sb.hist);
        } else {
            CK(cudaMemsetAsync(sb.hist, 0, 256 * sizeof(u32), st));
            LAUNCH(KC_RERANK, 4.0 * m, k_bin_count, min(cdiv(cdiv(m, 4), 256), 148u * 8u), 256, pos, m, shift, sb.hist);
            LAUNCH(KC_RERANK, 0, k_radix_hist_scan, 1, 256, sb.hist);
        }
        do { ctx->epoch = (g_epoch.fetch_add(1) + 1) & 0x3fffffffu; } while (ctx->epoch == 0);
        LAUNCH_REC(KC_RERANK, 16.0 * m, "k_onesweep_pass<u32> bin",
                   k_onesweep_pass<u32, 384, 12, 3, 4><<<cdiv(m, 384 * 12), 384, OsSmem<u32, 384, 12>::bytes, st>>>(
                       pos, nr, bin_pos, bin_val, m, shift, sb.hist, sb.status, ctx->epoch));
        LAUNCH(KC_RERANK, 12.0 * m, k_scatter_pairs, cdiv(cdiv(m, 8), 256), 256, bin_pos, bin_val, m, rank);
        ctx->stats.binned_rounds++;
        return 0;
    };
    for (;;) {
        // ---- re-rank what was just sorted; S first, L appends to the same S stream
        ctx->phase = PH_ISA;
        CK(cudaMemsetAsync(rrc, 0, 2 * sizeof(RerankCounters), st));
        const LiveOut oS = {vS, grpS, gstS, nullptr};  // in place
        // The S set's ranks take the binned route as well while a third of them move per round (text: the first
        // small-group round resolves nearly every tie; C5 block 37.1 -> 35.7 ms).
        // Its idx array is compacted in place, so the kernel copies the positions out next to the ranks: three streams
        // of mS words in the idle key buffer (8n bytes), the binned ranks in kS once the kernel has read its keys.
        const bool binS = mS && sortedS && use_binned_scatter(n, kb) && g_tune_scatterbin != 3 && 3ull * mS + 16 <= 2ull * n &&
                          (g_tune_scatterbin == 4 || (n >= (1u << 27) && mS >= (1u << 20) && 3ull * changedS >= mS));
        const size_t mS4 = ((size_t)mS + 3) & ~(size_t)3;
        u32 *nrS = binS ? (u32 *)sb.k[sb.cur ^ 1] : (u32 *)nullptr, *posS = binS ? nrS + mS4 : (u32 *)nullptr;
        if (mS && sortedS) {
            CK(cudaMemsetAsync(rr_statusA, 0, rr_status_bytes(mS), st));
            CK(cudaMemsetAsync(rr_statusB, 0, rr_status_bytes(mS), st));
            if (t_on) {
                LAUNCH(KC_RERANK, 20.0 * mS, (k_rerank<2, u32>), cdiv(mS, RR_TILE), RR_NT, kS, vS, grpS, gstS, mS, 0, rank, oS,
                       (const u32 *)nullptr, none, rr_statusA, rr_statusB, rrc + 0, nrS, posS, nxtT[tc], tmax, thead);
            } else {
                LAUNCH(KC_RERANK, 20.0 * mS, (k_rerank<0, u32>), cdiv(mS, RR_TILE), RR_NT, kS, vS, grpS, gstS, mS, 0, rank, oS,
                       (const u32 *)nullptr, none, rr_statusA, rr_statusB, rrc + 0, nrS, posS, (u32 *)nullptr, 0u, 0u);
            }
            if (binS) {
                rc = scatter_binned(posS, nrS, mS, posS + mS4, kS);
                if (rc) return rc;
            }
        }
        if (mL && sortedL) {
            CK(cudaMemsetAsync(rr_statusA, 0, rr_status_bytes(mL), st));
            CK(cudaMemsetAsync(rr_statusB, 0, rr_status_bytes(mL), st));
            const LiveOut oL = {sb.v[sb.cur ^ 1], grp, gst, gid};  // grp / gst in place, idx into the idle half
            // First re-rank of a large input: all n ranks are written, at random text positions
            // (the kernel then runs at the DRAM random-access rate: 2.8 ms for 64 Mi elements, ncu:
            // 85 B moved per element).  Instead the ranks go out in sorted order, one u32 onesweep
            // pass bins the (position, rank) pairs by the top 8 bits of the position, and a
            // streaming kernel scatters them region by region through L2.
            // Later re-ranks do the same when a third of the set's ranks moved in the round before (k_rerank counts
            // them): the streams cost ~20 ps per slot, a directly scattered rank 36-50 ps.  The density of the set
            // does not matter -- the DRAM bytes per moved rank are the same either way, what the regions buy is
            // page and TLB locality (C4, sets of 15-18 % of the positions: forward 267.9 -> 259.0 ms).  From 128 Mi
            // bytes on: at 64 MiB (rank[] = twice the L2) the direct scatter is level or ahead (C2 8.30 against 8.39 ms).
            const bool binned = use_binned_scatter(n, kb) &&
                                (first || g_tune_scatterbin == 4 ||
                                 (g_tune_scatterbin != 3 && n >= (1u << 27) && mL >= (1u << 20) && 3ull * changedL >= mL));
            binned_now = binned;
            u32 *nr_out = binned ? (u32 *)sb.k[sb.cur ^ 1] : (u32 *)nullptr;  // the idle key buffer: 8n bytes
            if (g_tune_local) {
                LAUNCH(KC_RERANK, 24.0 * mL, (k_rerank<0, u64>), cdiv(mL, RR_TILE), RR_NT, sb.k[sb.cur], sb.v[sb.cur],
                       first ? (const u32 *)nullptr : grp, gst, mL, 0, rank, oL, (const u32 *)nullptr, none,
                       rr_statusA, rr_statusB, rrc + 1, nr_out, (u32 *)nullptr, (u32 *)nullptr, 0u, 0u);
            } else {
                LAUNCH(KC_RERANK, 24.0 * mL, (k_rerank<1, u64>), cdiv(mL, RR_TILE), RR_NT, sb.k[sb.cur], sb.v[sb.cur],
                       first ? (const u32 *)nullptr : grp, gst, mL, 0, rank, oS, (const u32 *)&rrc[0].keptS, oL,
                       rr_statusA, rr_statusB, rrc + 1, nr_out, (u32 *)nullptr, t_on ? nxtT[tc] : (u32 *)nullptr, t_on ? tmax : 0u, thead);
            }
        }
        if (mL && sortedL && binned_now) {
            // scratch: rank stream + binned positions in the idle key buffer, binned ranks in kS (the key2 array of the S
            // set is dead between its re-rank above and the warp-local sort of the coming round, which writes it)
            u32 *nr_buf = (u32 *)sb.k[sb.cur ^ 1], *bin_pos = nr_buf + (((size_t)n + 3) & ~(size_t)3), *bin_val = kS;
            rc = scatter_binned(sb.v[sb.cur], nr_buf, mL, bin_pos, bin_val);
            if (rc) return rc;
        }
        rc = readback(ctx, st, rrc, 2 * sizeof(RerankCounters) + 16);
        if (rc) return rc;
        const RerankCounters cS = ((const RerankCounters *)ctx->h_small)[0];
        const RerankCounters cL = ((const RerankCounters *)ctx->h_small)[1];
        // what the tuple round of the previous iteration left (zero when none ran) + this iteration's arrivals
        const u32 *tc_h = (const u32 *)((const RerankCounters *)ctx->h_small + 2);
        const bool splitT = tc_h[1] != 0;
        changedL = 16ull * ((u64)cL.changed[0] + cL.changed[1] + cL.changed[2] + cL.changed[3]);
        if (mS && sortedS) changedS = 16ull * ((u64)cS.changed[0] + cS.changed[1] + cS.changed[2] + cS.changed[3]);
        u32 headsS = 0, headsL = 0, kheadsS = 0, kheadsL_all = 0, enteredT = 0;
        for (int q = 0; q < RR_SPREAD; q++) {
            headsS += cS.heads[q]; headsL += cL.heads[q];
            kheadsS += cS.kheads[q]; kheadsL_all += cL.kheads[q];
            enteredT += cS.keptT[q] + cL.keptT[q];
        }
        mT = tc_h[0] + enteredT;
        if (first && !linear) {
            rc = readback(ctx, st, small + 1, 4);
            if (rc) return rc;
            lmax = ctx->h_small[0];
        }
        first = false;
        u32 newS, newL;
        if (g_tune_local) {  // routing off: the "S" stream of the L re-rank is the L set itself
            newS = 0;
            newL = cL.keptS;
        } else {
            newS = cS.keptS + cL.keptS;
            newL = cL.keptL;
        }
        ctx->stats.class_bytes[KC_RERANK] += 12.0 * ((double)newS + newL);
        const bool split = headsS + headsL != groups_before || splitT;
        // adopt the compacted arrays
        if (mL && sortedL) sb.cur ^= 1;   // idx of L now lives in sb.v[cur]
        mS = newS;
        mL = newL;
        groups_before = kheadsS + kheadsL_all;
        groupsL = g_tune_local ? 0 : cL.kheadsL;
        if (mS + mL + mT == 0) break;
        const bool deep_enough = !linear && k >= 2ull * lmax;  // Fine-Wilf: remaining ties are equal rotations
        if (!split || deep_enough) {
            if (linear) return BWTS_B200_EINTERNAL;  // suffixes are pairwise distinct
            // ties are final: give every member of a tie its own slot
            if (mS) {
                CK(cudaMemsetAsync(rr_statusA, 0, rr_status_bytes(mS), st));
                CK(cudaMemsetAsync(rr_statusB, 0, rr_status_bytes(mS), st));
                CK(cudaMemsetAsync(rrc, 0, sizeof(RerankCounters), st));
                LAUNCH(KC_RERANK, 16.0 * mS, (k_rerank<0, u32>), cdiv(mS, RR_TILE), RR_NT, (const u32 *)nullptr, vS,
                       grpS, gstS, mS, 1, rank, none, (const u32 *)nullptr, none, rr_statusA, rr_statusB, rrc,
                       (u32 *)nullptr, (u32 *)nullptr, (u32 *)nullptr, 0u, 0u);
            }
            if (mL) {
                CK(cudaMemsetAsync(rr_statusA, 0, rr_status_bytes(mL), st));
                CK(cudaMemsetAsync(rr_statusB, 0, rr_status_bytes(mL), st));
                CK(cudaMemsetAsync(rrc + 1, 0, sizeof(RerankCounters), st));
                LAUNCH(KC_RERANK, 16.0 * mL, (k_rerank<0, u64>), cdiv(mL, RR_TILE), RR_NT, (const u64 *)nullptr,
                       sb.v[sb.cur], grp, gst, mL, 1, rank, none, (const u32 *)nullptr, none, rr_statusA,
                       rr_statusB, rrc + 1, (u32 *)nullptr, (u32 *)nullptr, (u32 *)nullptr, 0u, 0u);
            }
            if (mT) {  // members of a final tie take consecutive slots in text order, the rings dissolve
                CK(cudaMemsetAsync(tcnt, 0, 16, st));
                if (theads) {
                    LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round_heads<false>, tgrid * 2, TUPLE_HNT, nxtT[tc], nxtT[tc ^ 1], drT,
                           rank, FS, cidx, n, (u32)k, 1, tcnt);
                } else {
                    LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round<false>, tgrid, 256, nxtT[tc], nxtT[tc ^ 1], drT, rank, FS, cidx,
                           n, (u32)k, 1, tcnt);
                }
                LAUNCH(KC_TUPLE, 4.0 * n + 13.0 * mT, k_tuple_apply, tgrid, 256, nxtT[tc], nxtT[tc ^ 1], drT, rank, n);
            }
            break;
        }
        // ---- one doubling round on both live sets
        ctx->phase = PH_FIX;
        if (ctx->stats.rounds == 0) ctx->stats.first_live = (long)mS + mL + mT;
        ctx->stats.rounds++;
        ctx->stats.live_sum += (long)mS + mL + mT;
        sortedS = sortedL = false;
        CK(cudaMemsetAsync(tcnt, 0, 16, st));
        if (mT) {
            // the tuple set first: phase A on old ranks and rings, phase B applies; the rank-ordered sets
            // gather afterwards (a group is refined as a whole, readers never see it at two depths)
            if (theads && !linear) {
                LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round_heads<false>, tgrid * 2, TUPLE_HNT, nxtT[tc], nxtT[tc ^ 1], drT,
                       rank, FS, cidx, n, (u32)k, 0, tcnt);
            } else if (theads) {
                LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round_heads<true>, tgrid * 2, TUPLE_HNT, nxtT[tc], nxtT[tc ^ 1], drT,
                       rank, FS, cidx, n, (u32)k, 0, tcnt);
            } else if (!linear) {
                LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round<false>, tgrid, 256, nxtT[tc], nxtT[tc ^ 1], drT, rank, FS, cidx,
                       n, (u32)k, 0, tcnt);
            } else {
                LAUNCH(KC_TUPLE, 4.0 * n + 30.0 * mT, k_tuple_round<true>, tgrid, 256, nxtT[tc], nxtT[tc ^ 1], drT, rank, FS, cidx,
                       n, (u32)k, 0, tcnt);
            }
            LAUNCH(KC_TUPLE, 4.0 * n + 13.0 * mT, k_tuple_apply, tgrid, 256, nxtT[tc], nxtT[tc ^ 1], drT, rank, n);
            tc ^= 1;
            ctx->stats.tuple_rounds++;
            ctx->stats.tuple_live_sum += (long)mT;
        }
        if (mS) {
            // every group fits a warp: gather + in-register ordering, no radix passes; sorted in place
            // The first small-group round also measures how many of its rotations stay tied: where most do,
            // the ties come from long repeats (DNA with copied segments: 98 %), neighbours in the text sit
            // in neighbouring groups and the tuple set's text-order sweeps beat one gather per rotation;
            // where few do (text: the ties end within a round or two) the set would only add random traffic.
            u32 *surv = (!t_decided && mS >= (n >> 5)) ? tcnt + 4 : (u32 *)nullptr;
            if (surv) CK(cudaMemsetAsync(surv, 0, 8, st));
            LAUNCH(KC_LOCAL_SORT, 24.0 * mS, k_local_sort_warp, cdiv((u64)cdiv(mS, 32) * 32, 256), 256, vS, gstS, mS, rank, FS,
                   cidx, (u32)k, kb, n, linear, kS, vS, surv);
            ctx->stats.local_rounds++;
            sortedS = true;
            if (surv) {
                rc = readback(ctx, st, surv, 8);
                if (rc) return rc;
                t_decided = true;
                if (ctx->h_small[0] && 2ull * ctx->h_small[1] >= ctx->h_small[0]) {
                    t_on = true;
                    CK(cudaMemsetAsync(nxtT[0], 0xff, (size_t)n * 4, st));
                    CK(cudaMemsetAsync(nxtT[1], 0xff, (size_t)n * 4, st));
                }
            }
        }
        if (mL) {
            // groups that fit one CTA: gather + bitonic network in shared memory, no radix passes
            bool cta_sorted = false;
            if (!g_tune_nocta) {
                CK(cudaMemsetAsync(small + 5, 0, 4, st));
                LAUNCH(KC_LOCAL_SORT, 0, k_ls_probe, cdiv(cdiv(mL, LS_T), 256), 256, gst, mL, small + 5);
                rc = readback(ctx, st, small + 5, 4);
                if (rc) return rc;
                if (ctx->h_small[0] == 0) {
                    if (g_tune_ctasort == 1)  // the bitonic network of round 1
                        LAUNCH_REC(KC_LOCAL_SORT, 32.0 * mL, "k_local_sort_cta",
                                   (!linear ? k_local_sort_cta<false> : k_local_sort_cta<true>)
                                       <<<cdiv(mL, LS_T), LS_NT, LS_CAP * sizeof(u64), st>>>(
                                       sb.v[sb.cur], gst, mL, rank, FS, cidx, (u32)k, kb, n, sb.k[sb.cur ^ 1], sb.v[sb.cur ^ 1]));
                    else
                        LAUNCH_REC(KC_LOCAL_SORT, 32.0 * mL, "k_local_sort_cta_radix",
                                   (!linear ? k_local_sort_cta_radix<false> : k_local_sort_cta_radix<true>)
                                       <<<cdiv(mL, LS_T), LSR_NT, LsrSmem::bytes, st>>>(
                                       sb.v[sb.cur], gst, mL, rank, FS, cidx, (u32)k, kb, n, sb.k[sb.cur ^ 1], sb.v[sb.cur ^ 1]));
                    sb.cur ^= 1;
                    ctx->stats.cta_rounds++;
                    cta_sorted = true;
                }
            }
            if (!cta_sorted) {
                // high part of the key: the dense group index (fewest bits); with routing off the
                // group start offset does the same job
                const u32 *hi = groupsL ? gid : gst;
                const int hibits = max(1, bit_length(groupsL ? (u64)groupsL - 1 : (u64)mL - 1));
                const int passes = max(1, (int)cdiv((u64)kb + hibits, 8));
                rc = radix_prepare(ctx, st, sb);
                if (rc) return rc;
                const u32 bgrid = min(cdiv(mL, 256), 148u * 8u);
                if (!linear) {
                    LAUNCH(KC_BUILD_KEYS, 20.0 * mL, k_build_keys<false>, bgrid, 256, sb.v[sb.cur], hi, mL, rank, FS,
                           cidx, n, (u32)k, kb, sb.k[sb.cur], passes, sb.hist);
                } else {
                    LAUNCH(KC_BUILD_KEYS, 20.0 * mL, k_build_keys<true>, bgrid, 256, sb.v[sb.cur], hi, mL, rank, FS,
                           cidx, n, (u32)k, kb, sb.k[sb.cur], passes, sb.hist);
                }
                rc = radix_sort(ctx, st, sb, mL, passes, false, true);
                if (rc) return rc;
            }
            sortedL = true;
        }
        k *= 2;
    }

    // -- emit
    ctx->phase = PH_EMIT;
    (void)PH_SORT0;
    const bool div = mode == FWD_DIVBWT || mode == FWD_FM;  // the byte emit below with emit_slot<true> (forward.cuh)
    if (!linear || div) {
        const bool emit_binned = g_tune_emit >= 2 || (g_tune_emit == 0 && n >= (512u << 20));
        if (emit_binned && kb >= 8 && g_tune_emit != 3) {
            // one packed word per element, binned by rank region, then scattered through L2: the bin pass reads
            // rank[] and the text, the value T[i-1] rides in the bits above the in-bin part of the rank
            u32 *packed = (u32 *)sb.k[0];
            const u32 shift = kb - 8;
            LAUNCH(KC_EMIT, 0, k_bin_bases, 1, 256, n, shift, sb.hist);
            do { ctx->epoch = (g_epoch.fetch_add(1) + 1) & 0x3fffffffu; } while (ctx->epoch == 0);
            LAUNCH_REC(KC_EMIT, 9.0 * n, "k_onesweep_pass<u32> pack",
                       k_onesweep_pass<u32, 384, 12, 3, 4, 2><<<cdiv(n, 384 * 12), 384, OsSmem<u32, 384, 12>::bytes, st>>>(
                           rank, (const u32 *)dT, (u32 *)nullptr, packed, n, shift, sb.hist, sb.status, ctx->epoch));
            if (div) LAUNCH(KC_EMIT, 5.0 * n, k_scatter_packed<true>, cdiv(cdiv(n, 4), 256), 256, packed, n, shift, d_out, rank);
            else LAUNCH(KC_EMIT, 5.0 * n, k_scatter_packed, cdiv(cdiv(n, 4), 256), 256, packed, n, shift, d_out);
        } else if (emit_binned && kb >= 8) {
            // (round 1, tune 9 = 3) (rank, byte) pairs as two u32 streams binned by rank region
            u32 *val = (u32 *)sb.k[0], *bin_pos = val + (((size_t)n + 3) & ~(size_t)3);
            u32 *bin_val = (u32 *)sb.k[1];
            const u32 shift = kb - 8;
            LAUNCH(KC_EMIT, 5.0 * n, k_emit_vals, cdiv(cdiv(n, 4), 256), 256, dT, n, val);
            LAUNCH(KC_EMIT, 0, k_bin_bases, 1, 256, n, shift, sb.hist);
            do { ctx->epoch = (g_epoch.fetch_add(1) + 1) & 0x3fffffffu; } while (ctx->epoch == 0);
            LAUNCH_REC(KC_EMIT, 16.0 * n, "k_onesweep_pass<u32> bin",
                       k_onesweep_pass<u32, 384, 12, 3, 4><<<cdiv(n, 384 * 12), 384, OsSmem<u32, 384, 12>::bytes, st>>>(
                           rank, val, bin_pos, bin_val, n, shift, sb.hist, sb.status, ctx->epoch));
            if (div) LAUNCH(KC_EMIT, 9.0 * n, k_scatter_bytes<true>, cdiv(cdiv(n, 4), 256), 256, bin_pos, bin_val, n, d_out, rank);
            else LAUNCH(KC_EMIT, 9.0 * n, k_scatter_bytes, cdiv(cdiv(n, 4), 256), 256, bin_pos, bin_val, n, d_out);
        } else {
            // rank windows of 64 Mi slots: the scatter target of one launch stays resident in the 126 MB L2
            const u32 win = (g_tune_emitwin >= 16 && g_tune_emitwin <= 1024) ? (u32)g_tune_emitwin << 20 : 64u << 20;
            for (u64 lo = 0; lo < n; lo += win) {
                const u32 hi = (u32)min((u64)n, lo + win);
                if (div)
                    LAUNCH(KC_EMIT, (lo == 0 ? 7.0 : 4.0) * n, k_emit<true>, cdiv(cdiv(n, 4), 256), 256, dT, n, rank, flags,
                           d_out, (u32)lo, hi);
                else
                    LAUNCH(KC_EMIT, (lo == 0 ? 7.0 : 4.0) * n, k_emit, cdiv(cdiv(n, 4), 256), 256, dT, n, rank, flags, d_out,
                           (u32)lo, hi);
            }
        }
        if (div) {  // slot 0 after every lane has stored; the row of suffix 0 is where the end of text stood
            LAUNCH(KC_EMIT, 0, k_divbwt_first, 1, 1, dT, n, d_out);
            rc = readback(ctx, st, rank, 4);
            if (rc) return rc;
            *primary = (long)ctx->h_small[0] + 1;
        } else {
            LAUNCH(KC_EMIT, 10.0 * F, k_emit_heads, cdiv(F, 256), 256, dT, FS, F, rank, d_out);
        }
        if (mode == FWD_BWT) {  // the row of rotation 0: ties are ranked in text order, so rotation 0 leads its own
            rc = readback(ctx, st, rank, 4);
            if (rc) return rc;
            *primary = (long)ctx->h_small[0];
        }
        if (mode == FWD_FM) LAUNCH(KC_EMIT, 8.0 * n, k_emit_sa, cdiv(n, 256), 256, rank, n, d_sa);
    } else if (mode == FWD_SA || mode == FWD_LZ) {
        // FWD_LZ: the suffix array and LCP array go to the S set's kS / vS, which the LCP stage does not use
        i32 *sa_out = mode == FWD_LZ ? (i32 *)kS : d_sa, *lcp_out = mode == FWD_LZ ? (i32 *)vS : d_lcp;
        LAUNCH(KC_EMIT, 8.0 * n, k_emit_sa, cdiv(n, 256), 256, rank, n, sa_out);
        if (lcp_out) {
            rc = lcp_stage(ctx, st, dT, n, sa_out, lcp_out, sb.v[0], grp, gst, sb.k[0], sb.k[1], small + 128);
            if (rc) return rc;
        }
        if (mode == FWD_LZ) {
            const LzScratch s = {(i32 *)rank, (i32 *)gid, {sb.v[1], FS, grpS, gstS, sb.v[0], grp}, gst, {sb.k[0], sb.k[1]},
                                 small + 160};
            rc = lz_stage(ctx, st, dT, n, sa_out, lcp_out, lz, s);
            if (rc) return rc;
        }
    } else {
        // FWD_LYNDON: rank[] is now the inverse suffix array; factor starts = its strict prefix minima
        const u32 pmt = cdiv(n, PM_TILE);
        LAUNCH(KC_LYNDON, 4.0 * n, k_tile_min_u32, pmt, 256, rank, n, tilecnt);
        LAUNCH(KC_LYNDON, 8.0 * pmt, k_tile_min_scan, 1, 1024, tilecnt, pmt);
        LAUNCH(KC_LYNDON, 5.0 * n, k_prefix_min_flags, pmt, 256, rank, n, tilecnt, d_out);
    }
    ctx->stats.factors = F;
    ctx->stats.longest_factor = lmax;
    return 0;
}

// ---- inverse -----------------------------------------------------------------------------------
// One attempt with the splitter hash h.  budget_k: step budget (in units of 1024 steps) of the
// fallback walks over cycles without splitters, 0 = unbounded; *over is set when it ran out.
// bwt_out != nullptr: classic inverse BWT from row `primary` into bwt_out; d_out then receives the
// BWTS layout, which the attempt rotates into bwt_out with its own sublist records (k_bwt_locate).
// div_primary > 0 (with bwt_out, primary 0): libdivsufsort's inverse_bw_transform, the same path over the
// map prev_s of k_inv_lf_rank<true>.
static int inverse_attempt(bwts_b200_ctx *ctx, const u8 *dB, u32 n, u8 *d_out, cudaStream_t st, SplHash h, u32 budget_k,
                           bool *over, u8 *bwt_out = nullptr, u32 primary = 0, u32 div_primary = 0)
{
    *over = false;
    const u32 shift = h.shift;
    const u32 ntiles = cdiv(n, INV_TILE), nchunks = cdiv(ntiles, INV_CHUNK);
    const u32 nst = cdiv(n, SP_TILE), nsc = cdiv(n, SC_TILE);

    u32 *tilehist = arena_take<u32>(ctx, (size_t)ntiles * 256);
    u32 *chunksum = arena_take<u32>(ctx, (size_t)nchunks * 256);
    u32 *prev = arena_take<u32>(ctx, n);
    const bool staged = g_tune_invpath == 0;
    // per-128 counts instead of one bit per element once the bitmap (n / 8 bytes) would no longer sit in L2
    // next to the walk's own traffic; below that the bitmap has fewer same-address atomics (tune 15: 1 / 2 force)
    const bool count_marks = staged && (g_tune_invmark == 2 || (g_tune_invmark == 0 && n > (256u << 20)));
    u32 *sid = staged ? (u32 *)nullptr : arena_take<u32>(ctx, n);  // two-walk path only (sparse element -> sublist map)
    u32 *len_at_min = arena_take<u32>(ctx, n);
    u32 *off = arena_take<u32>(ctx, n);
    uint2 *cyc = arena_take<uint2>(ctx, n);
    u32 *tilecnt = arena_take<u32>(ctx, max(nst, nsc) + 1);
    // [0] ns, [2] reached, [4] unreached handled, [5] fallback steps / 1024, [6] cycles, [8] scan total,
    // [10] deficient blocks, [12] budget exhausted, [16..18] classic BWT (d, L, off) of the primary,
    // [20] divbwt: the byte of the element whose prev_s is 0, [64..320] C
    u32 *small = arena_take<u32>(ctx, 512);
    if (!tilehist || !chunksum || !prev || (!staged && !sid) || !len_at_min || !off || !cyc || !tilecnt || !small)
        return BWTS_B200_EINTERNAL;
    u32 *Ctab = small + 64;
    CK(cudaMemsetAsync(small, 0, 64 * sizeof(u32), st));

    // -- LF map (phases: bwts_b200_phase_name(1, .))
    ctx->phase = 0;
    LAUNCH(KC_INV_HIST, 1.0 * n, k_inv_tile_hist, ntiles, INV_NT, dB, n, tilehist);
    LAUNCH(KC_INV_SCAN, 1024.0 * ntiles, k_inv_colsum, nchunks, 256, tilehist, ntiles, chunksum);
    LAUNCH(KC_INV_SCAN, 0, k_inv_chunk_scan, 1, 256, chunksum, nchunks, Ctab);
    LAUNCH(KC_INV_SCAN, 2048.0 * ntiles, k_inv_tile_base, nchunks, 256, tilehist, ntiles, chunksum);
    ctx->phase = 1;
    if (div_primary)
        LAUNCH(KC_INV_LF, 5.0 * n, k_inv_lf_rank<true>, ntiles, INV_NT, dB, n, tilehist, prev, div_primary, Ctab, small + 20);
    else
        LAUNCH(KC_INV_LF, 5.0 * n, k_inv_lf_rank, ntiles, INV_NT, dB, n, tilehist, prev);

    // -- splitters
    ctx->phase = 2;
    CK(cudaMemsetAsync(len_at_min, 0, (size_t)n * 4, st));
    LAUNCH(KC_INV_WALK, 0, k_inv_spl_count, nst, 256, n, h, tilecnt);
    LAUNCH(KC_INV_SCAN, 8.0 * nst, k_scan_excl_u32_block, 1, 1024, tilecnt, tilecnt, nst, small + 0);
    int rc = readback(ctx, st, small, 4);
    if (rc) return rc;
    const u32 ns = ctx->h_small[0];
    if (ns < 1 || ns > n) return BWTS_B200_EINTERNAL;
    u32 *spl = arena_take<u32>(ctx, ns);
    u64 *jm[3] = {arena_take<u64>(ctx, ns), arena_take<u64>(ctx, ns), arena_take<u64>(ctx, ns)};
    u64 *pv[2] = {arena_take<u64>(ctx, ns), arena_take<u64>(ctx, ns)};
    u32 *wlen = arena_take<u32>(ctx, ns);
    uint2 *minfo = arena_take<uint2>(ctx, ns);
    uint4 *srec = arena_take<uint4>(ctx, ns);
    if (!spl || !jm[0] || !jm[1] || !jm[2] || !pv[0] || !pv[1] || !wlen || !minfo || !srec) return BWTS_B200_EINTERNAL;
    u32 *blkoff = nullptr, *nxt = nullptr, *cont = nullptr;
    u8 *stage = nullptr;
    // bytes parked per sublist: 4 x the mean sublist length (e^-4 = 1.8 % of the elements lie beyond)
    const u32 slot = min((u32)INV_SLOT_MAX, max(32u, (4u << (32 - shift)) & ~31u));
    if (staged) {
        blkoff = arena_take<u32>(ctx, (size_t)(n >> 6) + 2);
        nxt = arena_take<u32>(ctx, ns);
        cont = arena_take<u32>(ctx, ns);
        stage = arena_take<u8>(ctx, (size_t)ns * slot);
        if (!blkoff || !nxt || !cont || !stage) return BWTS_B200_EINTERNAL;
    }
    LAUNCH(KC_INV_WALK, 8.0 * ns, k_inv_spl_write, nst, 256, n, h, tilecnt, spl, staged ? (u32 *)nullptr : sid, blkoff);
    // who gets reached: one bit per element, or (staged path) one 8-bit count per 128 elements
    const size_t vwords = (size_t)(n >> 5) + 2, cwords = (size_t)(n >> 9) + 2;
    u32 *visited = arena_take<u32>(ctx, vwords);
    u32 *vcnt = count_marks ? arena_take<u32>(ctx, cwords) : (u32 *)nullptr;
    if (!visited || (count_marks && !vcnt)) return BWTS_B200_EINTERNAL;
    if (count_marks) CK(cudaMemsetAsync(vcnt, 0, cwords * 4, st));
    else CK(cudaMemsetAsync(visited, 0, vwords * 4, st));
    if (staged) {
        // one full wave of warps (64 per SM), each owning a contiguous range of Q sublists
        const u32 wave = (u32)ctx->sm_count * 64u;
        u32 Q = g_tune_invq > 0 ? (u32)g_tune_invq : max(64u, cdiv(ns, wave));
        const u32 nwarps = cdiv(ns, Q);
        LAUNCH(KC_INV_WALK, 5.0 * n, k_inv_walk_stage, cdiv(nwarps, 8), 256, prev, h, spl, ns, Q, Ctab, nxt, wlen, minfo,
               stage, slot, cont, (g_tune_nomark || count_marks) ? (u32 *)nullptr : visited, g_tune_nomark ? (u32 *)nullptr : vcnt,
               small + 2);
        LAUNCH(KC_INV_WALK, 20.0 * ns, k_inv_resolve_next, cdiv(ns, 256), 256, nxt, minfo, blkoff, h, ns, jm[0]);
    } else {
        LAUNCH(KC_INV_WALK, 4.0 * n, k_inv_walk, cdiv(ns, 128), 128, prev, h, spl, ns, sid, jm[0], wlen, minfo,
               g_tune_nomark ? (u32 *)nullptr : visited, small + 2);
    }

    // -- reduced list: cycle minimum, then distance to the sublist holding it
    ctx->phase = 3;
    const int R = bit_length((u64)ns - 1) + 1;
    const u32 gs = cdiv(ns, 256);
    int cur = 0;
    for (int r = 0; r < R; r++) {
        const int dst = (cur == 1) ? 2 : 1;
        LAUNCH(KC_INV_JUMP, 24.0 * ns, k_inv_min_jump, gs, 256, jm[cur], jm[dst], ns);
        cur = dst;
    }
    u64 *jmR = jm[cur];
    LAUNCH(KC_INV_JUMP, 32.0 * ns, k_inv_sum_init, gs, 256, jm[0], jmR, wlen, minfo, ns, pv[0]);
    int pc = 0;
    for (int r = 0; r < R; r++) {
        LAUNCH(KC_INV_JUMP, 24.0 * ns, k_inv_sum_jump, gs, 256, pv[pc], pv[pc ^ 1], ns);
        pc ^= 1;
    }
    LAUNCH(KC_INV_JUMP, 24.0 * ns, k_inv_origin_publish, gs, 256, jmR, pv[pc], minfo, ns, len_at_min, cyc);

    // -- did the walks reach every element?  (they do unless a cycle holds no splitter)
    rc = readback(ctx, st, small + 2, 4);
    if (rc) return rc;
    const u32 reached = ctx->h_small[0];
    uint2 *urec = nullptr;
    const u32 nwords = cdiv(n, 32);
    const u32 bk = budget_k ? budget_k : 0xffffffffu;
    if (reached != n && !g_tune_nomark) {
        ctx->phase = 2;
        if (count_marks) {
            // the blocks of 128 whose count is short hold the unreached elements: few blocks (the usual case:
            // a handful of short last factors) -> test their elements one by one; many -> mark exactly
            const u32 cap = max(4096u, n >> 13);
            u32 *deflist = arena_take<u32>(ctx, cap);
            if (!deflist) return BWTS_B200_EINTERNAL;
            LAUNCH(KC_INV_WALK, (double)(n >> 7), k_inv_find_deficient, cdiv(cdiv(n, 128), 256), 256, vcnt, n, deflist, cap, small + 10);
            rc = readback(ctx, st, small + 10, 4);
            if (rc) return rc;
            const u32 ndef = ctx->h_small[0];
            if (ndef <= cap) {
                CK(cudaMemsetAsync(visited, 0xff, vwords * 4, st));
                LAUNCH(KC_INV_WALK, 512.0 * ndef, k_inv_verify_candidates, cdiv((u64)ndef * 128, 128), 128, prev, n, h, deflist, ndef,
                       visited, small + 4, bk, small + 12);
            } else {
                CK(cudaMemsetAsync(visited, 0, vwords * 4, st));
                LAUNCH(KC_INV_WALK, 4.0 * n, k_inv_walk_mark, cdiv(ns, 128), 128, prev, h, spl, ns, visited);
            }
        }
        urec = arena_take<uint2>(ctx, n);
        if (!urec) return BWTS_B200_EINTERNAL;
        LAUNCH(KC_INV_WALK, 12.0 * (n - reached), k_inv_self_walk, cdiv(nwords, 256), 256, prev, n, visited, urec,
               len_at_min, small + 4, bk, small + 12);
        // out of budget: the records of the unreached elements are incomplete, nothing below may read them
        rc = readback(ctx, st, small + 12, 4);
        if (rc) return rc;
        if (ctx->h_small[0]) { *over = true; return 0; }
        ctx->phase = 3;
    }

    // -- offsets of the cycles, in order of ascending smallest index
    LAUNCH(KC_INV_SCAN, 4.0 * n, k_tile_sum_u32, nsc, 256, len_at_min, n, tilecnt, small + 6);  // also counts the cycles
    LAUNCH(KC_INV_SCAN, 8.0 * nsc, k_scan_excl_u32_block, 1, 1024, tilecnt, tilecnt, nsc, small + 8);
    LAUNCH(KC_INV_SCAN, 8.0 * n, k_tile_scan_apply_u32, nsc, 256, len_at_min, off, n, tilecnt);

    // -- placement
    ctx->phase = 4;
    LAUNCH(KC_INV_PLACE, 44.0 * ns, k_inv_spl_record, gs, 256, jmR, pv[pc], cyc, off, ns, srec);
    if (staged) {
        LAUNCH(KC_INV_PLACE, 2.0 * n + 20.0 * ns, k_inv_place_copy, cdiv(ns, 8), 256, stage, wlen, srec, ns, n, slot, d_out);
        LAUNCH(KC_INV_PLACE, 8.0 * ns, k_inv_walk_tail, cdiv(ns, 128), 128, prev, n, h, wlen, cont, ns, slot, srec, Ctab, d_out);
    } else {
        LAUNCH(KC_INV_PLACE, 5.0 * n, k_inv_walk_place, cdiv(ns, 128), 128, prev, n, h, spl, ns, srec, Ctab, d_out);
    }
    if (urec)
        LAUNCH(KC_INV_PLACE, 14.0 * (n - reached), k_inv_place_unreached, cdiv(nwords, 256), 256, dB, n, visited, urec,
               off, d_out);

    rc = readback(ctx, st, small, 56);
    if (rc) return rc;
    if (g_tune_nomark) return 0;                            // timing experiment, the output is not checked
    if (ctx->h_small[8] != n) return BWTS_B200_EINTERNAL;  // cycle lengths must add up to n
    if (bwt_out) {
        u32 *loc = small + 16;
        if (div_primary)
            LAUNCH(KC_INV_PLACE, 0, k_bwt_locate<true>, 1, 1, prev, h, primary, sid, blkoff, srec, off, loc, d_out, n, small + 20);
        else
            LAUNCH(KC_INV_PLACE, 0, k_bwt_locate, 1, 1, prev, h, primary, sid, blkoff, srec, off, loc);
        LAUNCH(KC_INV_PLACE, 2.0 * n, k_bwt_rotate, cdiv(cdiv(n, 16), 256), 256, d_out, n, loc, bwt_out);
    }
    ctx->stats.splitters = ns;
    ctx->stats.unreached = ctx->h_small[4];
    ctx->stats.factors = ctx->h_small[6];
    return 0;
}

// primary >= 0: classic inverse BWT (the BWTS layout goes to an n-byte scratch S in the workspace first);
// div: libdivsufsort's inverse_bw_transform with primary in [1, n], the classic path from row 0
static int inverse_core(bwts_b200_ctx *ctx, const u8 *dB, u32 n, u8 *d_out, cudaStream_t st, long primary = -1,
                        bool div = false)
{
    int rc = arena_reserve(ctx, workspace_bytes(n));
    if (rc) return rc;
    // A cycle that holds no splitter is ranked by its own members walking it: L steps each, L^2 per
    // cycle.  With random-looking hashing such cycles are short (a cycle of L elements is missed with
    // probability e^(-L / 64): at most ~24 steps per element on any input), so 32 n steps are a
    // generous budget; an input built against the public hash exceeds it and the inverse starts
    // again with another multiplier -- and four times the splitter density where the workspace has
    // room for it -- the last attempt unbounded.
    static const u32 muls[4] = {0x9E3779B1u, 0x85EBCA6Bu, 0xC2B2AE35u, 0x27D4EB2Fu};
    // one splitter per 64 elements; per 128 from 256 MiB on, where the 2 x 26 pointer-jumping rounds over the sublists
    // cost more than the longer sublists do (C4 inverse 57.1 -> 49.5 ms with 512-byte slots, C5 block 13.6 -> 13.2 ms; C2: 3.79 -> 4.25 ms)
    u32 shift = g_tune_spl_shift ? (u32)g_tune_spl_shift : (n >= (1u << 28) ? 25u : 26u);
    ctx->stats.inverse_attempts = 0;
    for (int a = 0; a < 4; a++) {
        ctx->arena_used = ctx->io_end;
        const u64 steps = g_tune_invbudget > 0 ? (u64)g_tune_invbudget : 32ull * n;
        u64 bk64 = steps >> 10;
        if (bk64 < 1) bk64 = 1;
        if (bk64 > 0xfffffffeull) bk64 = 0xfffffffeull;
        const u32 budget_k = (a == 3) ? 0u : (u32)bk64;
        bool over = false;
        ctx->stats.inverse_attempts++;
        if (primary >= 0) {
            u8 *S = arena_take<u8>(ctx, n);
            if (!S) return BWTS_B200_EINTERNAL;
            rc = inverse_attempt(ctx, dB, n, S, st, SplHash{muls[a], shift}, budget_k, &over, d_out, div ? 0u : (u32)primary,
                                 div ? (u32)primary : 0u);
        } else {
            rc = inverse_attempt(ctx, dB, n, d_out, st, SplHash{muls[a], shift}, budget_k, &over);
        }
        if (rc || !over) return rc;
        if (shift < 30) {
            // denser splitters if ~(80 + slot) bytes per sublist fit behind the per-element arrays (~33 n)
            const u32 s2 = shift + 2;
            const u64 ns2 = ((u64)n >> (32 - s2)) + 1024;
            u64 slot2 = (4ull << (32 - s2)) & ~31ull;
            if (slot2 < 32) slot2 = 32;
            if (slot2 > INV_SLOT_MAX) slot2 = INV_SLOT_MAX;
            const u64 need = (primary >= 0 ? 35ull : 34ull) * n + ns2 * (80 + slot2) * 5 / 4 + ctx->io_end + (16u << 20);
            if (need <= ctx->arena_bytes) shift = s2;
        }
    }
    return BWTS_B200_EINTERNAL;
}

// ---- contexts -------------------------------------------------------------------------------------
extern "C" int bwts_b200_device_count(void)
{
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
    return c;
}

extern "C" bwts_b200_ctx *bwts_b200_create(int device)
{
    if (device < 0 || device >= bwts_b200_device_count()) return nullptr;
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    // the sort kernels use > 48 KB of dynamic shared memory and want the large carveout
#define OS_ATTR(K_, NT_, IPT_, MINB_, LB_)                                                                          \
    cudaFuncSetAttribute(k_onesweep_pass<K_, NT_, IPT_, MINB_, LB_>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                         (int)OsSmem<K_, NT_, IPT_>::bytes);                                                         \
    cudaFuncSetAttribute(k_onesweep_pass<K_, NT_, IPT_, MINB_, LB_>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)
    OS_ATTR(u64, 384, 12, 3, 4);
    OS_ATTR(u64, 384, 12, 3, 8);
    OS_ATTR(u64, 384, 12, 3, 2);
    OS_ATTR(u64, 512, 8, 3, 8);
    OS_ATTR(u64, 256, 16, 3, 8);
    OS_ATTR(u32, 384, 12, 3, 4);
    cudaFuncSetAttribute(k_onesweep_pass<u32, 384, 12, 3, 4, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)OsSmem<u32, 384, 12>::bytes);
    cudaFuncSetAttribute(k_onesweep_pass<u32, 384, 12, 3, 4, 2>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaFuncSetAttribute(k_init_keys, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768);  // + 18.7 KB static: above 48 KB in all
    cudaFuncSetAttribute(k_local_sort_cta_radix<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LsrSmem::bytes);
    cudaFuncSetAttribute(k_local_sort_cta_radix<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LsrSmem::bytes);
    cudaFuncSetAttribute(k_local_sort_cta<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(LS_CAP * sizeof(u64)));
    cudaFuncSetAttribute(k_local_sort_cta<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(LS_CAP * sizeof(u64)));
    cudaFuncSetAttribute(k_lpf_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 << LZ_TB_MAX);
#undef OS_ATTR
    bwts_b200_ctx *ctx = new bwts_b200_ctx();
    ctx->device = device;
    if (cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || ctx->sm_count < 1)
        ctx->sm_count = 148;
    memset(&ctx->stats, 0, sizeof ctx->stats);
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaHostAlloc((void **)&ctx->h_small, 4096, cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer((void **)&ctx->h_small_dev, ctx->h_small, 0) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_begin) != cudaSuccess || cudaEventCreate(&ctx->ev_end) != cudaSuccess ||
        cudaEventCreate(&ctx->ev_io0) != cudaSuccess || cudaEventCreate(&ctx->ev_io1) != cudaSuccess) {
        bwts_b200_destroy(ctx);
        return nullptr;
    }
    return ctx;
}

extern "C" void bwts_b200_destroy(bwts_b200_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) { cudaStreamSynchronize(ctx->own_stream); cudaStreamDestroy(ctx->own_stream); }
    for (cudaEvent_t e : ctx->pool) cudaEventDestroy(e);
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->ev_io0) cudaEventDestroy(ctx->ev_io0);
    if (ctx->ev_io1) cudaEventDestroy(ctx->ev_io1);
    pipe_state_destroy(ctx);
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->h_small) cudaFreeHost(ctx->h_small);
    delete ctx;
}

extern "C" int bwts_b200_reserve(bwts_b200_ctx *ctx, long max_len)
{
    if (!ctx || max_len <= 0) return BWTS_B200_EINVAL;
    if (max_len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    CK(cudaSetDevice(ctx->device));
    // sized for the host-buffer calls too (their input and output live in front of the workspace)
    return arena_reserve(ctx, workspace_bytes((size_t)max_len) + 2 * (size_t)max_len + 1024);
}

// ---- the call frame --------------------------------------------------------------------------------
// host <-> device copies of the host-buffer entry points: pinned buffers go as one async copy,
// pageable ones (the tools' mmap'ed input, map_file.c, and malloc'ed output) through the context's
// ring of pinned chunks -- the memcpy into chunk c+1 runs while chunk c is on the bus, where a
// pageable cudaMemcpy stages serially inside the driver.  Defined behind PinnedRing.
static int stage_h2d(bwts_b200_ctx *ctx, u8 *d_dst, const u8 *src, size_t len, cudaStream_t st);
static int stage_d2h(bwts_b200_ctx *ctx, u8 *dst, const u8 *d_src, size_t len, cudaStream_t st);

// copies into the arena at byte `at` before the core runs, and out of it after
struct CopyIn { size_t at; const void *src; size_t bytes; };
struct CopyOut { size_t at; void *dst; size_t bytes; };
// What an entry point states about one call: the stats header, the arena bytes it reserves (workspace and I/O
// region), the I/O region's end (the cores allocate their workspace from there up) and its copies.  A host form
// copies in[] host -> device and out[] device -> host, timed into stats.h2d_ms / d2h_ms; a device form copies in[]
// device -> device (an input its kernels cannot read where it lies) and has no out[].
struct Frame {
    long len;
    int direction;
    size_t arena, io_end;
    bool host;
    CopyIn in[2];
    CopyOut out[2];  // the core may set the sizes of what is known only once it has run
};

// The bracket around every entry point's core: device, stream (stream: a device form's, else nullptr for the
// context's own), workspace, limits, copies in, stats, core, stats, copies out.  On an error of the core the stream
// is drained, the error cleared and the code returned without stats_end.
template <typename Core>
static int run_frame(bwts_b200_ctx *ctx, void *stream, Frame &f, Core &&core)
{
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->own_stream;
    int rc = arena_reserve(ctx, f.arena);
    if (rc) return rc;
    apply_device_limits();
    if (f.host) CK(cudaEventRecord(ctx->ev_io0, st));
    for (const CopyIn &c : f.in) {
        if (!c.bytes) continue;
        if (!f.host) CK(cudaMemcpyAsync(ctx->arena + c.at, c.src, c.bytes, cudaMemcpyDeviceToDevice, st));
        else if ((rc = stage_h2d(ctx, ctx->arena + c.at, (const u8 *)c.src, c.bytes, st))) return rc;
    }
    ctx->io_end = f.io_end;
    stats_begin(ctx, f.len, f.direction, st);
    rc = core(st);
    ctx->io_end = 0;
    if (rc) { cudaStreamSynchronize(st); cudaGetLastError(); return rc; }
    stats_end(ctx, st);
    if (!f.host) {
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { ctx->last_cuda = (int)e; return BWTS_B200_ECUDA; }
        return 0;
    }
    size_t copied = 0;
    for (const CopyOut &c : f.out) {
        if (!c.bytes) continue;
        if ((rc = stage_d2h(ctx, (u8 *)c.dst, ctx->arena + c.at, c.bytes, st))) return rc;
        copied += c.bytes;
    }
    CK(cudaEventRecord(ctx->ev_io1, st));
    CK(cudaStreamSynchronize(st));
    float t = 0;
    if (cudaEventElapsedTime(&t, ctx->ev_io0, ctx->ev_begin) == cudaSuccess) ctx->stats.h2d_ms = t;
    if (copied && cudaEventElapsedTime(&t, ctx->ev_end, ctx->ev_io1) == cudaSuccess) ctx->stats.d2h_ms = t;
    return 0;
}

// A device form over a text.  The text kernels read 16-byte vectors: a text that is not 16-byte aligned (a slice
// of a larger buffer) is first copied to the bottom of the arena, and the core reads it there.
template <typename Core>
static int run_text_device(bwts_b200_ctx *ctx, const void *d_in, long len, int direction, void *stream, Core &&core)
{
    const bool copy = (uintptr_t)d_in & 15;
    Frame f = {len, direction, workspace_bytes((size_t)len) + (copy ? 2 * (size_t)len + 1024 : 0), copy ? r256(len) : 0,
               false};
    if (copy) f.in[0] = {0, d_in, (size_t)len};
    return run_frame(ctx, stream, f, [&](cudaStream_t st) { return core(copy ? ctx->arena : (const u8 *)d_in, st); });
}

static int check_len(const void *in, long len, void *out)
{
    if (!in || !out || len <= 0) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    return 0;
}

// What a call computes.  The classic BWT and divbwt ops take a primary index: the forward writes it, the
// inverse reads it (classic: a row in [0, len); divbwt: where the end of text stood, in [1, len]).
enum Op { OP_FORWARD = 0, OP_INVERSE = 1, OP_BWT_FORWARD = 2, OP_BWT_INVERSE = 3, OP_DIVBWT_FORWARD = 4, OP_DIVBWT_INVERSE = 5 };
static inline int op_direction(int op) { return op & 1; }  // stats.direction: 0 forward, 1 inverse

static int check_primary(int op, long len, const long *primary)
{
    if (op < OP_BWT_FORWARD) return 0;
    if (!primary) return BWTS_B200_EINVAL;
    if (op == OP_BWT_INVERSE && (*primary < 0 || *primary >= len)) return BWTS_B200_EINVAL;
    if (op == OP_DIVBWT_INVERSE && (*primary < 1 || *primary > len)) return BWTS_B200_EINVAL;
    return 0;
}

static int run_core(bwts_b200_ctx *ctx, int op, const u8 *d_in, u32 n, u8 *d_out, long *primary, cudaStream_t st)
{
    switch (op) {
    case OP_FORWARD: return forward_core(ctx, d_in, n, d_out, nullptr, FWD_BWTS, st);
    case OP_INVERSE: return inverse_core(ctx, d_in, n, d_out, st);
    case OP_BWT_FORWARD: return forward_core(ctx, d_in, n, d_out, nullptr, FWD_BWT, st, primary);
    case OP_BWT_INVERSE: return inverse_core(ctx, d_in, n, d_out, st, *primary);
    case OP_DIVBWT_FORWARD: return forward_core(ctx, d_in, n, d_out, nullptr, FWD_DIVBWT, st, primary);
    case OP_DIVBWT_INVERSE: return inverse_core(ctx, d_in, n, d_out, st, *primary, true);
    }
    return BWTS_B200_EINVAL;
}

static int run_device(bwts_b200_ctx *ctx, int op, const void *d_in, long len, void *d_out, void *stream,
                      long *primary = nullptr)
{
    if (!ctx) return BWTS_B200_EINVAL;
    int rc = check_len(d_in, len, d_out);
    if (!rc) rc = check_primary(op, len, primary);
    if (rc) return rc;
    return run_text_device(ctx, d_in, len, op_direction(op), stream, [&](const u8 *d_text, cudaStream_t st) {
        return run_core(ctx, op, d_text, (u32)len, (u8 *)d_out, primary, st);
    });
}

extern "C" int bwts_b200_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, void *stream)
{
    return run_device(ctx, OP_FORWARD, d_in, len, d_out, stream);
}
extern "C" int bwts_b200_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, void *stream)
{
    return run_device(ctx, OP_INVERSE, d_in, len, d_out, stream);
}
extern "C" int bwts_b200_bwt_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, long *primary,
                                            void *stream)
{
    return run_device(ctx, OP_BWT_FORWARD, d_in, len, d_out, stream, primary);
}
extern "C" int bwts_b200_bwt_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, long primary, void *d_out,
                                            void *stream)
{
    return run_device(ctx, OP_BWT_INVERSE, d_in, len, d_out, stream, &primary);
}
extern "C" int bwts_b200_divbwt_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, long *primary,
                                               void *stream)
{
    return run_device(ctx, OP_DIVBWT_FORWARD, d_in, len, d_out, stream, primary);
}
extern "C" int bwts_b200_divbwt_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, long primary, void *d_out,
                                               void *stream)
{
    return run_device(ctx, OP_DIVBWT_INVERSE, d_in, len, d_out, stream, &primary);
}

#define MAX_DEV 64
static std::mutex g_dev_mutex[MAX_DEV];
static bwts_b200_ctx *g_dev_ctx[MAX_DEV];

// The per-device context behind the one-call entry points and the block dealer, created on first use and returned
// with the device's mutex held in lock.  Nobody can ask it for statistics, so it records no per-launch events (two
// cudaEventRecord per kernel are a quarter of a small transform's time: ~120 launches for a 1 MiB input).
// BWTS_B200_PROFILE=1 switches them back on.
static int default_ctx(int device, std::unique_lock<std::mutex> &lock, bwts_b200_ctx *&ctx)
{
    const int ndev = bwts_b200_device_count();
    if (ndev == 0) return BWTS_B200_ENODEV;
    if (device < 0 || device >= ndev || device >= MAX_DEV) return BWTS_B200_EINVAL;
    lock = std::unique_lock<std::mutex>(g_dev_mutex[device]);
    if (!g_dev_ctx[device]) {
        g_dev_ctx[device] = bwts_b200_create(device);
        if (g_dev_ctx[device] && !getenv("BWTS_B200_PROFILE") && !getenv("BWTS_B200_TRACE")) g_dev_ctx[device]->profile = false;
    }
    ctx = g_dev_ctx[device];
    return ctx ? 0 : BWTS_B200_ENODEV;
}

static int run_host(bwts_b200_ctx *ctx, int op, const unsigned char *in, long len, unsigned char *out,
                    long *primary = nullptr)
{
    if (!ctx) return BWTS_B200_EINVAL;
    int rc = check_len(in, len, out);
    if (!rc) rc = check_primary(op, len, primary);
    if (rc) return rc;
    // the input and the output in front of the workspace
    const size_t io = r256((size_t)len);
    Frame f = {len, op_direction(op), workspace_bytes((size_t)len) + 2 * (size_t)len + 1024, 2 * io, true};
    f.in[0] = {0, in, (size_t)len};
    f.out[0] = {io, out, (size_t)len};
    return run_frame(ctx, nullptr, f, [&](cudaStream_t st) {
        return run_core(ctx, op, ctx->arena, (u32)len, ctx->arena + io, primary, st);
    });
}

extern "C" int bwts_b200_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out)
{
    return run_host(ctx, OP_FORWARD, in, len, out);
}
extern "C" int bwts_b200_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out)
{
    return run_host(ctx, OP_INVERSE, in, len, out);
}
extern "C" int bwts_b200_bwt_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out,
                                          long *primary)
{
    return run_host(ctx, OP_BWT_FORWARD, in, len, out, primary);
}
extern "C" int bwts_b200_bwt_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, long primary,
                                          unsigned char *out)
{
    return run_host(ctx, OP_BWT_INVERSE, in, len, out, &primary);
}
extern "C" int bwts_b200_divbwt_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out,
                                             long *primary)
{
    return run_host(ctx, OP_DIVBWT_FORWARD, in, len, out, primary);
}
extern "C" int bwts_b200_divbwt_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, long primary,
                                             unsigned char *out)
{
    return run_host(ctx, OP_DIVBWT_INVERSE, in, len, out, &primary);
}

// ---- one-call entry points ---------------------------------------------------------------------------

static int with_default_ctx(int device, int op, const unsigned char *in, long len, unsigned char *out,
                            long *primary = nullptr)
{
    int rc = check_len(in, len, out);
    if (!rc) rc = check_primary(op, len, primary);
    std::unique_lock<std::mutex> lock;
    bwts_b200_ctx *ctx = nullptr;
    if (!rc) rc = default_ctx(device, lock, ctx);
    return rc ? rc : run_host(ctx, op, in, len, out, primary);
}

extern "C" int bwts_b200_forward(const unsigned char *in, long len, unsigned char *out, int device)
{
    return with_default_ctx(device, OP_FORWARD, in, len, out);
}
extern "C" int bwts_b200_inverse(const unsigned char *in, long len, unsigned char *out, int device)
{
    return with_default_ctx(device, OP_INVERSE, in, len, out);
}
extern "C" int bwts_b200_bwt_forward(const unsigned char *in, long len, unsigned char *out, long *primary, int device)
{
    return with_default_ctx(device, OP_BWT_FORWARD, in, len, out, primary);
}
extern "C" int bwts_b200_bwt_inverse(const unsigned char *in, long len, long primary, unsigned char *out, int device)
{
    return with_default_ctx(device, OP_BWT_INVERSE, in, len, out, &primary);
}
// libdivsufsort's signatures.  A (its temporary array) is never touched; U may be T: the input is on the
// device before the first output byte comes back.
extern "C" int bwts_b200_divbwt(const unsigned char *T, unsigned char *U, int *A, int n, int device)
{
    (void)A;
    if (!T || !U || n < 0) return BWTS_B200_EINVAL;
    if (n == 0) return 0;
    long primary = 0;
    const int rc = with_default_ctx(device, OP_DIVBWT_FORWARD, T, n, U, &primary);
    return rc ? rc : (int)primary;
}
extern "C" int bwts_b200_inverse_bw_transform(const unsigned char *T, unsigned char *U, int *A, int n, int idx, int device)
{
    (void)A;
    if (!T || !U || n < 0 || idx < 0 || idx > n || (idx == 0 && n > 0)) return BWTS_B200_EINVAL;
    if (n == 0) return 0;
    long primary = idx;
    return with_default_ctx(device, OP_DIVBWT_INVERSE, T, n, U, &primary);
}

// ---- independent blocks: per device a three-stage pipeline ------------------------------------------
// SURVEY.md 8f row 1 (the steps either side of the hot path: map_file.c:16-46 before it,
// mk_bwts_sa.c:60 / unbwts.c:173 after it).  For the blocks dealt to one device:
//     loader    host bytes -> pinned chunk ring -> H2D on its own stream      (block b+1)
//     compute   the transform on the context's stream                        (block b)
//     drainer   D2H on its own stream -> pinned chunk ring -> caller's bytes  (block b-1)
// Two device input and two device output buffers; counting semaphores hand blocks from stage
// to stage.  Caller buffers that are already pinned (cudaHostAlloc / cudaHostRegister) skip the
// chunk rings and are copied directly.  tune(5, 1) turns the overlap off (one block at a time).
#include <condition_variable>

struct Sema {
    std::mutex m;
    std::condition_variable cv;
    long count;
    explicit Sema(long c) : count(c) {}
    void release() { { std::lock_guard<std::mutex> l(m); count++; } cv.notify_one(); }
    void acquire() { std::unique_lock<std::mutex> l(m); cv.wait(l, [&] { return count > 0; }); count--; }
};

#define PIPE_CHUNK ((size_t)8 << 20)
#define PIPE_NCHUNK 4

static bool host_ptr_is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

struct PinnedRing {
    u8 *buf[PIPE_NCHUNK] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev[PIPE_NCHUNK] = {nullptr, nullptr, nullptr, nullptr};
    bool busy[PIPE_NCHUNK] = {false, false, false, false};
    int init()
    {
        for (int i = 0; i < PIPE_NCHUNK; i++) {
            if (cudaHostAlloc((void **)&buf[i], PIPE_CHUNK, cudaHostAllocDefault) != cudaSuccess) return BWTS_B200_ENOMEM;
            if (cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming) != cudaSuccess) return BWTS_B200_ECUDA;
        }
        return 0;
    }
    void destroy()
    {
        for (int i = 0; i < PIPE_NCHUNK; i++) {
            if (ev[i]) cudaEventDestroy(ev[i]);
            if (buf[i]) cudaFreeHost(buf[i]);
        }
    }
};

static void pipe_state_destroy(bwts_b200_ctx *ctx)
{
    if (ctx->pipe_ring_in) { ctx->pipe_ring_in->destroy(); delete ctx->pipe_ring_in; ctx->pipe_ring_in = nullptr; }
    if (ctx->pipe_ring_out) { ctx->pipe_ring_out->destroy(); delete ctx->pipe_ring_out; ctx->pipe_ring_out = nullptr; }
    for (int i = 0; i < 2; i++)
        if (ctx->pipe_ev_loaded[i]) { cudaEventDestroy(ctx->pipe_ev_loaded[i]); ctx->pipe_ev_loaded[i] = nullptr; }
    if (ctx->pipe_s_in) { cudaStreamDestroy(ctx->pipe_s_in); ctx->pipe_s_in = nullptr; }
    if (ctx->pipe_s_out) { cudaStreamDestroy(ctx->pipe_s_out); ctx->pipe_s_out = nullptr; }
    if (ctx->pipe_io) { cudaFree(ctx->pipe_io); ctx->pipe_io = nullptr; ctx->pipe_io_bytes = 0; }
}

// host -> device, through the ring when the source is pageable; returns after the copies are ISSUED
static int pipe_h2d(PinnedRing &ring, bool pinned, u8 *d_dst, const u8 *src, size_t len, cudaStream_t st, size_t &seq)
{
    if (pinned) return cudaMemcpyAsync(d_dst, src, len, cudaMemcpyHostToDevice, st) == cudaSuccess ? 0 : BWTS_B200_ECUDA;
    for (size_t off = 0; off < len; off += PIPE_CHUNK, seq++) {
        const int c = (int)(seq % PIPE_NCHUNK);
        const size_t l = len - off < PIPE_CHUNK ? len - off : PIPE_CHUNK;
        if (ring.busy[c] && cudaEventSynchronize(ring.ev[c]) != cudaSuccess) return BWTS_B200_ECUDA;
        memcpy(ring.buf[c], src + off, l);
        if (cudaMemcpyAsync(d_dst + off, ring.buf[c], l, cudaMemcpyHostToDevice, st) != cudaSuccess ||
            cudaEventRecord(ring.ev[c], st) != cudaSuccess)
            return BWTS_B200_ECUDA;
        ring.busy[c] = true;
    }
    return 0;
}

// device -> host, complete on return; the copy of chunk i+1 runs while chunk i is moved to the caller's buffer
static int pipe_d2h(PinnedRing &ring, bool pinned, u8 *dst, const u8 *d_src, size_t len, cudaStream_t st)
{
    if (pinned) {
        if (cudaMemcpyAsync(dst, d_src, len, cudaMemcpyDeviceToHost, st) != cudaSuccess) return BWTS_B200_ECUDA;
        return cudaStreamSynchronize(st) == cudaSuccess ? 0 : BWTS_B200_ECUDA;
    }
    const size_t nch = (len + PIPE_CHUNK - 1) / PIPE_CHUNK;
    for (size_t i = 0; i <= nch; i++) {
        if (i < nch) {
            const int c = (int)(i % PIPE_NCHUNK);
            const size_t off = i * PIPE_CHUNK, l = len - off < PIPE_CHUNK ? len - off : PIPE_CHUNK;
            if (cudaMemcpyAsync(ring.buf[c], d_src + off, l, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaEventRecord(ring.ev[c], st) != cudaSuccess)
                return BWTS_B200_ECUDA;
        }
        if (i >= 1) {  // chunk i-1 has been in flight while chunk i was issued
            const int c = (int)((i - 1) % PIPE_NCHUNK);
            const size_t off = (i - 1) * PIPE_CHUNK, l = len - off < PIPE_CHUNK ? len - off : PIPE_CHUNK;
            if (cudaEventSynchronize(ring.ev[c]) != cudaSuccess) return BWTS_B200_ECUDA;
            memcpy(dst + off, ring.buf[c], l);
        }
    }
    return 0;
}

static int stage_h2d(bwts_b200_ctx *ctx, u8 *d_dst, const u8 *src, size_t len, cudaStream_t st)
{
    bool pinned = len < 2 * PIPE_CHUNK || host_ptr_is_pinned(src);
    if (!pinned && !ctx->pipe_ring_in) {
        ctx->pipe_ring_in = new PinnedRing();
        if (ctx->pipe_ring_in->init() != 0) {  // no pinned memory to be had: the plain copy still works
            ctx->pipe_ring_in->destroy(); delete ctx->pipe_ring_in; ctx->pipe_ring_in = nullptr;
            cudaGetLastError();
            pinned = true;
        }
    }
    if (pinned) {
        CK(cudaMemcpyAsync(d_dst, src, len, cudaMemcpyHostToDevice, st));
        return 0;
    }
    size_t seq = 0;
    const int rc = pipe_h2d(*ctx->pipe_ring_in, false, d_dst, src, len, st, seq);
    if (rc) ctx->last_cuda = (int)cudaGetLastError();
    return rc;
}
static int stage_d2h(bwts_b200_ctx *ctx, u8 *dst, const u8 *d_src, size_t len, cudaStream_t st)
{
    bool pinned = len < 2 * PIPE_CHUNK || host_ptr_is_pinned(dst);
    if (!pinned && !ctx->pipe_ring_out) {
        ctx->pipe_ring_out = new PinnedRing();
        if (ctx->pipe_ring_out->init() != 0) {
            ctx->pipe_ring_out->destroy(); delete ctx->pipe_ring_out; ctx->pipe_ring_out = nullptr;
            cudaGetLastError();
            pinned = true;
        }
    }
    if (pinned) {
        CK(cudaMemcpyAsync(dst, d_src, len, cudaMemcpyDeviceToHost, st));
        return 0;
    }
    const int rc = pipe_d2h(*ctx->pipe_ring_out, false, dst, d_src, len, st);
    if (rc) ctx->last_cuda = (int)cudaGetLastError();
    return rc;
}

static long g_tune_pipeline = 0;  // 1 = no overlap between blocks on one device

// all blocks b = first, first + stride, ... < nblocks on device `dev`; primary[b]: block b's primary index
// (classic BWT and divbwt ops only, else nullptr)
static int run_blocks_on_device(int op, const u8 *in, long len, long block_len, u8 *out, long *primary, int dev,
                                long first, long stride, long nblocks)
{
    std::vector<long> mine;
    for (long b = first; b < nblocks; b += stride) mine.push_back(b);
    if (mine.empty()) return 0;
    // the device's cached context (and its workspace) serves all blocks of this call
    std::unique_lock<std::mutex> lock;
    bwts_b200_ctx *ctx = nullptr;
    if (const int rc = default_ctx(dev, lock, ctx)) return rc;
    if (cudaSetDevice(dev) != cudaSuccess) return BWTS_B200_ECUDA;
    auto blk_off = [&](long b) { return b * block_len; };
    auto blk_len = [&](long b) { return (blk_off(b) + block_len <= len) ? block_len : len - blk_off(b); };

    if (g_tune_pipeline == 1 || mine.size() == 1) {
        int rc = 0;
        for (size_t i = 0; i < mine.size() && rc == 0; i++)
            rc = run_host(ctx, op, in + blk_off(mine[i]), blk_len(mine[i]), out + blk_off(mine[i]),
                          primary ? primary + mine[i] : nullptr);
        return rc;
    }

    const bool dbg = getenv("BWTS_B200_PIPE_DEBUG") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
    const bool in_pinned = host_ptr_is_pinned(in), out_pinned = host_ptr_is_pinned(out);
    const size_t slot_bytes = ((size_t)block_len + 255) & ~(size_t)255;
    std::atomic<int> status{0};
    auto fail = [&](int rc) { int z = 0; status.compare_exchange_strong(z, rc); };

    int rc = arena_reserve(ctx, workspace_bytes((size_t)block_len));
    if (rc == 0 && ctx->pipe_io_bytes < 4 * slot_bytes) {
        if (ctx->pipe_io) { cudaFree(ctx->pipe_io); ctx->pipe_io = nullptr; ctx->pipe_io_bytes = 0; }
        if (cudaMalloc((void **)&ctx->pipe_io, 4 * slot_bytes) != cudaSuccess) { cudaGetLastError(); rc = BWTS_B200_ENOMEM; }
        else ctx->pipe_io_bytes = 4 * slot_bytes;
    }
    if (rc == 0 && !ctx->pipe_s_in &&
        (cudaStreamCreateWithFlags(&ctx->pipe_s_in, cudaStreamNonBlocking) != cudaSuccess ||
         cudaStreamCreateWithFlags(&ctx->pipe_s_out, cudaStreamNonBlocking) != cudaSuccess ||
         cudaEventCreateWithFlags(&ctx->pipe_ev_loaded[0], cudaEventDisableTiming) != cudaSuccess ||
         cudaEventCreateWithFlags(&ctx->pipe_ev_loaded[1], cudaEventDisableTiming) != cudaSuccess))
        rc = BWTS_B200_ECUDA;
    if (rc == 0 && !in_pinned && !ctx->pipe_ring_in) {
        ctx->pipe_ring_in = new PinnedRing();
        rc = ctx->pipe_ring_in->init();
    }
    if (rc == 0 && !out_pinned && !ctx->pipe_ring_out) {
        ctx->pipe_ring_out = new PinnedRing();
        rc = ctx->pipe_ring_out->init();
    }
    if (rc) {  // a half-built pipeline must not survive into the next call
        pipe_state_destroy(ctx);
        return rc;
    }
    u8 *d_io = ctx->pipe_io;
    cudaStream_t s_in = ctx->pipe_s_in, s_out = ctx->pipe_s_out;
    cudaEvent_t *ev_loaded = ctx->pipe_ev_loaded;
    PinnedRing dummy_ring;
    PinnedRing &ring_in = ctx->pipe_ring_in ? *ctx->pipe_ring_in : dummy_ring;
    PinnedRing &ring_out = ctx->pipe_ring_out ? *ctx->pipe_ring_out : dummy_ring;
    for (int c = 0; c < PIPE_NCHUNK; c++) { ring_in.busy[c] = false; }
    if (dbg) fprintf(stderr, "[pipe dev %d] setup %.2f ms (pinned in/out %d/%d, %zu blocks)\n", dev, since(), (int)in_pinned, (int)out_pinned, mine.size());
    if (rc == 0) {
        u8 *d_in[2] = {d_io, d_io + slot_bytes}, *d_out[2] = {d_io + 2 * slot_bytes, d_io + 3 * slot_bytes};
        Sema in_free(2), in_ready(0), out_free(2), out_ready(0);
        const size_t K = mine.size();

        std::thread loader([&]() {
            cudaSetDevice(dev);
            size_t seq = 0;
            for (size_t i = 0; i < K; i++) {
                in_free.acquire();
                if (status.load() == 0) {
                    const long b = mine[i];
                    int r = pipe_h2d(ring_in, in_pinned, d_in[i & 1], in + blk_off(b), (size_t)blk_len(b), s_in, seq);
                    if (r == 0 && cudaEventRecord(ev_loaded[i & 1], s_in) != cudaSuccess) r = BWTS_B200_ECUDA;
                    if (r) fail(r);
                }
                in_ready.release();
            }
        });
        std::thread drainer([&]() {
            cudaSetDevice(dev);
            for (size_t i = 0; i < K; i++) {
                out_ready.acquire();
                if (status.load() == 0) {
                    const long b = mine[i];
                    const int r = pipe_d2h(ring_out, out_pinned, out + blk_off(b), d_out[i & 1], (size_t)blk_len(b), s_out);
                    if (r) fail(r);
                }
                out_free.release();
            }
        });
        // compute stage on this thread
        cudaStream_t st = ctx->own_stream;
        for (size_t i = 0; i < K; i++) {
            in_ready.acquire();
            out_free.acquire();
            if (status.load() == 0) {
                const long b = mine[i];
                int r = 0;
                if (cudaStreamWaitEvent(st, ev_loaded[i & 1], 0) != cudaSuccess) r = BWTS_B200_ECUDA;
                const double t0 = since();
                if (r == 0)
                    r = run_device(ctx, op, d_in[i & 1], blk_len(b), d_out[i & 1], nullptr, primary ? primary + b : nullptr);
                if (dbg) fprintf(stderr, "[pipe dev %d] block %zu: waited until %.2f, transform %.2f ms (device %.2f)\n", dev, i, t0, since() - t0, ctx->stats.total_ms);
                if (r) fail(r);
            }
            in_free.release();
            out_ready.release();
        }
        loader.join();
        drainer.join();
        rc = status.load();
    }
    if (dbg) fprintf(stderr, "[pipe dev %d] pipeline done at %.2f ms\n", dev, since());
    cudaStreamSynchronize(s_in);
    cudaStreamSynchronize(s_out);
    if (dbg) fprintf(stderr, "[pipe dev %d] teardown done at %.2f ms\n", dev, since());
    return rc;
}

static int run_blocks(int op, const unsigned char *in, long len, long block_len, unsigned char *out, long *primary,
                      const int *devices, int ndev)
{
    if (!in || !out || len <= 0 || ndev < 1) return BWTS_B200_EINVAL;
    if (block_len <= 0 || block_len > len) block_len = len;
    if (block_len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    if (op >= OP_BWT_FORWARD && !primary) return BWTS_B200_EINVAL;
    if (op == OP_BWT_INVERSE || op == OP_DIVBWT_INVERSE) {  // every block's index against that block's length, before any work
        const long lo = op == OP_DIVBWT_INVERSE ? 1 : 0;      // [0, len) for the classic row, [1, len] for divbwt
        for (long b = 0, off = 0; off < len; b++, off += block_len)
            if (primary[b] < lo || primary[b] >= (len - off < block_len ? len - off : block_len) + lo) return BWTS_B200_EINVAL;
    }
    const int have = bwts_b200_device_count();
    if (have == 0) return BWTS_B200_ENODEV;
    std::vector<int> dev(ndev);
    for (int i = 0; i < ndev; i++) {
        dev[i] = devices ? devices[i] : i;
        if (dev[i] < 0 || dev[i] >= have) return BWTS_B200_EINVAL;
    }
    const long nblocks = (len + block_len - 1) / block_len;
    std::vector<int> status(ndev, 0);
    std::vector<std::thread> workers;
    for (int w = 0; w < ndev; w++)
        workers.emplace_back([&, w]() {
            status[w] = run_blocks_on_device(op, in, len, block_len, out, primary, dev[w], w, ndev, nblocks);
        });
    for (std::thread &t : workers) t.join();
    for (int w = 0; w < ndev; w++)
        if (status[w]) return status[w];
    return 0;
}

extern "C" int bwts_b200_forward_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                        const int *devices, int ndev)
{
    return run_blocks(OP_FORWARD, in, len, block_len, out, nullptr, devices, ndev);
}
extern "C" int bwts_b200_inverse_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                        const int *devices, int ndev)
{
    return run_blocks(OP_INVERSE, in, len, block_len, out, nullptr, devices, ndev);
}
extern "C" int bwts_b200_bwt_forward_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                            long *primary, const int *devices, int ndev)
{
    return run_blocks(OP_BWT_FORWARD, in, len, block_len, out, primary, devices, ndev);
}
extern "C" int bwts_b200_bwt_inverse_blocks(const unsigned char *in, long len, long block_len, const long *primary,
                                            unsigned char *out, const int *devices, int ndev)
{
    // read only: the inverse never writes through it
    return run_blocks(OP_BWT_INVERSE, in, len, block_len, out, (long *)primary, devices, ndev);
}
extern "C" int bwts_b200_divbwt_forward_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                               long *primary, const int *devices, int ndev)
{
    return run_blocks(OP_DIVBWT_FORWARD, in, len, block_len, out, primary, devices, ndev);
}
extern "C" int bwts_b200_divbwt_inverse_blocks(const unsigned char *in, long len, long block_len, const long *primary,
                                               unsigned char *out, const int *devices, int ndev)
{
    return run_blocks(OP_DIVBWT_INVERSE, in, len, block_len, out, (long *)primary, devices, ndev);
}

// ---- suffix array and LCP array ----------------------------------------------------------------------
// [a, a + na) and [b, b + nb) share a byte
static bool spans_overlap(const void *a, size_t na, const void *b, size_t nb)
{
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return x < y + nb && y < x + na;
}
// the bwts_b200_bwt_* rules, plus: no two of in, sa and lcp (if wanted) share a byte
static int check_sa_args(const void *in, long len, const void *sa, const void *lcp, bool want_lcp)
{
    if (!in || !sa || (want_lcp && !lcp) || len <= 0) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    const size_t n = (size_t)len;
    if (spans_overlap(in, n, sa, 4 * n)) return BWTS_B200_EINVAL;
    if (want_lcp && (spans_overlap(in, n, lcp, 4 * n) || spans_overlap(sa, 4 * n, lcp, 4 * n))) return BWTS_B200_EINVAL;
    return 0;
}

static int run_sa_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_sa, void *d_lcp, void *stream,
                         bool want_lcp)
{
    if (!ctx) return BWTS_B200_EINVAL;
    int rc = check_sa_args(d_in, len, d_sa, d_lcp, want_lcp);
    if (rc) return rc;
    if (((uintptr_t)d_sa & 3) || ((uintptr_t)d_lcp & 3)) return BWTS_B200_EINVAL;
    return run_text_device(ctx, d_in, len, 0, stream, [&](const u8 *d_text, cudaStream_t st) {
        return forward_core(ctx, d_text, (u32)len, nullptr, (i32 *)d_sa, FWD_SA, st, nullptr, want_lcp ? (i32 *)d_lcp : nullptr);
    });
}

// host buffers: the text, the suffix array and the LCP array (if wanted) in the I/O region in front of the
// workspace, 1 + 4 + 4 bytes per input byte; arguments already checked
static int run_sa_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *sa, int *lcp)
{
    const size_t io = r256((size_t)len), sa_bytes = r256((size_t)len * 4);
    const size_t out_bytes = lcp ? 2 * sa_bytes : sa_bytes;
    Frame f = {len, 0, workspace_bytes((size_t)len) + io + out_bytes + 1024, io + out_bytes, true};
    f.in[0] = {0, in, (size_t)len};
    f.out[0] = {io, sa, (size_t)len * 4};
    if (lcp) f.out[1] = {io + sa_bytes, lcp, (size_t)len * 4};
    return run_frame(ctx, nullptr, f, [&](cudaStream_t st) {
        return forward_core(ctx, ctx->arena, (u32)len, nullptr, (i32 *)(ctx->arena + io), FWD_SA, st, nullptr,
                            lcp ? (i32 *)(ctx->arena + io + sa_bytes) : nullptr);
    });
}

extern "C" int bwts_b200_sa_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *sa)
{
    if (!ctx) return BWTS_B200_EINVAL;
    const int rc = check_sa_args(in, len, sa, nullptr, false);
    return rc ? rc : run_sa_host(ctx, in, len, sa, nullptr);
}
extern "C" int bwts_b200_sa_lcp_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *sa, int *lcp)
{
    if (!ctx) return BWTS_B200_EINVAL;
    const int rc = check_sa_args(in, len, sa, lcp, true);
    return rc ? rc : run_sa_host(ctx, in, len, sa, lcp);
}
extern "C" int bwts_b200_sa_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_sa, void *stream)
{
    return run_sa_device(ctx, d_in, len, d_sa, nullptr, stream, false);
}
extern "C" int bwts_b200_sa_lcp_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_sa, void *d_lcp,
                                       void *stream)
{
    return run_sa_device(ctx, d_in, len, d_sa, d_lcp, stream, true);
}

// the one-call forms, on the per-device context of the other one-call functions; n == 0 returns 0
// libdivsufsort's seam
extern "C" int bwts_b200_divsufsort(const unsigned char *T, int *SA, int n, int device)
{
    if (!T || !SA || n < 0) return BWTS_B200_EINVAL;
    if (n == 0) return 0;
    std::unique_lock<std::mutex> lock;
    bwts_b200_ctx *ctx = nullptr;
    const int rc = default_ctx(device, lock, ctx);
    return rc ? rc : run_sa_host(ctx, T, n, SA, nullptr);
}
extern "C" int bwts_b200_sa_lcp(const unsigned char *T, int *SA, int *LCP, int n, int device)
{
    if (!T || !SA || !LCP || n < 0) return BWTS_B200_EINVAL;
    if (n == 0) return 0;
    int rc = check_sa_args(T, n, SA, LCP, true);
    std::unique_lock<std::mutex> lock;
    bwts_b200_ctx *ctx = nullptr;
    if (!rc) rc = default_ctx(device, lock, ctx);
    return rc ? rc : run_sa_host(ctx, T, n, SA, LCP);
}

// ---- longest-previous-factor array and LZ77 parse ---------------------------------------------------------------
// the bwts_b200_sa_* rules: no two of in, lpf and prev share a byte
static int check_lpf_args(const bwts_b200_ctx *ctx, const void *in, long len, const void *lpf, const void *prev)
{
    if (!ctx || !in || !lpf || !prev || len <= 0) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    const size_t n = (size_t)len;
    if (spans_overlap(in, n, lpf, 4 * n) || spans_overlap(in, n, prev, 4 * n) || spans_overlap(lpf, 4 * n, prev, 4 * n))
        return BWTS_B200_EINVAL;
    return 0;
}
// in and factors[0 .. 2 cap) share no byte; z is required, cap >= 0
static int check_lz_args(const bwts_b200_ctx *ctx, const void *in, long len, const void *factors, long cap, const long *z)
{
    if (!ctx || !in || !factors || !z || len <= 0 || cap < 0) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    if (spans_overlap(in, (size_t)len, factors, 8 * (size_t)min(cap, 1L << 56))) return BWTS_B200_EINVAL;
    return 0;
}

static int run_lz_device(bwts_b200_ctx *ctx, const void *d_in, long len, LzOut *lz, void *stream)
{
    return run_text_device(ctx, d_in, len, 0, stream, [&](const u8 *d_text, cudaStream_t st) {
        return forward_core(ctx, d_text, (u32)len, nullptr, nullptr, FWD_LZ, st, nullptr, nullptr, lz);
    });
}

// host buffers: the text and LPF + PREV, or up to n factor pairs, in the I/O region in front of the workspace,
// 1 + 8 bytes per input byte; arguments already checked
static int run_lz_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *lpf, int *prev, int *factors,
                       long cap, long *z)
{
    const size_t io = r256((size_t)len), w_bytes = r256((size_t)len * 4);
    Frame f = {len, 0, workspace_bytes((size_t)len) + io + 2 * w_bytes + 1024, io + 2 * w_bytes, true};
    f.in[0] = {0, in, (size_t)len};
    if (lpf) {
        f.out[0] = {io, lpf, (size_t)len * 4};
        f.out[1] = {io + w_bytes, prev, (size_t)len * 4};
    }
    return run_frame(ctx, nullptr, f, [&](cudaStream_t st) {
        LzOut o;
        if (lpf) { o.lpf = (i32 *)(ctx->arena + io); o.prev = (i32 *)(ctx->arena + io + w_bytes); }
        else { o.factors = (i32 *)(ctx->arena + io); o.cap = cap; }
        const int rc = forward_core(ctx, ctx->arena, (u32)len, nullptr, nullptr, FWD_LZ, st, nullptr, nullptr, &o);
        if (z && o.z >= 0) *z = o.z;
        if (!lpf && o.z > 0) f.out[0] = {io, factors, (size_t)o.z * 8};
        return rc;
    });
}

extern "C" int bwts_b200_lpf_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *lpf, int *prev)
{
    const int rc = check_lpf_args(ctx, in, len, lpf, prev);
    return rc ? rc : run_lz_host(ctx, in, len, lpf, prev, nullptr, 0, nullptr);
}
extern "C" int bwts_b200_lpf_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_lpf, void *d_prev, void *stream)
{
    const int rc = check_lpf_args(ctx, d_in, len, d_lpf, d_prev);
    if (rc) return rc;
    if (((uintptr_t)d_lpf & 3) || ((uintptr_t)d_prev & 3)) return BWTS_B200_EINVAL;
    LzOut o;
    o.lpf = (i32 *)d_lpf;
    o.prev = (i32 *)d_prev;
    return run_lz_device(ctx, d_in, len, &o, stream);
}
extern "C" int bwts_b200_lz77_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *factors, long cap, long *z)
{
    const int rc = check_lz_args(ctx, in, len, factors, cap, z);
    return rc ? rc : run_lz_host(ctx, in, len, nullptr, nullptr, factors, cap, z);
}
extern "C" int bwts_b200_lz77_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_factors, long cap, long *z,
                                     void *stream)
{
    int rc = check_lz_args(ctx, d_in, len, d_factors, cap, z);
    if (rc) return rc;
    if ((uintptr_t)d_factors & 3) return BWTS_B200_EINVAL;
    LzOut o;
    o.factors = (i32 *)d_factors;
    o.cap = cap;
    rc = run_lz_device(ctx, d_in, len, &o, stream);
    if (o.z >= 0) *z = o.z;
    return rc;
}

// ---- FM-index (fm.cuh) --------------------------------------------------------------------------------------
// One cudaMalloc per index, laid out in this order, every array rounded up to 256 bytes:
//     U n, S 4 sg (n/65536 + 1), B 2 sg (n/256 + 1), marks 4 ceil(n/32), dir 4 (n/256 + 1), samples 4 ceil(n/sample),
//     C 4 x 257, map 256
struct bwts_b200_fm {
    int device;
    u32 n, primary, sample, sg;
    u8 *mem;
    size_t bytes;
    FmView v;
};

static size_t fm_layout(u32 n, u32 sg, u32 sample, size_t off[9])
{
    const size_t sz[8] = {(size_t)n, 4ull * sg * ((n >> 16) + 1), 2ull * sg * ((n >> 8) + 1), 4ull * ((n + 31ull) / 32),
                          4ull * ((n >> 8) + 1), 4ull * ((n + (u64)sample - 1) / sample), 4 * 257, 256};
    off[0] = 0;
    for (int k = 0; k < 8; k++) off[k + 1] = off[k] + r256(sz[k]);
    return off[8];
}
static bool fm_sample_ok(int sample) { return sample >= 1 && sample <= 1024 && (sample & (sample - 1)) == 0; }

// The build: the byte histogram (C, the symbol map, sg, and so the index's size), the FWD_FM sort -- divbwt bytes
// into the index's U, the suffix array into the I/O region -- then the checkpoints, marks, directory and samples.
// The text lies at the bottom of the arena, in the I/O region (fm_build_io) the caller reserved.  *out is set once
// every launch is queued.
static int fm_build_core(bwts_b200_ctx *ctx, u32 n, u32 sample, bwts_b200_fm **out, cudaStream_t st)
{
    const u32 nb = (n >> 8) + 1, ns = (n >> 16) + 1;
    const u32 nt = cdiv(nb, SC_TILE);
    const u8 *d_text = ctx->arena;
    u8 *p = ctx->arena + r256(n);
    i32 *d_sa = (i32 *)p;            p += r256(4ull * n);
    u32 *dircnt = (u32 *)p;          p += r256(4ull * nb);
    u32 *tiles = (u32 *)p;           p += r256(4ull * (nt + 1));
    u32 *hist = (u32 *)p;            p += 1024;
    u8 *syms = p;                    p += 256;
    if ((size_t)(p - ctx->arena) > ctx->io_end) return BWTS_B200_EINTERNAL;

    ctx->phase = 3;
    CK(cudaMemsetAsync(hist, 0, 1024, st));
    LAUNCH(KC_EMIT, 1.0 * n, k_fm_hist, min(cdiv(n, 256), (u32)ctx->sm_count * 8), 256, d_text, n, hist);
    int rc = readback(ctx, st, hist, 1024);
    if (rc) return rc;
    ctx->phase = 0;
    std::vector<u32> C(257);
    std::vector<u8> map(256, 0), sy;
    u32 acc = 1;  // the end of text
    for (int c = 0; c < 256; c++) {
        C[c] = acc;
        acc += ctx->h_small[c];
        if (ctx->h_small[c]) { map[c] = (u8)sy.size(); sy.push_back((u8)c); }
    }
    C[256] = acc;
    const u32 sg = (u32)sy.size();
    size_t off[9];
    const size_t bytes = fm_layout(n, sg, sample, off);
    bwts_b200_fm *fm = new bwts_b200_fm();
    fm->device = ctx->device; fm->n = n; fm->sample = sample; fm->sg = sg; fm->bytes = bytes;
    const cudaError_t ea = cudaMalloc((void **)&fm->mem, bytes);
    if (ea != cudaSuccess) {
        delete fm;
        ctx->last_cuda = (int)ea;
        cudaGetLastError();
        return ea == cudaErrorMemoryAllocation ? BWTS_B200_ENOMEM : BWTS_B200_ECUDA;
    }
    u8 *U = fm->mem + off[0];
    u32 *S = (u32 *)(fm->mem + off[1]);
    u16 *B = (u16 *)(fm->mem + off[2]);
    u32 *marks = (u32 *)(fm->mem + off[3]), *dir = (u32 *)(fm->mem + off[4]), *samples = (u32 *)(fm->mem + off[5]);
    u32 *dC = (u32 *)(fm->mem + off[6]);
    u8 *dmap = fm->mem + off[7];
    const auto fail = [&](int code) { cudaStreamSynchronize(st); cudaGetLastError(); cudaFree(fm->mem); delete fm; return code; };
#define FCK(call) do { const cudaError_t e__ = (call); if (e__ != cudaSuccess) { ctx->last_cuda = (int)e__; return fail(BWTS_B200_ECUDA); } } while (0)
    FCK(cudaMemcpyAsync(dC, C.data(), 4 * 257, cudaMemcpyHostToDevice, st));
    FCK(cudaMemcpyAsync(dmap, map.data(), 256, cudaMemcpyHostToDevice, st));
    FCK(cudaMemcpyAsync(syms, sy.data(), sg, cudaMemcpyHostToDevice, st));
    FCK(cudaStreamSynchronize(st));  // the host vectors go out of scope below
    long primary = 0;
    rc = forward_core(ctx, d_text, n, U, d_sa, FWD_FM, st, &primary);
    if (rc) return fail(rc);
    fm->primary = (u32)primary;
    // the k_fm_* build kernels, booked like the LCP stage: class emit, phase 3
    ctx->phase = 3;
    rc = [&]() -> int {
        LAUNCH(KC_EMIT, 1.0 * n + 2.0 * sg * nb, k_fm_block_counts, cdiv(nb, 8), 256, U, n, syms, sg, B);
        LAUNCH(KC_EMIT, 4.0 * sg * nb + 4.0 * sg * ns, k_fm_block_scan, ns, 256, n, sg, B, S);
        LAUNCH(KC_EMIT, 8.0 * sg * ns, k_fm_super_scan, sg, 32, n, sg, S);
        LAUNCH(KC_EMIT, 4.0 * n + n / 8.0 + 4.0 * nb, k_fm_marks, nb, 256, d_sa, n, sample, marks, dircnt);
        LAUNCH(KC_EMIT, 4.0 * nb, k_tile_sum_u32, nt, 256, dircnt, nb, tiles, nullptr);
        LAUNCH(KC_EMIT, 8.0 * nt, k_scan_excl_u32_block, 1, 1024, tiles, tiles, nt, nullptr);
        LAUNCH(KC_EMIT, 8.0 * nb, k_tile_scan_apply_u32, nt, 256, dircnt, dir, nb, tiles);
        LAUNCH(KC_EMIT, 4.0 * n + n / 8.0 + 4.0 * n / sample, k_fm_samples, cdiv(n, 256), 256, d_sa, n, sample, marks, dir,
               samples);
        return 0;
    }();
    if (rc) return fail(rc);
#undef FCK
    fm->v.U = U; fm->v.S = S; fm->v.B = B; fm->v.marks = marks; fm->v.dir = dir; fm->v.samples = samples;
    fm->v.C = dC; fm->v.map = dmap;
    fm->v.n = n; fm->v.primary = fm->primary; fm->v.sample = sample; fm->v.sg = sg;
    *out = fm;
    return 0;
}

// I/O region of a build: the text, the suffix array, the directory's block counts and its tile sums, the histogram
// and the symbol list
static size_t fm_build_io(size_t n)
{
    const size_t nb = (n >> 8) + 1;
    return r256(n) + r256(4 * n) + r256(4 * nb) + r256(4 * (cdiv(nb, SC_TILE) + 1)) + 1024 + 256;
}
static int fm_build_args(bwts_b200_ctx *ctx, const void *in, long len, int sample, bwts_b200_fm **fm)
{
    if (fm) *fm = nullptr;
    if (!ctx || !in || !fm || len <= 0 || !fm_sample_ok(sample)) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    return 0;
}
// the device form copies the text next to the suffix array whatever its alignment: one n-byte copy
static int fm_build(bwts_b200_ctx *ctx, const void *src, long len, int sample, bwts_b200_fm **fm, void *stream, bool host)
{
    const size_t io = fm_build_io((size_t)len);
    Frame f = {len, 0, workspace_bytes((size_t)len) + io + 1024, io, host};
    f.in[0] = {0, src, (size_t)len};
    const int rc = run_frame(ctx, stream, f, [&](cudaStream_t st) { return fm_build_core(ctx, (u32)len, (u32)sample, fm, st); });
    if (rc && *fm) { bwts_b200_fm_free(*fm); *fm = nullptr; }
    return rc;
}

extern "C" int bwts_b200_fm_build_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int sample,
                                       bwts_b200_fm **fm)
{
    const int rc = fm_build_args(ctx, in, len, sample, fm);
    return rc ? rc : fm_build(ctx, in, len, sample, fm, nullptr, true);
}
extern "C" int bwts_b200_fm_build_device(bwts_b200_ctx *ctx, const void *d_in, long len, int sample, bwts_b200_fm **fm,
                                         void *stream)
{
    const int rc = fm_build_args(ctx, d_in, len, sample, fm);
    return rc ? rc : fm_build(ctx, d_in, len, sample, fm, stream, false);
}
extern "C" void bwts_b200_fm_free(bwts_b200_fm *fm)
{
    if (!fm) return;
    cudaSetDevice(fm->device);
    cudaFree(fm->mem);
    delete fm;
}
extern "C" long bwts_b200_fm_bytes(const bwts_b200_fm *fm)
{
    return fm ? (long)fm->bytes : 0;
}

// Queries run on the context's arena: 64 bytes of counters at its start, then (host forms) the staged arrays.
// direction 1, phase 2 ("Walk sublists"): the searches and walks in class inv_walk, the checks and the offsets
// scan in class inv_scan.  f: the staged arrays and the arena they need.
template <typename Core>
static int run_fm_query(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, void *stream, Frame &f, Core &&core)
{
    if (ctx->device != fm->device) return BWTS_B200_EINVAL;
    f.len = fm->n;
    f.direction = 1;
    f.arena = max(f.arena, (size_t)4096);
    return run_frame(ctx, stream, f, [&](cudaStream_t st) {
        ctx->phase = 2;
        return core(st);
    });
}
static u64 h_small_u64(const bwts_b200_ctx *ctx, int w) { return (u64)ctx->h_small[w] | ((u64)ctx->h_small[w + 1] << 32); }

// arguments and stream set up by the caller; check_off: the device form's offsets check
static int fm_count_core(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const u8 *d_pat, long pat_len, const long long *d_off,
                         long npat, i32 *d_range, long *total, bool check_off, cudaStream_t st)
{
    u32 *flags = (u32 *)ctx->arena;  // [0] bad offsets, [2..3] sum of hi - lo, [4..5] bytes read
    unsigned long long *cnt = (unsigned long long *)(flags + 2);
    CK(cudaMemsetAsync(flags, 0, 64, st));
    if (check_off)
        LAUNCH(KC_INV_SCAN, 8.0 * (npat + 1), k_fm_check_off, min(cdiv((u64)npat + 1, 256), (u32)ctx->sm_count * 8), 256,
               d_off, (u64)npat, (long long)pat_len, flags);
    LAUNCH(KC_INV_WALK, 16.0 * npat, k_fm_count, min(cdiv((u64)npat, 8), (u32)ctx->sm_count * 64), 256, fm->v, d_pat,
           d_off, (u64)npat, d_range, flags, cnt);
    const size_t rec = ctx->recs.size() - 1;
    int rc = readback(ctx, st, flags, 24);
    if (rc) return rc;
    if (ctx->h_small[0]) return BWTS_B200_EINVAL;
    ctx->recs[rec].bytes += (double)h_small_u64(ctx, 4);
    if (total) *total = (long)h_small_u64(ctx, 2);
    return 0;
}

// the rules of off on the host: off[0] == 0, non-decreasing, off[npat] == pat_len
static bool fm_off_ok(const long *off, long npat, long pat_len)
{
    if (off[0] != 0 || off[npat] != pat_len) return false;
    for (long k = 0; k < npat; k++)
        if (off[k] > off[k + 1]) return false;
    return true;
}

extern "C" int bwts_b200_fm_count_host(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const unsigned char *pat, long pat_len,
                                       const long *off, long npat, int *range, long *total)
{
    if (!ctx || !fm || npat < 0 || pat_len < 0) return BWTS_B200_EINVAL;
    if (npat == 0) { if (total) *total = 0; return 0; }
    if (!off || !range || (pat_len > 0 && !pat)) return BWTS_B200_EINVAL;
    if (!fm_off_ok(off, npat, pat_len)) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    const size_t a_pat = 256, a_off = a_pat + r256((size_t)pat_len), a_range = a_off + r256(8 * ((size_t)npat + 1));
    Frame f = {0, 0, a_range + r256(8 * (size_t)npat), 0, true};
    f.in[0] = {a_pat, pat, (size_t)pat_len};
    f.in[1] = {a_off, off, 8 * ((size_t)npat + 1)};
    f.out[0] = {a_range, range, 8 * (size_t)npat};
    return run_fm_query(ctx, fm, nullptr, f, [&](cudaStream_t st) {
        return fm_count_core(ctx, fm, ctx->arena + a_pat, pat_len, (const long long *)(ctx->arena + a_off), npat,
                             (i32 *)(ctx->arena + a_range), total, false, st);
    });
}
extern "C" int bwts_b200_fm_count_device(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const void *d_pat, long pat_len,
                                         const void *d_off, long npat, void *d_range, long *total, void *stream)
{
    if (!ctx || !fm || npat < 0 || pat_len < 0) return BWTS_B200_EINVAL;
    if (npat == 0) { if (total) *total = 0; return 0; }
    if (!d_off || !d_range || (pat_len > 0 && !d_pat)) return BWTS_B200_EINVAL;
    if (((uintptr_t)d_off & 7) || ((uintptr_t)d_range & 3)) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    Frame f = {0, 0, 4096, 0, false};
    return run_fm_query(ctx, fm, stream, f, [&](cudaStream_t st) {
        return fm_count_core(ctx, fm, (const u8 *)d_pat, pat_len, (const long long *)d_off, npat, (i32 *)d_range, total,
                             true, st);
    });
}

// offsets of the ranges at arena + 256 (nrange + 1 u64); a bad range or a total above cap is EINVAL, nothing written
static int fm_locate_core(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const i32 *d_range, long nrange, i32 *d_pos, long cap,
                          long *total, cudaStream_t st)
{
    u32 *flags = (u32 *)ctx->arena;  // [0] bad range, [1] over cap, [2..3] total, [4..5] bytes read
    unsigned long long *offs = (unsigned long long *)(ctx->arena + 256);
    CK(cudaMemsetAsync(flags, 0, 64, st));
    LAUNCH(KC_INV_SCAN, 16.0 * nrange, k_fm_range_scan, 1, 1024, d_range, (u64)nrange, fm->n, (u64)cap, offs, flags);
    int rc = readback(ctx, st, flags, 16);
    if (rc) return rc;
    if (ctx->h_small[0] || ctx->h_small[1]) return BWTS_B200_EINVAL;
    const u64 tot = h_small_u64(ctx, 2);
    if (tot) {
        LAUNCH(KC_INV_WALK, 4.0 * tot, k_fm_locate, (u32)min((tot + 15) / 16, (u64)ctx->sm_count * 64), 256, fm->v, d_range,
               (u64)nrange, offs, tot, d_pos, (unsigned long long *)(flags + 4));
        const size_t rec = ctx->recs.size() - 1;
        rc = readback(ctx, st, flags, 24);
        if (rc) return rc;
        ctx->recs[rec].bytes += (double)h_small_u64(ctx, 4);
    }
    if (total) *total = (long)tot;
    return 0;
}

extern "C" int bwts_b200_fm_locate_host(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const int *range, long nrange,
                                        int *pos, long cap, long *total)
{
    if (!ctx || !fm || nrange < 0 || cap < 0) return BWTS_B200_EINVAL;
    if (nrange == 0) { if (total) *total = 0; return 0; }
    if (!range || !pos) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    u64 tot = 0;
    for (long k = 0; k < nrange; k++) {
        const int lo = range[2 * k], hi = range[2 * k + 1];
        if (lo < 0 || lo > hi || (u32)hi > fm->n) return BWTS_B200_EINVAL;
        tot += (u64)(hi - lo);
    }
    if (tot > (u64)cap) return BWTS_B200_EINVAL;
    const size_t a_range = 256 + r256(8 * ((size_t)nrange + 1)), a_pos = a_range + r256(8 * (size_t)nrange);
    Frame f = {0, 0, a_pos + r256(4 * tot), 0, true};
    f.in[0] = {a_range, range, 8 * (size_t)nrange};
    f.out[0] = {a_pos, pos, 4 * tot};
    return run_fm_query(ctx, fm, nullptr, f, [&](cudaStream_t st) {
        return fm_locate_core(ctx, fm, (const i32 *)(ctx->arena + a_range), nrange, (i32 *)(ctx->arena + a_pos), cap, total, st);
    });
}
extern "C" int bwts_b200_fm_locate_device(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const void *d_range, long nrange,
                                          void *d_pos, long cap, long *total, void *stream)
{
    if (!ctx || !fm || nrange < 0 || cap < 0) return BWTS_B200_EINVAL;
    if (nrange == 0) { if (total) *total = 0; return 0; }
    if (!d_range || !d_pos || ((uintptr_t)d_range & 3) || ((uintptr_t)d_pos & 3)) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    Frame f = {0, 0, 256 + r256(8 * ((size_t)nrange + 1)), 0, false};
    return run_fm_query(ctx, fm, stream, f, [&](cudaStream_t st) {
        return fm_locate_core(ctx, fm, (const i32 *)d_range, nrange, (i32 *)d_pos, cap, total, st);
    });
}

// Extract's scratch from the arena's start: 256 bytes of counters, the byte offsets and the segment offsets of the
// ranges (nrange + 1 u64 each) and the inverse table of the samples (ceil(n / sample) + 1 u32).  A host form stages
// its ranges and output above fm_extract_scratch.
static size_t fm_extract_scratch(const bwts_b200_fm *fm, long nrange)
{
    const size_t nsamp = ((size_t)fm->n + fm->sample - 1) / fm->sample;
    return 256 + 2 * r256(8 * ((size_t)nrange + 1)) + r256(4 * (nsamp + 1));
}

// The checks and byte offsets of k_fm_range_scan, then -- when some range is non-empty -- the segment offsets, the
// inverse table and the walk; a bad range or a total above cap is EINVAL with nothing written
static int fm_extract_core(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const i32 *d_range, long nrange, u8 *d_out, long cap,
                           long *total, cudaStream_t st)
{
    u32 *flags = (u32 *)ctx->arena;  // [0] bad range, [1] over cap, [2..3] total, [4..5] bytes read
    unsigned long long *offs = (unsigned long long *)(ctx->arena + 256);
    unsigned long long *segs = (unsigned long long *)(ctx->arena + 256 + r256(8 * ((size_t)nrange + 1)));
    u32 *isa = (u32 *)(ctx->arena + 256 + 2 * r256(8 * ((size_t)nrange + 1)));
    const u32 sh = (u32)__builtin_ctz(fm->sample), nsamp = cdiv(fm->n, fm->sample), nblk = cdiv(fm->n, FM_BLOCK);
    CK(cudaMemsetAsync(flags, 0, 64, st));
    LAUNCH(KC_INV_SCAN, 16.0 * nrange, k_fm_range_scan, 1, 1024, d_range, (u64)nrange, fm->n, (u64)cap, offs, flags);
    int rc = readback(ctx, st, flags, 16);
    if (rc) return rc;
    if (ctx->h_small[0] || ctx->h_small[1]) return BWTS_B200_EINVAL;
    const u64 tot = h_small_u64(ctx, 2);
    if (tot) {
        LAUNCH(KC_INV_SCAN, 16.0 * nrange, k_fm_seg_scan, 1, 1024, d_range, (u64)nrange, sh, segs);
        // marks and directory, the samples read and the table written
        LAUNCH(KC_INV_SCAN, fm->n / 8.0 + 4.0 * nblk + 8.0 * nsamp, k_fm_isa, cdiv(nblk, 8), 256, fm->v, sh, isa);
        // every segment holds at least one output byte, so at most tot half-warps have work
        LAUNCH(KC_INV_WALK, 1.0 * tot, k_fm_extract, (u32)min((tot + 15) / 16, (u64)ctx->sm_count * 64), 256, fm->v, isa,
               sh, d_range, (u64)nrange, offs, segs, d_out, (unsigned long long *)(flags + 4));
        const size_t rec = ctx->recs.size() - 1;
        rc = readback(ctx, st, flags, 24);
        if (rc) return rc;
        ctx->recs[rec].bytes += (double)h_small_u64(ctx, 4);
    }
    if (total) *total = (long)tot;
    return 0;
}

extern "C" int bwts_b200_fm_extract_host(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const int *range, long nrange,
                                         unsigned char *out, long cap, long *total)
{
    if (!ctx || !fm || nrange < 0 || cap < 0) return BWTS_B200_EINVAL;
    if (nrange == 0) { if (total) *total = 0; return 0; }
    if (!range || !out) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    u64 tot = 0;
    for (long k = 0; k < nrange; k++) {
        const int lo = range[2 * k], hi = range[2 * k + 1];
        if (lo < 0 || lo > hi || (u32)hi > fm->n) return BWTS_B200_EINVAL;
        tot += (u64)(hi - lo);
    }
    if (tot > (u64)cap) return BWTS_B200_EINVAL;
    const size_t a_range = fm_extract_scratch(fm, nrange), a_out = a_range + r256(8 * (size_t)nrange);
    Frame f = {0, 0, a_out + r256(tot), 0, true};
    f.in[0] = {a_range, range, 8 * (size_t)nrange};
    f.out[0] = {a_out, out, tot};
    return run_fm_query(ctx, fm, nullptr, f, [&](cudaStream_t st) {
        return fm_extract_core(ctx, fm, (const i32 *)(ctx->arena + a_range), nrange, ctx->arena + a_out, cap, total, st);
    });
}
extern "C" int bwts_b200_fm_extract_device(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const void *d_range, long nrange,
                                           void *d_out, long cap, long *total, void *stream)
{
    if (!ctx || !fm || nrange < 0 || cap < 0) return BWTS_B200_EINVAL;
    if (nrange == 0) { if (total) *total = 0; return 0; }
    if (!d_range || !d_out || ((uintptr_t)d_range & 3)) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    Frame f = {0, 0, fm_extract_scratch(fm, nrange), 0, false};
    return run_fm_query(ctx, fm, stream, f, [&](cudaStream_t st) {
        return fm_extract_core(ctx, fm, (const i32 *)d_range, nrange, (u8 *)d_out, cap, total, st);
    });
}

// ---- LZ77 decoding (lzd.cuh) -----------------------------------------------------------------------------------
// Scratch from the end of the I/O region on: the words v, the starts p (z <= n), the two live lists, 4 n bytes each; the
// tile sums, 8 per 4096 factors; 256 bytes of counters.
static size_t lzd_scratch_bytes(size_t n)
{
    return 4 * r256(4 * n) + r256(8 * ((size_t)cdiv(n, LZD_TILE) + 1)) + 256;
}
// the bwts_b200_lz77_* rules: factors[0 .. 2z) and out[0 .. len) share no byte
static int check_lzd_args(const bwts_b200_ctx *ctx, const void *factors, long z, const void *out, long len)
{
    if (!ctx || !factors || !out || z <= 0 || len <= 0) return BWTS_B200_EINVAL;
    if (len > BWTS_B200_MAX_LEN) return BWTS_B200_ETOOBIG;
    if (z > len || spans_overlap(factors, 8 * (size_t)z, out, (size_t)len)) return BWTS_B200_EINVAL;
    return 0;
}

// d_f: z pairs on the device, 4-byte aligned; d_out: n bytes.  The content rules are checked before anything is
// written to d_out.  Direction 1: the checks and the scan in class inv_scan / phase 0, the chunks in inv_walk / 2,
// the global rounds in inv_jump / 3, the bytes in inv_place / 4.
static int lzd_core(bwts_b200_ctx *ctx, const i32 *d_f, u32 z, u8 *d_out, u32 n, cudaStream_t st)
{
    const u32 nt = cdiv(z, LZD_TILE);
    u8 *a = ctx->arena + ctx->io_end;
    u32 *v = (u32 *)a;                a += r256(4ull * n);
    u32 *p = (u32 *)a;                a += r256(4ull * n);
    u32 *live[2] = {(u32 *)a, nullptr}; a += r256(4ull * n);
    live[1] = (u32 *)a;               a += r256(4ull * n);
    u64 *tsum = (u64 *)a;             a += r256(8ull * (nt + 1));
    u32 *cnt = (u32 *)a;  // [0] bad, [2..3] the sum of max(1, len_k), [4] / [5] the live counts
    ctx->stats.factors = z;
    CK(cudaMemsetAsync(cnt, 0, 32, st));
    // pairs 8 per factor (twice), p 4, tile sums
    LAUNCH(KC_INV_SCAN, 8.0 * z + 8.0 * nt, k_lzd_tile_sum, nt, 256, d_f, (u64)z, tsum, cnt);
    LAUNCH(KC_INV_SCAN, 16.0 * nt, k_lzd_tile_scan, 1, 1024, tsum, nt, (u64 *)(cnt + 2));
    LAUNCH(KC_INV_SCAN, 12.0 * z + 8.0 * nt, k_lzd_apply, nt, 256, d_f, (u64)z, tsum, p, cnt);
    int rc = readback(ctx, st, cnt, 16);
    if (rc) return rc;
    if (ctx->h_small[0] || h_small_u64(ctx, 2) != n) return BWTS_B200_EINVAL;

    const u32 tb = lz_tile_bits(n), nc = cdiv(n, 1u << tb);
    ctx->phase = 2;
    // per position the word 4 and the live entry 4 (at most), per factor its start 4 and its pair 8
    LAUNCH_SMEM(KC_INV_WALK, 8.0 * n + 12.0 * z, k_lzd_chunk, nc, 256, (size_t)8 << tb, d_f, p, z, n, tb, v, live[0],
                cnt + 4);
    rc = readback(ctx, st, cnt + 4, 4);
    if (rc) return rc;
    u32 m = ctx->h_small[0];
    const int bound = bit_length((u64)nc - 1) + 1;  // ceil(log2 nc) + 1
    ctx->phase = 3;
    int cur = 0;
    while (m) {
        if (ctx->stats.rounds == bound) return BWTS_B200_EINTERNAL;
        CK(cudaMemsetAsync(cnt + 5 - cur, 0, 4, st));
        // the list 4, the two words read 8, the word written 4, the next list 4 (at most)
        LAUNCH(KC_INV_JUMP, 20.0 * m, k_lzd_jump, cdiv(m, 256), 256, v, live[cur], m, live[cur ^ 1], cnt + 5 - cur);
        ctx->stats.rounds++;
        ctx->stats.live_sum += m;
        rc = readback(ctx, st, cnt + 5 - cur, 4);
        if (rc) return rc;
        m = ctx->h_small[0];
        cur ^= 1;
    }
    ctx->phase = 4;
    LAUNCH(KC_INV_PLACE, 5.0 * n, k_lzd_bytes, cdiv(n, 1024), 256, v, n, d_out);
    return 0;
}

extern "C" int bwts_b200_lz77_decode_host(bwts_b200_ctx *ctx, const int *factors, long z, unsigned char *out, long len)
{
    int rc = check_lzd_args(ctx, factors, z, out, len);
    if (rc) return rc;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    // I/O region: the pairs, then the text
    const size_t fb = r256(8 * (size_t)z), io = fb + r256((size_t)len);
    Frame f = {len, 1, io + lzd_scratch_bytes((size_t)len), io, true};
    f.in[0] = {0, factors, 8 * (size_t)z};
    f.out[0] = {fb, out, (size_t)len};
    return run_frame(ctx, nullptr, f, [&](cudaStream_t st) {
        return lzd_core(ctx, (const i32 *)ctx->arena, (u32)z, ctx->arena + fb, (u32)len, st);
    });
}
extern "C" int bwts_b200_lz77_decode_device(bwts_b200_ctx *ctx, const void *d_factors, long z, void *d_out, long len,
                                            void *stream)
{
    int rc = check_lzd_args(ctx, d_factors, z, d_out, len);
    if (rc) return rc;
    if ((uintptr_t)d_factors & 3) return BWTS_B200_EINVAL;
    if (bwts_b200_device_count() == 0) return BWTS_B200_ENODEV;
    Frame f = {len, 1, lzd_scratch_bytes((size_t)len), 0, false};
    return run_frame(ctx, stream, f, [&](cudaStream_t st) {
        return lzd_core(ctx, (const i32 *)d_factors, (u32)z, (u8 *)d_out, (u32)len, st);
    });
}

// ---- introspection --------------------------------------------------------------------------------------
extern "C" int bwts_b200_get_stats(const bwts_b200_ctx *ctx, bwts_b200_stats *out)
{
    if (!ctx || !out) return BWTS_B200_EINVAL;
    *out = ctx->stats;
    return 0;
}
extern "C" const char *bwts_b200_class_name(int cls)
{
    return (cls >= 0 && cls < BWTS_B200_NCLASS) ? kclass_names[cls] : nullptr;
}
extern "C" const char *bwts_b200_phase_name(int direction, int phase)
{
    static const char *fwd[] = {"Suffix sort", "Compute ISA", "Fix sort order", "Generate BWTS"};
    static const char *inv[] = {"Count bytes", "LF map", "Walk sublists", "Rank sublists", "Place bytes"};
    if (phase < 0) return nullptr;
    if (direction == 0) return phase < 4 ? fwd[phase] : nullptr;
    return phase < 5 ? inv[phase] : nullptr;
}
extern "C" int bwts_b200_set_profile(bwts_b200_ctx *ctx, int on)
{
    if (!ctx) return BWTS_B200_EINVAL;
    ctx->profile = on != 0;
    return 0;
}
extern "C" const char *bwts_b200_strerror(int code)
{
    switch (code) {
    case BWTS_B200_OK: return "ok";
    case BWTS_B200_EINVAL: return "invalid argument";
    case BWTS_B200_ETOOBIG: return "input of 2^31 bytes or more per block";
    case BWTS_B200_ENODEV: return "no usable CUDA device (there is no CPU fallback)";
    case BWTS_B200_ENOMEM: return "out of device or pinned host memory";
    case BWTS_B200_ECUDA: return "CUDA error";
    case BWTS_B200_EINTERNAL: return "internal invariant violated";
    default: return "unknown error";
    }
}
extern "C" int bwts_b200_last_cuda_error(const bwts_b200_ctx *ctx) { return ctx ? ctx->last_cuda : 0; }
extern "C" const char *bwts_b200_version(void) { return BWTS_VERSION; }
#ifdef BWTS_PROFILE_PHASES
// diagnostic builds only (make profile-lib): per-phase cycle sums of the instrumented kernels
extern "C" int bwts_b200_debug_phases(unsigned long long *out32, int reset)
{
    if (out32 && cudaMemcpyFromSymbol(out32, g_phase, 32 * sizeof(unsigned long long)) != cudaSuccess) return BWTS_B200_ECUDA;
    if (reset) {
        unsigned long long z[32] = {0};
        if (cudaMemcpyToSymbol(g_phase, z, sizeof z) != cudaSuccess) return BWTS_B200_ECUDA;
    }
    return 0;
}
#endif
extern "C" int bwts_b200_tune(int key, long value)
{
    if (key == 0) { if (value < 0) return BWTS_B200_EINVAL; g_tune_chunk = value; return 0; }
    if (key == 1) { if (value != 0 && (value < 20 || value > 31)) return BWTS_B200_EINVAL; g_tune_spl_shift = value; return 0; }
    if (key == 3) { g_tune_local = value; return 0; }
    if (key == 4) { g_tune_lyndon = value; return 0; }
    if (key == 2) { if (value < 0 || value > 4) return BWTS_B200_EINVAL; g_tune_onesweep = value; return 0; }
    if (key == 5) { g_tune_pipeline = value; return 0; }
    if (key == 6) { g_tune_keybits = value; return 0; }
    if (key == 7) { g_tune_scatterbin = value; return 0; }
    if (key == 8) { g_tune_nocta = value; return 0; }
    if (key == 9) { g_tune_emit = value; return 0; }
    if (key == 10) { g_tune_l2gran = value; return 0; }
    if (key == 11) { g_tune_nomark = value; return 0; }
    if (key == 12) { g_tune_invpath = value; return 0; }
    if (key == 14) { if (value < 0 || value > 32) return BWTS_B200_EINVAL; g_tune_tmax = value; return 0; }
    if (key == 15) { g_tune_invmark = value; return 0; }
    if (key == 17) { g_tune_lyscan = value; return 0; }
    if (key == 18) { g_tune_ctasort = value; return 0; }
    if (key == 20) { g_tune_tmode = value; return 0; }
    if (key == 21) { g_tune_hist = value; return 0; }
    if (key == 22) { g_tune_partial = value; return 0; }
    if (key == 23) { g_tune_emitwin = value; return 0; }
    if (key == 16) { if (value < 0) return BWTS_B200_EINVAL; g_tune_invbudget = value; return 0; }
    if (key == 13) { if (value < 0) return BWTS_B200_EINVAL; g_tune_invq = value; return 0; }
    if (key == 24) { if (value < 0 || value > 2) return BWTS_B200_EINVAL; g_tune_lcp = value; return 0; }
    if (key == 25) {
        if (value != 0 && (value < LZ_TB_MIN || value > LZ_TB_MAX)) return BWTS_B200_EINVAL;
        g_tune_lz = value;
        return 0;
    }
    return BWTS_B200_EINVAL;
}

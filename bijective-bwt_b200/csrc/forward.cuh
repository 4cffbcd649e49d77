// forward.cuh -- forward BWTS kernels around the radix sort: alphabet compaction, packed
// initial keys, one prefix-doubling round (key build, re-rank + live-set compaction), emit.
//
// State of the doubling (all u32, live arrays indexed by position j in the live array):
//   rank[i]   for every text position: number of rotations strictly smaller at the current
//             depth (= global slot of the head of i's group)
//   idx[j]    text position of the j-th live rotation; live = its group has > 1 member;
//             the live array is ordered by rank, groups are contiguous
//   grp[j]    rank of the group that owns live slot j      (position-indexed, not sorted)
//   gst[j]    live-array offset at which that group starts (position-indexed, not sorted)
// A round sorts (gst | rank[succ^k(idx)]) inside the live array, splits groups where the
// sorted keys change, drops rotations that became unique, and doubles k.
#pragma once
#include "common.cuh"

// ---- alphabet compaction ------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_byte_presence(const u8 *__restrict__ T, u32 n, u32 *__restrict__ present)
{
    __shared__ u8 seen[256];  // racing stores of the same value are fine
    seen[threadIdx.x] = 0;
    __syncthreads();
    const u32 nvec = n / 16;
    for (u32 v = blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += gridDim.x * blockDim.x) {
        const uint4 x = ldg_stream_u4((const uint4 *)T + v);
        const u32 w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int q = 0; q < 4; q++)
#pragma unroll
            for (int s = 0; s < 32; s += 8) seen[(w[q] >> s) & 255] = 1;
    }
    if (blockIdx.x == 0)
        for (u32 p = nvec * 16 + threadIdx.x; p < n; p += blockDim.x) seen[T[p]] = 1;
    __syncthreads();
    const u32 bits = __ballot_sync(FULL_MASK, seen[threadIdx.x] != 0);  // warp w covers bytes 32w..32w+31
    if (lane_id() == 0 && bits) atomicOr(present + (threadIdx.x >> 5), bits);
}

// code[c] = number of present bytes below c; *sigma = number of present bytes
__global__ void k_code_table(const u32 *__restrict__ present, u8 *__restrict__ code, u32 *__restrict__ sigma)
{
    const u32 c = threadIdx.x;  // 256 threads
    u32 below = 0;
    for (u32 w = 0; w < (c >> 5); w++) below += __popc(present[w]);
    below += __popc(present[c >> 5] & ((1u << (c & 31)) - 1));
    code[c] = (u8)below;
    if (c == 255) *sigma = below + ((present[7] >> 31) & 1);
}

// ---- initial keys: k0 packed symbols of the rotation starting at i -------------------------
// Thread owns 8 consecutive positions; inside one factor and away from its end the window
// slides by one symbol per position.  The keys leave through shared memory: a thread storing its own
// eight keys one by one puts 32 lanes on 32 different sectors per store instruction (ncu: 5.4 ms for the
// 8 GiB of keys of C4, the L2 transaction rate); staged, consecutive lanes write consecutive 16 bytes.
// rows of 8 keys + 1 pad word pair: the 64-byte stride of the thread rows would put 16 lanes on one bank pair
#define IK_SLOT(l_) ((l_) + ((l_) >> 3))
#define IK_WORDS (2048 + 256)
static __device__ __forceinline__ void init_keys_flush(const u64 *s_keys, u64 *__restrict__ keys, u32 base, u32 n)
{
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const u32 t = q * 256 + threadIdx.x;
        if (base + t < n) keys[base + t] = s_keys[IK_SLOT(t)];
    }
}
// Digit histograms of the initial sort without eight shared atomics per key (k_radix_hist: 7.7 ms at 1 GiB, exactly
// the 4 lanes per clock and SM that ATOMS sustains; copies per lane group changed nothing).  A radix digit of the
// packed key is a bit slice of w consecutive symbols, w = 2..4 -- and the symbols t .. t+w-1 of rotation i are the
// first w symbols of rotation i + t (cyclic inside the factor): over all i of a factor that is every rotation once.
// So ONE histogram of the leading w symbols (`whist`, 2^(w * bits) <= 2^14 bins, one shared atomic per key, taken here
// while the key is in a register) holds all eight digit histograms; k_digit_hists reads them off.
// Grid-stride over tiles of 2048 positions: the window histogram is flushed once per CTA.
// `extra` > 0: the bits the k0 whole symbols leave free in the 64-bit key (4 of them for 6-bit alphabets) hold the top
// bits of symbol k0 + 1.  Ranks that are finer than "order by k0 symbols" but still consistent with the order of the
// rotations are as good for the doubling as the exact ones (a round only needs ties to mean "equal on at least k
// symbols"), and on text a third of the ties of the initial sort end there: fewer rotations enter the doubling rounds.
__global__ void __launch_bounds__(256) k_init_keys(const u8 *__restrict__ T, u32 n, const u32 *__restrict__ FS,
                                                   const u32 *__restrict__ cidx, const u8 *__restrict__ code,
                                                   u32 bits, u32 k0, u32 extra, u64 *__restrict__ keys,
                                                   u32 *__restrict__ whist, u32 wshift, u32 wbins)
{
    // window histogram (when whist != nullptr): one word per bin up to 4096 bins; beyond (7-bit alphabets: 2^14 bins)
    // two 16-bit counts per word, flushed every 31 tiles -- a CTA adds at most 31 * 2048 < 2^16 to a count in between
    extern __shared__ u32 s_wh[];
    __shared__ u8 s_code[256];
    __shared__ u64 s_keys[IK_WORDS];
    const bool wpack = wbins > 4096;
    const u32 wwords = wpack ? wbins / 2 : wbins;
    s_code[threadIdx.x] = code[threadIdx.x];
    if (whist)
        for (u32 b = threadIdx.x; b < wwords; b += 256) s_wh[b] = 0;
    __syncthreads();
    u32 tiles_done = 0;
    const u32 l0 = threadIdx.x * 8;
    const u64 mask = (k0 * bits >= 64) ? ~0ull : ((1ull << (k0 * bits)) - 1);
    const u32 look = k0 + (extra ? 1u : 0u);  // symbols a key reads
    const u32 pshift = bits - extra;          // the partial symbol keeps its top `extra` bits
    const u32 ntiles = (n + 2047u) / 2048u;
    for (u32 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const u32 i0 = tile * 2048u + l0;
        const u32 iend = min(n, i0 + 8);
        u32 i = i0;
        while (i < iend) {
            const u32 f = factor_of(FS, cidx, i);
            const u32 s = FS[f], e = FS[f + 1];
            // first key of this stretch, symbol by symbol with cyclic wrap
            u64 key = 0;
            u32 pos = i;
            for (u32 c = 0; c < k0; c++) {
                key = (key << bits) | s_code[T[pos]];
                pos = (pos + 1 == e) ? s : pos + 1;
            }
            u32 nextc = extra ? (u32)s_code[T[pos]] : 0u;  // symbol k0 + 1 of this rotation
            u64 full = extra ? ((key << extra) | (u64)(nextc >> pshift)) : key;
            s_keys[IK_SLOT(l0 + (i - i0))] = full;
            if (whist) {
                const u32 w = (u32)(full >> wshift);
                if (wpack) atomicAdd(&s_wh[w >> 1], 1u << (16 * (w & 1))); else atomicAdd(&s_wh[w], 1u);
            }
            i++;
            // slide while the window [i, i + look) stays inside the factor
            while (i < iend && i < e && (u64)i + look <= e) {
                if (extra) {
                    key = ((key << bits) | nextc) & mask;
                    nextc = s_code[T[i + k0]];
                    full = (key << extra) | (u64)(nextc >> pshift);
                } else {
                    key = ((key << bits) | s_code[T[i + k0 - 1]]) & mask;
                    full = key;
                }
                s_keys[IK_SLOT(l0 + (i - i0))] = full;
                if (whist) {
                    const u32 w = (u32)(full >> wshift);
                    if (wpack) atomicAdd(&s_wh[w >> 1], 1u << (16 * (w & 1))); else atomicAdd(&s_wh[w], 1u);
                }
                i++;
            }
        }
        init_keys_flush(s_keys, keys, tile * 2048u, n);
        __syncthreads();  // the staging rows are free again (and every count of this tile is in)
        if (whist && wpack && ++tiles_done == 31) {
            tiles_done = 0;
            for (u32 b = threadIdx.x; b < wwords; b += 256) {
                const u32 c = s_wh[b];
                if (c) {
                    if (c & 0xffffu) atomicAdd(whist + 2 * b, c & 0xffffu);
                    if (c >> 16) atomicAdd(whist + 2 * b + 1, c >> 16);
                    s_wh[b] = 0;
                }
            }
            __syncthreads();
        }
    }
    if (whist) {
        for (u32 b = threadIdx.x; b < wwords; b += 256) {
            const u32 c = s_wh[b];
            if (!c) continue;
            if (wpack) {
                if (c & 0xffffu) atomicAdd(whist + 2 * b, c & 0xffffu);
                if (c >> 16) atomicAdd(whist + 2 * b + 1, c >> 16);
            } else {
                atomicAdd(whist + b, c);
            }
        }
    }
}
// ghist[p][d] = sum of whist[W] over the windows W whose slice for digit p is d.  Digit p = key bits [8p, 8p + 8).
// The key is the packing K of k0' = k0 (+ 1 with a partial symbol) symbols, symbol t at K bits [bits * (k0'-1-t),
// bits * (k0'-t)), shifted right by d = bits - extra (0 without a partial symbol): key bit b = K bit b + d.  With
// t_lo / t_hi the symbols holding the lowest / highest K bit of the digit (clipped to the key width), the digit is a
// slice of the first t_lo - t_hi + 1 symbols of the window that starts t_hi symbols into the rotation.  One block per digit.
__global__ void __launch_bounds__(256) k_digit_hists(const u32 *__restrict__ whist, u32 wbins, u32 wsyms, u32 bits, u32 k0,
                                                     u32 extra, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[256];
    const u32 p = blockIdx.x;
    sh[threadIdx.x] = 0;
    __syncthreads();
    const u32 k0p = k0 + (extra ? 1u : 0u), d = extra ? bits - extra : 0u;
    const u32 lo_bit = 8 * p + d, hi_bit = min(8 * p + 7 + d, k0p * bits - 1);
    const u32 t_lo = k0p - 1 - lo_bit / bits, t_hi = k0p - 1 - hi_bit / bits;
    const u32 wp = t_lo - t_hi + 1;                    // symbols the digit touches (<= wsyms)
    const u32 drop = bits * (wsyms - wp);              // trailing symbols of the window the digit does not see
    const u32 sh_r = lo_bit - bits * (k0p - 1 - t_lo);  // digit's lowest bit inside symbol t_lo
    for (u32 w = threadIdx.x; w < wbins; w += 256) {
        const u32 c = whist[w];
        if (c) atomicAdd(&sh[((w >> drop) >> sh_r) & 255u], c);
    }
    __syncthreads();
    ghist[p * 256 + threadIdx.x] = sh[threadIdx.x];
}

// suffix-array variant: no factors, symbols are code+1, positions past the end read as 0
__global__ void __launch_bounds__(256) k_init_keys_linear(const u8 *__restrict__ T, u32 n, const u8 *__restrict__ code,
                                                          u32 bits, u32 k0, u64 *__restrict__ keys)
{
    __shared__ u8 s_code[256];
    __shared__ u64 s_keys[IK_WORDS];
    s_code[threadIdx.x] = code[threadIdx.x];
    __syncthreads();
    const u32 l0 = threadIdx.x * 8;
    const u32 i0 = blockIdx.x * 2048u + l0;
    if (i0 < n) {
        const u32 iend = min(n, i0 + 8);
        const u64 mask = (k0 * bits >= 64) ? ~0ull : ((1ull << (k0 * bits)) - 1);
        u64 key = 0;
        for (u32 c = 0; c < k0; c++) {
            const u64 p = (u64)i0 + c;
            key = (key << bits) | (p < n ? (u64)s_code[T[p]] + 1 : 0ull);
        }
        s_keys[IK_SLOT(l0)] = key;
        for (u32 i = i0 + 1; i < iend; i++) {
            const u64 p = (u64)i + k0 - 1;
            key = ((key << bits) | (p < n ? (u64)s_code[T[p]] + 1 : 0ull)) & mask;
            s_keys[IK_SLOT(l0 + (i - i0))] = key;
        }
    }
    init_keys_flush(s_keys, keys, blockIdx.x * 2048u, n);
}

// ---- key build of one doubling round ---------------------------------------------------------
// key[j] = hi[j] << kb | rank[succ^k(idx[j])] (hi = dense group index, or gst), and -- while the key is in a register and the
// kernel waits on its random gather anyway -- the digit histograms of all radix passes
// (same shared-memory scheme as k_radix_hist, which this replaces for the doubling rounds).
// Grid-stride over warps of 32 slots; ghist: [8][256], zeroed by the host.
template <bool LINEAR>
__global__ void __launch_bounds__(256) k_build_keys(const u32 *__restrict__ idx, const u32 *__restrict__ hi, u32 m,
                                                    const u32 *__restrict__ rank, const u32 *__restrict__ FS,
                                                    const u32 *__restrict__ cidx, u32 n, u32 k, u32 kb,
                                                    u64 *__restrict__ keys, int passes, u32 *__restrict__ ghist)
{
    __shared__ u32 sh[8][256];
    for (u32 i = threadIdx.x; i < 8 * 256; i += blockDim.x) ((u32 *)sh)[i] = 0;
    __syncthreads();
    const u32 lane = lane_id();
    const u32 stride = gridDim.x * blockDim.x;
    for (u32 jb = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); jb < m; jb += stride) {
        const u32 j = jb + lane;
        const bool valid = j < m;
        u64 key = 0;
        if (valid) {
            const u32 i = ldg_stream_u32(idx + j);
            u32 r;
            if (LINEAR) {
                const u64 t = (u64)i + k;
                r = (t < n) ? __ldg(rank + (u32)t) + 1 : 0;
            } else {
                const u32 f = factor_of(FS, cidx, i);
                const u32 s = __ldg(FS + f), len = __ldg(FS + f + 1) - s;
                u32 o = i - s;
                if (len > 1) {
                    o += (k < len) ? k : k % len;  // < 2 * len <= 2^31
                    if (o >= len) o -= len;
                }
                r = __ldg(rank + s + o);
            }
            key = ((u64)ldg_stream_u32(hi + j) << kb) | (u64)r;  // hi: any index that grows with the group
            keys[j] = key;
        }
        const bool whole = __all_sync(FULL_MASK, valid);
        for (int p = 0; p < passes; p++) {
            const u32 d = (u32)(key >> (p * 8)) & 255;
            const u32 d0 = __shfl_sync(FULL_MASK, d, 0);
            if (whole && __all_sync(FULL_MASK, d == d0)) {
                if (lane == 0) atomicAdd(&sh[p][d0], 32u);
            } else if (valid) {
                atomicAdd(&sh[p][d], 1u);
            }
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < (u32)passes * 256; i += blockDim.x) {
        const u32 c = ((u32 *)sh)[i];
        if (c) atomicAdd(ghist + i, c);
    }
}

// ---- re-rank + compaction -----------------------------------------------------------------------
// One pass over a freshly sorted live array: split groups where the sorted keys change, write
// the new ranks, drop rotations that became unique and compact the rest into the next live
// arrays.  Two output streams: S takes groups known to have at most 32 members (they are
// re-sorted by k_local_sort_warp from then on), L the others (global radix path).  A group's
// size is taken from the tile's own head flags; a group that touches a tile border counts
// as large -- that only costs speed, never correctness.
#define RR_NT 256
#ifndef RR_MINB
#define RR_MINB 4  // CTAs per SM the re-rank is compiled for (64 registers at 4; experiments: -DRR_MINB=5 / 6)
#endif
#define RR_IPT 8
#define RR_TILE (RR_NT * RR_IPT)
#define RR_FLAG_AGG 1ull
#define RR_FLAG_PREFIX 2ull
#define RR_SMALL 32
// status words: A = flag[63:62] | (last head position + 1)[61:31] | kept in S [30:0]
//               B = flag[63:62] | kept group heads in L [61:31] | kept in L [30:0]
static __device__ __forceinline__ u64 rr_packA(u64 flag, u32 headp1, u32 keep)
{
    return (flag << 62) | ((u64)headp1 << 31) | (u64)keep;
}
static __device__ __forceinline__ u64 rr_packB(u64 flag, u32 heads, u32 keep)
{
    return (flag << 62) | ((u64)heads << 31) | (u64)keep;
}

// Totals of one re-rank launch, zeroed before it.  heads / kheads are sums of per-tile counts:
// one atomic per tile, spread over RR_SPREAD words (the ncu launch list showed the kernel at
// 40 ns per tile with two same-address atomics per WARP: 0.5 M serialised L2 atomics per
// launch).  The kept totals are the last tile's inclusive prefix: no atomics at all.
#define RR_SPREAD 16
struct RerankCounters {
    u32 heads[RR_SPREAD];   // groups after the split (all of them)
    u32 kheads[RR_SPREAD];  // groups that stay live (both streams)
    u32 keptS;              // live elements compacted into the S stream
    u32 keptL;              // live elements compacted into the L stream
    u32 kheadsL;            // groups in the L stream
    u32 changed[4];         // ranks that changed, counted in every 16th tile (x 16 = estimate for the launch)
    u32 pad[1];
    u32 keptT[RR_SPREAD];   // live elements handed to the tuple set (rings by text position)
};

struct LiveOut {  // one compaction stream
    u32 *idx, *grp, *gst;
    u32 *gid;     // L stream only: dense index of the group inside the stream (radix key high part)
};

// grp == nullptr (with gst ignored): both arrays are all zero -- the first re-rank after the
// initial sort, where the whole text is one group of rank 0 starting at slot 0.
// ROUTE: decide S/L per group (otherwise everything kept goes to S, used for the S set itself).
// KeyT: u64 radix keys (L set) or the bare u32 key2 = rank[succ^k] (S set: inside a group the high
// part of the radix key is the same for all members, so equal key2 <=> equal key).
// finalize != 0: every element becomes its own group (ties are known to be final); no outputs.
// baseS: device word holding the number of elements already in the S stream (nullptr = 0).
// nr_out != nullptr: the new rank of slot j is stored at nr_out[j] instead of being scattered to
// rank[idx[j]]; the caller bins the (idx, rank) pairs by text region and scatters them with
// locality (first re-rank of large inputs, where every one of the n ranks is written; later re-ranks that
// move a third of their set's ranks).  pos_out != nullptr: idx[j] is copied to pos_out[j] as well (sets compacted in place).
//
// IN PLACE: outS / outL may alias the input arrays (idx, grp, gst).  A tile writes its kept
// elements at [exclusive prefix, +kept), which never lies beyond its own input region, and it
// learns that prefix only after every earlier tile has published its counts.  A tile publishes
// after a barrier that follows a shared-memory store of a value computed from EVERY input word
// it loaded (s_sink): its input is in registers -- not merely requested -- before any later
// tile can start writing.  Inputs are read with ld.global.cg (L2, coherent), not through the
// non-coherent path.  This halves the doubling state: one grp / gst / idx array per set.
// MODE 0: no routing, everything kept goes to outS (routing switched off, finalize).
// MODE 1: L set -- a kept group goes to the tuple set T (at most tmax members, tmax >= 2), to S (at
//         most 32) or stays in L; sizes are taken from the tile's own head bits, a group that
//         touches a tile border counts as large.
// MODE 2: S set -- T or S.
// Tuple set: the members of a group are linked into a ring by text position, nxtT[idx] = idx of
// the next member (k_tuple_round); they leave the rank-ordered arrays for good.
template <int MODE, typename KeyT>
__global__ void __launch_bounds__(RR_NT, RR_MINB) k_rerank(const KeyT *__restrict__ keys, const u32 *idx,
                                                  const u32 *grp, const u32 *gst, u32 m,
                                                  int finalize, u32 *__restrict__ rank, LiveOut outS,
                                                  const u32 *__restrict__ baseS, LiveOut outL,
                                                  u64 *__restrict__ statusA, u64 *__restrict__ statusB,
                                                  RerankCounters *__restrict__ ctr, u32 *__restrict__ nr_out,
                                                  u32 *__restrict__ pos_out, u32 *__restrict__ nxtT, u32 tmax, u32 head_flag)
{
    // compaction staging (outputs phase) -- and, before the look-back, st_idx doubles as `s_all`: idx by tile
    // slot for the ring links of the tuple set (every thread is past the routing when the staging starts:
    // two barriers lie between)
    __shared__ u32 st_idx[RR_TILE], st_grp[RR_TILE], st_aux[RR_TILE], st_gid[RR_TILE];
    u32 *s_all = st_idx;
    __shared__ u32 s_nt[RR_NT / 32];
    __shared__ __align__(16) u32 s_hw[RR_NT / 4 + 4];  // head flags of the tile as a bit array (slot = bit), + the slots after it
    __shared__ u32 s_sink[RR_NT];
    __shared__ u32 s_wh[RR_NT / 32], s_ws[RR_NT / 32], s_wl[RR_NT / 32], s_wg[RR_NT / 32];
    __shared__ u32 s_nh[RR_NT / 32], s_nk[RR_NT / 32];
    __shared__ u32 s_exh, s_exs, s_exl, s_exg;
    u8 *s_hb = (u8 *)s_hw;  // byte t = the 8 slots of thread t

    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    PH_INIT();
    if (tid < 4) s_hw[RR_NT / 4 + tid] = 0;
    __syncthreads();
    // tile = blockIdx.x: CTAs are dispatched in index order, so the tiles a look-back waits for
    // are resident or finished (same assumption as the onesweep kernel)
    const u32 tile = blockIdx.x, base = tile * RR_TILE;
    const u32 j0 = base + tid * RR_IPT;

    // ---- my 8 slots, loaded up front (vector loads when the whole stretch is in range)
    u32 vi[RR_IPT], vg[RR_IPT], vs[RR_IPT];
    KeyT vk[RR_IPT];
    const bool full = (u64)j0 + RR_IPT <= m;
    if (full) {
#pragma unroll
        for (int q = 0; q < RR_IPT / 4; q++) {
            const uint4 a = __ldcg((const uint4 *)(idx + j0) + q);
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            const uint4 b = grp ? __ldcg((const uint4 *)(grp + j0) + q) : z4;
            const uint4 c = grp ? __ldcg((const uint4 *)(gst + j0) + q) : z4;
            vi[4 * q] = a.x; vi[4 * q + 1] = a.y; vi[4 * q + 2] = a.z; vi[4 * q + 3] = a.w;
            vg[4 * q] = b.x; vg[4 * q + 1] = b.y; vg[4 * q + 2] = b.z; vg[4 * q + 3] = b.w;
            vs[4 * q] = c.x; vs[4 * q + 1] = c.y; vs[4 * q + 2] = c.z; vs[4 * q + 3] = c.w;
        }
        if (!finalize) {
            if (sizeof(KeyT) == 8) {
#pragma unroll
                for (int q = 0; q < RR_IPT / 2; q++) {
                    const uint4 a = __ldcg((const uint4 *)(keys + j0) + q);
                    vk[2 * q] = (KeyT)(((u64)a.y << 32) | a.x);
                    vk[2 * q + 1] = (KeyT)(((u64)a.w << 32) | a.z);
                }
            } else {
#pragma unroll
                for (int q = 0; q < RR_IPT / 4; q++) {
                    const uint4 a = __ldcg((const uint4 *)(keys + j0) + q);
                    vk[4 * q] = (KeyT)a.x; vk[4 * q + 1] = (KeyT)a.y; vk[4 * q + 2] = (KeyT)a.z; vk[4 * q + 3] = (KeyT)a.w;
                }
            }
        }
    } else {
#pragma unroll
        for (int q = 0; q < RR_IPT; q++) {
            const bool in = (u64)j0 + q < m;
            vi[q] = in ? __ldcg(idx + j0 + q) : 0;
            vg[q] = (in && grp) ? __ldcg(grp + j0 + q) : 0;
            vs[q] = (in && grp) ? __ldcg(gst + j0 + q) : 0;
            vk[q] = (in && !finalize) ? __ldcg(keys + j0 + q) : (KeyT)0;
        }
    }
    const u32 mine = (j0 >= m) ? 0u : min((u32)RR_IPT, m - j0);  // slots of mine that exist
    // head flags of my slots and of the slot right after them
    u32 hbits = 0;  // bit q = slot j0+q starts a group; bit 8 = slot j0+8 does (or is past the end)
    if (finalize) {
        hbits = 0x1ffu;
    } else {
        KeyT prevk = 0;
        if (j0 > 0 && j0 < m) prevk = __ldcg(keys + j0 - 1);
#pragma unroll
        for (int q = 0; q < RR_IPT; q++) {
            if ((u32)q < mine) {
                const bool h = (vs[q] == j0 + q) || (vk[q] != (q ? vk[q - 1] : prevk));
                hbits |= (u32)h << q;
            }
        }
        const u64 jn = (u64)j0 + RR_IPT;
        bool hn = true;
        if (jn < m) hn = ((grp ? __ldcg(gst + jn) : 0u) == (u32)jn) || (__ldcg(keys + jn) != vk[RR_IPT - 1]);
        hbits |= (u32)hn << RR_IPT;
    }
    if (mine < RR_IPT) hbits |= 1u << mine;  // the slot after the last live slot acts as a head
    {
        // every input word is in a register before the barrier below (see IN PLACE above)
        u32 x = hbits;
#pragma unroll
        for (int q = 0; q < RR_IPT; q++) x ^= vi[q] ^ vg[q] ^ vs[q];
        s_sink[tid] = x;
        if (MODE) {
#pragma unroll
            for (int q = 0; q < RR_IPT; q++) s_all[tid * RR_IPT + q] = vi[q];
        }
    }
    s_hb[tid] = (u8)hbits;
    if (tid == RR_NT - 1) s_hb[RR_NT] = (u8)(hbits >> RR_IPT);
    PH(16);  // loads + head flags
    __syncthreads();
    PH(17);

    // ---- per slot: keep?  which stream?
    // A group goes to S when its head and the next head both lie in this tile's bit array and are at
    // most 32 slots apart.  Bit scans over the head bits (64-bit windows assembled from the words).
    auto head_at_or_before = [&](u32 x) -> int {  // tile slot of the last head in (x - 32, x], or -1
        const u32 w = x >> 5;
        const u64 two = ((u64)s_hw[w] << 32) | (u64)(w ? s_hw[w - 1] : 0u);
        const u32 pos = 32 + (x & 31);  // bit of slot x inside `two`
        const u64 upto = two & ((pos == 63) ? ~0ull : (((u64)2 << pos) - 1));
        if (!upto) return -1;
        const u32 hb = 63u - (u32)__clzll((long long)upto);
        if (pos - hb >= 32) return -1;
        return (int)(x - (pos - hb));
    };
    auto heads_after = [&](u32 hs) -> u32 {  // head bits of the 32 slots after tile slot hs (bit 0 = slot hs + 1)
        const u32 b0 = hs + 1, w = b0 >> 5;
        return __funnelshift_r(s_hw[w], s_hw[w + 1], b0 & 31);
    };
    u32 kbits = 0, sbits = 0;  // keep in a stream, keep-in-S
    u32 lasth = 0, nS = 0, nL = 0, nG = 0, nhead = 0, nkhead = 0, nT = 0;  // nG: kept heads that go to L
    {
        // the group my first slot continues: its head is an earlier slot of this tile (or outside it)
        int route = -1;  // -1 unknown yet, 0 = L, 1 = S, 2 = T
        u32 g_hs = 0, g_end = 0;  // tile slots [g_hs, g_end) of the current group when it is routed to T
#pragma unroll
        for (int q = 0; q < RR_IPT; q++) {
            if ((u32)q < mine) {
                const u32 h = (hbits >> q) & 1, hn = (hbits >> (q + 1)) & 1;
                const u32 keep = !(h && hn);
                if (h) {
                    lasth = j0 + q + 1;
                    nhead++;
                    route = -1;
                }
                if (keep) {
                    const u32 x = tid * RR_IPT + q;
                    if (MODE == 0) {
                        route = 1;
                    } else if (route < 0) {
                        const int hs = h ? (int)x : head_at_or_before(x);
                        route = (MODE == 2) ? 1 : 0;
                        if (hs >= 0) {
                            const u32 w32 = heads_after((u32)hs);
                            if (w32) {  // the group has __ffs(w32) <= 32 members, all inside this tile
                                const u32 sz = (u32)__ffs(w32);
                                route = 1;
                                if (sz <= tmax) { route = 2; g_hs = (u32)hs; g_end = (u32)hs + sz; }
                            }
                        }
                    }
                    if (route == 2) {
                        // ring link: the next member in tile order, the head after the last one
                        nT++;
                        const u32 nx = (x + 1 < g_end) ? x + 1 : g_hs;
                        nxtT[vi[q]] = s_all[MODE ? nx : 0] | (x == g_hs ? head_flag : 0u);  // k_tuple_round_heads: the head does the group's work
                    } else {
                        nkhead += h;
                        kbits |= 1u << q;
                        if (route == 1) { sbits |= 1u << q; nS++; } else { nL++; nG += h; }
                    }
                }
            }
        }
    }

    PH(18);  // keep / route
    // ---- block-wide scans of (max lasth, sum nS, sum nL)
    const u32 ih = warp_incl_max(lasth), is = warp_incl_sum(nS), il = warp_incl_sum(nL), ig = warp_incl_sum(nG);
    if (lane == 31) { s_wh[warp] = ih; s_ws[warp] = is; s_wl[warp] = il; s_wg[warp] = ig; }
    const u32 th = warp_sum(nhead), tkh = warp_sum(nkhead), tnt = warp_sum(nT);
    if (lane == 0) { s_nh[warp] = th; s_nk[warp] = tkh; s_nt[warp] = tnt; }
    __syncthreads();
    if (tid == 0) {
        u32 bh = 0, bk = 0, bt = 0;
#pragma unroll
        for (int w = 0; w < RR_NT / 32; w++) { bh += s_nh[w]; bk += s_nk[w]; bt += s_nt[w]; }
        if (bh) atomicAdd(&ctr->heads[tile % RR_SPREAD], bh);
        if (bk) atomicAdd(&ctr->kheads[tile % RR_SPREAD], bk);
        if (bt) atomicAdd(&ctr->keptT[tile % RR_SPREAD], bt);
    }
    u32 offh = 0, offs = 0, offl = 0, offg = 0, toth = 0, tots = 0, totl = 0, totg = 0;
#pragma unroll
    for (int w = 0; w < RR_NT / 32; w++) {
        if (w < (int)warp) { offh = max(offh, s_wh[w]); offs += s_ws[w]; offl += s_wl[w]; offg += s_wg[w]; }
        toth = max(toth, s_wh[w]);
        tots += s_ws[w];
        totl += s_wl[w];
        totg += s_wg[w];
    }

    PH(19);  // scans
    // ---- decoupled look-back on (max, sum, sum, sum), by warp 0, over TWO levels of status words.
    // With ~600 tiles in flight a one-level walk reads ~16 windows of 32 tile words before it meets a
    // prefix (ncu: `barrier` 14-37 stalls per issue -- seven warps wait for this walk).  Here tiles form
    // blocks of 32: a tile sums the words of its own block before it (one window), the last tile of a
    // block publishes what the block adds, and the walk over earlier BLOCKS covers 1024 tiles per window:
    // two or three L2 round trips in all.  Block words live behind the tile words (status[gridDim.x + block]).
    if (warp == 0) {
        u32 exh = 0, exs = 0, exl = 0, exg = 0;
        u64 *blkA = statusA + gridDim.x, *blkB = statusB + gridDim.x;
        const u32 blk = tile >> 5, r = tile & 31;
        if (lane == 0) {
            const u64 f = tile == 0 ? RR_FLAG_PREFIX : RR_FLAG_AGG;
            st_relaxed_u64(statusB + tile, rr_packB(f, totg, totl));
            st_relaxed_u64(statusA + tile, rr_packA(f, toth, tots));
        }
        bool done = tile == 0;  // the exclusive prefix is complete
        if (!done && r > 0) {
            // step 1: the tiles of my block before me, lane <-> tile 32 blk + lane
            const u32 need = (1u << r) - 1;
            const bool mine_ = lane < r;
            for (;;) {
                const u64 va = mine_ ? ld_relaxed_u64(statusA + blk * 32 + lane) : 0ull;
                const u64 vb = mine_ ? ld_relaxed_u64(statusB + blk * 32 + lane) : 0ull;
                const u32 fa = (u32)(va >> 62), fb = (u32)(vb >> 62);
                const u32 flag = (fa == fb) ? fa : 0u;  // a tile counts once both of its words carry the same kind of flag
                const u32 empties = __ballot_sync(FULL_MASK, mine_ && flag == 0);
                const u32 prefixes = __ballot_sync(FULL_MASK, mine_ && flag == (u32)RR_FLAG_PREFIX);
                u32 take = need;
                if (prefixes) take &= ~((1u << (31 - __clz(prefixes))) - 1);  // from the prefix closest to me on
                if (empties & take) continue;                                 // somebody in between has not published yet
                const bool on = (take >> lane) & 1;
                exh = warp_max(on ? (u32)((va >> 31) & 0x7fffffffu) : 0u);
                exs = warp_sum(on ? (u32)(va & 0x7fffffffu) : 0u);
                exl = warp_sum(on ? (u32)(vb & 0x7fffffffu) : 0u);
                exg = warp_sum(on ? (u32)((vb >> 31) & 0x7fffffffu) : 0u);
                done = prefixes != 0;  // a prefix word already holds everything before it
                break;
            }
        }
        if (!done && r == 31 && lane == 0) {  // what this block adds (if a prefix was met, the block's own prefix follows below)
            st_relaxed_u64(blkB + blk, rr_packB(RR_FLAG_AGG, exg + totg, exl + totl));
            st_relaxed_u64(blkA + blk, rr_packA(RR_FLAG_AGG, max(exh, toth), exs + tots));
        }
        if (!done && blk > 0) {
            // step 2: the blocks before mine, 32 block words per window, until one carries a prefix
            int t = (int)blk - 1;
            for (;;) {
                const int q = t - (int)lane;
                const u64 va = (q >= 0) ? ld_relaxed_u64(blkA + q) : rr_packA(RR_FLAG_PREFIX, 0, 0);
                const u64 vb = (q >= 0) ? ld_relaxed_u64(blkB + q) : rr_packB(RR_FLAG_PREFIX, 0, 0);
                const u32 fa = (u32)(va >> 62), fb = (u32)(vb >> 62);
                const u32 flag = (fa == fb) ? fa : 0u;
                const u32 empties = __ballot_sync(FULL_MASK, flag == 0);
                const u32 prefixes = __ballot_sync(FULL_MASK, flag == (u32)RR_FLAG_PREFIX);
                u32 take;
                if (prefixes) {
                    const u32 fp = __ffs(prefixes) - 1;
                    take = (fp == 31) ? FULL_MASK : ((2u << fp) - 1);
                    if (empties & take) continue;  // a closer block has not published yet
                } else {
                    if (empties) continue;
                    take = FULL_MASK;
                }
                const bool on = (take >> lane) & 1;
                exh = max(exh, warp_max(on ? (u32)((va >> 31) & 0x7fffffffu) : 0u));
                exs += warp_sum(on ? (u32)(va & 0x7fffffffu) : 0u);
                exl += warp_sum(on ? (u32)(vb & 0x7fffffffu) : 0u);
                exg += warp_sum(on ? (u32)((vb >> 31) & 0x7fffffffu) : 0u);
                if (prefixes) break;
                t -= 32;
            }
        }
        if (lane == 0) {
            if (tile != 0) {
                st_relaxed_u64(statusB + tile, rr_packB(RR_FLAG_PREFIX, exg + totg, exl + totl));
                st_relaxed_u64(statusA + tile, rr_packA(RR_FLAG_PREFIX, max(exh, toth), exs + tots));
            }
            if (r == 31) {  // the inclusive prefix of the last tile of a block is the block's
                st_relaxed_u64(blkB + blk, rr_packB(RR_FLAG_PREFIX, exg + totg, exl + totl));
                st_relaxed_u64(blkA + blk, rr_packA(RR_FLAG_PREFIX, max(exh, toth), exs + tots));
            }
            s_exh = exh; s_exs = exs; s_exl = exl; s_exg = exg;
            if (tile == gridDim.x - 1) {  // the last tile's inclusive prefix = the totals
                ctr->keptS = exs + tots;
                ctr->keptL = exl + totl;
                ctr->kheadsL = exg + totg;
            }
        }
    }
    PH(20);  // look-back (thread 0 is in warp 0)
    __syncthreads();
    PH(21);

    // ---- outputs.  Ranks: 8 consecutive slots per thread (vector store) or a scatter of the
    // changed ones.  Compaction: through shared memory, S members packed from slot 0, L members
    // behind them, so that both streams leave the tile with consecutive threads on consecutive
    // addresses (per-thread runs cost 32 four-byte transactions per store instruction).
    u32 eh = __shfl_up_sync(FULL_MASK, ih, 1);
    u32 es = __shfl_up_sync(FULL_MASK, is, 1);
    u32 el = __shfl_up_sync(FULL_MASK, il, 1);
    u32 eg = __shfl_up_sync(FULL_MASK, ig, 1);
    if (lane == 0) { eh = 0; es = 0; el = 0; eg = 0; }
    u32 curh = max(s_exh, max(offh, eh));
    u32 ls = offs + es;          // tile-local slot in the S stream
    u32 ll = tots + offl + el;   // tile-local slot in the L stream, staged behind the S members
    u32 curg = s_exg + offg + eg;  // kept L heads up to and including the current slot
    u32 nrv[RR_IPT];
    u32 nchg = 0;
#pragma unroll
    for (int q = 0; q < RR_IPT; q++) {
        nrv[q] = 0;
        if ((u32)q < mine) {
            const u32 j = j0 + q;
            if ((hbits >> q) & 1) curh = j + 1;
            const u32 jh = curh - 1;  // every slot has a head at or before it (slot gst[j] is one)
            const u32 nr = vg[q] + (jh - vs[q]);
            nrv[q] = nr;
            nchg += nr != vg[q];
            if (!nr_out && nr != vg[q]) rank[vi[q]] = nr;
            if ((kbits >> q) & 1) {
                u32 slot;
                if ((sbits >> q) & 1) {
                    slot = ls++;
                } else {
                    curg += (hbits >> q) & 1;
                    slot = ll++;
                    st_gid[slot] = curg - 1;
                }
                st_idx[slot] = vi[q];
                st_grp[slot] = nr;
                st_aux[slot] = j - jh;  // distance to the group head: gst = own position - distance
            }
        }
    }
    if ((tile & 15) == 0) {  // how many ranks moved: the driver's cue for the binned scatter of the next round
        const u32 c = warp_sum(nchg);
        if (lane == 0 && c) atomicAdd(&ctr->changed[warp & 3], c);
    }
    if (nr_out) {
        if (full) {
            ((uint4 *)(nr_out + j0))[0] = make_uint4(nrv[0], nrv[1], nrv[2], nrv[3]);
            ((uint4 *)(nr_out + j0))[1] = make_uint4(nrv[4], nrv[5], nrv[6], nrv[7]);
        } else {
#pragma unroll
            for (int q = 0; q < RR_IPT; q++)
                if ((u32)q < mine) nr_out[j0 + q] = nrv[q];
        }
    }
    if (pos_out) {  // the S set compacts idx in place: the bin pass needs its own copy of the positions
        if (full) {
            ((uint4 *)(pos_out + j0))[0] = make_uint4(vi[0], vi[1], vi[2], vi[3]);
            ((uint4 *)(pos_out + j0))[1] = make_uint4(vi[4], vi[5], vi[6], vi[7]);
        } else {
#pragma unroll
            for (int q = 0; q < RR_IPT; q++)
                if ((u32)q < mine) pos_out[j0 + q] = vi[q];
        }
    }
    PH(22);  // ranks + staging
    if (tots + totl == 0) return;  // uniform over the block
    __syncthreads();
    PH(23);
    const u32 gS0 = (baseS ? *baseS : 0u) + s_exs, gL0 = s_exl;
    for (u32 t = tid; t < tots; t += RR_NT) {
        const u32 p = gS0 + t;
        outS.idx[p] = st_idx[t];
        outS.grp[p] = st_grp[t];
        outS.gst[p] = p - st_aux[t];
    }
    for (u32 t = tid; t < totl; t += RR_NT) {
        const u32 p = gL0 + t, u = tots + t;
        outL.idx[p] = st_idx[u];
        outL.grp[p] = st_grp[u];
        outL.gst[p] = p - st_aux[u];
        outL.gid[p] = st_gid[u];
    }
    PH(24);  // coalesced stream writes
}

// ---- local sort: one doubling round when every live group has at most 32 members ---------------
// Warp w owns the whole groups between the group holding live slot 32w and the group holding
// slot 32w+32 (at most 63 slots): gather key2 = rank[succ^k(idx)], order the slots by
// (group, key2) by counting, write keys / idx in the layout the radix path would have produced.
// keys_out receives the bare key2 (u32): the group part of the key is position-indexed state (gst).
// idx_out may alias idx: a warp reads all of its slots before it writes any, and no other warp
// touches them.
__global__ void __launch_bounds__(256) k_local_sort_warp(const u32 *idx, const u32 *__restrict__ gst,
                                                         u32 m, const u32 *__restrict__ rank,
                                                         const u32 *__restrict__ FS, const u32 *__restrict__ cidx,
                                                         u32 k, u32 kb, u32 n, int linear,
                                                         u32 *__restrict__ keys_out, u32 *idx_out,
                                                         u32 *__restrict__ surv)
{
    // surv != nullptr: every 16th block reports (slots, slots still tied with a member of their group)
    // -- the host's estimate of how long the repeats behind the small groups are (tuple set on / off)
    __shared__ u32 s_surv[2];
    const bool sample = surv != nullptr && (blockIdx.x & 15u) == 0;
    if (sample) {
        if (threadIdx.x < 2) s_surv[threadIdx.x] = 0;
        __syncthreads();
    }
    const u32 w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const u32 lane = lane_id();
    if ((u64)w * 32 >= m) {
        if (sample) {  // keep the block's barrier count
            __syncthreads();
            if (threadIdx.x < 2 && s_surv[threadIdx.x]) atomicAdd(surv + threadIdx.x, s_surv[threadIdx.x]);
        }
        return;
    }
    const u32 lo = __ldg(gst + w * 32);
    const u32 hi = ((u64)(w + 1) * 32 < m) ? __ldg(gst + (w + 1) * 32) : m;
    const u32 cnt = hi - lo;  // 1 .. 63
    u64 key[2];
    u32 pay[2];
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const u32 t = lane + 32 * h;
        key[h] = ~0ull;
        pay[h] = 0;
        if (t < cnt) {
            const u32 j = lo + t;
            const u32 i = __ldcg(idx + j);
            const u32 g = ldg_stream_u32(gst + j);
            u32 r;
            if (linear) {
                const u64 tt = (u64)i + k;
                r = (tt < n) ? __ldg(rank + (u32)tt) + 1 : 0;
            } else {
                const u32 f = factor_of(FS, cidx, i);
                const u32 s = __ldg(FS + f), len = __ldg(FS + f + 1) - s;
                u32 o = i - s;
                if (len > 1) {
                    o += (k < len) ? k : k % len;
                    if (o >= len) o -= len;
                }
                r = __ldg(rank + s + o);
            }
            key[h] = ((u64)g << kb) | (u64)r;
            pay[h] = i;
        }
    }
    // Groups are contiguous runs of slots; a slot's position inside its group = number of
    // members that order before it (ties broken by slot number).  The loop runs over the
    // offset inside the group, so its trip count is the largest group of the warp (2-4 for
    // DNA-like inputs), not the number of slots.
    const u64 gmask = ((u64)1 << kb) - 1;
    const bool head0 = (lane < cnt) && ((key[0] >> kb) == (u64)(lo + lane));
    const bool head1 = (lane + 32 < cnt) && ((key[1] >> kb) == (u64)(lo + lane + 32));
    const u64 H = (u64)__ballot_sync(FULL_MASK, head0) | ((u64)__ballot_sync(FULL_MASK, head1) << 32);
    u32 gs[2], ge[2], r[2];
    u32 maxlen = 0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const u32 s = lane + 32 * h;
        const u64 upto = (s == 63) ? ~0ull : (((u64)2 << s) - 1);  // slots 0..s
        const u64 below = H & upto, above = H & ~upto;
        gs[h] = below ? 63u - (u32)__clzll((long long)below) : 0u;
        ge[h] = above ? (u32)__ffsll((long long)above) - 1u : cnt;
        r[h] = (u32)(key[h] & gmask);
        if (s < cnt) maxlen = max(maxlen, ge[h] - gs[h]);
    }
    maxlen = warp_max(maxlen);
    u32 pos[2] = {0, 0};
    for (u32 o = 0; o < maxlen; o++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const u32 t = gs[h] + o;  // a member of my group while t < ge
            const u32 a = __shfl_sync(FULL_MASK, r[0], t & 31);
            const u32 b = __shfl_sync(FULL_MASK, r[1], t & 31);
            const u32 other = (t & 32) ? b : a;
            const u32 me = lane + 32 * h;
            pos[h] += (t < ge[h]) && ((other < r[h]) || (other == r[h] && t < me));
        }
    }
    if (sample) {  // block-uniform; the sampled blocks run the member loop a second time for the tie count
        u32 tied[2] = {0, 0};
        for (u32 o = 0; o < maxlen; o++) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const u32 t = gs[h] + o;
                const u32 a = __shfl_sync(FULL_MASK, r[0], t & 31);
                const u32 b = __shfl_sync(FULL_MASK, r[1], t & 31);
                const u32 other = (t & 32) ? b : a;
                tied[h] |= (t < ge[h]) && (other == r[h]) && (t != lane + 32 * h);
            }
        }
        const u32 c = warp_sum((u32)(lane < cnt) + (u32)(lane + 32 < cnt));
        const u32 t = warp_sum(((lane < cnt) ? tied[0] : 0u) + ((lane + 32 < cnt) ? tied[1] : 0u));
        if (lane == 0) { atomicAdd(&s_surv[0], c); atomicAdd(&s_surv[1], t); }
    }
#pragma unroll
    for (int h = 0; h < 2; h++)
        if (lane + 32 * h < cnt) {
            keys_out[lo + gs[h] + pos[h]] = r[h];
            idx_out[lo + gs[h] + pos[h]] = pay[h];
        }
    if (sample) {
        __syncthreads();
        if (threadIdx.x < 2 && s_surv[threadIdx.x]) atomicAdd(surv + threadIdx.x, s_surv[threadIdx.x]);
    }
}

// ---- tuple set: doubling rounds in TEXT order for groups of a few members ---------------------
// A group of g <= tmax members (pairs and triples of long repeats: 60 % of a DNA text with copied
// segments stays in such groups for log2(repeat length / k0) rounds) needs neither a sort nor a
// compaction: with the members linked into a ring by text position (nxt[i] = next member of i's
// group, NONE32 = i is not in the set),
//     new rank(i) = rank(i) + #{members m of the ring : rank[succ^k(m)] < rank[succ^k(i)]}
// and the ring of i's new group = the members with the same key2, in ring order.  The point is
// locality: neighbours in the text sit in neighbouring rings (the partner of i + 1 is the partner
// of i, + 1, for as long as the repeat runs), so a warp that sweeps 32 consecutive positions reads
// nxt[], rank[i + k] and rank[partner + k] as a few contiguous lines -- where the rank-ordered
// sets pay one DRAM access per gathered rank (20 ms per round for 0.65 G rotations of the 1 GiB
// DNA input, against the same round here as two streaming sweeps).
//   k_tuple_round   phase A, reads old ranks and old rings only: dr[i] = the rank increment,
//                   nxt_out[i] = next member with an equal key2 (NONE32: i became unique).
//                   finalize: key2 := the text position -- members of a final tie (equal rotations)
//                   get consecutive slots, every ring dissolves.
//   k_tuple_apply   phase B: rank[i] += dr[i]; ring entries of resolved positions are cleared in the
//                   old buffer too (both buffers hold NONE32 for every position outside the set).
// Phase B completes before the rank-ordered sets gather their key2 of the same round: a group is
// refined as a whole, so readers never see one group at two depths.
#define TUPLE_MAX_STEPS 64  // a ring has at most 32 members; corrupt links must not hang the kernel

template <bool LINEAR>
static __device__ __forceinline__ u32 tuple_key2(const u32 *__restrict__ rank, const u32 *__restrict__ FS,
                                                 const u32 *__restrict__ cidx, u32 n, u32 k, u32 i)
{
    if (LINEAR) {
        const u64 t = (u64)i + k;
        return (t < n) ? __ldg(rank + (u32)t) + 1 : 0;
    }
    const u32 f = factor_of(FS, cidx, i);
    const u32 s = __ldg(FS + f), len = __ldg(FS + f + 1) - s;
    u32 o = i - s;
    if (len > 1) {
        o += (k < len) ? k : k % len;
        if (o >= len) o -= len;
    }
    return __ldg(rank + s + o);
}

// Is the tuple set worth switching on?  Sample of the freshly sorted initial keys: among the sampled
// neighbours that tie on their k0 symbols, how many still agree on the `extra` bytes that follow?
// Long repeats (copied DNA segments) answer "nearly all", text answers "hardly any".  Factor
// boundaries are ignored (the cyclic wrap inside short factors cannot matter for a vote).
// counters[0] += tied pairs sampled, counters[1] += those that agree further.
__global__ void __launch_bounds__(256) k_sample_lcp(const u64 *__restrict__ keys, const u32 *__restrict__ idx,
                                                    const u8 *__restrict__ T, u32 n, u32 samples, u32 k0, u32 extra,
                                                    u32 *__restrict__ counters)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    u32 tied = 0, deep = 0;
    if (t < samples) {
        const u32 j = (u32)(((u64)t * (n - 1)) / samples);  // < n - 1
        if (keys[j] == keys[j + 1]) {
            tied = 1;
            const u64 a = (u64)idx[j] + k0, b = (u64)idx[j + 1] + k0;
            if (a + extra <= n && b + extra <= n) {
                deep = 1;
                for (u32 e = 0; e < extra; e++)
                    if (T[a + e] != T[b + e]) { deep = 0; break; }
            }
        }
    }
    tied = warp_sum(tied); deep = warp_sum(deep);
    if (lane_id() == 0) {
        if (tied) atomicAdd(counters, tied);
        if (deep) atomicAdd(counters + 1, deep);
    }
}

// One ring member's share of phase A: walks the ring from m (the member after i), key2 of i given.
template <bool LINEAR>
static __device__ __forceinline__ void tuple_walk(const u32 *__restrict__ nxt_in, const u32 *__restrict__ rank,
                                                  const u32 *__restrict__ FS, const u32 *__restrict__ cidx, u32 n, u32 k,
                                                  int finalize, u32 i, u32 ki, u32 m, u32 km, u32 mn, u32 &less, u32 &eqn,
                                                  u32 &diff)
{
    // (m, km, mn) = first member after i, its key2 and its successor, already loaded by the caller
    less = km < ki;
    diff = km != ki;
    eqn = (km == ki) ? m : NONE32;
    m = mn;
    for (int step = 0; m != i && step < TUPLE_MAX_STEPS; step++) {
        const u32 kq = finalize ? m : tuple_key2<LINEAR>(rank, FS, cidx, n, k, m);
        less += kq < ki;
        diff |= kq != ki;
        if (kq == ki && eqn == NONE32) eqn = m;
        m = __ldg(nxt_in + m) & ~0x80000000u;
    }
}

// counters[0] += elements still in the set after this round, counters[1] += elements that saw a
// member with a different key2 (their group split), counters[2] += elements processed.
// A thread owns 4 consecutive positions: one 16-byte load tells it whether any of them is in the
// set (the sweep over the n positions costs 4 bytes each), and the loads of the four first ring
// steps -- key2 of the position, key2 and successor of its ring neighbour -- are all issued before
// the first of them is used (the kernel is bound by memory latency, not by bytes).
template <bool LINEAR>
__global__ void __launch_bounds__(256) k_tuple_round(const u32 *__restrict__ nxt_in, u32 *__restrict__ nxt_out,
                                                     u8 *__restrict__ dr, const u32 *__restrict__ rank,
                                                     const u32 *__restrict__ FS, const u32 *__restrict__ cidx, u32 n,
                                                     u32 k, int finalize, u32 *__restrict__ counters)
{
    __shared__ u32 s_cnt[3];
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x * 4;
    u32 remain = 0, split = 0, seen = 0;
    for (u64 i64 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 4; i64 < n; i64 += stride) {
        const u32 i0 = (u32)i64;
        u32 m[4];
        if (i64 + 4 <= n) {
            const uint4 v = ldg_stream_u4((const uint4 *)(nxt_in + i0));
            m[0] = v.x; m[1] = v.y; m[2] = v.z; m[3] = v.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++) m[q] = (i64 + q < n) ? nxt_in[i0 + q] : NONE32;
        }
        if ((m[0] & m[1] & m[2] & m[3]) == NONE32) continue;
        u32 ki[4], km[4], mn[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            ki[q] = km[q] = 0; mn[q] = NONE32;
            if (m[q] != NONE32) {
                ki[q] = finalize ? i0 + q : tuple_key2<LINEAR>(rank, FS, cidx, n, k, i0 + q);
                km[q] = finalize ? m[q] : tuple_key2<LINEAR>(rank, FS, cidx, n, k, m[q]);
                mn[q] = __ldg(nxt_in + m[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (m[q] == NONE32) continue;
            u32 less, eqn, diff;
            tuple_walk<LINEAR>(nxt_in, rank, FS, cidx, n, k, finalize, i0 + q, ki[q], m[q], km[q], mn[q], less, eqn, diff);
            if (finalize) eqn = NONE32;
            nxt_out[i0 + q] = eqn;
            dr[i0 + q] = (u8)less;
            seen++;
            remain += eqn != NONE32;
            split += diff;
        }
    }
    remain = warp_sum(remain); split = warp_sum(split); seen = warp_sum(seen);
    if (lane_id() == 0) {
        if (remain) atomicAdd(&s_cnt[0], remain);
        if (split) atomicAdd(&s_cnt[1], split);
        if (seen) atomicAdd(&s_cnt[2], seen);
    }
    __syncthreads();
    if (threadIdx.x < 3 && s_cnt[threadIdx.x]) atomicAdd(counters + threadIdx.x, s_cnt[threadIdx.x]);
}

// Phase A, one thread per GROUP (round 2b).  In the per-member form above every member walks the whole
// ring: g^2 loads per group, which is why that form stops at 8 members.  Here the re-rank marks one member
// of every ring (TUPLE_HEAD in its link word); the thread that sweeps over a marked position collects the
// ring (g dependent link loads), gathers the g keys (independent), and writes the increment and the new
// link of EVERY member: g loads per group, and groups of up to 32 can join the set (tmax 32), which takes
// the warp-local sorts and their re-ranks out of the rounds of inputs with long repeats.  Locality is the
// same: the heads of neighbouring rings are neighbours in the text, and so are their members.
#define TUPLE_HEAD 0x80000000u
#define TUPLE_CAP 32
#define TUPLE_HNT 128
template <bool LINEAR>
__global__ void __launch_bounds__(TUPLE_HNT) k_tuple_round_heads(const u32 *__restrict__ nxt_in, u32 *__restrict__ nxt_out,
                                                                 u8 *__restrict__ dr, const u32 *__restrict__ rank,
                                                                 const u32 *__restrict__ FS, const u32 *__restrict__ cidx,
                                                                 u32 n, u32 k, int finalize, u32 *__restrict__ counters)
{
    __shared__ u32 s_m[TUPLE_CAP][TUPLE_HNT], s_k[TUPLE_CAP][TUPLE_HNT];  // members / keys of my group, column = thread
    __shared__ u32 s_cnt[3];
    const u32 tid = threadIdx.x;
    if (tid < 3) s_cnt[tid] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * blockDim.x * 4;
    u32 remain = 0, split = 0, seen = 0;
    for (u64 i64 = ((u64)blockIdx.x * blockDim.x + tid) * 4; i64 < n; i64 += stride) {
        const u32 i0 = (u32)i64;
        u32 v[4];
        if (i64 + 4 <= n) {
            const uint4 x = ldg_stream_u4((const uint4 *)(nxt_in + i0));
            v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
        } else {
#pragma unroll
            for (int q = 0; q < 4; q++) v[q] = (i64 + q < n) ? nxt_in[i0 + q] : NONE32;
        }
        if ((v[0] & v[1] & v[2] & v[3]) == NONE32) continue;
#pragma unroll 1
        for (int q = 0; q < 4; q++) {
            if (v[q] == NONE32 || !(v[q] & TUPLE_HEAD)) continue;
            const u32 i = i0 + q;
            u32 g = 1, m = v[q] & ~TUPLE_HEAD;
            s_m[0][tid] = i;
            while (m != i && g < TUPLE_CAP) {
                s_m[g][tid] = m;
                g++;
                m = __ldg(nxt_in + m) & ~TUPLE_HEAD;
            }
            for (u32 j = 0; j < g; j++) {
                const u32 mj = s_m[j][tid];
                s_k[j][tid] = finalize ? mj : tuple_key2<LINEAR>(rank, FS, cidx, n, k, mj);
            }
            for (u32 j = 0; j < g; j++) {
                const u32 kj = s_k[j][tid];
                u32 less = 0, diff = 0, after = NONE32, wrap = NONE32;
                for (u32 l = 0; l < g; l++) {
                    const u32 kl = s_k[l][tid];
                    less += kl < kj;
                    diff |= kl != kj;
                    if (kl == kj && l != j) {
                        if (l < j) { if (wrap == NONE32) wrap = l; }
                        else if (after == NONE32) after = l;
                    }
                }
                // the new ring of j's class keeps the collection order; its first member becomes the head
                u32 nx = (after != NONE32) ? after : wrap;
                if (finalize) nx = NONE32;
                const u32 mj = s_m[j][tid];
                nxt_out[mj] = (nx == NONE32) ? NONE32 : (s_m[nx][tid] | (wrap == NONE32 ? TUPLE_HEAD : 0u));
                dr[mj] = (u8)less;
                seen++;
                remain += nx != NONE32;
                split += diff;
            }
        }
    }
    remain = warp_sum(remain); split = warp_sum(split); seen = warp_sum(seen);
    if (lane_id() == 0) {
        if (remain) atomicAdd(&s_cnt[0], remain);
        if (split) atomicAdd(&s_cnt[1], split);
        if (seen) atomicAdd(&s_cnt[2], seen);
    }
    __syncthreads();
    if (tid < 3 && s_cnt[tid]) atomicAdd(counters + tid, s_cnt[tid]);
}

__global__ void __launch_bounds__(256) k_tuple_apply(u32 *__restrict__ nxt_old, const u32 *__restrict__ nxt_new,
                                                     const u8 *__restrict__ dr, u32 *__restrict__ rank, u32 n)
{
    const u64 stride = (u64)gridDim.x * blockDim.x * 4;
    for (u64 i64 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 4; i64 < n; i64 += stride) {
        const u32 i0 = (u32)i64;
        if (i64 + 4 <= n) {
            uint4 o = *(const uint4 *)(nxt_old + i0);
            if ((o.x & o.y & o.z & o.w) == NONE32) continue;
            const uint4 nw = ldg_stream_u4((const uint4 *)(nxt_new + i0));
            const u32 d4 = *(const u32 *)(dr + i0);
            uint4 r = *(const uint4 *)(rank + i0);
            const u32 l0 = o.x != NONE32, l1 = o.y != NONE32, l2 = o.z != NONE32, l3 = o.w != NONE32;
            r.x += l0 ? (d4 & 255u) : 0u;
            r.y += l1 ? ((d4 >> 8) & 255u) : 0u;
            r.z += l2 ? ((d4 >> 16) & 255u) : 0u;
            r.w += l3 ? (d4 >> 24) : 0u;
            *(uint4 *)(rank + i0) = r;
            // a position that became unique leaves the set in both buffers
            if (l0 && nw.x == NONE32) o.x = NONE32;
            if (l1 && nw.y == NONE32) o.y = NONE32;
            if (l2 && nw.z == NONE32) o.z = NONE32;
            if (l3 && nw.w == NONE32) o.w = NONE32;
            *(uint4 *)(nxt_old + i0) = o;
        } else {
            for (u32 i = i0; i < n; i++) {
                if (nxt_old[i] == NONE32) continue;
                const u32 d = dr[i];
                if (d) rank[i] += d;
                if (nxt_new[i] == NONE32) nxt_old[i] = NONE32;
            }
        }
    }
}

// ---- CTA-local sort: one doubling round of a live set whose groups fit one CTA ------------------
// Same ownership rule as the warp kernel, one level up: CTA c owns the whole groups between the
// group holding live slot c*LS_T and the group holding slot (c+1)*LS_T.  With every group at most
// LS_T members that is at most 2*LS_T - 1 slots; they are gathered once, ordered by
// (group, key2, slot) with a bitonic network in shared memory and written once -- against
// 6-8 onesweep passes over HBM on the global path (the 4096-copy classes of the tiled C3 input
// stay at this size for ~19 rounds).
#define LS_NT 512
#define LS_T 4096
#define LS_CAP (2 * LS_T)

// *oversize = 1 if some CTA of k_local_sort_cta would own more than LS_CAP slots
__global__ void k_ls_probe(const u32 *__restrict__ gst, u32 m, u32 *__restrict__ oversize)
{
    const u32 c = blockIdx.x * blockDim.x + threadIdx.x;
    if ((u64)c * LS_T >= m) return;
    const u32 lo = __ldg(gst + c * LS_T);
    const u32 hi = ((u64)(c + 1) * LS_T < m) ? __ldg(gst + (c + 1) * LS_T) : m;
    if (hi - lo > LS_CAP) *oversize = 1u;
}

template <bool LINEAR>
__global__ void __launch_bounds__(LS_NT, 2) k_local_sort_cta(const u32 *__restrict__ idx, const u32 *__restrict__ gst,
                                                             u32 m, const u32 *__restrict__ rank,
                                                             const u32 *__restrict__ FS, const u32 *__restrict__ cidx,
                                                             u32 k, u32 kb, u32 n, u64 *__restrict__ keys_out,
                                                             u32 *__restrict__ idx_out)
{
    extern __shared__ __align__(16) u64 s_key[];  // LS_CAP words
    const u32 tid = threadIdx.x;
    const u32 c = blockIdx.x;
    const u32 lo = __ldg(gst + c * LS_T);
    const u32 hi = ((u64)(c + 1) * LS_T < m) ? __ldg(gst + (c + 1) * LS_T) : m;
    const u32 cnt = hi - lo;
    if (cnt == 0 || cnt > LS_CAP) return;  // nothing owned / refused by k_ls_probe beforehand
    u32 P = 64;
    while (P < cnt) P <<= 1;

    // gather: key = local group start (13 bits) | key2 (31 bits) | slot (13 bits)
    for (u32 s = tid; s < P; s += LS_NT) {
        u64 key = ~0ull;
        if (s < cnt) {
            const u32 j = lo + s;
            const u32 i = ldg_stream_u32(idx + j);
            const u32 g = ldg_stream_u32(gst + j) - lo;
            u32 r;
            if (LINEAR) {
                const u64 t = (u64)i + k;
                r = (t < n) ? __ldg(rank + (u32)t) + 1 : 0;
            } else {
                const u32 f = factor_of(FS, cidx, i);
                const u32 fs = __ldg(FS + f), len = __ldg(FS + f + 1) - fs;
                u32 o = i - fs;
                if (len > 1) {
                    o += (k < len) ? k : k % len;
                    if (o >= len) o -= len;
                }
                r = __ldg(rank + fs + o);
            }
            key = ((u64)g << 44) | ((u64)r << 13) | (u64)s;
        }
        s_key[s] = key;
    }
    __syncthreads();

    // Already in order?  On repetitive inputs (the tiled C3 text) most groups see one and the same
    // key2 for all of their members in most rounds -- the network would move nothing.  One pass
    // over the staged words decides; keys are distinct (the slot is part of them).
    bool unsorted = false;
    for (u32 s = tid; s + 1 < cnt; s += LS_NT) unsorted |= s_key[s] > s_key[s + 1];
    const bool need_sort = __syncthreads_or(unsorted);

    // bitonic network; strides below 8 run in registers on 8 consecutive words per thread
    for (u32 k2 = 2; need_sort && k2 <= P; k2 <<= 1) {
        u32 j = k2 >> 1;
        for (; j >= 8; j >>= 1) {
            for (u32 t = tid; t < P / 2; t += LS_NT) {
                const u32 i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const u32 l = i + j;
                const bool up = (i & k2) == 0;
                const u64 a = s_key[i], b = s_key[l];
                if ((a > b) == up) { s_key[i] = b; s_key[l] = a; }
            }
            __syncthreads();
        }
        for (u32 base = tid * 8; base < P; base += LS_NT * 8) {
            u64 v[8];
#pragma unroll
            for (int q = 0; q < 8; q++) v[q] = s_key[base + q];
            const bool up = (base & k2) == 0;  // k2 >= 8 here or the whole 8-block shares the direction bits below
#pragma unroll
            for (int jj = 4; jj > 0; jj >>= 1) {
                if ((u32)jj > j) continue;
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    if (q & jj) continue;
                    const bool upq = (k2 >= 8) ? up : (((base + q) & k2) == 0);
                    const u64 a = v[q], b = v[q + jj];
                    if ((a > b) == upq) { v[q] = b; v[q + jj] = a; }
                }
            }
#pragma unroll
            for (int q = 0; q < 8; q++) s_key[base + q] = v[q];
        }
        __syncthreads();
    }

    for (u32 s = tid; s < cnt; s += LS_NT) {
        const u64 key = s_key[s];
        const u32 src = (u32)key & (LS_CAP - 1);
        const u32 r = (u32)(key >> 13) & 0x7fffffffu;
        const u32 g = (u32)(key >> 44);
        keys_out[lo + s] = ((u64)(lo + g) << kb) | (u64)r;
        idx_out[lo + s] = __ldg(idx + lo + src);
    }
}

// ---- CTA-local sort, radix form ---------------------------------------------------------------------
// Same ownership and gather as k_local_sort_cta; the bitonic network (91 stages over 8192 words,
// ~24 warp instructions per slot, 15 ms per round of the tiled C3 text) gives way to a stable LSD
// radix sort inside shared memory: ceil(kb / 8) passes over key2, then two over the local group start
// when the CTA owns more than one group.  A pass = the onesweep kernel's ranking (digit byte,
// ballot masks, per-warp counters) on elements held in registers, a scan of the 256 digit counts,
// a scatter back into the same arrays.  Only (key2, source slot) move; the group start is looked up by
// source slot.  73 KB of shared memory, two CTAs per SM.
#define LSR_NT 512
#define LSR_IPT 16  // LS_CAP / LSR_NT
struct LsrSmem {
    static constexpr size_t r = 0;                                   // u32[LS_CAP] key2, current order
    static constexpr size_t s = r + sizeof(u32) * LS_CAP;            // u16[LS_CAP] source slot, current order
    static constexpr size_t g = s + sizeof(u16) * LS_CAP;            // u16[LS_CAP] local group start BY SOURCE SLOT
    static constexpr size_t wcnt = g + sizeof(u16) * LS_CAP;         // u16[16][256]
    static constexpr size_t dstart = wcnt + sizeof(u16) * (LSR_NT / 32) * 256;  // u32[256]
    static constexpr size_t wsum = dstart + sizeof(u32) * 256;       // u32[8]
    static constexpr size_t bytes = wsum + 64;
};

template <bool LINEAR>
__global__ void __launch_bounds__(LSR_NT, 2) k_local_sort_cta_radix(const u32 *__restrict__ idx, const u32 *__restrict__ gst,
                                                                    u32 m, const u32 *__restrict__ rank,
                                                                    const u32 *__restrict__ FS, const u32 *__restrict__ cidx,
                                                                    u32 k, u32 kb, u32 n, u64 *__restrict__ keys_out,
                                                                    u32 *__restrict__ idx_out)
{
    extern __shared__ __align__(16) u8 lsr_smem[];
    u32 *s_r = (u32 *)(lsr_smem + LsrSmem::r);
    u16 *s_s = (u16 *)(lsr_smem + LsrSmem::s);
    u16 *s_g = (u16 *)(lsr_smem + LsrSmem::g);
    u16(*s_wcnt)[256] = (u16(*)[256])(lsr_smem + LsrSmem::wcnt);
    u32 *s_dstart = (u32 *)(lsr_smem + LsrSmem::dstart);
    u32 *s_wsum = (u32 *)(lsr_smem + LsrSmem::wsum);
    constexpr int NW = LSR_NT / 32;

    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 c = blockIdx.x;
    const u32 lo = __ldg(gst + c * LS_T);
    const u32 hi = ((u64)(c + 1) * LS_T < m) ? __ldg(gst + (c + 1) * LS_T) : m;
    const u32 cnt = hi - lo;
    if (cnt == 0 || cnt > LS_CAP) return;  // nothing owned / refused by k_ls_probe beforehand
    const u32 ipt = (cnt + LSR_NT - 1) / LSR_NT;  // 1 .. 16 elements per thread
    const u32 P = ipt * LSR_NT;

    // gather; pads carry the largest key2 and a group start no real group has (groups have >= 2 members)
    bool multi = false;
    for (u32 s = tid; s < P; s += LSR_NT) {
        u32 r = 0xffffffffu, g = 0x1fffu;
        if (s < cnt) {
            const u32 j = lo + s;
            const u32 i = ldg_stream_u32(idx + j);
            g = ldg_stream_u32(gst + j) - lo;
            if (LINEAR) {
                const u64 t = (u64)i + k;
                r = (t < n) ? __ldg(rank + (u32)t) + 1 : 0;
            } else {
                const u32 f = factor_of(FS, cidx, i);
                const u32 fs = __ldg(FS + f), len = __ldg(FS + f + 1) - fs;
                u32 o = i - fs;
                if (len > 1) {
                    o += (k < len) ? k : k % len;
                    if (o >= len) o -= len;
                }
                r = __ldg(rank + fs + o);
            }
            multi |= g != 0;
        }
        s_r[s] = r;
        s_s[s] = (u16)s;
        s_g[s] = (u16)g;
    }
    __syncthreads();
    // already in order?  (most groups of a repetitive input see one key2 for all members in most rounds)
    bool unsorted = false;
    for (u32 s = tid; s + 1 < cnt; s += LSR_NT)
        unsorted |= (s_g[s] == s_g[s + 1]) && (s_r[s] > s_r[s + 1]);
    const bool need_sort = __syncthreads_or(unsorted);
    const bool many_groups = __syncthreads_or(multi);

    const int rp = (int)((kb + 7) / 8), gp = many_groups ? 2 : 0;
    const u32 lt = lanemask_lt();
    const u32 wpos = warp * (32 * ipt) + lane;  // warp-major: the order of (warp, j, lane) is the order of positions
    u16 *wc = s_wcnt[warp];
    for (int pass = 0; need_sort && pass < rp + gp; pass++) {
        for (u32 i = tid; i < NW * 256 / 2; i += LSR_NT) ((u32 *)s_wcnt)[i] = 0;
        __syncthreads();  // counters zeroed; the previous pass's scatter is complete
        u32 rr[LSR_IPT], dpk[LSR_IPT / 4];
        u32 sspk[LSR_IPT / 2], rnkpk[LSR_IPT / 2];  // source slots and in-warp ranks, two 16-bit values per word
#pragma unroll
        for (int h0 = 0; h0 < LSR_IPT; h0 += 8) {  // eight elements at a time: their peer masks live in registers
            u32 peers[8];
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int j = h0 + jj;
                if ((j & 3) == 0) dpk[j >> 2] = 0;
                if ((j & 1) == 0) { sspk[j >> 1] = 0; rnkpk[j >> 1] = 0; }
                peers[jj] = 0;
                rr[j] = 0;
                if ((u32)j < ipt) {
                    const u32 p = wpos + j * 32;
                    rr[j] = s_r[p];
                    const u32 sj = s_s[p];
                    sspk[j >> 1] |= sj << (16 * (j & 1));
                    const u32 dj = (pass < rp) ? ((rr[j] >> (8 * pass)) & 255u)
                                               : (((u32)s_g[sj] >> (8 * (pass - rp))) & 255u);
                    dpk[j >> 2] |= dj << (8 * (j & 3));
                    u32 pm = FULL_MASK;
#pragma unroll
                    for (int b = 0; b < 8; b++) {
                        const u32 bit = (dj >> b) & 1u;
                        const u32 bal = __ballot_sync(FULL_MASK, bit);
                        pm &= bal ^ (bit - 1u);
                    }
                    peers[jj] = pm;
                }
            }
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int j = h0 + jj;
                if ((u32)j < ipt) {
                    const u32 dj = (dpk[j >> 2] >> (8 * (j & 3))) & 255u;
                    const int leader = __ffs(peers[jj]) - 1;
                    u32 before = 0;
                    if ((int)lane == leader) {
                        before = wc[dj];
                        wc[dj] = (u16)(before + __popc(peers[jj]));
                    }
                    before = __shfl_sync(FULL_MASK, before, leader);
                    rnkpk[j >> 1] |= ((before + __popc(peers[jj] & lt)) & 0xffffu) << (16 * (j & 1));
                    __syncwarp();
                }
            }
        }
        __syncthreads();  // every element is in registers, every warp's counts are final
        u32 blockcnt = 0, dsum = 0;
        if (tid < 256) {
#pragma unroll
            for (int w = 0; w < NW; w++) {
                const u32 cw = s_wcnt[w][tid];
                s_wcnt[w][tid] = (u16)blockcnt;  // this warp's base inside the digit's run
                blockcnt += cw;
            }
            const u32 incl = warp_incl_sum(blockcnt);
            if (lane == 31) s_wsum[warp] = incl;
            dsum = incl - blockcnt;
        }
        __syncthreads();
        if (tid < 256) {
#pragma unroll
            for (int w = 0; w < 8; w++)
                if (w < (int)warp) dsum += s_wsum[w];
            s_dstart[tid] = dsum;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < LSR_IPT; j++) {
            if ((u32)j < ipt) {
                const u32 dj = (dpk[j >> 2] >> (8 * (j & 3))) & 255u;
                const u32 dst = s_dstart[dj] + wc[dj] + ((rnkpk[j >> 1] >> (16 * (j & 1))) & 0xffffu);
                s_r[dst] = rr[j];
                s_s[dst] = (u16)(sspk[j >> 1] >> (16 * (j & 1)));
            }
        }
        __syncthreads();  // the scatter read the warp bases: nobody may zero the counters before everyone is through
    }
    __syncthreads();
    for (u32 s = tid; s < cnt; s += LSR_NT) {
        const u32 src = s_s[s];
        const u32 g = s_g[src];
        keys_out[lo + s] = ((u64)(lo + g) << kb) | (u64)s_r[s];
        idx_out[lo + s] = __ldg(idx + lo + src);
    }
}

// ---- emit -----------------------------------------------------------------------------------------
// DIV: libdivsufsort's divbwt after the linear suffix sort.  Row r0 = rank[0] (suffix 0, whose byte
// would be the end of text) goes to slot 0, where k_divbwt_first writes T[n-1] afterwards; the rows
// in front of it move up by one.  One store per slot, so no two lanes write the same byte.  Without
// DIV the slot is the rank itself (BWTS and classic BWT).
template <bool DIV>
static __device__ __forceinline__ u32 emit_slot(u32 r, u32 r0)
{
    return DIV ? (r == r0 ? 0u : r + (r < r0)) : r;
}

// out[rank[i]] = T[i-1] for every position that does not start a factor and whose rank lies in
// [lo, hi).  Large outputs are emitted in rank windows small enough to stay in L2, so the
// one-byte scatter merges into full sectors there instead of read-modify-writing DRAM.
// DIV: out[emit_slot(rank[i])] for every position, windows over the slot; flags are not read.
template <bool DIV = false>
__global__ void __launch_bounds__(256) k_emit(const u8 *__restrict__ T, u32 n, const u32 *__restrict__ rank,
                                              const u8 *__restrict__ flags, u8 *__restrict__ out, u32 lo, u32 hi)
{
    const u32 i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i0 >= n) return;
    const u32 r0 = DIV ? __ldg(rank) : 0u;
    if (i0 + 4 <= n && i0 >= 4) {
        // every load is issued before the first store: the ranks, the four flags as one word, and
        // T[i0-1 .. i0+2] out of the aligned words around it (a word that holds a valid byte lies
        // inside the allocation)
        const uint4 r = ldg_stream_u4((const uint4 *)(rank + i0));
        const u32 fl = DIV ? 0u : *(const u32 *)(flags + i0);
        const uintptr_t a = (uintptr_t)(T + i0 - 1);
        const u32 *w = (const u32 *)(a & ~(uintptr_t)3);
        const u32 o = (u32)(a & 3);
        const u32 w0 = w[0], w1 = o ? w[1] : 0u;
        const u32 bytes = (u32)((((u64)w1 << 32) | w0) >> (8 * o));
        const u32 rr[4] = {emit_slot<DIV>(r.x, r0), emit_slot<DIV>(r.y, r0), emit_slot<DIV>(r.z, r0),
                           emit_slot<DIV>(r.w, r0)};
#pragma unroll
        for (int q = 0; q < 4; q++)
            if (rr[q] >= lo && rr[q] < hi && !((fl >> (8 * q)) & 0xffu)) out[rr[q]] = (u8)(bytes >> (8 * q));
    } else {
        for (u32 i = i0; i < min(n, i0 + 4); i++) {
            const u32 r = emit_slot<DIV>(rank[i], r0);
            if (r >= lo && r < hi && (DIV || !flags[i])) out[r] = (DIV && i == 0) ? (u8)0 : T[i - 1];
        }
    }
}
// Binned emit for outputs far larger than L2 (the windowed form above re-reads rank[] once per
// 64 Mi-slot window: 16 sweeps at 1 GiB).  val[i] = T[i-1] widened to 32 bits; one u32 onesweep
// pass bins the (rank[i], val[i]) pairs by the top 8 bits of the rank -- after the final re-rank
// the ranks are a permutation of 0..n-1, so the bin starts are known (k_bin_bases) -- and
// k_scatter_bytes writes them region by region.  Factor heads are overwritten afterwards.
__global__ void __launch_bounds__(256) k_emit_vals(const u8 *__restrict__ T, u32 n, u32 *__restrict__ val)
{
    const u32 i0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i0 >= n) return;
#pragma unroll
    for (int q = 0; q < 4; q++)
        if (i0 + q < n) val[i0 + q] = (i0 + q > 0) ? (u32)T[i0 + q - 1] : 0u;
}
// DIV: the store goes to emit_slot of the rank, rank0 = &rank[0] (unused otherwise)
template <bool DIV = false>
__global__ void __launch_bounds__(256) k_scatter_bytes(const u32 *__restrict__ pos, const u32 *__restrict__ val, u32 n,
                                                       u8 *__restrict__ out, const u32 *__restrict__ rank0 = nullptr)
{
    const u32 j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (j0 >= n) return;
    const u32 r0 = DIV ? __ldg(rank0) : 0u;
    if (j0 + 4 <= n) {
        const uint4 p = ldg_stream_u4((const uint4 *)(pos + j0));
        const uint4 v = ldg_stream_u4((const uint4 *)(val + j0));
        out[emit_slot<DIV>(p.x, r0)] = (u8)v.x; out[emit_slot<DIV>(p.y, r0)] = (u8)v.y;
        out[emit_slot<DIV>(p.z, r0)] = (u8)v.z; out[emit_slot<DIV>(p.w, r0)] = (u8)v.w;
    } else {
        for (u32 j = j0; j < n; j++) out[emit_slot<DIV>(pos[j], r0)] = (u8)val[j];
    }
}
// packed form of the same (k_onesweep_pass MODE 2): word j of the binned stream belongs to rank bin
// j >> shift (the bins hold exactly 2^shift ranks each: the ranks are a permutation of 0..n-1)
template <bool DIV = false>
__global__ void __launch_bounds__(256) k_scatter_packed(const u32 *__restrict__ packed, u32 n, u32 shift,
                                                        u8 *__restrict__ out, const u32 *__restrict__ rank0 = nullptr)
{
    const u32 j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (j0 >= n) return;
    const u32 mask = (1u << shift) - 1u;
    const u32 r0 = DIV ? __ldg(rank0) : 0u;
    if (j0 + 4 <= n) {
        const uint4 w = ldg_stream_u4((const uint4 *)(packed + j0));
        const u32 ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; q++)
            out[emit_slot<DIV>((((j0 + q) >> shift) << shift) | (ww[q] & mask), r0)] = (u8)(ww[q] >> shift);
    } else {
        for (u32 j = j0; j < n; j++) out[emit_slot<DIV>(((j >> shift) << shift) | (packed[j] & mask), r0)] = (u8)(packed[j] >> shift);
    }
}
// factor heads receive the last byte of their own factor
__global__ void __launch_bounds__(256) k_emit_heads(const u8 *__restrict__ T, const u32 *__restrict__ FS, u32 F,
                                                    const u32 *__restrict__ rank, u8 *__restrict__ out)
{
    const u32 f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    out[rank[FS[f]]] = T[FS[f + 1] - 1];
}
// suffix-array variant: SA[rank[i]] = i
__global__ void __launch_bounds__(256) k_emit_sa(const u32 *__restrict__ rank, u32 n, i32 *__restrict__ sa)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sa[ldg_stream_u32(rank + i)] = (i32)i;
}

// ---- binned rank scatter --------------------------------------------------------------------------
// bin b of the binning pass = text positions [b << shift, (b + 1) << shift): every position occurs
// exactly once among the n pairs, so the bin starts are known without counting
__global__ void k_bin_bases(u32 n, u32 shift, u32 *__restrict__ base)
{
    const u64 start = (u64)threadIdx.x << shift;  // 256 threads
    base[threadIdx.x] = (u32)min(start, (u64)n);
}
// later rounds: not every position is live, the bins are counted (then scanned by k_radix_hist_scan)
__global__ void __launch_bounds__(256) k_bin_count(const u32 *__restrict__ pos, u32 m, u32 shift, u32 *__restrict__ hist)
{
    __shared__ u32 h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const u32 m4 = m / 4;
    for (u32 j = blockIdx.x * blockDim.x + threadIdx.x; j < m4; j += gridDim.x * blockDim.x) {
        const uint4 p = ldg_stream_u4((const uint4 *)pos + j);
        atomicAdd(&h[p.x >> shift], 1u); atomicAdd(&h[p.y >> shift], 1u);
        atomicAdd(&h[p.z >> shift], 1u); atomicAdd(&h[p.w >> shift], 1u);
    }
    if (blockIdx.x == 0 && threadIdx.x < (m & 3u)) atomicAdd(&h[pos[m4 * 4 + threadIdx.x] >> shift], 1u);
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}
// rank[pos[j]] = val[j] over pairs that are grouped by text region: the targets of the CTAs
// running at any one time fall into a few MiB, so the 4-byte stores merge in L2
__global__ void __launch_bounds__(256) k_scatter_pairs(const u32 *__restrict__ pos, const u32 *__restrict__ val, u32 n,
                                                       u32 *__restrict__ rank)
{
    // 8 pairs per thread, all four vector loads in flight before the first store
    const u32 j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (j0 >= n) return;
    if (j0 + 8 <= n) {
        const uint4 p0 = ldg_stream_u4((const uint4 *)(pos + j0)), p1 = ldg_stream_u4((const uint4 *)(pos + j0) + 1);
        const uint4 v0 = ldg_stream_u4((const uint4 *)(val + j0)), v1 = ldg_stream_u4((const uint4 *)(val + j0) + 1);
        rank[p0.x] = v0.x; rank[p0.y] = v0.y; rank[p0.z] = v0.z; rank[p0.w] = v0.w;
        rank[p1.x] = v1.x; rank[p1.y] = v1.y; rank[p1.z] = v1.z; rank[p1.w] = v1.w;
    } else {
        for (u32 j = j0; j < n; j++) rank[pos[j]] = val[j];
    }
}

__global__ void k_set_u32(u32 *p, const u32 *idx_src, u32 value)
{
    p[*idx_src] = value;  // FS[F] = n
}

// classic BWT: the whole text is one factor [0, n) (F = small[0] = 1); its head is the only flagged
// position (flags zeroed by the host), so k_emit leaves out[rank[0]] to k_emit_heads
__global__ void k_one_factor(u32 n, u32 *__restrict__ FS, u8 *__restrict__ flags, u32 *__restrict__ small)
{
    FS[0] = 0;
    FS[1] = n;
    flags[0] = 1;
    small[0] = 1;
}

// divbwt: slot 0 holds the last byte of the text (the row of the end of text, "$T", ends with it)
__global__ void k_divbwt_first(const u8 *__restrict__ T, u32 n, u8 *__restrict__ out)
{
    out[0] = T[n - 1];
}

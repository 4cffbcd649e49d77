// lcp.cuh -- LCP array of the linear suffix sort, from the irreducible LCP values.
//
// Kärkkäinen, Manzini and Puglisi, "Permuted Longest-Common-Prefix Array" (CPM 2009).  With
// Phi(SA[r]) = SA[r-1] and PLCP[SA[r]] = LCP[r], position i is reducible when T[i-1] == T[Phi(i)-1],
// and then PLCP[i] = PLCP[i-1] - 1.  Only the irreducible pairs (i, Phi(i)) are compared; their
// values add up to at most 2 n log n, so the comparisons are work-bounded even on periodic text.
//   1. k_lcp_rows     one thread per row r in rank order: row r is irreducible when r == 0, SA[r] == 0,
//                     SA[r-1] == 0 or B[r] != B[r-1] (B[r] = T[SA[r]-1], the BWT's run boundaries).
//                     The thread compares the first LCP_T1 bytes of its pair; pairs still open go to
//   2. k_lcp_warp     one warp per pair, 1 KiB per step, up to LCP_T2 bytes; pairs still open go to
//   3. k_lcp_span     rounds over all open pairs: each pair's window of the round is cut into LCP_SEG
//                     segments, one CTA each, and the first mismatch per pair is an atomicMin; a CTA
//                     whose segment starts past a known mismatch returns at once.  k_lcp_span_close
//                     settles the pairs resolved in the round and compacts the rest.
//      Every tier writes PLCP[j] + j into the zeroed text-order array P at its irreducible j.
//   4. PLCP[i] + i never decreases with i, and is constant over a run of reducible positions, so
//      an inclusive max-scan of P gives PLCP[i] = scan[i] - i everywhere (position 0 is irreducible):
//      k_lcp_tile_max, k_lcp_tile_scan, k_lcp_plcp.
//   5. k_lcp_emit     LCP[r] = PLCP[SA[r]].
// Loads of the text never read past T[n-1]: the device input is the caller's buffer of exactly n bytes.
#pragma once
#include "common.cuh"

#define LCP_T1 32u            // bytes one thread compares before its pair goes to the warp tier
#define LCP_T2 (64u << 10)    // bytes one warp compares before its pair goes to the multi-CTA tier
#define LCP_SEG (16u << 10)   // bytes of one multi-CTA work item: 256 threads x 64
#define LCP_TILE 4096         // positions per CTA of the max-scan

// T[p .. p+8) as a little-endian word, bytes past T[n-1] read as 0 (never loaded).  T is 8-byte aligned.
static __device__ __forceinline__ u64 lcp_load8(const u8 *__restrict__ T, u32 n, u64 p)
{
    const u64 a = p & ~(u64)7;
    const u32 sh = (u32)(p & 7) * 8;
    if (a + 16 <= n) {
        const u64 lo = __ldg((const unsigned long long *)(T + a));
        if (sh == 0) return lo;
        const u64 hi = __ldg((const unsigned long long *)(T + a + 8));
        return (lo >> sh) | (hi << (64 - sh));
    }
    u64 v = 0;
#pragma unroll
    for (u32 k = 0; k < 8; k++)
        if (p + k < n) v |= (u64)__ldg(T + p + k) << (8 * k);
    return v;
}

// offset of the first difference of T[a..) and T[b..) in [off, hi), or hi if there is none
static __device__ __forceinline__ u32 lcp_scan_thread(const u8 *__restrict__ T, u32 n, u32 a, u32 b, u32 off, u32 hi)
{
    for (; off < hi; off += 8) {
        const u64 d = lcp_load8(T, n, (u64)a + off) ^ lcp_load8(T, n, (u64)b + off);
        if (d) return min(hi, off + (u32)(__ffsll((long long)d) - 1) / 8);
    }
    return hi;
}

// ---- 1. irreducible rows, first LCP_T1 bytes ----------------------------------------------------------
// mode 0: compare here; mode 1 / 2 (bwts_b200_tune key 24): every pair of an irreducible row goes on to
// the next tier.  list2 holds the open pairs as (i | Phi(i) << 32), *count2 their number.
// *bytes += the bytes of both suffixes compared, up to and including the first difference.
__global__ void __launch_bounds__(256) k_lcp_rows(const u8 *__restrict__ T, u32 n, const i32 *__restrict__ SA,
                                                  u32 *__restrict__ P, u64 *__restrict__ list2, u32 *__restrict__ count2,
                                                  u32 mode, unsigned long long *__restrict__ bytes)
{
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    const u32 lane = lane_id();
    const bool live = r < n;
    const u32 s = live ? (u32)__ldg(SA + r) : 0u;
    // B[r] = T[SA[r]-1], 256 for the row of suffix 0 (no preceding byte); the row before comes from the lane below
    const u32 b = (live && s > 0) ? (u32)__ldg(T + s - 1) : 256u;
    u32 p = __shfl_up_sync(FULL_MASK, s, 1), bp = __shfl_up_sync(FULL_MASK, b, 1);
    if (lane == 0 && live && r > 0) {
        p = (u32)__ldg(SA + r - 1);
        bp = p > 0 ? (u32)__ldg(T + p - 1) : 256u;
    }
    bool push = false;
    u32 cmp = 0;
    if (live) {
        if (r == 0) {
            P[s] = s;  // LCP[0] = 0
        } else if (b != bp || b == 256u) {
            const u32 L = n - max(s, p);  // the shorter suffix ends there
            if (mode == 0) {
                const u32 hi = min(L, LCP_T1);
                const u32 l = lcp_scan_thread(T, n, s, p, 0, hi);
                cmp = 2 * (l < hi ? l + 1 : hi);
                if (l < hi || hi == L) P[s] = l + s;
                else push = true;
            } else {
                push = true;
            }
        }
    }
    cmp = warp_sum(cmp);
    if (lane == 0 && cmp) atomicAdd(bytes, (unsigned long long)cmp);
    const u32 m = __ballot_sync(FULL_MASK, push);
    u32 base = 0;
    if (m) {
        const u32 leader = __ffs(m) - 1;
        if (lane == leader) base = atomicAdd(count2, (u32)__popc(m));
        base = __shfl_sync(FULL_MASK, base, leader);
    }
    if (push) list2[base + __popc(m & lanemask_lt())] = (u64)s | ((u64)p << 32);
}

// ---- 2. one warp per pair ---------------------------------------------------------------------------
// Warp q takes pair q of the m2 in list2 (the host read m2 back and launched m2 warps).  Bytes
// [start, min(L, cap)) in steps of 1 KiB (every lane 32 bytes); pairs open at cap go to list3.
__global__ void __launch_bounds__(256) k_lcp_warp(const u8 *__restrict__ T, u32 n, const u64 *__restrict__ list2, u32 m2,
                                                  u32 start, u32 cap, u32 *__restrict__ P, u64 *__restrict__ list3,
                                                  u32 *__restrict__ count3, unsigned long long *__restrict__ bytes)
{
    const u32 lane = lane_id();
    const u32 q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (q < m2) {  // warp-uniform
        const u64 e = list2[q];
        const u32 s = (u32)e, p = (u32)(e >> 32);
        const u32 L = n - max(s, p), hi = min(L, cap);
        u32 l = hi;
        for (u32 off = start; off < hi && l == hi; off += 1024) {
            const u32 lo = off + lane * 32, end = min(hi, lo + 32);
            const u32 mine = lo < hi ? lcp_scan_thread(T, n, s, p, lo, end) : hi;
            const u32 found = __ballot_sync(FULL_MASK, mine < end);
            if (found) l = __shfl_sync(FULL_MASK, mine, __ffs(found) - 1);
        }
        if (lane == 0) {
            if (l < hi || hi == L) P[s] = l + s;
            else list3[atomicAdd(count3, 1u)] = e;
            const u32 upto = l < hi ? l + 1 : hi;
            if (upto > start) atomicAdd(bytes, 2ull * (upto - start));
        }
    }
}

// ---- 3. many CTAs per pair --------------------------------------------------------------------------
// Round over the m open pairs of `list`, all compared up to `off`: item t = (pair t / S, segment t % S)
// covers [off + (t % S) * LCP_SEG, + LCP_SEG) of that pair, clipped to its L.  res[q] (0xff.. before the
// round) receives the first mismatch by atomicMin.  Consecutive CTAs take consecutive segments of
// one pair, so a single long pair runs over the whole GPU.
__global__ void __launch_bounds__(256) k_lcp_span(const u8 *__restrict__ T, u32 n, const u64 *__restrict__ list, u32 m,
                                                  u32 S, u32 off, u32 *__restrict__ res, unsigned long long *__restrict__ bytes)
{
    __shared__ u32 best;
    const u64 t = blockIdx.x + (u64)gridDim.x * blockIdx.y;
    const u32 q = (u32)(t / S);
    if (q >= m) return;
    const u64 e = list[q];
    const u32 s = (u32)e, p = (u32)(e >> 32);
    const u32 L = n - max(s, p);
    const u64 lo64 = (u64)off + (t % S) * LCP_SEG;
    if (lo64 >= L) return;
    const u32 lo = (u32)lo64, hi = (u32)min((u64)L, lo64 + LCP_SEG);
    if (threadIdx.x == 0) best = *(volatile u32 *)(res + q);
    __syncthreads();
    if (lo >= best) return;  // a mismatch before this segment is known
    u32 mine = NONE32;
    for (u32 k = 0; k < LCP_SEG / 2048; k++) {  // 256 threads x 8 bytes per step: coalesced
        const u32 o = lo + k * 2048 + threadIdx.x * 8;
        if (o < hi) {
            const u64 d = lcp_load8(T, n, (u64)s + o) ^ lcp_load8(T, n, (u64)p + o);
            if (d) {
                const u32 at = o + (u32)(__ffsll((long long)d) - 1) / 8;
                if (at < hi) mine = at;
            }
        }
        if (__syncthreads_or(mine != NONE32)) break;  // the step that holds the first mismatch ends the segment
    }
    mine = warp_min(mine);
    if (lane_id() == 0 && mine != NONE32) atomicMin(&best, mine);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (best < hi) atomicMin(res + q, best);  // found here: other CTAs' values lie outside [lo, hi)
        atomicAdd(bytes, 2ull * ((best < hi ? best + 1 : hi) - lo));
    }
}
// after the round over [off, end): settle the pairs with a mismatch or whose shorter suffix ended, move the
// rest to `next`
__global__ void __launch_bounds__(256) k_lcp_span_close(u32 n, const u64 *__restrict__ list, u32 m, u64 end,
                                                        const u32 *__restrict__ res, u32 *__restrict__ P,
                                                        u64 *__restrict__ next, u32 *__restrict__ count)
{
    const u32 q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const u64 e = list[q];
    const u32 s = (u32)e, p = (u32)(e >> 32);
    const u32 L = n - max(s, p);
    if (res[q] != NONE32) P[s] = res[q] + s;
    else if (end >= L) P[s] = L + s;
    else next[atomicAdd(count, 1u)] = e;
}

// ---- 4. PLCP by an inclusive max-scan of P ------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lcp_tile_max(const u32 *__restrict__ P, u32 n, u32 *__restrict__ tile_max)
{
    __shared__ u32 ws[8];
    const u32 base = blockIdx.x * LCP_TILE;
    u32 v = 0;
#pragma unroll
    for (int q = 0; q < LCP_TILE / 256; q++) {
        const u32 i = base + q * 256 + threadIdx.x;
        if (i < n) v = max(v, ldg_stream_u32(P + i));
    }
    v = warp_max(v);
    if (lane_id() == 0) ws[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
        for (int w = 0; w < 8; w++) t = max(t, ws[w]);
        tile_max[blockIdx.x] = t;
    }
}
// single block: exclusive prefix maximum of the tile maxima, in place
__global__ void __launch_bounds__(1024) k_lcp_tile_scan(u32 *__restrict__ tile_max, u32 ntiles)
{
    __shared__ u32 part[1024];
    const u32 per = (ntiles + 1023) / 1024;
    const u32 lo = min(ntiles, threadIdx.x * per), hi = min(ntiles, lo + per);
    u32 v = 0;
    for (u32 t = lo; t < hi; t++) v = max(v, tile_max[t]);
    part[threadIdx.x] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 run = 0;
        for (u32 t = 0; t < 1024; t++) { const u32 x = part[t]; part[t] = run; run = max(run, x); }
    }
    __syncthreads();
    u32 run = part[threadIdx.x];
    for (u32 t = lo; t < hi; t++) { const u32 x = tile_max[t]; tile_max[t] = run; run = max(run, x); }
}
// P[i] <- max(P[0..i]) - i = PLCP[i], in place (thread owns 16 consecutive positions)
__global__ void __launch_bounds__(256) k_lcp_plcp(u32 *__restrict__ P, u32 n, const u32 *__restrict__ tile_excl)
{
    __shared__ u32 ws[8];
    const u32 base = blockIdx.x * LCP_TILE + threadIdx.x * 16;
    u32 v[16];
    u32 mine = 0;
    if (base + 16 <= n) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint4 w = ldg_stream_u4((const uint4 *)(P + base) + q);
            v[4 * q] = w.x; v[4 * q + 1] = w.y; v[4 * q + 2] = w.z; v[4 * q + 3] = w.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 16; q++) v[q] = (base + q < n) ? P[base + q] : 0u;
    }
#pragma unroll
    for (int q = 0; q < 16; q++) mine = max(mine, v[q]);
    const u32 incl = warp_incl_max(mine);
    if (lane_id() == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    u32 run = __shfl_up_sync(FULL_MASK, incl, 1);
    if (lane_id() == 0) run = 0;
    run = max(run, tile_excl[blockIdx.x]);
    for (u32 w = 0; w < (threadIdx.x >> 5); w++) run = max(run, ws[w]);
#pragma unroll
    for (int q = 0; q < 16; q++) {
        run = max(run, v[q]);
        v[q] = run - (base + q);
    }
    if (base + 16 <= n) {
#pragma unroll
        for (int q = 0; q < 4; q++)
            ((uint4 *)(P + base))[q] = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else {
#pragma unroll
        for (int q = 0; q < 16; q++) if (base + q < n) P[base + q] = v[q];
    }
}

// ---- 5. LCP[r] = PLCP[SA[r]] ------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lcp_emit(const i32 *__restrict__ SA, u32 n, const u32 *__restrict__ plcp,
                                                  i32 *__restrict__ lcp)
{
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) lcp[r] = (i32)__ldg(plcp + (u32)ldg_stream_u32((const u32 *)SA + r));
}

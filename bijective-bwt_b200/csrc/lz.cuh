// lz.cuh -- longest-previous-factor array and greedy LZ77 parse, from the suffix array and LCP array.
//
// LPF[i] = max over j < i of lcp(i, j), PREV[i] its source (include/bwts_b200.h).  For row r with i = SA[r],
// l = the last row before r with SA[l] < i and g = the first row after r with SA[g] < i (the previous and
// next smaller values in rank order), a = min LCP[l+1..r], b = min LCP[r+1..g] (0 when the row does not
// exist): LPF[i] = max(a, b), PREV[i] = SA[l] if a >= b (and a > 0), else SA[g].
//   1. k_lpf_tile     one CTA of 1024 threads per tile of W = 2^tb rows: a min tree over the pair (SA, LCP) in
//                     shared memory (64 KiB: two CTAs per SM, four rows a thread).  Each row walks up to the
//                     first left (right) sibling whose SA minimum is below i, then down to the nearest such
//                     leaf, taking the LCP minimum of the nodes that cover the skipped span.  The tile's tree nodes over 32 rows and more go to gtree, its root to
//                     a leaf of the tile tree `top`.  Rows answered on both sides are stored in text order;
//                     the others (the tile's prefix / suffix minima of SA) keep their answered side in
//                     LPF[i] / PREV[i] and go to a list with the LCP minimum of their span inside the tile.
//      k_lpf_top      builds `top` level by level.
//   2. k_lpf_cross    one thread per listed row: the same walk over `top`, then down the target tile's
//                     gtree to a group of 32 rows, which the warp searches with one ballot.
//   Work: W log W per tile, log(n / W) + log W + 32 per listed row: O(n log n) for every input.
//
// Greedy parse: next(p) = p + max(1, LPF[p]), the factors are the chain from 0.  Level k blocks span W^k
// positions; X_k[p] = the first chain node from p at or past the end of p's level-k block.
//   3. k_lz_exit1     X_1 by tb rounds of pointer jumping in shared memory, one CTA per chunk.
//      k_lz_jump      X_k from X_(k-1) by tb rounds of in-place pointer jumping in global memory: an X_(k-1)
//                     hop crosses a level-(k-1) block, so W hops reach the level-k block's end.
//   4. k_lz_top       one thread walks X_L from 0 (at most W hops, L the lowest level with ceil(n / W^L)
//                     <= W) and marks the chain's entry into each level-L block; k_lz_down pushes the entries
//                     down a level, one thread per block, at most W hops each.
//   5. k_lz_chunk     one CTA per chunk walks the chain from its entry in shared memory: counts, then (after
//                     an exclusive scan of the counts) the factor pairs at their offsets.
//   Work: n tb in shared memory per level-1 pass, n tb per further level, plus n: O(n log n).
#pragma once
#include "common.cuh"

#define LZ_TB_MIN 5    // smallest tile / chunk: one 32-row group
#define LZ_TB_MAX 12   // largest (the default): 4096 rows, 64 KiB of tree in shared memory

static __device__ __forceinline__ uint2 lz_min2(uint2 a, uint2 b) { return make_uint2(min(a.x, b.x), min(a.y, b.y)); }

// a, b: the two LCP minima (0 where that side has no row), srcL / srcG their SA values
static __device__ __forceinline__ void lpf_put(i32 *__restrict__ lpf, i32 *__restrict__ prev, u32 i, u32 a, u32 srcL,
                                               u32 b, u32 srcG)
{
    if (a >= b) { lpf[i] = (i32)a; prev[i] = a ? (i32)srcL : -1; }
    else { lpf[i] = (i32)b; prev[i] = (i32)srcG; }
}

// ---- 1. in-tile nearest smaller values ----------------------------------------------------------------------
// Dynamic shared memory 16 W bytes: mS[2W], mL[2W] in heap order (root 1, leaves W..2W-1, padding rows NONE32).
// gtree: per tile, nodes 1 .. 2G-1 (G = W / 32: the nodes over 32 rows and more) at t * 2G + v.  top: leaf P + t.
// listed rows: listR = r, listP = (LCP minimum of [tile start, r], of (r, tile end]), capped at n, or NONE32
// where that side is answered in the tile.
__global__ void __launch_bounds__(1024) k_lpf_tile(const i32 *__restrict__ SA, const i32 *__restrict__ LCP, u32 n, u32 tb,
                                                  uint2 *__restrict__ gtree, uint2 *__restrict__ top, u32 P,
                                                  i32 *__restrict__ lpf, i32 *__restrict__ prev, u32 *__restrict__ listR,
                                                  uint2 *__restrict__ listP, u32 *__restrict__ count)
{
    extern __shared__ u32 lz_smem[];
    const u32 W = 1u << tb, G = W >> 5, t = blockIdx.x, base = t << tb;
    u32 *mS = lz_smem, *mL = lz_smem + 2 * W;
    for (u32 q = threadIdx.x; q < W; q += blockDim.x) {
        const u32 r = base + q;
        mS[W + q] = r < n ? (u32)__ldg(SA + r) : NONE32;
        mL[W + q] = r < n ? (u32)__ldg(LCP + r) : NONE32;
    }
    __syncthreads();
    for (u32 lv = W >> 1; lv >= 1; lv >>= 1) {
        for (u32 v = lv + threadIdx.x; v < 2 * lv; v += blockDim.x) {
            mS[v] = min(mS[2 * v], mS[2 * v + 1]);
            mL[v] = min(mL[2 * v], mL[2 * v + 1]);
        }
        __syncthreads();
    }
    for (u32 v = 1 + threadIdx.x; v < 2 * G; v += blockDim.x) gtree[(size_t)t * 2 * G + v] = make_uint2(mS[v], mL[v]);
    if (threadIdx.x == 0) top[P + t] = make_uint2(mS[1], mL[1]);
    const u32 lane = lane_id();
    for (u32 q0 = 0; q0 < W; q0 += blockDim.x) {  // uniform trip count: the list push below is warp-wide
        const u32 q = q0 + threadIdx.x, r = base + q;
        bool push = false;
        u32 pa = NONE32, pb = NONE32;
        if (q < W && r < n) {
            const u32 i = mS[W + q];
            // left: the span (l, r] includes LCP[r], excludes LCP[l]
            u32 a = mL[W + q], v = W + q, srcL = NONE32;
            bool fl = false;
            for (; v > 1; v >>= 1)
                if (v & 1) {
                    if (mS[v - 1] < i) { fl = true; v--; break; }
                    a = min(a, mL[v - 1]);
                }
            if (fl) {
                while (v < W) {
                    if (mS[2 * v + 1] < i) v = 2 * v + 1;
                    else { a = min(a, mL[2 * v + 1]); v = 2 * v; }
                }
                srcL = mS[v];
            }
            // right: the span (r, g] excludes LCP[r], includes LCP[g]
            u32 b = NONE32, srcG = NONE32;
            bool fr = false;
            for (v = W + q; v > 1; v >>= 1)
                if (!(v & 1)) {
                    if (mS[v + 1] < i) { fr = true; v++; break; }
                    b = min(b, mL[v + 1]);
                }
            if (fr) {
                while (v < W) {
                    if (mS[2 * v] < i) v = 2 * v;
                    else { b = min(b, mL[2 * v]); v = 2 * v + 1; }
                }
                b = min(b, mL[v]);
                srcG = mS[v];
            }
            if (i == 0 || (fl && fr)) {  // suffix 0 has no earlier position: LPF 0, PREV -1 from either form
                lpf_put(lpf, prev, i, fl ? a : 0u, srcL, fr ? b : 0u, srcG);
            } else {
                // the answered side waits in the output for k_lpf_cross
                lpf[i] = fl ? (i32)a : fr ? (i32)b : 0;
                prev[i] = fl ? (i32)srcL : fr ? (i32)srcG : -1;
                pa = fl ? NONE32 : min(a, n);
                pb = fr ? NONE32 : min(b, n);
                push = true;
            }
        }
        const u32 m = __ballot_sync(FULL_MASK, push);
        u32 at = 0;
        if (m) {
            const u32 leader = __ffs(m) - 1;
            if (lane == leader) at = atomicAdd(count, (u32)__popc(m));
            at = __shfl_sync(FULL_MASK, at, leader);
        }
        if (push) {
            at += __popc(m & lanemask_lt());
            listR[at] = r;
            listP[at] = make_uint2(pa, pb);
        }
    }
}

// nodes [half, 2 half) of top from their children; one CTA takes every level from `half` down when
// `all` (half <= 1024 then)
__global__ void __launch_bounds__(1024) k_lpf_top(uint2 *__restrict__ top, u32 half, u32 all)
{
    if (!all) {
        const u32 v = half + blockIdx.x * blockDim.x + threadIdx.x;
        if (v < 2 * half) top[v] = lz_min2(top[2 * v], top[2 * v + 1]);
        return;
    }
    for (; half >= 1; half >>= 1) {
        for (u32 v = half + threadIdx.x; v < 2 * half; v += blockDim.x) top[v] = lz_min2(top[2 * v], top[2 * v + 1]);
        __syncthreads();
    }
}

// ---- 2. rows whose answer lies outside their tile ------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lpf_cross(const i32 *__restrict__ SA, const i32 *__restrict__ LCP, u32 n, u32 tb,
                                                   const uint2 *__restrict__ gtree, const uint2 *__restrict__ top, u32 P,
                                                   i32 *__restrict__ lpf, i32 *__restrict__ prev,
                                                   const u32 *__restrict__ listR, const uint2 *__restrict__ listP, u32 m)
{
    const u32 e = blockIdx.x * blockDim.x + threadIdx.x, lane = lane_id();
    const u32 G = (1u << tb) >> 5;
    u32 i = 0, a = 0, b = 0, srcL = NONE32, srcG = NONE32, gL = 0, gR = 0;
    bool needL = false, needR = false;
    if (e < m) {
        const u32 r = listR[e];
        const uint2 pp = listP[e];
        i = (u32)SA[r];
        const u32 t = r >> tb;
        if (pp.x == NONE32) { a = (u32)lpf[i]; srcL = (u32)prev[i]; }
        if (pp.y == NONE32) { b = (u32)lpf[i]; srcG = (u32)prev[i]; }
        if (pp.x != NONE32) {
            a = pp.x;
            u32 v = P + t;
            bool f = false;
            for (; v > 1; v >>= 1)
                if (v & 1) {
                    const uint2 s = top[v - 1];
                    if (s.x < i) { f = true; v--; break; }
                    a = min(a, s.y);
                }
            if (f) {
                while (v < P) {
                    const uint2 c = top[2 * v + 1];
                    if (c.x < i) v = 2 * v + 1;
                    else { a = min(a, c.y); v = 2 * v; }
                }
                const u32 tt = v - P;
                const uint2 *tr = gtree + (size_t)tt * 2 * G;
                u32 u = 1;
                while (u < G) {
                    const uint2 c = tr[2 * u + 1];
                    if (c.x < i) u = 2 * u + 1;
                    else { a = min(a, c.y); u = 2 * u; }
                }
                gL = (tt << tb) + ((u - G) << 5);
                needL = true;
            } else {
                a = 0;
            }
        }
        if (pp.y != NONE32) {
            b = pp.y;
            u32 v = P + t;
            bool f = false;
            for (; v > 1; v >>= 1)
                if (!(v & 1)) {
                    const uint2 s = top[v + 1];
                    if (s.x < i) { f = true; v++; break; }
                    b = min(b, s.y);
                }
            if (f) {
                while (v < P) {
                    const uint2 c = top[2 * v];
                    if (c.x < i) v = 2 * v;
                    else { b = min(b, c.y); v = 2 * v + 1; }
                }
                const u32 tt = v - P;
                const uint2 *tr = gtree + (size_t)tt * 2 * G;
                u32 u = 1;
                while (u < G) {
                    const uint2 c = tr[2 * u];
                    if (c.x < i) u = 2 * u;
                    else { b = min(b, c.y); u = 2 * u + 1; }
                }
                gR = (tt << tb) + ((u - G) << 5);
                needR = true;
            } else {
                b = 0;
            }
        }
    }
    // the 32-row groups, one per ballot: the last (first) row with SA < i, and the LCP minimum of the rows
    // after it (up to and including it)
    for (u32 pend; (pend = __ballot_sync(FULL_MASK, needL)) != 0;) {
        const u32 src = __ffs(pend) - 1;
        const u32 row = __shfl_sync(FULL_MASK, gL, src) + lane, gi = __shfl_sync(FULL_MASK, i, src);
        const u32 s = row < n ? (u32)__ldg(SA + row) : NONE32, l = row < n ? (u32)__ldg(LCP + row) : NONE32;
        const u32 hi = 31 - __clz(__ballot_sync(FULL_MASK, s < gi));
        const u32 lm = warp_min(lane > hi ? l : NONE32), sv = __shfl_sync(FULL_MASK, s, hi);
        if (lane == src) { a = min(a, lm); srcL = sv; needL = false; }
    }
    for (u32 pend; (pend = __ballot_sync(FULL_MASK, needR)) != 0;) {
        const u32 src = __ffs(pend) - 1;
        const u32 row = __shfl_sync(FULL_MASK, gR, src) + lane, gi = __shfl_sync(FULL_MASK, i, src);
        const u32 s = row < n ? (u32)__ldg(SA + row) : NONE32, l = row < n ? (u32)__ldg(LCP + row) : NONE32;
        const u32 lo = __ffs(__ballot_sync(FULL_MASK, s < gi)) - 1;
        const u32 lm = warp_min(lane <= lo ? l : NONE32), sv = __shfl_sync(FULL_MASK, s, lo);
        if (lane == src) { b = min(b, lm); srcG = sv; needR = false; }
    }
    if (e < m) lpf_put(lpf, prev, i, a, srcL, b, srcG);
}

// ---- 3. chunk exits ----------------------------------------------------------------------------------------------
// Dynamic shared memory 4 W bytes.  X1[p] = the first chain node from p at or past the end of p's chunk (<= n).
__global__ void __launch_bounds__(256) k_lz_exit1(const i32 *__restrict__ lpf, u32 n, u32 tb, u32 *__restrict__ X1)
{
    extern __shared__ u32 lz_smem[];
    const u32 W = 1u << tb, base = blockIdx.x << tb, end = min(n, base + W);
    for (u32 q = threadIdx.x; q < W; q += blockDim.x) {
        const u32 p = base + q;
        lz_smem[q] = p < n ? p + max(1u, (u32)__ldg(lpf + p)) : n;
    }
    __syncthreads();
    for (u32 round = 0; round < tb; round++) {
        u32 v[(1 << LZ_TB_MAX) / 256];
#pragma unroll
        for (int k = 0; k < (1 << LZ_TB_MAX) / 256; k++) {
            const u32 q = threadIdx.x + k * 256;
            if (q < W) { const u32 x = lz_smem[q]; v[k] = x < end ? lz_smem[x - base] : x; }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < (1 << LZ_TB_MAX) / 256; k++) {
            const u32 q = threadIdx.x + k * 256;
            if (q < W) lz_smem[q] = v[k];
        }
        __syncthreads();
    }
    for (u32 q = threadIdx.x; q < W && base + q < n; q += blockDim.x) X1[base + q] = lz_smem[q];
}

// one round of Y[p] <- S[S[p]] while S[p] lies inside p's block of 2^sb positions: S = X_(k-1), Y = X_k in the
// first round, S = Y = X_k (in place) in the others.  A value read in place is a later iterate or the same one.
__global__ void __launch_bounds__(256) k_lz_jump(const u32 *S, u32 *Y, u32 n, u32 sb)
{
    const u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const u32 x = S[p];
    const u64 end = min((u64)n, (((u64)p >> sb) + 1) << sb);
    if (x < end) Y[p] = S[x];
    else if (S != Y) Y[p] = x;
}

// ---- 4. entries of the chain into the blocks ---------------------------------------------------------------------
// entry[b] = the chain's first node in block b of 2^sb positions, NONE32 (memset) where the chain skips it
__global__ void k_lz_top(const u32 *__restrict__ X, u32 n, u32 sb, u32 *__restrict__ entry)
{
    for (u32 p = 0; p < n; p = X[p]) entry[p >> sb] = p;
}
// from the entries of the blocks of 2^sb positions to those of 2^sb1 (X: that level's exits)
__global__ void __launch_bounds__(256) k_lz_down(const u32 *__restrict__ X, u32 n, u32 sb, u32 sb1,
                                                 const u32 *__restrict__ entry, u32 nblocks, u32 *__restrict__ entry1)
{
    const u32 b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    u32 p = entry[b];
    if (p == NONE32) return;
    const u32 end = (u32)min((u64)n, ((u64)b + 1) << sb);
    for (; p < end; p = X[p]) entry1[p >> sb1] = p;
}

// ---- 5. factors per chunk, then the factors ---------------------------------------------------------------------
// Dynamic shared memory 8 W bytes: the chunk's LPF values and its chain nodes.  EMIT = false: cnt[c] = the
// chunk's factors; EMIT = true: factor pairs (PREV[p], LPF[p]) or (T[p], 0) from pair off[c] on.
template <bool EMIT>
__global__ void __launch_bounds__(256) k_lz_chunk(const u8 *__restrict__ T, const i32 *__restrict__ lpf,
                                                  const i32 *__restrict__ prev, u32 n, u32 tb,
                                                  const u32 *__restrict__ entry1, u32 *__restrict__ cnt,
                                                  const u32 *__restrict__ off, i32 *__restrict__ factors)
{
    extern __shared__ u32 lz_smem[];
    __shared__ u32 k_s;
    const u32 W = 1u << tb, c = blockIdx.x, base = c << tb, end = min(n, base + W);
    const u32 e = entry1[c];
    if (e == NONE32) {  // block-uniform
        if (!EMIT && threadIdx.x == 0) cnt[c] = 0;
        return;
    }
    u32 *L = lz_smem, *list = lz_smem + W;
    for (u32 q = threadIdx.x; base + q < end; q += blockDim.x) L[q] = (u32)__ldg(lpf + base + q);
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 k = 0;
        for (u32 p = e; p < end; p += max(1u, L[p - base])) list[k++] = p;
        k_s = k;
    }
    __syncthreads();
    const u32 k = k_s;
    if (!EMIT) {
        if (threadIdx.x == 0) cnt[c] = k;
        return;
    }
    const size_t o = off[c];
    for (u32 j = threadIdx.x; j < k; j += blockDim.x) {
        const u32 p = list[j], l = L[p - base];
        factors[2 * (o + j)] = l ? __ldg(prev + p) : (i32)__ldg(T + p);
        factors[2 * (o + j) + 1] = (i32)l;
    }
}

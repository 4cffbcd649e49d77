// lzd.cuh -- LZ77 decoding: a factor list (include/bwts_b200.h, bwts_b200_lz77_decode_*) back into its text.
//
// Factor k covers [p_k, p_k + max(1, len_k)); a copy (src, len) sets out[p_k + j] = out[src + j] byte by byte, so
// a source may overlap its own factor and one byte may hang on a chain of earlier ones (n - 1 long on a^n).  Each
// position gets one word: bit 31 set = resolved, the byte in the low 8 bits; else the earlier position it copies.
//   1. k_lzd_tile_sum   per tile of 4096 factors: the literal / length rules and the sum of max(1, len_k) in u64;
//      k_lzd_tile_scan  exclusive scan of the tile sums in one CTA, the grand total;
//      k_lzd_apply      p_k (u32: the total is checked against n before any p_k is used) and the source rule.
//   2. k_lzd_chunk      one CTA per chunk of W = 2^tb positions: one binary search over p for the chunk's factor
//                       slice, one per position inside the slice (in shared memory), then tb rounds of pointer
//                       jumping in shared memory.  Every word ends resolved or pointing into an earlier chunk; the
//                       others go to the live list.
//   3. k_lzd_jump       v[i] <- v[v[i]] in place over the live list, compacting into the other list.  A chain now
//                       visits strictly earlier chunks, so it has at most ceil(n / W) - 1 hops and the rounds are
//                       bounded by ceil(log2 ceil(n / W)) + 1; a value read in place is the same or a later iterate.
//   4. k_lzd_bytes      out[i] = v[i] & 0xff.
//   Work: z + n log W in shared memory + live x rounds: O(n log n) for every input, whatever the factor lengths.
#pragma once
#include "common.cuh"

#define LZD_TILE 4096             // factors per scan tile: 256 threads x 16
#define LZD_RES 0x80000000u       // resolved word

static __device__ __forceinline__ u64 lzd_warp_incl_u64(u64 v)
{
    const u32 lane = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 y = __shfl_up_sync(FULL_MASK, v, o);
        if (lane >= (u32)o) v += y;
    }
    return v;
}

// exclusive sum over the CTA of 256 threads (ws: 8 words of shared memory); *all = the CTA's total
static __device__ __forceinline__ u64 lzd_cta_excl_u64(u64 v, u64 *ws, u64 *all)
{
    const u64 incl = lzd_warp_incl_u64(v);
    const u32 warp = threadIdx.x >> 5;
    if (lane_id() == 31) ws[warp] = incl;
    __syncthreads();
    u64 before = 0, tot = 0;
#pragma unroll
    for (u32 w = 0; w < 8; w++) {
        if (w < warp) before += ws[w];
        tot += ws[w];
    }
    *all = tot;
    return before + incl - v;
}

// ---- 1. checks and starts -------------------------------------------------------------------------------------
// bad[0] |= 1 on a literal byte outside [0, 255] or a negative length.  Pairs are read as two i32 loads: device
// factors need only be 4-byte aligned.
__global__ void __launch_bounds__(256) k_lzd_tile_sum(const i32 *__restrict__ f, u64 z, u64 *__restrict__ tsum,
                                                      u32 *__restrict__ bad)
{
    __shared__ u64 ws[8];
    const u64 base = (u64)blockIdx.x * LZD_TILE;
    u64 s = 0;
    bool b = false;
#pragma unroll 4
    for (int q = 0; q < 16; q++) {
        const u64 k = base + q * 256 + threadIdx.x;
        if (k < z) {
            const i32 a = __ldg(f + 2 * k), l = __ldg(f + 2 * k + 1);
            b |= l < 0 || (l == 0 && (u32)a > 255u);
            s += l > 0 ? (u64)l : 1u;
        }
    }
    u64 tot;
    lzd_cta_excl_u64(s, ws, &tot);
    if (__syncthreads_or(b) && threadIdx.x == 0) atomicOr(bad, 1u);
    if (threadIdx.x == 0) tsum[blockIdx.x] = tot;
}

// exclusive scan of the nt tile sums in place, one CTA of 1024 threads; *total = their sum
__global__ void __launch_bounds__(1024) k_lzd_tile_scan(u64 *__restrict__ tsum, u32 nt, u64 *__restrict__ total)
{
    __shared__ u64 ws[33];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    u64 carry = 0;
    for (u32 base = 0; base < nt; base += 1024) {
        const u32 k = base + threadIdx.x;
        const u64 v = k < nt ? tsum[k] : 0;
        const u64 incl = lzd_warp_incl_u64(v);
        if (lane == 31) ws[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const u64 w = ws[lane], wi = lzd_warp_incl_u64(w);
            ws[lane] = wi - w;
            if (lane == 31) ws[32] = wi;
        }
        __syncthreads();
        if (k < nt) tsum[k] = carry + ws[warp] + incl - v;
        carry += ws[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// p[k] = p_k (mod 2^32), thread t owning 16 consecutive factors of the tile; bad[0] |= 1 on a copy source outside
// [0, p_k).  The first rule's violations may give any p here: the caller rejects them by bad[0] and the total.
__global__ void __launch_bounds__(256) k_lzd_apply(const i32 *__restrict__ f, u64 z, const u64 *__restrict__ tsum,
                                                   u32 *__restrict__ p, u32 *__restrict__ bad)
{
    __shared__ u64 ws[8];
    const u64 k0 = (u64)blockIdx.x * LZD_TILE + threadIdx.x * 16;
    u64 s = 0;
#pragma unroll 4
    for (int q = 0; q < 16; q++) {
        const u64 k = k0 + q;
        if (k < z) {
            const i32 l = __ldg(f + 2 * k + 1);
            s += l > 0 ? (u64)l : 1u;
        }
    }
    u64 tot;
    u64 run = tsum[blockIdx.x] + lzd_cta_excl_u64(s, ws, &tot);
    bool b = false;
#pragma unroll 4
    for (int q = 0; q < 16; q++) {
        const u64 k = k0 + q;
        if (k < z) {
            const i32 a = __ldg(f + 2 * k), l = __ldg(f + 2 * k + 1);
            if (l > 0) b |= a < 0 || (u64)a >= run;
            p[k] = (u32)run;
            run += l > 0 ? (u64)l : 1u;
        }
    }
    if (__syncthreads_or(b) && threadIdx.x == 0) atomicOr(bad, 1u);
}

// ---- 2. chunks ---------------------------------------------------------------------------------------------------
// Dynamic shared memory 8 W bytes: the chunk's words, then the starts of its factor slice (at most W factors: all
// but the first start inside the chunk).  v: the words, live / *nlive: the positions left unresolved.
__global__ void __launch_bounds__(256) k_lzd_chunk(const i32 *__restrict__ f, const u32 *__restrict__ p, u32 z, u32 n,
                                                   u32 tb, u32 *__restrict__ v, u32 *__restrict__ live,
                                                   u32 *__restrict__ nlive)
{
    extern __shared__ u32 lzd_smem[];
    __shared__ u32 k_s[2];
    const u32 W = 1u << tb, base = blockIdx.x << tb, end = min(n, base + W);
    u32 *w = lzd_smem, *sp = lzd_smem + W;
    if (threadIdx.x < 2) {  // the factors holding base and end - 1: the last k with p[k] <= x
        const u32 x = threadIdx.x ? end - 1 : base;
        u32 lo = 0, hi = z;  // p[lo] <= x < p[hi] (p[z] = n)
        while (hi - lo > 1) {
            const u32 mid = lo + (hi - lo) / 2;
            if (__ldg(p + mid) <= x) lo = mid;
            else hi = mid;
        }
        k_s[threadIdx.x] = lo;
    }
    __syncthreads();
    const u32 k0 = k_s[0], m = k_s[1] - k0 + 1;
    for (u32 j = threadIdx.x; j < m; j += blockDim.x) sp[j] = __ldg(p + k0 + j);
    __syncthreads();
    for (u32 q = threadIdx.x; base + q < end; q += blockDim.x) {
        const u32 i = base + q;
        u32 lo = 0, hi = m;  // sp[lo] <= i < sp[hi]
        while (hi - lo > 1) {
            const u32 mid = (lo + hi) >> 1;
            if (sp[mid] <= i) lo = mid;
            else hi = mid;
        }
        const u32 k = k0 + lo;
        const i32 a = __ldg(f + 2 * (size_t)k), l = __ldg(f + 2 * (size_t)k + 1);
        w[q] = l == 0 ? (LZD_RES | (u32)a) : (u32)a + (i - sp[lo]);
    }
    __syncthreads();
    // pointer jumping inside the chunk: a chain inside it has fewer than W hops, so tb rounds resolve it or leave
    // it pointing below base
    for (u32 round = 0; round < tb; round++) {
        u32 t[(1 << LZ_TB_MAX) / 256];
        bool moved = false;
#pragma unroll
        for (int c = 0; c < (1 << LZ_TB_MAX) / 256; c++) {
            const u32 q = threadIdx.x + c * 256;
            if (q < W && base + q < end) {
                const u32 x = w[q];
                const bool in = !(x & LZD_RES) && x >= base;
                t[c] = in ? w[x - base] : x;
                moved |= in;
            }
        }
        if (!__syncthreads_or(moved)) break;
#pragma unroll
        for (int c = 0; c < (1 << LZ_TB_MAX) / 256; c++) {
            const u32 q = threadIdx.x + c * 256;
            if (q < W && base + q < end) w[q] = t[c];
        }
        __syncthreads();
    }
    const u32 lane = lane_id();
    for (u32 q0 = 0; q0 < W; q0 += blockDim.x) {  // uniform trip count: the append below is warp-wide
        const u32 q = q0 + threadIdx.x;
        bool push = false;
        if (q < W && base + q < end) {
            const u32 x = w[q];
            v[base + q] = x;
            push = !(x & LZD_RES);
        }
        const u32 msk = __ballot_sync(FULL_MASK, push);
        u32 at = 0;
        if (msk) {
            const u32 leader = __ffs(msk) - 1;
            if (lane == leader) at = atomicAdd(nlive, (u32)__popc(msk));
            at = __shfl_sync(FULL_MASK, at, leader);
        }
        if (push) live[at + __popc(msk & lanemask_lt())] = base + q;
    }
}

// ---- 3. global rounds ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_lzd_jump(u32 *v, const u32 *__restrict__ cur, u32 m, u32 *__restrict__ nxt,
                                                  u32 *__restrict__ nnxt)
{
    const u32 e = blockIdx.x * blockDim.x + threadIdx.x, lane = lane_id();
    bool push = false;
    u32 i = 0;
    if (e < m) {
        i = cur[e];
        const u32 y = v[v[i]];
        v[i] = y;
        push = !(y & LZD_RES);
    }
    const u32 msk = __ballot_sync(FULL_MASK, push);
    u32 at = 0;
    if (msk) {
        const u32 leader = __ffs(msk) - 1;
        if (lane == leader) at = atomicAdd(nnxt, (u32)__popc(msk));
        at = __shfl_sync(FULL_MASK, at, leader);
    }
    if (push) nxt[at + __popc(msk & lanemask_lt())] = i;
}

// ---- 4. bytes ------------------------------------------------------------------------------------------------------
// four positions a thread: one 16-byte load of words (v is 256-byte aligned), one 4-byte store where out allows it
__global__ void __launch_bounds__(256) k_lzd_bytes(const u32 *__restrict__ v, u32 n, u8 *__restrict__ out)
{
    const u64 i0 = 4 * ((u64)blockIdx.x * blockDim.x + threadIdx.x);
    if (i0 >= n) return;
    if (i0 + 4 <= n) {
        const uint4 x = ldg_stream_u4((const uint4 *)(v + i0));
        const u32 b = (x.x & 0xff) | (x.y & 0xff) << 8 | (x.z & 0xff) << 16 | (x.w & 0xff) << 24;
        if (((uintptr_t)(out + i0) & 3) == 0) {
            *(u32 *)(out + i0) = b;
        } else {
            out[i0] = (u8)b; out[i0 + 1] = (u8)(b >> 8); out[i0 + 2] = (u8)(b >> 16); out[i0 + 3] = (u8)(b >> 24);
        }
    } else {
        for (u64 i = i0; i < n; i++) out[i] = (u8)v[i];
    }
}

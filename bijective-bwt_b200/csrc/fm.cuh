// fm.cuh -- FM-index over libdivsufsort's BWT: the build kernels after the FWD_FM sort and the count / locate / extract
// queries (DESIGN.md section 4.9).
//
// Rows are those of T$: row 0 is the end-of-text suffix, row i >= 1 is SA row i-1.  The L column is the divbwt
// output U with the $ row (row `primary`) cut out, so row i's byte is U[i - (i > primary)] and
// occ(c, i) = occ_U(c, i - (i > primary)); C[c] = 1 + #{bytes < c}.  occ_U(c, j) comes from three levels:
//     S[(j >> 16) * sg + k]   u32, occurrences of symbol k before the superblock
//     B[(j >> 8) * sg + k]    u16, occurrences from the superblock start to the block start
//     U[j & ~255 .. j)        counted by 16 lanes with 16-byte loads
// k = map[c] indexes the sg symbols that occur in T; a byte with C[c + 1] == C[c] is absent and occ = 0 (all 256
// symbol indices are taken when every byte occurs).  Sampled SA: SA row r is marked
// when SA[r] % sample == 0 (bit r of marks), dir[r >> 8] counts the marked rows before r & ~255, and the marked
// rows' SA values lie in row order in samples[].
#pragma once
#include "common.cuh"

#define FM_BLOCK 256
#define FM_SUPER 65536

struct FmView {
    const u8 *U;
    const u32 *S;
    const u16 *B;
    const u32 *marks, *dir, *samples, *C;  // C[0..256], C[256] = n + 1
    const u8 *map;
    u32 n, primary, sample, sg;
};

// ---- build ----------------------------------------------------------------------------------------------
// byte histogram of T (256 words, zeroed by the caller)
__global__ void __launch_bounds__(256) k_fm_hist(const u8 *__restrict__ T, u32 n, u32 *__restrict__ hist)
{
    __shared__ u32 h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    for (u64 i = (u64)blockIdx.x * 256 + threadIdx.x; i < n; i += (u64)gridDim.x * 256) atomicAdd(&h[T[i]], 1u);
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

// one warp per 256-byte block of U (blocks 0 .. n >> 8, the last one possibly empty): B[b * sg + k] = occurrences of
// symbol k in the block; syms[k] = the byte of symbol k
__global__ void __launch_bounds__(256) k_fm_block_counts(const u8 *__restrict__ U, u32 n, const u8 *__restrict__ syms,
                                                         u32 sg, u16 *__restrict__ B)
{
    const u32 b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = lane_id();
    if (b > (n >> 8)) return;
    const u64 p = (u64)b * FM_BLOCK + lane * 8;
    u32 w0 = 0, w1 = 0, valid = 0;  // lane's 8 bytes and how many of them lie before n
    if (p < n) {
        valid = (u32)min((u64)8, n - p);
        if (valid == 8) {
            const uint2 v = *(const uint2 *)(U + p);
            w0 = v.x; w1 = v.y;
        } else {
            for (u32 q = 0; q < valid; q++) {
                const u32 x = U[p + q];
                if (q < 4) w0 |= x << (8 * q); else w1 |= x << (8 * (q - 4));
            }
        }
    }
    const u32 m0 = valid >= 4 ? 0x01010101u : (0x01010101u & ((1u << (8 * valid)) - 1u));
    const u32 m1 = valid >= 8 ? 0x01010101u : valid <= 4 ? 0u : (0x01010101u & ((1u << (8 * (valid - 4))) - 1u));
    for (u32 k = 0; k < sg; k++) {
        const u32 cc = 0x01010101u * syms[k];
        const u32 c = __popc(__vcmpeq4(w0, cc) & m0) + __popc(__vcmpeq4(w1, cc) & m1);
        const u32 t = __reduce_add_sync(FULL_MASK, c);
        if (lane == 0) B[(size_t)b * sg + k] = (u16)t;
    }
}

// one thread per symbol and superblock: the block counts of superblock s become exclusive prefixes inside it,
// and S[s * sg + k] receives the superblock's total (scanned by k_fm_super_scan)
__global__ void __launch_bounds__(256) k_fm_block_scan(u32 n, u32 sg, u16 *__restrict__ B, u32 *__restrict__ S)
{
    const u32 s = blockIdx.x, k = threadIdx.x;
    if (k >= sg) return;
    const u32 b0 = s << 8, b1 = min((n >> 8) + 1, b0 + 256);
    u32 run = 0;
    for (u32 b = b0; b < b1; b++) {
        const u32 v = B[(size_t)b * sg + k];
        B[(size_t)b * sg + k] = (u16)run;
        run += v;
    }
    S[(size_t)s * sg + k] = run;
}

// one warp per symbol: exclusive scan of the superblock totals over s = 0 .. n >> 16, in place
__global__ void __launch_bounds__(32) k_fm_super_scan(u32 n, u32 sg, u32 *__restrict__ S)
{
    const u32 k = blockIdx.x, lane = lane_id(), ns = (n >> 16) + 1;
    u32 carry = 0;
    for (u32 s0 = 0; s0 < ns; s0 += 32) {
        const u32 s = s0 + lane;
        const u32 v = s < ns ? S[(size_t)s * sg + k] : 0u;
        const u32 incl = warp_incl_sum(v);
        if (s < ns) S[(size_t)s * sg + k] = carry + incl - v;
        carry += __shfl_sync(FULL_MASK, incl, 31);
    }
}

// one CTA per 256 rows (n / 256 + 1 CTAs): the mark bits and the directory's per-block counts
__global__ void __launch_bounds__(256) k_fm_marks(const i32 *__restrict__ sa, u32 n, u32 sample, u32 *__restrict__ marks,
                                                  u32 *__restrict__ dir)
{
    const u32 r = blockIdx.x * 256 + threadIdx.x;
    const bool m = r < n && ((u32)sa[r] & (sample - 1)) == 0;
    const u32 w = __ballot_sync(FULL_MASK, m);
    if (lane_id() == 0 && r < n) marks[r >> 5] = w;
    const u32 c = __syncthreads_count(m);
    if (threadIdx.x == 0) dir[blockIdx.x] = c;
}

// rank of SA row r among the marked rows (r marked or not)
static __device__ __forceinline__ u32 fm_mark_rank(const u32 *__restrict__ marks, const u32 *__restrict__ dir, u32 r)
{
    u32 k = __ldg(dir + (r >> 8));
    for (u32 w = (r >> 8) << 3; w < (r >> 5); w++) k += __popc(__ldg(marks + w));
    return k + __popc(__ldg(marks + (r >> 5)) & ((1u << (r & 31)) - 1u));
}

__global__ void __launch_bounds__(256) k_fm_samples(const i32 *__restrict__ sa, u32 n, u32 sample,
                                                    const u32 *__restrict__ marks, const u32 *__restrict__ dir,
                                                    u32 *__restrict__ samples)
{
    const u32 r = blockIdx.x * 256 + threadIdx.x;
    if (r >= n) return;
    const u32 v = (u32)sa[r];
    if ((v & (sample - 1)) == 0) samples[fm_mark_rank(marks, dir, r)] = v;
}

// ---- queries ---------------------------------------------------------------------------------------------
// occ_U(c, j) for the 16 lanes of one half-warp (hl = lane & 15, hmask its lanes); every lane gets the result.
// *rd adds the bytes read (lane 0 of the half)
static __device__ __forceinline__ u32 fm_occ_u(const FmView &f, const u32 *sC, const u8 *smap, u32 c, u32 j, u32 hl,
                                               u32 hmask, u64 *rd)
{
    if (sC[c + 1] == sC[c]) return 0;
    const u32 k = smap[c];
    const u32 base = j & ~(u32)(FM_BLOCK - 1), r = j & (FM_BLOCK - 1), o = hl * 16;
    u32 cnt = 0;
    if (o < r) {  // base + o < j <= n: the 16-byte load ends inside U's allocation (rounded up to 256)
        const uint4 w = __ldg((const uint4 *)(f.U + base + o));
        const u32 cc = 0x01010101u * c, v = min(16u, r - o);
        const u32 ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const u32 vq = v > 4u * q ? min(4u, v - 4u * q) : 0u;
            const u32 m = vq == 4 ? 0x01010101u : (0x01010101u & ((1u << (8 * vq)) - 1u));
            cnt += __popc(__vcmpeq4(ws[q], cc) & m);
        }
    }
#pragma unroll
    for (int d = 8; d > 0; d >>= 1) cnt += __shfl_xor_sync(hmask, cnt, d, 16);
    if (hl == 0) *rd += 6 + ((r + 15) & ~15u);
    return __ldg(f.S + (size_t)(j >> 16) * f.sg + k) + __ldg(f.B + (size_t)(j >> 8) * f.sg + k) + cnt;
}
static __device__ __forceinline__ u32 fm_occ(const FmView &f, const u32 *sC, const u8 *smap, u32 c, u32 i, u32 hl,
                                             u32 hmask, u64 *rd)
{
    return fm_occ_u(f, sC, smap, c, i - (i > f.primary), hl, hmask, rd);
}

// Device-form checks, before any other work: off[0] == 0, off non-decreasing, off[npat] == pat_len.  *bad = 1 on
// a violation (zeroed by the caller); k_fm_count does nothing when it is set.
__global__ void __launch_bounds__(256) k_fm_check_off(const long long *__restrict__ off, u64 npat, long long pat_len,
                                                      u32 *__restrict__ bad)
{
    for (u64 k = (u64)blockIdx.x * 256 + threadIdx.x; k <= npat; k += (u64)gridDim.x * 256) {
        const long long v = off[k];
        bool ok = k == npat ? v == pat_len : v <= off[k + 1];
        if (k == 0) ok = ok && v == 0;
        if (!ok) atomicOr(bad, 1u);
    }
}

// Backward search, one warp per pattern (grid-stride): lanes 0-15 carry sp, lanes 16-31 ep, both through every
// byte of the pattern read from its end.  range[2k] = lo = sp - 1 (0 for the empty pattern), range[2k+1] = hi =
// ep - 1.  cnt[0] += sum of (hi - lo), cnt[1] += bytes read.
__global__ void __launch_bounds__(256) k_fm_count(FmView f, const u8 *__restrict__ pat, const long long *__restrict__ off,
                                                  u64 npat, i32 *__restrict__ range, const u32 *__restrict__ bad,
                                                  unsigned long long *__restrict__ cnt)
{
    __shared__ u32 sC[257];
    __shared__ u8 smap[256];
    if (*bad) return;
    for (u32 t = threadIdx.x; t < 257; t += 256) sC[t] = f.C[t];
    smap[threadIdx.x] = f.map[threadIdx.x];
    __syncthreads();
    const u32 lane = lane_id(), hl = lane & 15, hmask = lane < 16 ? 0x0000ffffu : 0xffff0000u;
    const u64 warps = (u64)gridDim.x * 8;
    u64 hits = 0, rd = 0;
    for (u64 k = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); k < npat; k += warps) {
        const long long a = off[k], e = off[k + 1];
        const u64 m = (u64)(e - a);
        u32 x = lane < 16 ? 0u : f.n + 1;  // sp = 0, ep = n + 1: every row of T$
        u32 chunk = 0;
        for (u64 s = 0; s < m; s++) {
            if ((s & 31) == 0) {  // 32 bytes of the pattern, from its end, one per lane
                const u64 q = s + lane;
                chunk = q < m ? pat[e - 1 - (long long)q] : 0u;
                rd += 32;
            }
            const u32 c = __shfl_sync(FULL_MASK, chunk, (u32)(s & 31));
            x = sC[c] + fm_occ(f, sC, smap, c, x, hl, hmask, &rd);
        }
        const u32 sp = __shfl_sync(FULL_MASK, x, 0), ep = __shfl_sync(FULL_MASK, x, 16);
        const u32 lo = m ? sp - 1 : 0u, hi = ep - 1;
        if (lane == 0) {
            range[2 * k] = (i32)lo;
            range[2 * k + 1] = (i32)hi;
            hits += hi - lo;
            rd += 16 + 8;
        }
    }
    if (lane == 0 && (hits || rd)) {
        atomicAdd(cnt, (unsigned long long)hits);
        atomicAdd(cnt + 1, (unsigned long long)rd);
    }
}

// One CTA: checks every range (0 <= lo <= hi <= n), writes the exclusive offsets of hi - lo to offs[0..nrange]
// (offs[nrange] = the total).  flags[0] = 1 on a bad range, flags[1] = 1 when the total exceeds cap, flags[2..3] =
// the total (u64, 8-byte aligned).
__global__ void __launch_bounds__(1024) k_fm_range_scan(const i32 *__restrict__ range, u64 nrange, u32 n, u64 cap,
                                                        unsigned long long *__restrict__ offs, u32 *__restrict__ flags)
{
    __shared__ unsigned long long ws[33];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    unsigned long long carry = 0;
    bool bad = false;
    for (u64 base = 0; base < nrange; base += 1024) {
        const u64 k = base + threadIdx.x;
        unsigned long long v = 0;
        if (k < nrange) {
            const i32 lo = range[2 * k], hi = range[2 * k + 1];
            if (lo < 0 || lo > hi || (u32)hi > n) bad = true;
            else v = (unsigned long long)(hi - lo);
        }
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long y = __shfl_up_sync(FULL_MASK, incl, o);
            if (lane >= (u32)o) incl += y;
        }
        if (lane == 31) ws[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long w = ws[lane];
            unsigned long long wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long y = __shfl_up_sync(FULL_MASK, wi, o);
                if (lane >= (u32)o) wi += y;
            }
            ws[lane] = wi - w;
            if (lane == 31) ws[32] = wi;
        }
        __syncthreads();
        if (k < nrange) offs[k] = carry + ws[warp] + incl - v;
        carry += ws[32];
        __syncthreads();
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) {
        offs[nrange] = carry;
        flags[0] = bad;
        flags[1] = carry > cap;
        *(unsigned long long *)(flags + 2) = carry;
    }
}

// Locate, one half-warp per output slot p (grid-stride): the range k with offs[k] <= p < offs[k+1] by binary search,
// SA row r = lo_k + p - offs[k], then LF from FM row r + 1 until a marked row: pos[p] = sample value + steps.
// Position 0 is marked, so no walk reaches the $ row.  cnt[0] += bytes read.
__global__ void __launch_bounds__(256) k_fm_locate(FmView f, const i32 *__restrict__ range, u64 nrange,
                                                   const unsigned long long *__restrict__ offs, u64 total,
                                                   i32 *__restrict__ pos, unsigned long long *__restrict__ cnt)
{
    __shared__ u32 sC[257];
    __shared__ u8 smap[256];
    for (u32 t = threadIdx.x; t < 257; t += 256) sC[t] = f.C[t];
    smap[threadIdx.x] = f.map[threadIdx.x];
    __syncthreads();
    const u32 lane = lane_id(), hl = lane & 15, hmask = lane < 16 ? 0x0000ffffu : 0xffff0000u;
    const u64 halves = (u64)gridDim.x * 16;
    u64 rd = 0;
    for (u64 p = (u64)blockIdx.x * 16 + (threadIdx.x >> 4); p < total; p += halves) {
        u64 a = 0, b = nrange;  // largest k with offs[k] <= p
        while (b - a > 1) {
            const u64 mid = (a + b) >> 1;
            if (offs[mid] <= p) a = mid; else b = mid;
            rd += 8;
        }
        u32 r = (u32)(range[2 * a] + (p - offs[a]));
        u32 steps = 0;
        rd += 8 + 16;  // offs[a], the range
        for (;;) {
            const u32 w = __ldg(f.marks + (r >> 5));
            rd += 4;
            if ((w >> (r & 31)) & 1u) break;
            const u32 i = r + 1;  // FM row; never the $ row (i != primary: that row's SA value, 0, is marked)
            const u32 c = __ldg(f.U + (i - (i > f.primary)));
            r = sC[c] + fm_occ(f, sC, smap, c, i, hl, hmask, &rd) - 1;
            rd += 1;
            steps++;
        }
        if (hl == 0) {
            pos[p] = (i32)(__ldg(f.samples + fm_mark_rank(f.marks, f.dir, r)) + steps);
            rd += 4 + 4 + 32 + 4;
        }
    }
    if (lane == 0 || lane == 16) {
        if (rd) atomicAdd(cnt, (unsigned long long)rd);
    }
}

// ---- extract ---------------------------------------------------------------------------------------------
// The inverse of the samples, derived per call: isa[v >> sh] = FM row of text position v for every sampled v
// (sample = 2^sh), and isa[ceil(n / sample)] = 0, the $ row, which is the row of position n.  Segment q of the text
// is [q << sh, min((q + 1) << sh, n)); it is decoded from the row isa[q + 1] of its end by LF steps, each giving
// the byte before the current position: T[p - 1] = L[row].

// One warp per 256-row block of the marks: lane l takes rows 8l .. 8l + 7 of the block, its marked rows' ranks
// follow from dir and a warp scan, and each marked row r with value v = samples[rank] sets isa[v >> sh] = r + 1.
__global__ void __launch_bounds__(256) k_fm_isa(FmView f, u32 sh, u32 *__restrict__ isa)
{
    const u32 b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = lane_id();
    if (blockIdx.x == 0 && threadIdx.x == 0) isa[(f.n + (1u << sh) - 1) >> sh] = 0;
    if ((u64)b * FM_BLOCK >= f.n) return;
    const u32 w = b * 8 + (lane >> 2);
    const u32 bits = w < (f.n + 31) / 32 ? (__ldg(f.marks + w) >> ((lane & 3) * 8)) & 0xffu : 0u;
    const u32 c = __popc(bits);
    u32 rank = __ldg(f.dir + b) + warp_incl_sum(c) - c;
    for (u32 m = bits; m; m &= m - 1) {
        const u32 r = b * FM_BLOCK + lane * 8 + (__ffs(m) - 1);
        isa[__ldg(f.samples + rank++) >> sh] = r + 1;
    }
}

static __device__ __forceinline__ u64 fm_warp_incl_u64(u64 v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 y = __shfl_up_sync(FULL_MASK, v, o);
        if (lane_id() >= (u32)o) v += y;
    }
    return v;
}

// One CTA, after k_fm_range_scan accepted the ranges: segs[k] = exclusive 64-bit prefix of the segment counts
// ceil(b_k / s) - floor(a_k / s) (0 for an empty range), segs[nrange] = the number of segments.
__global__ void __launch_bounds__(1024) k_fm_seg_scan(const i32 *__restrict__ range, u64 nrange, u32 sh,
                                                      unsigned long long *__restrict__ segs)
{
    __shared__ u64 ws[33];
    const u32 lane = lane_id(), warp = threadIdx.x >> 5;
    u64 carry = 0;
    for (u64 base = 0; base < nrange; base += 1024) {
        const u64 k = base + threadIdx.x;
        u64 v = 0;
        if (k < nrange) {
            const u32 a = (u32)range[2 * k], b = (u32)range[2 * k + 1];
            v = a < b ? (u64)(((b - 1) >> sh) - (a >> sh) + 1) : 0u;
        }
        const u64 incl = fm_warp_incl_u64(v);
        if (lane == 31) ws[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const u64 x = ws[lane], xi = fm_warp_incl_u64(x);
            ws[lane] = xi - x;
            if (lane == 31) ws[32] = xi;
        }
        __syncthreads();
        if (k < nrange) segs[k] = carry + ws[warp] + incl - v;
        carry += ws[32];
        __syncthreads();
    }
    if (threadIdx.x == 0) segs[nrange] = carry;
}

// Extract, one half-warp per segment (grid-stride): the range k with segs[k] <= g < segs[k+1] by binary search,
// its segment q = a_k / s + g - segs[k], then LF from isa[q + 1] down to position max(a_k, q s); the bytes at
// positions inside [a_k, b_k) go to out[offs[k] + p - a_k].  A walk stops at position >= 0 before reading row
// primary, so the $ is never read.  cnt[0] += bytes read.
__global__ void __launch_bounds__(256) k_fm_extract(FmView f, const u32 *__restrict__ isa, u32 sh,
                                                    const i32 *__restrict__ range, u64 nrange,
                                                    const unsigned long long *__restrict__ offs,
                                                    const unsigned long long *__restrict__ segs, u8 *__restrict__ out,
                                                    unsigned long long *__restrict__ cnt)
{
    __shared__ u32 sC[257];
    __shared__ u8 smap[256];
    for (u32 t = threadIdx.x; t < 257; t += 256) sC[t] = f.C[t];
    smap[threadIdx.x] = f.map[threadIdx.x];
    __syncthreads();
    const u32 lane = lane_id(), hl = lane & 15, hmask = lane < 16 ? 0x0000ffffu : 0xffff0000u;
    const u64 halves = (u64)gridDim.x * 16, nseg = segs[nrange];
    u64 rd = 0;
    for (u64 g = (u64)blockIdx.x * 16 + (threadIdx.x >> 4); g < nseg; g += halves) {
        u64 lo = 0, hi = nrange;  // largest k with segs[k] <= g: the non-empty range after any empty ones
        while (hi - lo > 1) {
            const u64 mid = (lo + hi) >> 1;
            if (segs[mid] <= g) lo = mid; else hi = mid;
            rd += 8;
        }
        const u32 a = (u32)range[2 * lo], b = (u32)range[2 * lo + 1];
        const u32 q = (a >> sh) + (u32)(g - segs[lo]);
        const u32 first = max(a, q << sh);
        const u64 base = offs[lo] - a;  // out[base + p] holds T[p]
        u32 p = min((q + 1) << sh, f.n);
        u32 i = __ldg(isa + q + 1);
        rd += 8 + 8 + 8 + 4;  // segs[k], offs[k], the range, the start row
        for (;;) {
            const u32 c = __ldg(f.U + (i - (i > f.primary)));
            rd += 1;
            p--;
            if (hl == 0 && p < b) out[base + p] = (u8)c;
            if (p == first) break;
            i = sC[c] + fm_occ(f, sC, smap, c, i, hl, hmask, &rd);
        }
    }
    if (lane == 0 || lane == 16) {
        if (rd) atomicAdd(cnt, (unsigned long long)rd);
    }
}

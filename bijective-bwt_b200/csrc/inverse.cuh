// inverse.cuh -- inverse BWTS kernels.
//
// Reference: /root/reference/unbwts.c:31-86.  prev[i] = C[B[i]] + occ(B[i], i) is the
// stable LF map (:31-52); its cycles are the Lyndon factors.  The reference walks them one
// byte at a time (:62-86): cycles in order of ascending smallest index, the first one
// landing at the END of the output, bytes of a cycle written at descending positions
// starting from the cycle's smallest index.  Closed form used here:
//     out[n-1 - off(c) - d(i)] = B[i]
// d(i) = prev-steps from the smallest index of i's cycle to i, off(c) = total length of
// the cycles whose smallest index is below c's.
//
// d and off come from list ranking with hashed splitters.  Every splitter walks its sublist
// (k_inv_walk: length, smallest index, next sublist -- it only READS prev), the reduced list
// of splitters is ranked by pointer jumping (min, then suffix sums cut at the sublist holding
// the cycle minimum), an exclusive scan over the cycle lengths parked at the cycle minima
// gives off, and every splitter walks its sublist a second time (k_inv_walk_place) writing
// its bytes at descending, consecutive output positions; the byte of element i is recovered
// from prev[i] alone (it is the byte whose C-range holds prev[i]).  Random traffic is two
// 4-byte reads per element and nothing else.  Cycles without any splitter (detected by the
// sublist lengths not adding up to n; the first walk also sets a visited bit per element, the
// bitmap stays in L2) take the fallback: walk themselves, place.
#pragma once
#include "common.cuh"

#define INV_TILE 8192  // bytes per tile, 256 threads x 32
#define INV_NT 256
#define INV_CHUNK 256  // tiles per column-scan chunk

// ---- byte counts per tile -------------------------------------------------------------------
__global__ void __launch_bounds__(INV_NT) k_inv_tile_hist(const u8 *__restrict__ B, u32 n, u32 *__restrict__ tilehist)
{
    __shared__ u32 wh[INV_NT / 32][256];
    const u32 tid = threadIdx.x, warp = tid >> 5;
    for (u32 i = tid; i < (INV_NT / 32) * 256; i += INV_NT) ((u32 *)wh)[i] = 0;
    __syncthreads();
    const u32 base = blockIdx.x * INV_TILE;
    u32 *h = wh[warp];
    // two 16-byte vectors per thread; runs of equal bytes are folded before the atomic
#pragma unroll
    for (int v = 0; v < 2; v++) {
        const u32 p = base + (v * INV_NT + tid) * 16;
        if (p + 16 <= n) {
            const uint4 x = ldg_stream_u4((const uint4 *)(B + p));
            const u32 w[4] = {x.x, x.y, x.z, x.w};
            u32 cur = w[0] & 255, run = 0;
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int s = 0; s < 32; s += 8) {
                    const u32 c = (w[q] >> s) & 255;
                    if (c == cur) run++;
                    else { atomicAdd(&h[cur], run); cur = c; run = 1; }
                }
            atomicAdd(&h[cur], run);
        } else {
            for (u32 q = p; q < n && q < p + 16; q++) atomicAdd(&h[B[q]], 1u);
        }
    }
    __syncthreads();
    u32 s = 0;
#pragma unroll
    for (int w = 0; w < INV_NT / 32; w++) s += wh[w][tid];
    tilehist[(u64)blockIdx.x * 256 + tid] = s;
}

// column sums over chunks of INV_CHUNK tiles (grid = nchunks, block = 256)
__global__ void __launch_bounds__(256) k_inv_colsum(const u32 *__restrict__ tilehist, u32 ntiles,
                                                    u32 *__restrict__ chunksum)
{
    const u32 lo = blockIdx.x * INV_CHUNK, hi = min(ntiles, lo + INV_CHUNK);
    u32 s = 0;
    for (u32 t = lo; t < hi; t++) s += tilehist[(u64)t * 256 + threadIdx.x];
    chunksum[blockIdx.x * 256 + threadIdx.x] = s;
}

// single block: per byte exclusive scan over chunks, then add C[byte]
__global__ void __launch_bounds__(256) k_inv_chunk_scan(u32 *__restrict__ chunksum, u32 nchunks,
                                                        u32 *__restrict__ Cout /*[257]*/)
{
    __shared__ u32 ws[8];
    const u32 d = threadIdx.x;
    u32 run = 0;
    for (u32 c = 0; c < nchunks; c++) {
        const u32 v = chunksum[c * 256 + d];
        chunksum[c * 256 + d] = run;
        run += v;
    }
    const u32 incl = warp_incl_sum(run);
    if (lane_id() == 31) ws[d >> 5] = incl;
    __syncthreads();
    u32 C = incl - run;
    for (u32 w = 0; w < (d >> 5); w++) C += ws[w];
    for (u32 c = 0; c < nchunks; c++) chunksum[c * 256 + d] += C;
    Cout[d] = C;
    if (d == 255) Cout[256] = C + run;
}

// tilehist -> exclusive base per (tile, byte), in place
__global__ void __launch_bounds__(256) k_inv_tile_base(u32 *__restrict__ tilehist, u32 ntiles,
                                                       const u32 *__restrict__ chunksum)
{
    const u32 lo = blockIdx.x * INV_CHUNK, hi = min(ntiles, lo + INV_CHUNK);
    u32 run = chunksum[blockIdx.x * 256 + threadIdx.x];
    for (u32 t = lo; t < hi; t++) {
        const u32 v = tilehist[(u64)t * 256 + threadIdx.x];
        tilehist[(u64)t * 256 + threadIdx.x] = run;
        run += v;
    }
}

// ---- stable LF map ------------------------------------------------------------------------------
// DIV (libdivsufsort's inverse_bw_transform, `primary` in [1, n]): B is the sentinel BWT with its end of
// text removed, and prev receives the map with that row cut out of the cycle,
//     p = 1 + LF(i),  prev_s(i) = (p == primary) ? 0 : p - (p > primary),
// a permutation of [0, n) whatever B and primary are; out[n-1-j] = B[prev_s^j(0)] is the classic walk
// from row 0.  The placement kernels recover the byte of i from prev[i] through C (byte_of_rank), so
// block 0 also rewrites Ctab to C'[c] = C[c] + (C[c] < primary): then byte_of_rank(C', prev_s(i)) = B[i]
// for every prev_s(i) > 0.  The one element with prev_s = 0 gets byte 0 there; its byte c*, the c with
// C[c] < primary <= C[c+1], goes to *cstar and k_bwt_locate<true> puts it in place.
template <bool DIV = false>
__global__ void __launch_bounds__(INV_NT) k_inv_lf_rank(const u8 *__restrict__ B, u32 n,
                                                        const u32 *__restrict__ tilebase, u32 *__restrict__ prev,
                                                        u32 primary = 0, u32 *__restrict__ Ctab = nullptr,
                                                        u32 *__restrict__ cstar = nullptr)
{
    __shared__ __align__(16) u8 s_b[INV_TILE];
    __shared__ u32 s_wcnt[INV_NT / 32][256];
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const u32 base = blockIdx.x * INV_TILE;
    if (DIV && blockIdx.x == 0) {  // block-uniform
        const u32 c = Ctab[tid], c1 = Ctab[tid + 1];
        __syncthreads();
        if (c < primary && primary <= c1) *cstar = tid;
        Ctab[tid] = c + (c < primary);
    }
    for (u32 i = tid; i < (INV_NT / 32) * 256; i += INV_NT) ((u32 *)s_wcnt)[i] = 0;
#pragma unroll
    for (int v = 0; v < 2; v++) {
        const u32 o = (v * INV_NT + tid) * 16;
        if (base + o + 16 <= n) {
            *(uint4 *)(s_b + o) = ldg_stream_u4((const uint4 *)(B + base + o));
        } else {
            for (u32 q = 0; q < 16; q++) s_b[o + q] = (base + o + q < n) ? B[base + o + q] : 0;
        }
    }
    __syncthreads();
    // warp w ranks bytes [w*1024, (w+1)*1024) of the tile, 32 at a time, in order
    constexpr int ROUNDS = INV_TILE / INV_NT;  // 32
    const u32 wo = warp * (32 * ROUNDS);
    u32 *wc = s_wcnt[warp];
    const u32 lt = lanemask_lt();
    u16 rnk[ROUNDS];
#pragma unroll
    for (int j = 0; j < ROUNDS; j++) {
        const u32 o = wo + j * 32 + lane;
        const bool valid = base + o < n;
        const u32 d = valid ? s_b[o] : 256u + lane;  // invalid lanes match nobody
        const u32 peers = __match_any_sync(FULL_MASK, d);
        const int leader = __ffs(peers) - 1;
        u32 before = 0;
        if (valid && (int)lane == leader) {
            before = wc[d];
            wc[d] = before + __popc(peers);
        }
        before = __shfl_sync(FULL_MASK, before, leader);
        rnk[j] = (u16)(before + __popc(peers & lt));
        __syncwarp();
    }
    __syncthreads();
    {
        const u32 d = tid;
        u32 run = __ldg(tilebase + (u64)blockIdx.x * 256 + d);
#pragma unroll
        for (int w = 0; w < INV_NT / 32; w++) {
            const u32 c = s_wcnt[w][d];
            s_wcnt[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < ROUNDS; j++) {
        const u32 o = wo + j * 32 + lane;
        if (base + o < n) {
            u32 v = wc[s_b[o]] + rnk[j];
            if (DIV) {
                const u32 p = v + 1;
                v = p == primary ? 0u : p - (p > primary);
            }
            prev[base + o] = v;
        }
    }
}

// ---- splitters ------------------------------------------------------------------------------------
// Splitters are picked by a multiplicative hash of the index: density 2^-(32 - shift).  The
// multiplier is a parameter: when the self-walk fallback runs over its work budget (a long cycle
// that the hash happens to miss -- it is public and fixed, so an input can be built against it),
// the host starts the inverse again with another multiplier and a denser set.
struct SplHash { u32 mul, shift; };
static __device__ __forceinline__ bool is_splitter(u32 i, SplHash h) { return ((i * h.mul) >> h.shift) == 0; }

#define SP_TILE 4096
__global__ void __launch_bounds__(256) k_inv_spl_count(u32 n, SplHash shift, u32 *__restrict__ tilecnt)
{
    __shared__ u32 ws[8];
    const u32 base = blockIdx.x * SP_TILE + threadIdx.x * 16;
    u32 c = 0;
#pragma unroll
    for (int q = 0; q < 16; q++) c += (base + q < n) && is_splitter(base + q, shift);
    c = warp_sum(c);
    if (lane_id() == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 s = 0;
        for (int w = 0; w < 8; w++) s += ws[w];
        tilecnt[blockIdx.x] = s;
    }
}
// sid (two-walk path): sparse map element -> sublist id, written at splitter slots only.
// blkoff (staged path): blkoff[b] = number of splitters below element 64 b; the id of the sublist
// that starts at splitter p is blkoff[p >> 6] + the splitters in [p & ~63, p) (sid_of).
__global__ void __launch_bounds__(256) k_inv_spl_write(u32 n, SplHash shift, const u32 *__restrict__ tileoff,
                                                       u32 *__restrict__ spl, u32 *__restrict__ sid,
                                                       u32 *__restrict__ blkoff)
{
    __shared__ u32 ws[8];
    const u32 base = blockIdx.x * SP_TILE + threadIdx.x * 16;
    u32 c = 0;
#pragma unroll
    for (int q = 0; q < 16; q++) c += (base + q < n) && is_splitter(base + q, shift);
    const u32 incl = warp_incl_sum(c);
    if (lane_id() == 31) ws[threadIdx.x >> 5] = incl;
    __syncthreads();
    u32 s = tileoff[blockIdx.x] + incl - c;
    for (u32 w = 0; w < (threadIdx.x >> 5); w++) s += ws[w];
    if (blkoff && (threadIdx.x & 3) == 0 && base < n) blkoff[base >> 6] = s;  // SP_TILE and 16 divide 64-blocks evenly
#pragma unroll
    for (int q = 0; q < 16; q++)
        if ((base + q < n) && is_splitter(base + q, shift)) {
            spl[s] = base + q;
            if (sid) sid[base + q] = s;
            s++;
        }
}
static __device__ __forceinline__ u32 sid_of(const u32 *__restrict__ blkoff, u32 p, SplHash shift)
{
    u32 s = __ldg(blkoff + (p >> 6));
    for (u32 q = p & ~63u; q < p; q++) s += is_splitter(q, shift);
    return s;
}

// first walk: one thread per splitter follows prev until the next splitter.  (A persistent
// variant with dynamic work fetch was measured slower: the limit is the dependent random
// access rate, not warp divergence.)
// jm[s] = next sublist << 32 | smallest index; wlen[s] = sublist length; minfo[s] = (smallest
// index, its offset).  visited (optional) gets one bit per element reached.  *total += lengths.
__global__ void __launch_bounds__(128) k_inv_walk(const u32 *__restrict__ prev, SplHash shift,
                                                  const u32 *__restrict__ spl, u32 ns, const u32 *__restrict__ sid,
                                                  u64 *__restrict__ jm, u32 *__restrict__ wlen,
                                                  uint2 *__restrict__ minfo, u32 *__restrict__ visited,
                                                  u32 *__restrict__ total)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    u32 o = 0;
    if (s < ns) {
        const u32 i0 = spl[s];
        u32 mn = i0, mo = 0;
        o = 1;
        if (visited) atomicOr(visited + (i0 >> 5), 1u << (i0 & 31));
        u32 i = prev[i0];
        while (!is_splitter(i, shift)) {
            if (visited) atomicOr(visited + (i >> 5), 1u << (i & 31));
            if (i < mn) { mn = i; mo = o; }
            i = prev[i];
            o++;
        }
        jm[s] = ((u64)sid[i] << 32) | mn;
        wlen[s] = o;
        minfo[s] = make_uint2(mn, mo);
    }
    if (total) {
        o = warp_sum(o);
        if (lane_id() == 0 && o) atomicAdd(total, o);
    }
}

// second walk: srec[s] = (d of the splitter element, cycle length L, cycle offset off);
// element at offset o of the sublist has d = (A + o) mod L and lands at out[n-1-off-d].
__global__ void __launch_bounds__(128) k_inv_walk_place(const u32 *__restrict__ prev, u32 n, SplHash shift,
                                                        const u32 *__restrict__ spl, u32 ns,
                                                        const uint4 *__restrict__ srec,
                                                        const u32 *__restrict__ Ctab, u8 *__restrict__ out)
{
    __shared__ u32 sC[257];
    for (u32 t = threadIdx.x; t < 257; t += blockDim.x) sC[t] = Ctab[t];
    __syncthreads();
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const uint4 r = srec[s];
    const u32 L = r.y, top = n - 1 - r.z;
    u32 d = r.x;
    u32 i = spl[s];
    do {
        const u32 p = prev[i];
        // byte of element i: largest c with C[c] <= p
        u32 c = 0;
#pragma unroll
        for (u32 step = 128; step > 0; step >>= 1)
            if (sC[c + step] <= p) c += step;
        out[top - d] = (u8)c;
        if (++d == L) d = 0;
        i = p;
    } while (!is_splitter(i, shift));
}

// pointer jumping with min: (jmp, mn) <- (jmp[jmp], min(mn, mn[jmp]))
__global__ void __launch_bounds__(256) k_inv_min_jump(const u64 *__restrict__ in, u64 *__restrict__ out, u32 ns)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const u64 a = in[s];
    const u64 b = in[(u32)(a >> 32)];
    out[s] = (b & 0xffffffff00000000ull) | (u64)min((u32)a, (u32)b);
}

// suffix sums over the reduced list, cut in front of the sublist that holds the cycle minimum.
// pv[s] = ptr << 32 | val
__global__ void __launch_bounds__(256) k_inv_sum_init(const u64 *__restrict__ jm0, const u64 *__restrict__ jmR,
                                                      const u32 *__restrict__ wlen, const uint2 *__restrict__ minfo,
                                                      u32 ns, u64 *__restrict__ pv)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const u32 nxt = (u32)(jm0[s] >> 32);
    const u32 cm = (u32)jmR[s];
    const bool next_is_origin = minfo[nxt].x == cm;
    pv[s] = ((u64)(next_is_origin ? NONE32 : nxt) << 32) | wlen[s];
}
__global__ void __launch_bounds__(256) k_inv_sum_jump(const u64 *__restrict__ in, u64 *__restrict__ out, u32 ns)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    u64 a = in[s];
    const u32 p = (u32)(a >> 32);
    if (p != NONE32) {
        const u64 b = in[p];
        a = (b & 0xffffffff00000000ull) | (u64)((u32)a + (u32)b);
    }
    out[s] = a;
}

// the sublist holding the cycle minimum publishes the cycle: length at the minimum's index
// (for the offsets scan) and (length, offset of the minimum inside that sublist)
__global__ void __launch_bounds__(256) k_inv_origin_publish(const u64 *__restrict__ jmR, const u64 *__restrict__ pvR,
                                                            const uint2 *__restrict__ minfo, u32 ns,
                                                            u32 *__restrict__ len_at_min, uint2 *__restrict__ cyc)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const u32 cm = (u32)jmR[s];
    const uint2 mi = minfo[s];
    if (mi.x == cm) {
        const u32 L = (u32)pvR[s];
        len_at_min[cm] = L;
        cyc[cm] = make_uint2(L, mi.y);
    }
}

// fallback: elements no walk reached belong to cycles without a splitter: walk the whole cycle.
// One thread per word of the visited bitmap.  urec[i] = (smallest index, d(i)), written (and
// later read) only for unreached elements.
// counters[0] += elements handled; counters[1] += steps (in units of 1024); *abort is raised once the
// steps exceed budget_k x 1024: cycles of length L cost L steps per member here, L^2 per cycle.
__global__ void __launch_bounds__(256) k_inv_self_walk(const u32 *__restrict__ prev, u32 n,
                                                       const u32 *__restrict__ visited, uint2 *__restrict__ urec,
                                                       u32 *__restrict__ len_at_min, u32 *__restrict__ counters,
                                                       u32 budget_k, u32 *__restrict__ abort)
{
    const u32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if ((u64)w * 32 >= n) return;
    u32 todo = ~visited[w];
    if ((u64)w * 32 + 32 > n) todo &= (1u << (n - w * 32)) - 1;
    u32 spent = 0;
    while (todo) {
        const u32 i = w * 32 + (__ffs(todo) - 1);
        todo &= todo - 1;
        u32 j = prev[i], steps = 1, mn = i, mstep = 0;
        while (j != i) {
            if (j < mn) { mn = j; mstep = steps; }
            j = prev[j];
            steps++;
            if ((++spent & 1023u) == 0) {
                if (atomicAdd(counters + 1, 1u) >= budget_k) atomicExch(abort, 1u);
                if (*(volatile u32 *)abort) return;
            }
        }
        urec[i] = make_uint2(mn, (mstep == 0) ? 0 : steps - mstep);
        if (mn == i) len_at_min[i] = steps;
        atomicAdd(counters, 1u);
    }
}

// ---- finding the elements no walk reached, from the per-128 counts --------------------------------
// deflist[0..*ndef) = blocks of 128 elements whose count is short (capacity cap; *ndef keeps counting)
__global__ void __launch_bounds__(256) k_inv_find_deficient(const u32 *__restrict__ vcnt, u32 n, u32 *__restrict__ deflist,
                                                            u32 cap, u32 *__restrict__ ndef)
{
    const u32 b = blockIdx.x * blockDim.x + threadIdx.x;  // block of 128 elements
    if ((u64)b * 128 >= n) return;
    const u32 expect = min(128u, n - b * 128);
    const u32 c = (vcnt[b >> 2] >> (8 * (b & 3))) & 255u;
    if (c != expect) {
        const u32 at = atomicAdd(ndef, 1u);
        if (at < cap) deflist[at] = b;
    }
}
// one thread per element of a deficient block: an element that some walk reached meets a splitter
// when it follows prev (the end of its sublist); one that meets itself first lies on a cycle without
// splitters and gets its bit in `visited` cleared (the bitmap starts all ones).  Same step budget.
__global__ void __launch_bounds__(128) k_inv_verify_candidates(const u32 *__restrict__ prev, u32 n, SplHash h,
                                                               const u32 *__restrict__ deflist, u32 ndef,
                                                               u32 *__restrict__ visited, u32 *__restrict__ counters,
                                                               u32 budget_k, u32 *__restrict__ abort)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if ((t >> 7) >= ndef) return;
    const u32 i = deflist[t >> 7] * 128 + (t & 127);
    if (i >= n) return;
    u32 j = i, spent = 0;
    for (;;) {
        if (is_splitter(j, h)) return;  // reached
        j = prev[j];
        if (j == i) break;              // a cycle without splitters
        if ((++spent & 1023u) == 0) {
            if (atomicAdd(counters + 1, 1u) >= budget_k) atomicExch(abort, 1u);
            if (*(volatile u32 *)abort) return;
        }
    }
    atomicAnd(visited + (i >> 5), ~(1u << (i & 31)));
}
// many deficient blocks (inputs with very many short cycles): mark exactly, one bit per element
__global__ void __launch_bounds__(128) k_inv_walk_mark(const u32 *__restrict__ prev, SplHash h,
                                                       const u32 *__restrict__ spl, u32 ns, u32 *__restrict__ visited)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    u32 i = spl[s];
    do {
        atomicOr(visited + (i >> 5), 1u << (i & 31));
        i = prev[i];
    } while (!is_splitter(i, h));
}

__global__ void __launch_bounds__(256) k_inv_place_unreached(const u8 *__restrict__ B, u32 n,
                                                             const u32 *__restrict__ visited,
                                                             const uint2 *__restrict__ urec,
                                                             const u32 *__restrict__ off, u8 *__restrict__ out)
{
    const u32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if ((u64)w * 32 >= n) return;
    u32 todo = ~visited[w];
    if ((u64)w * 32 + 32 > n) todo &= (1u << (n - w * 32)) - 1;
    while (todo) {
        const u32 i = w * 32 + (__ffs(todo) - 1);
        todo &= todo - 1;
        const uint2 r = urec[i];
        out[n - 1 - off[r.x] - r.y] = B[i];
    }
}

// per sublist: (A, L, off) with d(i) = (A + offset(i)) mod L
__global__ void __launch_bounds__(256) k_inv_spl_record(const u64 *__restrict__ jmR, const u64 *__restrict__ pvR,
                                                        const uint2 *__restrict__ cyc, const u32 *__restrict__ off,
                                                        u32 ns, uint4 *__restrict__ srec)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    const u32 cm = (u32)jmR[s];
    const uint2 c = cyc[cm];  // (L, offset of the minimum in the origin sublist)
    const u32 L = c.x;
    u32 A = (L - (u32)pvR[s]) + (L - c.y);  // P(s) + L - o(m), both terms in (0, L]
    while (A >= L) A -= L;
    srec[s] = make_uint4(A, L, off[cm], 0u);
}


// ---- staged single walk (default path) ----------------------------------------------------------
// The two-walk form above chases every element twice (ncu, round 1: 89 B of DRAM traffic per
// 4-byte step, 22x the algorithmic bytes, lanes idle 3/4 of the time because a warp runs until its
// longest sublist ends).  Here the first walk already recovers the bytes: the byte of element i is
// the c with C[c] <= prev[i] < C[c+1], and the walker of sublist s parks it at stage[s][offset]
// (slot bytes per sublist, written as full 32-byte sectors).  After the list ranking a
// streaming kernel copies every slot to its place in the output (a sublist is at most two
// descending runs there); only the 1.8 % of the elements beyond offset slot of their sublist
// are chased a second time, from the element the first walk parked in cont[s].
// Lanes are refilled: warp w owns the sublists [w Q, (w+1) Q) and a lane whose sublist ended takes
// the next one of the warp's range (ballot + popc, no atomics), so the warp stays full until its
// range runs dry.
#define INV_SLOT_MAX 512  // staged bytes per sublist (`slot`): 4 x the mean sublist length, a multiple of 32, at most this

static __device__ __forceinline__ u32 byte_of_rank(const u32 *sC, u32 p)
{
    u32 c = 0;  // largest c with C[c] <= p
#pragma unroll
    for (u32 step = 128; step > 0; step >>= 1)
        if (sC[c + step] <= p) c += step;
    return c;
}

__global__ void __launch_bounds__(256) k_inv_walk_stage(const u32 *__restrict__ prev, SplHash shift,
                                                        const u32 *__restrict__ spl, u32 ns, u32 Q,
                                                        const u32 *__restrict__ Ctab, u32 *__restrict__ nxt,
                                                        u32 *__restrict__ wlen, uint2 *__restrict__ minfo,
                                                        u8 *__restrict__ stage, u32 slot, u32 *__restrict__ cont,
                                                        u32 *__restrict__ visited, u32 *__restrict__ vcnt,
                                                        u32 *__restrict__ total)
{
    __shared__ u32 sC[257];
    for (u32 t = threadIdx.x; t < 257; t += blockDim.x) sC[t] = Ctab[t];
    __syncthreads();
    const u32 lane = lane_id(), lt = lanemask_lt();
    const u64 lo64 = ((u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * Q;
    if (lo64 >= ns) return;  // warp-uniform
    u32 next = (u32)lo64;
    const u32 hi = (u32)min((u64)ns, lo64 + Q);
    u32 s = NONE32, i = 0, o = 0, mn = 0, mo = 0, sum = 0;
    u64 a0 = 0, a1 = 0, a2 = 0, a3 = 0;  // 32 staged bytes
    for (;;) {
        const u32 idle = __ballot_sync(FULL_MASK, s == NONE32);
        if (idle) {
            if (s == NONE32) {
                const u32 cand = next + __popc(idle & lt);
                if (cand < hi) {
                    s = cand;
                    i = __ldg(spl + s);
                    o = 0; mn = i; mo = 0;
                    a0 = a1 = a2 = a3 = 0;
                }
            }
            next = min(hi, next + (u32)__popc(idle));  // saturates: a long walk next to idle lanes must not wrap the cursor
            if (__all_sync(FULL_MASK, s == NONE32)) break;
        }
        if (s != NONE32) {
            const u32 p = ldg_stream_u32(prev + i);  // evict-first: keeps the reach marks resident in L2 (default policy: C5 block inverse 13.5 -> 14.7 ms)
            // who was reached?  Either one bit per element (n / 8 bytes: beyond ~512 MiB of input the
            // bitmap falls out of L2 and every mark becomes a DRAM read-modify-write) or one 8-bit
            // count per 128 elements (n / 128 bytes, L2-resident at every size; k_inv_find_deficient)
            if (vcnt) atomicAdd(vcnt + (i >> 9), 1u << (8 * ((i >> 7) & 3)));
            else if (visited) atomicOr(visited + (i >> 5), 1u << (i & 31));
            if (o < slot) {
                const u32 c = byte_of_rank(sC, p);
                const u32 b = o & 31, q = b >> 3;
                const u64 v = (u64)c << (8 * (b & 7));
                a0 |= (q == 0) ? v : 0ull;
                a1 |= (q == 1) ? v : 0ull;
                a2 |= (q == 2) ? v : 0ull;
                a3 |= (q == 3) ? v : 0ull;
                if (b == 31) {
                    uint4 *dst = (uint4 *)(stage + (u64)s * slot + (o & ~31u));
                    dst[0] = make_uint4((u32)a0, (u32)(a0 >> 32), (u32)a1, (u32)(a1 >> 32));
                    dst[1] = make_uint4((u32)a2, (u32)(a2 >> 32), (u32)a3, (u32)(a3 >> 32));
                    a0 = a1 = a2 = a3 = 0;
                }
            } else if (o == slot) {
                cont[s] = i;  // the element at offset slot: where k_inv_walk_tail resumes
            }
            o++;
            if (is_splitter(p, shift)) {
                if (o <= slot && (o & 31)) {
                    uint4 *dst = (uint4 *)(stage + (u64)s * slot + ((o - 1) & ~31u));
                    dst[0] = make_uint4((u32)a0, (u32)(a0 >> 32), (u32)a1, (u32)(a1 >> 32));
                    dst[1] = make_uint4((u32)a2, (u32)(a2 >> 32), (u32)a3, (u32)(a3 >> 32));
                }
                nxt[s] = p;  // the splitter that starts the next sublist (resolved to its id afterwards)
                wlen[s] = o;
                minfo[s] = make_uint2(mn, mo);
                sum += o;
                s = NONE32;
            } else {
                i = p;
                if (p < mn) { mn = p; mo = o; }
            }
        }
    }
    sum = warp_sum(sum);
    if (lane == 0 && sum) atomicAdd(total, sum);
}

// jm[s] = id of the next sublist << 32 | smallest index of sublist s
__global__ void __launch_bounds__(256) k_inv_resolve_next(const u32 *__restrict__ nxt, const uint2 *__restrict__ minfo,
                                                          const u32 *__restrict__ blkoff, SplHash shift, u32 ns,
                                                          u64 *__restrict__ jm)
{
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns) return;
    jm[s] = ((u64)sid_of(blkoff, nxt[s], shift) << 32) | (u64)minfo[s].x;
}

// one warp per sublist: its staged bytes go to out[top - d], d = (A + offset) mod L
__global__ void __launch_bounds__(256) k_inv_place_copy(const u8 *__restrict__ stage, const u32 *__restrict__ wlen,
                                                        const uint4 *__restrict__ srec, u32 ns, u32 n, u32 slot,
                                                        u8 *__restrict__ out)
{
    const u64 s = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= ns) return;
    const u32 len = min(__ldg(wlen + s), slot);
    const uint4 r = __ldg(srec + s);
    const u32 L = r.y, top = n - 1 - r.z;
    const u8 *src = stage + s * slot;
    for (u32 o = lane_id(); o < len; o += 32) {
        u32 d = r.x + o;  // A < L and o < len <= L
        if (d >= L) d -= L;
        out[top - d] = src[o];
    }
}

// ---- classic inverse BWT: out[n-1-j] = B[LF^j(primary)] ------------------------------------------
// The BWTS layout S (above) holds the cycle c of `primary` as S[n-1-off(c)-d(i)] = B[i], and d grows by
// one per prev-step (mod L), so the classic output is that window of L bytes rotated to start at
// d(primary) and repeated (once when the input came from the forward: then L = n):
//     out[n-1-j] = S[n-1-off - ((d(primary) + j) mod L)]
// One thread finds (d(primary), L, off): it walks prev from primary to the first splitter p, t steps,
// where d(p) = A of the sublist p starts; a cycle without splitters brings the walk back to primary
// (t = L), and the walk's own minimum gives d as in k_inv_self_walk.  loc = (d, L, off).
// DIV (primary = 0, prev = prev_s of k_inv_lf_rank<true>): the element whose prev_s is 0 is the last of
// the cycle of 0 (d = L - 1, and off = 0: no cycle has a smaller index), so its byte sits at
// S[n - off - L]; that byte is written here from *cstar, before k_bwt_rotate reads the window.
template <bool DIV = false>
__global__ void k_bwt_locate(const u32 *__restrict__ prev, SplHash h, u32 primary, const u32 *__restrict__ sid,
                             const u32 *__restrict__ blkoff, const uint4 *__restrict__ srec,
                             const u32 *__restrict__ off, u32 *__restrict__ loc, u8 *__restrict__ S = nullptr,
                             u32 n = 0, const u32 *__restrict__ cstar = nullptr)
{
    u32 j = primary, t = 0, mn = primary, mstep = 0;
    while (!is_splitter(j, h)) {
        j = prev[j];
        t++;
        if (j == primary) break;
        if (j < mn) { mn = j; mstep = t; }
    }
    if (is_splitter(j, h)) {
        const uint4 r = srec[sid ? sid[j] : sid_of(blkoff, j, h)];  // (A, L, off); t < L
        loc[0] = r.x >= t ? r.x - t : r.x + r.y - t;
        loc[1] = r.y;
        loc[2] = r.z;
    } else {
        loc[0] = mstep == 0 ? 0 : t - mstep;
        loc[1] = t;
        loc[2] = off[mn];
    }
    if (DIV) S[n - loc[2] - loc[1]] = (u8)*cstar;
}

// 16 output bytes per thread: the source runs forward through the window [n - off - L, n - off) and wraps
__global__ void __launch_bounds__(256) k_bwt_rotate(const u8 *__restrict__ S, u32 n, const u32 *__restrict__ loc,
                                                    u8 *__restrict__ out)
{
    const u64 q0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 16;
    if (q0 >= n) return;
    const u32 d = __ldg(loc), L = __ldg(loc + 1), base = n - __ldg(loc + 2) - L;
    // out[q] = S[base + g(q)], g(q) = L-1 - ((d + n-1-q) mod L), and g(q+1) = g(q) + 1 mod L
    u32 g = L - 1 - (u32)(((u64)d + (n - 1 - (u32)q0)) % L);
    u8 v[16];
#pragma unroll
    for (int e = 0; e < 16; e++) {
        v[e] = (q0 + e < n) ? S[base + g] : 0;
        if (++g == L) g = 0;
    }
    u8 *dst = out + q0;
    if (q0 + 16 <= n && ((uintptr_t)dst & 15) == 0) {
        uint4 w;
        memcpy(&w, v, 16);
        *(uint4 *)dst = w;
    } else {
        for (int e = 0; e < 16 && q0 + e < n; e++) dst[e] = v[e];
    }
}

// the elements beyond offset slot of their sublist: a second walk from cont[s]
__global__ void __launch_bounds__(128) k_inv_walk_tail(const u32 *__restrict__ prev, u32 n, SplHash shift,
                                                       const u32 *__restrict__ wlen, const u32 *__restrict__ cont,
                                                       u32 ns, u32 slot, const uint4 *__restrict__ srec,
                                                       const u32 *__restrict__ Ctab, u8 *__restrict__ out)
{
    __shared__ u32 sC[257];
    for (u32 t = threadIdx.x; t < 257; t += blockDim.x) sC[t] = Ctab[t];
    __syncthreads();
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= ns || wlen[s] <= slot) return;
    const uint4 r = srec[s];
    const u32 L = r.y, top = n - 1 - r.z;
    u32 d = r.x + slot;  // < 2 L
    if (d >= L) d -= L;
    u32 i = cont[s];
    do {
        const u32 p = ldg_stream_u32(prev + i);  // evict-first: keeps the reach marks resident in L2 (default policy: C5 block inverse 13.5 -> 14.7 ms)
        out[top - d] = (u8)byte_of_rank(sC, p);
        if (++d == L) d = 0;
        i = p;
    } while (!is_splitter(i, shift));
}

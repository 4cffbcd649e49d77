/*
 * bwts_b200.h -- C ABI of libbwts_b200.so: the bijective Burrows-Wheeler transform
 * (BWTS, Gil & Scott) and its inverse as hand-written CUDA for NVIDIA B200 (sm_100a).
 *
 * The reference (NealB/Bijective-BWT) has no library API: its hot paths are the bodies
 * of three `main`s working on file-scope globals.  Each entry point below replaces one
 * such seam; a reference-side caller keeps `map_in(...)` before it and `fwrite(...)`
 * after it (see INTEGRATION.md).
 *
 *   bwts_b200_forward   replaces  mk_bwts_sa.c:47-52      (malloc sa; divsufsort; make_bwts_sa)
 *                       and       mk_bwts_sa_new.c:50-55  (same, refactored)
 *   bwts_b200_inverse   replaces  unbwts.c:31-86          (counts, scan, LF map, cycle walk)
 *   bwts_b200_*_blocks  additive: independent fixed-size blocks dealt over several GPUs
 *                       (the reference transforms the whole file as one block).
 *   bwts_b200_bwt_*     additive: the classic Burrows-Wheeler transform with a primary index
 *                       and its inverse, on the same kernels (see the section below).
 *   bwts_b200_divbwt*, bwts_b200_inverse_bw_transform
 *                       additive: libdivsufsort's end-of-text BWT (divbwt / inverse_bw_transform),
 *                       on the same kernels (see the section below).
 *   bwts_b200_sa_*, bwts_b200_sa_lcp
 *                       additive: the suffix array and the LCP array on the context, device and
 *                       one-call entry points (see the section below).
 *   bwts_b200_fm_*      additive: an FM-index over the divbwt output, counting and locating many
 *                       patterns on the GPU (see the section below).
 *   bwts_b200_lpf_*, bwts_b200_lz77_*
 *                       additive: the longest-previous-factor array and the greedy LZ77 parse,
 *                       from the suffix array and LCP array on the GPU (see the last section).
 *
 * Byte layout is the reference's: `len` raw input bytes in, exactly `len` raw bytes
 * out, no header, no primary index, no terminator (mk_bwts_sa.c:60, unbwts.c:173).
 * Bytes order as unsigned char (mk_bwts_sa.c:24,86).
 *
 * Ownership: the caller owns `in` and `out` (never aliased); the library owns all
 * device memory.  Every function returns 0 on success or a negative BWTS_B200_E*
 * code; nothing prints, nothing calls exit() -- the host tools turn a failure into
 * the reference's "message to stderr, exit(1)" convention.  There is no CPU
 * fallback: without a CUDA device every transform fails with BWTS_B200_ENODEV.
 *
 * Limits: 1 <= len < 2^31 per block, the reference's own range (`int` / `saidx_t`,
 * mk_bwts_sa.c:26-27, unbwts.c:12-13).  The device workspace is 71 bytes per input byte (+ 64 MiB,
 * + 2 per byte for the host-buffer calls): 2 GiB blocks need ~157 GB of the B200's 192 GB.
 */
#ifndef BWTS_B200_H
#define BWTS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define BWTS_B200_OK         0
#define BWTS_B200_EINVAL    -1   /* NULL pointer, len <= 0, bad device / block size      */
#define BWTS_B200_ETOOBIG   -2   /* len > BWTS_B200_MAX_LEN                               */
#define BWTS_B200_ENODEV    -3   /* no usable CUDA device (no CPU fallback exists)        */
#define BWTS_B200_ENOMEM    -4   /* device or pinned-host allocation failed               */
#define BWTS_B200_ECUDA     -5   /* a CUDA call or kernel failed; see bwts_b200_last_cuda_error */
#define BWTS_B200_EINTERNAL -6   /* invariant violated (a bug)                            */

#define BWTS_B200_MAX_LEN ((1L << 31) - 1)

typedef struct bwts_b200_ctx bwts_b200_ctx;

/* ---- one-call entry points (host buffers) -------------------------------------- */

/* Forward BWTS of in[0..len) into out[0..len) on CUDA device `device`.
 * Replaces: sa = malloc(...); divsufsort(T, sa, len); bwts = make_bwts_sa();
 * (/root/reference/mk_bwts_sa.c:47-52, mk_bwts_sa_new.c:50-55).                     */
int bwts_b200_forward(const unsigned char *in, long len, unsigned char *out, int device);

/* Inverse BWTS.  Replaces /root/reference/unbwts.c:31-86.                            */
int bwts_b200_inverse(const unsigned char *in, long len, unsigned char *out, int device);

/* Independent blocks of `block_len` bytes (last one shorter), block j = bytes
 * [j*block_len, min((j+1)*block_len, len)); output block j = transform of input block
 * j at the same offsets.  Blocks are dealt round-robin over devices[0..ndev); per device
 * a three-stage pipeline (pinned staging + H2D of block b+1 | transform of block b | D2H
 * + un-staging of block b-1, each on its own stream and host thread) overlaps the copies
 * with the kernels; no inter-GPU traffic.  block_len <= 0 or
 * >= len means "whole input is one block" (= the reference's behaviour).
 * devices == NULL means devices 0..ndev-1.                                           */
int bwts_b200_forward_blocks(const unsigned char *in, long len, long block_len,
                             unsigned char *out, const int *devices, int ndev);
int bwts_b200_inverse_blocks(const unsigned char *in, long len, long block_len,
                             unsigned char *out, const int *devices, int ndev);

/* ---- context API (reusable workspace; one context per device per host thread) ---- */

int  bwts_b200_device_count(void);                 /* >= 0, or 0 when no driver/device */
bwts_b200_ctx *bwts_b200_create(int device);       /* NULL on failure                   */
void bwts_b200_destroy(bwts_b200_ctx *ctx);
int  bwts_b200_reserve(bwts_b200_ctx *ctx, long max_len);   /* pre-size the workspace   */

/* host buffers: pinned staging + H2D, transform, D2H; blocks until `out` is complete  */
int bwts_b200_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out);
int bwts_b200_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out);

/* device-resident buffers (d_in, d_out: device pointers on ctx's device, not aliased; any
 * alignment -- an input that is not 16-byte aligned costs one device-to-device copy).
 * Work is issued on `stream` (a cudaStream_t passed as void*; NULL = the context's own
 * stream).  The call returns after the result is complete in d_out (the driver loop
 * reads a few counters back per doubling round).                                      */
int bwts_b200_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, void *stream);
int bwts_b200_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, void *stream);

/* ---- classic Burrows-Wheeler transform with a primary index ------------------------ */
/* The index-carrying counterpart of BWTS (Gil & Scott), as in bzip2-style block sorting.
 * Bytes compare as unsigned char; n = len, 1 <= len <= BWTS_B200_MAX_LEN.
 *
 * Forward: the rows are the n cyclic rotations of T, sorted; rows that tie (only when T = u^k)
 * are ordered by start position.  out[r] = T[(s_r - 1) mod n], s_r the start of row r, and
 * *primary = the row of rotation 0 = the number of rotations strictly smaller than T.
 * So a Lyndon word T gives the BWTS output and *primary == 0, every rotation of T gives the
 * same out, and out[*primary] == T[n-1].
 *
 * Inverse: out[n-1-j] = in[LF^j(primary)] for j = 0..n-1, LF the stable LF map
 * (C[c] + occ(c, i), unbwts.c:50-52).  For a pair made by the forward this is T again, and
 * for a row r other than the primary it is rotation s_r of T.  Any other pair still has a
 * defined result (the LF cycle through `primary`, written repeatedly): the inverse fails on
 * bad arguments only, never because of the content.
 *
 * Arguments: a NULL `primary`, or a `primary` outside [0, len), is BWTS_B200_EINVAL; the
 * *_blocks inverse checks every block's index against that block's length before any work.
 * Block layout and devices are those of the BWTS *_blocks calls, with one primary index per
 * block.  Statistics: a forward reports factors = 1, longest_factor = n, lyndon_fallback = 0;
 * an inverse reports its cycles in `factors` and books the final rotation of the cycle layout
 * into the output (one n-byte copy) to phase 4, "Place bytes".  The workspace is that of the
 * BWTS call of the same length.                                                         */
int bwts_b200_bwt_forward(const unsigned char *in, long len, unsigned char *out, long *primary, int device);
int bwts_b200_bwt_inverse(const unsigned char *in, long len, long primary, unsigned char *out, int device);
int bwts_b200_bwt_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out,
                               long *primary);
int bwts_b200_bwt_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, long primary,
                               unsigned char *out);
int bwts_b200_bwt_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, long *primary,
                                 void *stream);
int bwts_b200_bwt_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, long primary, void *d_out,
                                 void *stream);
int bwts_b200_bwt_forward_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                 long *primary /* one per block */, const int *devices, int ndev);
int bwts_b200_bwt_inverse_blocks(const unsigned char *in, long len, long block_len, const long *primary,
                                 unsigned char *out, const int *devices, int ndev);

/* ---- introspection --------------------------------------------------------------- */

#define BWTS_B200_NCLASS 16
#define BWTS_B200_NPHASE 8
typedef struct {
    long   len;                 /* length of the last transform                         */
    int    direction;           /* 0 forward, 1 inverse                                 */
    long   factors;             /* forward: Lyndon factors; inverse: cycles             */
    long   longest_factor;      /* forward only                                         */
    int    alphabet_bits;       /* forward: bits per packed symbol                      */
    int    initial_depth;       /* forward: symbols in the initial key (k0)             */
    int    rounds;              /* forward: doubling rounds after the initial sort      */
    int    radix_passes;        /* forward: onesweep passes launched                    */
    int    local_rounds;        /* forward: rounds served by the warp-local sort        */
    int    cta_rounds;          /* forward: rounds whose large-group set was sorted CTA-locally */
    long   live_sum;            /* forward: sum over rounds of live elements            */
    long   splitters;           /* inverse: sublists                                    */
    long   unreached;           /* inverse: elements ranked by the self-walk fallback   */
    long   launches;            /* kernels launched by the last transform               */
    double total_ms;            /* device time of the last transform (CUDA events)      */
    /* per kernel class: launches, summed CUDA-event milliseconds, summed algorithmic
     * bytes (DESIGN.md section 4 states the per-element figures)                       */
    long   class_launches[BWTS_B200_NCLASS];
    double class_ms[BWTS_B200_NCLASS];
    double class_bytes[BWTS_B200_NCLASS];
    /* host-buffer entry points only: CUDA-event times of the two copies around the transform */
    double h2d_ms;
    double d2h_ms;
    int    lyndon_fallback;     /* forward: 1 if the Lyndon boundaries came from the suffix-sort fallback */
    /* device time per phase, the counterpart of the reference's MARK_TIME marks
     * (/root/reference/mk_bwts_sa.c:13-22,50,124,168,190); names: bwts_b200_phase_name       */
    double phase_ms[BWTS_B200_NPHASE];
    long   arena_bytes;         /* device workspace held by the context after this transform */
    long   first_live;          /* forward: rotations still tied after the initial sort      */
    int    tuple_rounds;        /* forward: rounds in which the text-ordered tuple set ran   */
    long   tuple_live_sum;      /* forward: sum over those rounds of its members             */
    int    inverse_attempts;    /* inverse: 1 + restarts with another splitter hash (fallback over budget) */
    int    binned_rounds;       /* forward: re-ranks whose ranks went out through the binned scatter */
} bwts_b200_stats;

int bwts_b200_get_stats(const bwts_b200_ctx *ctx, bwts_b200_stats *out);
const char *bwts_b200_class_name(int cls);          /* NULL when cls is out of range   */
/* forward (direction 0): "Suffix sort", "Compute ISA", "Fix sort order", "Generate BWTS" -- the
 * reference's own labels, in its order; inverse (direction 1): "Count bytes", "LF map",
 * "Walk sublists", "Rank sublists", "Place bytes".  NULL past the last phase.           */
const char *bwts_b200_phase_name(int direction, int phase);
int bwts_b200_set_profile(bwts_b200_ctx *ctx, int on);   /* per-launch events (default on) */

const char *bwts_b200_strerror(int code);
int bwts_b200_last_cuda_error(const bwts_b200_ctx *ctx);  /* cudaError_t of the last failure */
const char *bwts_b200_version(void);

/* Test hooks: override tuning constants so that small inputs exercise the multi-tile /
 * multi-chunk paths.  key: 0 = Lyndon chunk bytes (>= 1), 1 = inverse splitter shift
 * (density 2^-(32-shift), 20..31), 2 = onesweep tile shape (0..4), 3 = disable the
 * warp-local sort path (1), 4 = force the suffix-sort fallback for the Lyndon boundaries (1),
 * 5 = no copy/compute overlap between the blocks of one device (1), 6 = cap on the bits of
 * the initial packed key (8..64), 7 = binned rank scatter of the re-ranks (1 = never, 2 = the first
 * re-rank of inputs of any size, 3 = the first re-rank only, 4 = every re-rank of both rank-ordered sets; default:
 * the first re-rank of inputs of 4 Mi bytes and more, later ones from 128 Mi bytes on when a third of the set's
 * ranks moved in the round before), 8 = never sort the large-group set
 * CTA-locally (1), 9 = emit through rank windows (1), binned by rank region as one packed word per
 * element (2; default from 512 Mi bytes) or as (rank, byte) pairs in two streams (3), 10 = cudaLimitMaxL2FetchGranularity (32 / 64 / 128; measured: no
 * effect), 12 = inverse through two read-only walks (1) instead of the staged single walk, 13 =
 * sublists per warp of the staged walk, 14 = largest group the text-ordered tuple set takes (1 =
 * set switched off, 2..32; default 8), 15 = inverse marks reached elements with one bit each (1) or one
 * count per 128 (2; default: counts above 256 MiB), 16 = step budget of the inverse's fallback walks per attempt
 * (default 32 n), 17 = Lyndon chunk-minimum scan (1 = Hillis-Steele levels, 2 = CTA-wide levels; default:
 * chosen by the match lengths of the first level), 18 = CTA-local sort as the bitonic network of
 * round 1 (1) instead of the radix sort in shared memory, 20 = tuple set with one thread per group and
 * groups of up to 32 (1; measured slower than one thread per member), 21 = digit histograms of the initial sort by a
 * sweep over the keys (1) instead of the window histogram taken while the keys are built, 22 = initial keys of whole
 * symbols only (1; default: spare key bits hold the top bits of the next symbol), 23 = MiB of output per emit window
 * (16..1024; default 64: the scatter target of one sweep stays in L2), 24 = LCP array: every irreducible pair
 * through the warp tier (1) or the multi-CTA tier (2) instead of by its length, 25 = LPF array and LZ77 parse: log2 of
 * the tile and chunk width (5..12; default 12), so that small inputs take the cross-tile and multi-level paths.
 * value 0 = default. */
int bwts_b200_tune(int key, long value);

/* ---- "next" row (SURVEY.md 8f.2): suffix array behind libdivsufsort's own seam ----- */
/* Same contract as divsufsort(T, SA, n) (/root/reference/mk_bwts_sa.c:48): SA[0..n) =
 * start offsets of the suffixes of T in ascending order; returns 0 or a negative code. */
int bwts_b200_divsufsort(const unsigned char *T, int *SA, int n, int device);

/* ---- libdivsufsort's BWT: divbwt and inverse_bw_transform ---------------------------- */
/* The end-of-text ("sentinel") BWT of libdivsufsort, the form FM-index and DNA tools read.
 * Bytes compare as unsigned char; n = len.  SA is the suffix array of T with the end of text
 * smaller than every byte (the order of the suffixes of T$, bwts_b200_divsufsort).
 *
 * Forward (divbwt): B[r] = T[SA[r] - 1] for SA[r] > 0, r0 the row with SA[r0] == 0,
 *     U = T[n-1] . B[0..r0) . B[r0+1..n),   primary = r0 + 1, in [1, n].
 * That is the BWT of T$ with the $ removed, and primary is where the $ stood.  Examples:
 * banana -> (annbaa, 4), abracadabra -> (ardrcaaaabb, 3), mississippi -> (ipssmpissii, 5),
 * aaaa -> (aaaa, 4), a -> (a, 1).
 *
 * Inverse (inverse_bw_transform): prev the stable LF map over U (C[c] + occ(c, i)), p = 1 + prev[u],
 *     prev_s[u] = (p == primary) ? 0 : p - (p > primary),   out[n-1-j] = U[prev_s^j(0)], j = 0..n-1.
 * prev_s is a permutation of [0, n) for every U and every primary in [1, n], so every pair has a
 * defined result (the cycle through 0, written repeatedly); for a pair made by the forward it is
 * one n-cycle and the result is T.  The inverse fails on bad arguments only.  (libdivsufsort's
 * own inverse is defined on the pairs its forward makes; there the two agree.)
 *
 * The one-call functions keep libdivsufsort's signatures and argument rules: a NULL T or U,
 * n < 0, idx < 0, idx > n, or idx == 0 with n > 0 is BWTS_B200_EINVAL; n == 0 returns 0;
 * U may be T; A (libdivsufsort's temporary array) may be NULL and is never touched.
 * bwts_b200_divbwt returns primary (> 0) or a negative code, bwts_b200_inverse_bw_transform
 * 0 or a negative code.  They run on the per-device context of the other one-call functions.
 *
 * The context and block calls have the shape of the bwts_b200_bwt_* calls: len bytes, never
 * aliased, a NULL `primary` or an inverse `primary` outside [1, len] is BWTS_B200_EINVAL, and the
 * *_blocks inverse checks every block's index against [1, that block's length] before any work.
 * Statistics: a forward reports factors = 1, longest_factor = n, lyndon_fallback = 0; an inverse
 * reports its cycles in `factors` (1 for a pair made by the forward) and books the rotation into
 * the output to phase 4, "Place bytes".  The workspace is that of the BWTS call of the same length. */
int bwts_b200_divbwt(const unsigned char *T, unsigned char *U, int *A, int n, int device);
int bwts_b200_inverse_bw_transform(const unsigned char *T, unsigned char *U, int *A, int n, int idx, int device);
int bwts_b200_divbwt_forward_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, unsigned char *out,
                                  long *primary);
int bwts_b200_divbwt_inverse_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, long primary,
                                  unsigned char *out);
int bwts_b200_divbwt_forward_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_out, long *primary,
                                    void *stream);
int bwts_b200_divbwt_inverse_device(bwts_b200_ctx *ctx, const void *d_in, long len, long primary, void *d_out,
                                    void *stream);
int bwts_b200_divbwt_forward_blocks(const unsigned char *in, long len, long block_len, unsigned char *out,
                                    long *primary /* one per block */, const int *devices, int ndev);
int bwts_b200_divbwt_inverse_blocks(const unsigned char *in, long len, long block_len, const long *primary,
                                    unsigned char *out, const int *devices, int ndev);

/* ---- suffix array and LCP array ------------------------------------------------------ */
/* n = len, 1 <= len <= BWTS_B200_MAX_LEN.  Bytes compare as unsigned char and the end of text is
 * smaller than every byte (the order of bwts_b200_divsufsort).  Both arrays are int32:
 *     SA[0..n)   the start offsets of the suffixes of in, ascending;
 *     LCP[0] = 0, and for r >= 1 LCP[r] = the length of the longest common prefix of the suffixes
 *                starting at SA[r-1] and SA[r] (Kasai's convention).
 * Examples:  banana       SA [5,3,1,0,4,2]              LCP [0,1,3,0,0,2]
 *            mississippi  SA [10,7,4,1,0,9,8,6,3,5,2]   LCP [0,1,1,4,0,0,1,0,2,1,3]
 *            abracadabra  SA [10,7,0,3,5,8,1,4,6,9,2]   LCP [0,1,4,1,1,0,3,0,0,0,2]
 *            aaaa         SA [3,2,1,0]                  LCP [0,1,2,3]
 *            a            SA [0]                        LCP [0]
 * and in general a^n gives SA[r] = n-1-r, LCP[r] = r.
 *
 * The LCP array is computed on the GPU after the suffix sort from the irreducible LCP values
 * (Kärkkäinen, Manzini and Puglisi, CPM 2009; DESIGN.md section 4.8): only the pairs at the BWT's run
 * boundaries are compared, in tiers of one thread, one warp and many CTAs per pair, and the rest
 * follows from one max-scan.
 *
 * Arguments follow the bwts_b200_bwt_* calls: a NULL pointer or len <= 0 is BWTS_B200_EINVAL,
 * len > BWTS_B200_MAX_LEN is BWTS_B200_ETOOBIG, and no two of in, sa and lcp may share a byte
 * (BWTS_B200_EINVAL).  The device calls take device addresses: sa and lcp must be 4-byte
 * aligned (else BWTS_B200_EINVAL), the input may lie at any offset.  bwts_b200_sa_lcp takes the rules of
 * bwts_b200_divsufsort: n == 0 returns 0, n < 0 is BWTS_B200_EINVAL; it runs on the per-device
 * context of the other one-call functions.  Without a device every call returns BWTS_B200_ENODEV.
 *
 * Device memory: the workspace of the BWTS call of the same length (71 bytes per input byte + 64 MiB);
 * the LCP stage takes its scratch from the sort's buffers, which are dead by then.  The host and one-call
 * forms add an I/O region of 5 bytes per input byte (text, SA), 9 with the LCP array: ~80 bytes per
 * byte in all, 172 GB at len = 2^31 - 1.  The device forms add nothing for an input at a 16-byte aligned
 * address (2 bytes per byte otherwise, as the other device calls).
 * Statistics: direction 0, factors = 1, longest_factor = n; the LCP kernels (k_lcp_*) are booked to
 * kernel class "emit" and phase 3, beside k_emit_sa. */
int bwts_b200_sa_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *sa);
int bwts_b200_sa_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_sa, void *stream);
int bwts_b200_sa_lcp_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *sa, int *lcp);
int bwts_b200_sa_lcp_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_sa, void *d_lcp, void *stream);
int bwts_b200_sa_lcp(const unsigned char *T, int *SA, int *LCP, int n, int device);   /* divsufsort-shaped */

/* ---- FM-index: count and locate over libdivsufsort's BWT ----------------------------------- */
/* Bytes compare as unsigned char and the end of text is smaller than every byte (the order of
 * bwts_b200_divsufsort and bwts_b200_sa_*); SA is the suffix array of the text T, n = len,
 * 1 <= len <= BWTS_B200_MAX_LEN.  An index is built once from T and answers batches of patterns.
 *
 * Count: for a pattern P of m >= 0 bytes,
 *     lo = #{ i : T[i..n) < P },   hi = #{ i : T[i..n)[0..m) <= P },   0 <= lo <= hi <= n,
 * with a suffix that is a proper prefix of P smaller than P.  P occurs hi - lo times, at SA[lo..hi); when it
 * does not occur, lo == hi is its insertion point among the sorted suffixes; the empty pattern gives [0, n).
 * (bisect_left / bisect_right over the sorted suffixes.)
 * Locate: for ranges [lo_k, hi_k) with 0 <= lo_k <= hi_k <= n, pos = SA[lo_0..hi_0) . SA[lo_1..hi_1) . ...,
 * in range order and in SA row order inside each range -- no sorting by position.
 *     banana       ana -> (1, 3) [3, 1]     a -> (0, 3) [5, 3, 1]    na -> (4, 6) [4, 2]
 *                  anan -> (2, 3) [1]       banana -> (3, 4) [0]     bananas -> (4, 4) []
 *                  nab -> (5, 5) []         z -> (6, 6) []           \x00 -> (0, 0) []
 *                  (empty) -> (0, 6) [5, 3, 1, 0, 4, 2]
 *     mississippi  ssi -> (9, 11) [5, 2]    issi -> (2, 4) [4, 1]    ppp -> (7, 7) []
 *     aaaa         aa -> (1, 4) [2, 1, 0]   aaaaa -> (4, 4) []
 *
 * Index (DESIGN.md section 4.9): the divbwt output U and its primary as the L column of T$, occurrence
 * checkpoints for the sg distinct bytes of T (u32 per 65536 rows, u16 per 256 rows), and the SA values at
 * the rows whose text position is a multiple of `sample`, found by a bit vector with a directory.  Counting
 * is backward search, one warp per pattern; locating walks LF from each row to a sampled one, at most
 * sample - 1 steps.  `sample` is a power of two in [1, 1024], else BWTS_B200_EINVAL.
 * bwts_b200_fm_bytes, with every term rounded up to a multiple of 256:
 *     n + 4 sg (n/65536 + 1) + 2 sg (n/256 + 1) + 4 ceil(n/32) + 4 (n/256 + 1) + 4 ceil(n/sample) + 1028 + 256
 * (/ is integer division): ~1.17 n + 4n/sample for DNA, ~3.16 n + 4n/sample with all 256 byte values.
 * The build needs the workspace of the SA call of the same length plus an I/O region of ~5 bytes per byte
 * (text and suffix array); it books like bwts_b200_sa_*: direction 0, factors = 1, the k_fm_* build kernels to
 * class "emit" and phase 3.  A query resets the statistics: direction 1, backward search and LF walks
 * (k_fm_count, k_fm_locate) in class "inv_walk", the argument checks and the offsets scan in class
 * "inv_scan", all in phase 2.
 *
 * Patterns: pattern k = pat[off[k] .. off[k+1]); off int64[npat + 1] with off[0] == 0, non-decreasing,
 * off[npat] == pat_len.  range int32[2 npat] = (lo_k, hi_k).  *total (may be NULL) = the sum of hi_k - lo_k.
 * Locate: pos int32[cap]; a sum of hi_k - lo_k above cap is BWTS_B200_EINVAL and nothing is written.
 *
 * Arguments: a NULL ctx or fm, npat < 0, nrange < 0, pat_len < 0, cap < 0, a NULL array the call needs is
 * BWTS_B200_EINVAL; npat == 0 (nrange == 0) returns 0 with *total = 0.  The host forms check the offsets and the
 * ranges on the host; the device forms check the same rules in a validation kernel before any other work and
 * report a violation as BWTS_B200_EINVAL.  No kernel reads outside the buffers it was given, whatever they
 * hold.  Device offsets must be 8-byte aligned, ranges and positions 4-byte aligned; patterns may start at
 * any address.  Without a device every call returns BWTS_B200_ENODEV after the checks that need no index
 * (the ranges against n and the index's device are checked after it).
 * Device and lifetime: the index owns one device allocation on the device of the context that built it and
 * outlives that context; any context on that device may query it (another device is BWTS_B200_EINVAL).
 * Queries only read the index, so host threads with their own contexts may query one index at once. */
typedef struct bwts_b200_fm bwts_b200_fm;   /* device-resident index, owned by the caller until fm_free */

int  bwts_b200_fm_build_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int sample, bwts_b200_fm **fm);
int  bwts_b200_fm_build_device(bwts_b200_ctx *ctx, const void *d_in, long len, int sample, bwts_b200_fm **fm,
                               void *stream);
void bwts_b200_fm_free(bwts_b200_fm *fm);                 /* NULL is a no-op */
long bwts_b200_fm_bytes(const bwts_b200_fm *fm);          /* device bytes the index holds; 0 for NULL */
int bwts_b200_fm_count_host(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const unsigned char *pat, long pat_len,
                            const long *off, long npat, int *range, long *total);
int bwts_b200_fm_count_device(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const void *d_pat, long pat_len,
                              const void *d_off, long npat, void *d_range, long *total, void *stream);
int bwts_b200_fm_locate_host(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const int *range, long nrange,
                             int *pos, long cap, long *total);
int bwts_b200_fm_locate_device(bwts_b200_ctx *ctx, const bwts_b200_fm *fm, const void *d_range, long nrange,
                               void *d_pos, long cap, long *total, void *stream);

/* ---- longest-previous-factor array and greedy LZ77 parse ------------------------------------ */
/* Bytes compare as unsigned char and the end of text is smaller than every byte (the order of
 * bwts_b200_sa_*); n = len, 1 <= len <= BWTS_B200_MAX_LEN; lcp(i, j) is the length of the longest
 * common prefix of T[i..n) and T[j..n).
 *     LPF[i]  = max over j < i of lcp(i, j): 0 for i = 0 and for a byte that has not occurred before.
 *     PREV[i] = -1 when LPF[i] == 0.  Otherwise, among the j < i with lcp(i, j) == LPF[i]: if some of
 *               their suffixes are smaller than T[i..n), the one whose suffix is the largest of those;
 *               else the one whose suffix is the smallest.  (The previous smaller value in suffix array
 *               order, else the next smaller value, the previous one on a tie.)
 *     LZ77    the greedy parse, a source may overlap its factor: p_0 = 0; factor k at p_k is
 *               (PREV[p_k], LPF[p_k]) when LPF[p_k] >= 1, else the literal (T[p_k], 0);
 *               p_(k+1) = p_k + max(1, LPF[p_k]); z factors, int32 pairs (src_or_byte, len).
 * Examples:  banana       LPF [0,0,0,3,2,1]  PREV [-1,-1,-1,1,2,3]  LZ77 (98,0) (97,0) (110,0) (1,3)
 *            abracadabra  LPF [0,0,0,1,0,1,0,4,3,2,1]  PREV [-1,-1,-1,0,-1,3,-1,0,1,2,7]
 *                         LZ77 (97,0) (98,0) (114,0) (0,1) (99,0) (3,1) (100,0) (0,4)
 *            mississippi  LPF [0,0,0,1,4,3,2,1,0,1,1]  PREV [-1,-1,-1,2,1,2,3,4,-1,8,7]
 *                         LZ77 (109,0) (105,0) (115,0) (2,1) (1,4) (112,0) (8,1) (7,1)
 *            aaaa         LPF [0,3,2,1]  PREV [-1,0,1,2]  LZ77 (97,0) (0,3)
 *            a            LPF [0]  PREV [-1]  LZ77 (97,0)
 * and in general a^n gives LPF[i] = n - i, PREV[i] = i - 1 for i >= 1, LZ77 (97,0) (0,n-1).
 *
 * GPU path (DESIGN.md section 4.10): the suffix sort and LCP stage of bwts_b200_sa_lcp_*, then the
 * previous / next smaller values in suffix array order with the LCP minimum over each span (a min tree per
 * tile of 4096 rows in shared memory, a tree over the tiles for the rest), then the greedy parse by levels of
 * pointer jumping over chunks of 4096 positions.  Both are O(n log n) for every input.
 *
 * Arguments follow bwts_b200_sa_*: a NULL ctx, in or output pointer, or len <= 0 is BWTS_B200_EINVAL,
 * len > BWTS_B200_MAX_LEN is BWTS_B200_ETOOBIG; no two of in, lpf and prev may share a byte, nor in and
 * factors[0 .. 2 cap) (BWTS_B200_EINVAL).  Device outputs must be 4-byte aligned, the input may lie at any
 * offset.  LZ77: z must not be NULL and cap >= 0 (else BWTS_B200_EINVAL); *z is set to the number of factors
 * whenever the parse ran; z > cap is BWTS_B200_EINVAL and nothing is written to factors.  z <= n, so
 * cap = len always suffices.  Without a device every call returns BWTS_B200_ENODEV.
 *
 * Device memory: the device forms need the workspace of the SA call of the same length (71 bytes per input
 * byte + 64 MiB) and nothing more for an input at a 16-byte aligned address (2 bytes per byte otherwise);
 * every stage takes its scratch from the sort's buffers.  The host forms add an I/O region of 9 bytes per
 * input byte (text, LPF and PREV, or up to n factor pairs): ~80 bytes per byte in all, 172 GB at
 * len = 2^31 - 1, as bwts_b200_sa_lcp_host.
 * Statistics: direction 0, factors = 1, longest_factor = n; the LPF and parse kernels (k_lpf_*, k_lz_*) are
 * booked to kernel class "emit" and phase 3, beside k_lcp_*. */
int bwts_b200_lpf_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *lpf, int *prev);
int bwts_b200_lpf_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_lpf, void *d_prev, void *stream);
int bwts_b200_lz77_host(bwts_b200_ctx *ctx, const unsigned char *in, long len, int *factors, long cap, long *z);
int bwts_b200_lz77_device(bwts_b200_ctx *ctx, const void *d_in, long len, void *d_factors, long cap, long *z,
                          void *stream);

#ifdef __cplusplus
}
#endif

#endif /* BWTS_B200_H */

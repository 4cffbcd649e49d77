/*
 * TEST INFRASTRUCTURE ONLY -- never linked into the product library.
 *
 * CPU statement of libdivsufsort's end-of-text BWT (include/bwts_b200.h, bwts_b200_divbwt /
 * bwts_b200_inverse_bw_transform), the checker of the GPU path:
 *   oracle_divbwt = suffix array of T (oracle/sais.c), then libdivsufsort's copy rule:
 *                   U[0] = T[n-1], the row of suffix 0 drops out, returns primary = its row + 1.
 *   oracle_inverse_bw_transform = libdivsufsort's own forward walk: per byte the end of its bucket
 *                   (C, over the bytes present, D), the successor of each row in B, and the byte
 *                   of a row by binary search over C.  It walks T front to back, the GPU walks it
 *                   back to front, so the two share no step.  The walk is only defined on pairs the
 *                   forward makes: on others it would read B[-1] and returns -4 instead.
 * Built on its own as oracle/libdivbwt_oracle.so (with sais.c; __graft_entry__.build and
 * tests/divbwt_oracle.py), so the other oracle libraries stay as they are.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "shim/divsufsort.h"

int oracle_divbwt(const unsigned char *T, unsigned char *U, long n, long *primary)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !U || !primary) return -1;
    int32_t *sa = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!sa) return -2;
    if (divsufsort(T, sa, (int32_t)n) != 0) { free(sa); return -3; }
    long r0 = 0;
    while (sa[r0] != 0) r0++;
    U[0] = T[n - 1];
    for (long r = 0; r < r0; r++) U[r + 1] = T[sa[r] - 1];
    for (long r = r0 + 1; r < n; r++) U[r] = T[sa[r] - 1];
    free(sa);
    *primary = r0 + 1;
    return 0;
}

/* first i in [0, size) with A[i] >= value */
static int32_t lower_bound_i32(const int32_t *A, int32_t size, int32_t value)
{
    int32_t lo = 0, hi = size;
    while (lo < hi) {
        const int32_t mid = lo + (hi - lo) / 2;
        if (A[mid] < value) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

int oracle_inverse_bw_transform(const unsigned char *T, unsigned char *U, long n, long idx)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !U || idx < 1 || idx > n) return -1;
    int32_t C[256];
    unsigned char D[256];
    int32_t d = 0;
    memset(C, 0, sizeof C);
    for (long i = 0; i < n; i++) C[T[i]]++;
    for (int32_t c = 0, i = 0; c < 256; c++) {
        const int32_t k = C[c];
        if (k > 0) {
            C[c] = i;
            D[d++] = (unsigned char)c;
            i += k;
        }
    }
    int32_t *B = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!B) return -2;
    long i = 0;
    for (; i < idx; i++) B[C[T[i]]++] = (int32_t)i;
    for (; i < n; i++) B[C[T[i]]++] = (int32_t)(i + 1);
    for (int32_t c = 0; c < d; c++) C[c] = C[D[c]];  /* end of each present byte's bucket */
    int32_t p = (int32_t)idx;
    for (i = 0; i < n; i++) {
        if (p == 0) { free(B); return -4; }
        U[i] = D[lower_bound_i32(C, d, p)];
        p = B[p - 1];
    }
    free(B);
    return 0;
}

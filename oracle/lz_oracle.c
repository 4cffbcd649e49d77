/*
 * TEST INFRASTRUCTURE ONLY -- never linked into the product library.
 *
 * CPU statement of the longest-previous-factor array and the greedy LZ77 parse (include/bwts_b200.h,
 * bwts_b200_lpf_* / bwts_b200_lz77_*), the checker of the GPU path:
 *   oracle_lpf  = suffix array of T (SA-IS, oracle/sais.c), one stack pass over it for the previous and next
 *                 smaller values (psv, nsv: the sources whose suffixes are the nearest smaller / larger ones
 *                 among the earlier positions), stored in text order; then lcp(i, psv(i)) and lcp(i, nsv(i))
 *                 by direct byte comparison, each starting from its value at i - 1 minus 1 (Kärkkäinen, Kempa
 *                 and Puglisi, "Linear time Lempel-Ziv factorization: simple, fast, small", CPM 2013).  It
 *                 never uses the LCP array or a range minimum, unlike the GPU.
 *   oracle_lz77 = oracle_lpf, then the sequential greedy parse.
 * Built on its own as oracle/liblz_oracle.so (with sais.c; __graft_entry__.build and tests/lz_oracle.py).
 */
#include <stdint.h>
#include <stdlib.h>

#include "shim/divsufsort.h"

static long match(const unsigned char *T, long n, long i, long j, long h)
{
    while (i + h < n && j + h < n && T[i + h] == T[j + h]) h++;
    return h;
}

int oracle_lpf(const unsigned char *T, int32_t *LPF, int32_t *PREV, long n)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !LPF || !PREV) return -1;
    int32_t *SA = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int32_t *psv = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int32_t *nsv = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int32_t *stk = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!SA || !psv || !nsv || !stk) { free(SA); free(psv); free(nsv); free(stk); return -2; }
    if (divsufsort(T, SA, (int32_t)n) != 0) { free(SA); free(psv); free(nsv); free(stk); return -3; }
    /* the stack holds the rows' text positions, increasing from the bottom: a row pops every larger one
     * above it (those find their next smaller value here), and what stays below is its previous smaller value */
    long top = 0;
    for (long r = 0; r < n; r++) {
        const int32_t i = SA[r];
        while (top > 0 && stk[top - 1] > i) nsv[stk[--top]] = i;
        psv[i] = top > 0 ? stk[top - 1] : -1;
        stk[top++] = i;
    }
    while (top > 0) nsv[stk[--top]] = -1;
    long a = 0, b = 0;
    for (long i = 0; i < n; i++) {
        a = psv[i] < 0 ? 0 : match(T, n, i, psv[i], a > 0 ? a - 1 : 0);
        b = nsv[i] < 0 ? 0 : match(T, n, i, nsv[i], b > 0 ? b - 1 : 0);
        if (a >= b) { LPF[i] = (int32_t)a; PREV[i] = a > 0 ? psv[i] : -1; }
        else { LPF[i] = (int32_t)b; PREV[i] = nsv[i]; }
    }
    free(SA); free(psv); free(nsv); free(stk);
    return 0;
}

/* factors int32[2 cap]; *z = the number of factors; returns 1 (nothing written) when z > cap */
int oracle_lz77(const unsigned char *T, long n, int32_t *factors, long cap, long *z)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !z || cap < 0) return -1;
    int32_t *LPF = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    int32_t *PREV = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!LPF || !PREV) { free(LPF); free(PREV); return -2; }
    int rc = oracle_lpf(T, LPF, PREV, n);
    if (rc) { free(LPF); free(PREV); return rc; }
    long k = 0;
    for (long p = 0; p < n; p += LPF[p] > 0 ? LPF[p] : 1) k++;
    *z = k;
    if (k > cap || !factors) { free(LPF); free(PREV); return k > cap ? 1 : 0; }
    k = 0;
    for (long p = 0; p < n; p += LPF[p] > 0 ? LPF[p] : 1, k++) {
        factors[2 * k] = LPF[p] > 0 ? PREV[p] : (int32_t)T[p];
        factors[2 * k + 1] = LPF[p];
    }
    free(LPF); free(PREV);
    return 0;
}

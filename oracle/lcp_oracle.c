/*
 * TEST INFRASTRUCTURE ONLY -- never linked into the product library.
 *
 * CPU statement of the suffix array and LCP array (include/bwts_b200.h, bwts_b200_sa_lcp), the
 * checker of the GPU path:
 *   oracle_sa_lcp = suffix array of T (SA-IS, oracle/sais.c), then Kasai, Lee, Arimura, Arikawa and
 *                   Park's sequential LCP construction (CPM 2001): rank = SA^-1, and for i = 0..n-1 the
 *                   lcp h of suffix i and the suffix ranked just before it, starting from the previous
 *                   h minus 1.  It shares no step with the GPU's irreducible-pair formulation.
 * Built on its own as oracle/liblcp_oracle.so (with sais.c; __graft_entry__.build and
 * tests/lcp_oracle.py), so the other oracle libraries stay as they are.
 */
#include <stdint.h>
#include <stdlib.h>

#include "shim/divsufsort.h"

/* LCP[0] = 0, LCP[r] = lcp(T[SA[r-1]..), T[SA[r]..)) for r >= 1 */
int oracle_kasai(const unsigned char *T, const int32_t *SA, int32_t *LCP, long n)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !SA || !LCP) return -1;
    int32_t *rank = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!rank) return -2;
    for (long r = 0; r < n; r++) rank[SA[r]] = (int32_t)r;
    long h = 0;
    LCP[0] = 0;
    for (long i = 0; i < n; i++) {
        const long r = rank[i];
        if (r == 0) { h = 0; continue; }
        const long j = SA[r - 1];
        while (i + h < n && j + h < n && T[i + h] == T[j + h]) h++;
        LCP[r] = (int32_t)h;
        if (h > 0) h--;
    }
    free(rank);
    return 0;
}

int oracle_sa_lcp(const unsigned char *T, int32_t *SA, int32_t *LCP, long n)
{
    if (n <= 0 || n > 0x7fffffffL || !T || !SA) return -1;
    if (divsufsort(T, SA, (int32_t)n) != 0) return -3;
    return LCP ? oracle_kasai(T, SA, LCP, n) : 0;
}

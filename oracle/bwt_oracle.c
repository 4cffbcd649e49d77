/*
 * TEST INFRASTRUCTURE ONLY -- never linked into the product library.
 *
 * CPU statement of the classic Burrows-Wheeler transform with a primary index
 * (include/bwts_b200.h, bwts_b200_bwt_*), the checker of the GPU path:
 *   forward = suffix array of T.T (oracle/sais.c); the suffixes that start below
 *             n are the rotations of T in sorted order (two distinct rotations
 *             differ within n bytes).  T.T leaves tied rows in no particular
 *             order, so the primary index is computed directly: the number of
 *             rotations strictly smaller than T, i.e. the first row whose
 *             rotation equals T.  Needs 2n < 2^31.
 *   inverse = the plain n-step walk of the stable LF map (unbwts.c:50-52).
 * Built on its own as oracle/libbwt_oracle.so (with sais.c; __graft_entry__.build
 * and tests/bwt_oracle.py), so liboracle.so stays as it is.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "shim/divsufsort.h"

int oracle_bwt_forward(const unsigned char *in, long len, unsigned char *out, long *primary)
{
    if (len <= 0 || len > 0x3fffffffL || !in || !out || !primary) return -1;
    const int32_t n = (int32_t)len;

    /* rotation j equals T exactly when p divides j, p the smallest period of T that divides n
     * (KMP failure function) */
    int32_t *fail = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
    if (!fail) return -2;
    fail[0] = 0;
    for (int32_t i = 1, k = 0; i < n; i++) {
        while (k > 0 && in[i] != in[k]) k = fail[k - 1];
        if (in[i] == in[k]) k++;
        fail[i] = k;
    }
    int32_t p = n - fail[n - 1];
    if (n % p) p = n;
    free(fail);

    unsigned char *tt = (unsigned char *)malloc(2 * (size_t)n);
    int32_t *sa = (int32_t *)malloc(sizeof(int32_t) * 2 * (size_t)n);
    if (!tt || !sa) { free(tt); free(sa); return -2; }
    memcpy(tt, in, (size_t)n);
    memcpy(tt + n, in, (size_t)n);
    if (divsufsort(tt, sa, 2 * n) != 0) { free(tt); free(sa); return -3; }
    long r = 0, prim = -1;
    for (int32_t k = 0; k < 2 * n; k++) {
        const int32_t s = sa[k];
        if (s >= n) continue;
        out[r] = in[s == 0 ? n - 1 : s - 1];
        if (prim < 0 && s % p == 0) prim = r;
        r++;
    }
    free(tt);
    free(sa);
    *primary = prim;
    return 0;
}

int oracle_bwt_inverse(const unsigned char *in, long len, long primary, unsigned char *out)
{
    if (len <= 0 || len > 0x7fffffffL || !in || !out || primary < 0 || primary >= len) return -1;
    int32_t *lf = (int32_t *)malloc(sizeof(int32_t) * (size_t)len);
    if (!lf) return -2;
    int32_t first[256];
    memset(first, 0, sizeof first);
    for (long i = 0; i < len; i++) first[in[i]]++;
    for (int32_t c = 0, run = 0; c < 256; c++) {
        const int32_t k = first[c];
        first[c] = run;
        run += k;
    }
    for (long i = 0; i < len; i++) lf[i] = first[in[i]]++;
    int32_t q = (int32_t)primary;
    for (long j = 0; j < len; j++) {
        out[len - 1 - j] = in[q];
        q = lf[q];
    }
    free(lf);
    return 0;
}

/*
 * TEST INFRASTRUCTURE ONLY -- never linked into the product library.
 *
 * CPU statement of LZ77 decoding (include/bwts_b200.h, bwts_b200_lz77_decode_*), the checker of the GPU path:
 * the content rules in one pass over the factors, then the sequential byte-by-byte copy.  It accepts any valid
 * factor list, greedy or not.  Built on its own as oracle/liblz_decode_oracle.so (__graft_entry__.build and
 * tests/lz_decode_oracle.py).
 */
#include <stdint.h>

/* factors int32[2 z] -> out[0 .. n); returns 0, or -1 (nothing written) on bad arguments or a bad list: a literal
 * byte outside [0, 255], a negative length, a copy source outside [0, p_k), or sum of max(1, len_k) != n */
int oracle_lz77_decode(const int32_t *factors, long z, unsigned char *out, long n)
{
    if (!factors || !out || z <= 0 || n <= 0 || z > n || n > 0x7fffffffL) return -1;
    long p = 0;
    for (long k = 0; k < z; k++) {
        const int32_t a = factors[2 * k], l = factors[2 * k + 1];
        if (l < 0 || (l == 0 && (a < 0 || a > 255)) || (l > 0 && (a < 0 || a >= p))) return -1;
        p += l > 0 ? l : 1;
        if (p > n) return -1;
    }
    if (p != n) return -1;
    p = 0;
    for (long k = 0; k < z; k++) {
        const int32_t a = factors[2 * k], l = factors[2 * k + 1];
        if (l == 0) { out[p++] = (unsigned char)a; continue; }
        for (long j = 0; j < l; j++, p++) out[p] = out[a + j];
    }
    return 0;
}

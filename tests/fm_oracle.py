"""Checkers of the FM-index (include/bwts_b200.h, bwts_b200_fm_*): the brute-force definition of count and locate
(bisection over the sorted suffixes), the oracle (the suffix array of oracle/lcp_oracle.c plus bisection on the
text), and FmModel, a numpy restatement of the GPU index (bijective-bwt_b200/csrc/fm.cuh) -- U and its primary,
C, both checkpoint levels, the marks, their directory, the samples, backward search and the LF walk -- its
executable specification.  Nothing in the product imports this module."""
import bisect

import numpy as np

import lcp_oracle

KNOWN = [(b"banana", b"ana", 1, 3, [3, 1]), (b"banana", b"a", 0, 3, [5, 3, 1]), (b"banana", b"na", 4, 6, [4, 2]),
         (b"banana", b"anan", 2, 3, [1]), (b"banana", b"banana", 3, 4, [0]), (b"banana", b"bananas", 4, 4, []),
         (b"banana", b"nab", 5, 5, []), (b"banana", b"z", 6, 6, []), (b"banana", b"\x00", 0, 0, []),
         (b"banana", b"", 0, 6, [5, 3, 1, 0, 4, 2]), (b"mississippi", b"ssi", 9, 11, [5, 2]),
         (b"mississippi", b"issi", 2, 4, [4, 1]), (b"mississippi", b"ppp", 7, 7, []), (b"aaaa", b"aa", 1, 4, [2, 1, 0]),
         (b"aaaa", b"aaaaa", 4, 4, [])]
SAMPLES = (1, 2, 32, 1024)


def r256(b):
    return (b + 255) & ~255


def fm_bytes(n, sg, sample):
    """bwts_b200_fm_bytes: U, S, B, marks, directory, samples, C, map, each rounded up to 256 bytes"""
    sizes = [n, 4 * sg * ((n >> 16) + 1), 2 * sg * ((n >> 8) + 1), 4 * ((n + 31) // 32), 4 * ((n >> 8) + 1),
             4 * ((n + sample - 1) // sample), 4 * 257, 256]
    return sum(r256(s) for s in sizes)


def brute_count(x, p):
    """(lo, hi) = bisect_left / bisect_right of p over the sorted suffixes, truncated to len(p) for hi"""
    x, p = bytes(x), bytes(p)
    suf = sorted(x[i:] for i in range(len(x)))
    return bisect.bisect_left(suf, p), bisect.bisect_right([s[:len(p)] for s in suf], p)


def brute_sa(x):
    x = bytes(x)
    return sorted(range(len(x)), key=lambda s: x[s:])


def dollar_row_text(k, m):
    """b a^k c^m: the k suffixes a^j c^m (1 <= j <= k) sort before suffix 0 and every c^j after it, so suffix 0 sits
    at SA row k and the $ row of the FM-index at row k + 1"""
    return b"b" + b"a" * k + b"c" * m


class FmOracle:
    """count by bisection over the suffix array, locate by slicing it"""

    def __init__(self, x, sa=None):
        self.x = bytes(x)
        self.sa = lcp_oracle.LcpOracle().sa_lcp(self.x)[0] if sa is None else np.asarray(sa, dtype=np.int32)

    def _bound(self, p, upper):
        x, sa, m = self.x, self.sa, len(p)
        lo, hi = 0, len(sa)
        while lo < hi:
            mid = (lo + hi) // 2
            s = x[int(sa[mid]):int(sa[mid]) + m]
            if s < p or (upper and s == p):
                lo = mid + 1
            else:
                hi = mid
        return lo

    def count(self, p):
        p = bytes(p)
        return self._bound(p, False), self._bound(p, True)

    def count_many(self, patterns):
        r = np.array([self.count(p) for p in patterns], dtype=np.int32).reshape(-1, 2)
        return r[:, 0].copy(), r[:, 1].copy()

    def locate(self, lo, hi):
        return np.concatenate([self.sa[a:b] for a, b in zip(lo, hi)] + [np.zeros(0, np.int32)]).astype(np.int32)


class FmModel:
    """the GPU index, array for array (fm.cuh): rows of T$, row 0 the end of text, row i >= 1 SA row i - 1"""

    def __init__(self, x, sample, sa=None):
        self.x = bytes(x)
        t = np.frombuffer(self.x, dtype=np.uint8)
        n = self.n = len(t)
        self.sample = sample
        sa = lcp_oracle.LcpOracle().sa_lcp(self.x)[0] if sa is None else np.asarray(sa)
        sa = sa.astype(np.int64)
        # U, primary: the divbwt output (bwts_b200_divbwt): T[n-1], then B[r] = T[SA[r]-1] without the row of SA 0
        r0 = int(np.nonzero(sa == 0)[0][0])
        b = t[np.maximum(sa - 1, 0)]
        self.U = np.concatenate([t[n - 1:], b[:r0], b[r0 + 1:]]).astype(np.uint8)
        self.primary = r0 + 1
        hist = np.bincount(t, minlength=256)
        self.C = np.concatenate([[0], np.cumsum(hist)]).astype(np.int64) + 1    # C[c] = 1 + #{bytes < c}, C[256] = n+1
        self.syms = np.nonzero(hist)[0]
        self.sg = len(self.syms)
        self.map = np.zeros(256, dtype=np.int64)      # absent bytes: C[c + 1] == C[c], occ = 0
        self.map[self.syms] = np.arange(self.sg)
        # checkpoints: occ_U at every 256-byte block start, split into S (per 65536) and B (relative, u16)
        nb, ns = (n >> 8) + 1, (n >> 16) + 1
        onehot = self.U[:, None] == self.syms[None, :].astype(np.uint8)
        cum = np.vstack([np.zeros((1, self.sg), np.int64), np.cumsum(onehot, axis=0)])   # occ_U(k, j), j = 0..n
        self.S = cum[np.arange(ns) << 16].astype(np.uint32)
        blocks = np.arange(nb) << 8
        self.B = (cum[blocks] - cum[(blocks >> 16) << 16]).astype(np.uint16)
        assert int(self.B.max(initial=0)) < 65536
        # sampled SA: marks by SA row, directory per 256 rows, the marked rows' values in row order
        marked = (sa % sample) == 0
        self.marks = marked
        padded = np.zeros(nb * 256, dtype=bool)
        padded[:n] = marked
        self.dir = np.concatenate([[0], np.cumsum(padded.reshape(nb, 256).sum(axis=1))[:-1]]).astype(np.int64)
        self.samples = sa[marked].astype(np.int64)
        self.sa = sa

    def nbytes(self):
        return fm_bytes(self.n, self.sg, self.sample)

    def occ_u(self, c, j):
        if self.C[c + 1] == self.C[c]:
            return 0
        k = self.map[c]
        base = j & ~255
        inblock = int(np.count_nonzero(self.U[base:j] == c))
        return int(self.S[j >> 16, k]) + int(self.B[j >> 8, k]) + inblock

    def occ(self, c, i):
        return self.occ_u(c, i - (i > self.primary))

    def count(self, p):
        """backward search from the end of p through every byte; lo = sp - 1 (0 for the empty pattern)"""
        sp, ep = 0, self.n + 1
        for c in reversed(bytes(p)):
            sp = int(self.C[c]) + self.occ(c, sp)
            ep = int(self.C[c]) + self.occ(c, ep)
        return (sp - 1 if len(p) else 0), ep - 1

    def mark_rank(self, r):
        base = (r >> 8) << 8
        return int(self.dir[r >> 8]) + int(np.count_nonzero(self.marks[base:r]))

    def locate_row(self, r):
        """LF from FM row r + 1 to a marked row: sample value + steps"""
        steps = 0
        while not self.marks[r]:
            i = r + 1
            assert i != self.primary
            c = int(self.U[i - (i > self.primary)])
            r = int(self.C[c]) + self.occ(c, i) - 1
            steps += 1
        assert steps < self.sample
        return int(self.samples[self.mark_rank(r)]) + steps

    def locate(self, lo, hi):
        return np.array([self.locate_row(r) for a, b in zip(lo, hi) for r in range(a, b)], dtype=np.int32)


def golden_patterns(x, seed, count=4096):
    """the seeded pattern set of tests/golden/fm_fullsize.json: count substrings of 1..64 bytes, a quarter of them
    with one byte changed, and count / 8 random strings of 1..16 bytes"""
    rng = np.random.default_rng(seed)
    n = len(x)
    out = []
    for k in range(count):
        a = int(rng.integers(0, n))
        p = bytearray(x[a:a + int(rng.integers(1, 65))])
        if k % 4 == 3:
            p[int(rng.integers(0, len(p)))] ^= int(rng.integers(1, 256))
        out.append(bytes(p))
    for _ in range(count // 8):
        out.append(rng.integers(0, 256, size=int(rng.integers(1, 17)), dtype=np.uint8).tobytes())
    return out


def golden_locate_ranges(lo, hi, cap=4096):
    """each range cut to its first cap rows, so that short patterns on tiled text stay small"""
    lo = np.asarray(lo, dtype=np.int64)
    return lo.astype(np.int32), np.minimum(np.asarray(hi, dtype=np.int64), lo + cap).astype(np.int32)


def golden_hashes(lo, hi, pos):
    import hashlib
    rng = np.empty(2 * len(lo), dtype="<i4")
    rng[0::2], rng[1::2] = lo, hi
    return {"ranges_sha256": hashlib.sha256(rng.tobytes()).hexdigest(),
            "positions_sha256": hashlib.sha256(np.asarray(pos, dtype="<i4").tobytes()).hexdigest(),
            "hits": int((np.asarray(hi, np.int64) - lo).sum()), "located": int(len(pos))}

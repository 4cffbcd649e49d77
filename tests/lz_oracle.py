"""Checkers of the longest-previous-factor array and the greedy LZ77 parse (include/bwts_b200.h, bwts_b200_lpf_*,
bwts_b200_lz77_*): the C oracle oracle/liblz_oracle.so (oracle/lz_oracle.c: SA-IS, a stack pass for the previous and
next smaller values, direct byte comparison; built on demand with gcc), the brute-force definition, and a restatement
of the GPU's two stages (bijective-bwt_b200/csrc/lz.cuh) at any tile width, their executable specification.  Nothing
in the product imports this module."""
import ctypes
import subprocess

import numpy as np

import helpers

SO = helpers.ORACLE_DIR / "liblz_oracle.so"
NONE32 = 0xFFFFFFFF


def build():
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-I", str(helpers.ORACLE_DIR), "-o", str(SO),
                           str(helpers.ORACLE_DIR / "lz_oracle.c"), str(helpers.ORACLE_DIR / "sais.c")])


class LzOracle:
    def __init__(self):
        if not SO.exists():
            build()
        self.lib = ctypes.CDLL(str(SO))
        vp = ctypes.c_void_p
        self.lib.oracle_lpf.argtypes = [vp, vp, vp, ctypes.c_long]
        self.lib.oracle_lpf.restype = ctypes.c_int
        self.lib.oracle_lz77.argtypes = [vp, ctypes.c_long, vp, ctypes.c_long, ctypes.POINTER(ctypes.c_long)]
        self.lib.oracle_lz77.restype = ctypes.c_int

    def lpf(self, data):
        """-> (LPF, PREV), int32 numpy arrays"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        lpf = np.empty(len(src), dtype=np.int32)
        prev = np.empty(len(src), dtype=np.int32)
        rc = self.lib.oracle_lpf(src.ctypes.data, lpf.ctypes.data, prev.ctypes.data, len(src))
        if rc != 0:
            raise RuntimeError(f"oracle_lpf returned {rc}")
        return lpf, prev

    def lz77(self, data):
        """-> int32 array [z, 2] of (src_or_byte, len)"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty((len(src), 2), dtype=np.int32)
        z = ctypes.c_long(-1)
        rc = self.lib.oracle_lz77(src.ctypes.data, len(src), out.ctypes.data, len(src), ctypes.byref(z))
        if rc != 0:
            raise RuntimeError(f"oracle_lz77 returned {rc}")
        return out[:z.value].copy()


def common_prefix(x, i, j):
    k = 0
    while i + k < len(x) and j + k < len(x) and x[i + k] == x[j + k]:
        k += 1
    return k


def brute_lpf(x):
    """the definition: LPF[i] = max over j < i of lcp(i, j); PREV[i] among the j reaching it, the one with the
    largest suffix smaller than T[i..), else the one with the smallest suffix (-1 when LPF[i] == 0)"""
    x = bytes(x)
    n = len(x)
    lpf = np.zeros(n, dtype=np.int32)
    prev = np.full(n, -1, dtype=np.int32)
    for i in range(1, n):
        best = max(common_prefix(x, i, j) for j in range(i))
        lpf[i] = best
        if best == 0:
            continue
        cand = [j for j in range(i) if common_prefix(x, i, j) == best]
        smaller = [j for j in cand if x[j:] < x[i:]]
        prev[i] = max(smaller, key=lambda j: x[j:]) if smaller else min(cand, key=lambda j: x[j:])
    return lpf, prev


def parse(x, lpf, prev):
    """the greedy parse from LPF / PREV -> int32 [z, 2]"""
    out = []
    p = 0
    while p < len(x):
        out.append((int(prev[p]), int(lpf[p])) if lpf[p] > 0 else (x[p], 0))
        p += max(1, int(lpf[p]))
    return np.array(out, dtype=np.int32).reshape(-1, 2)


def tile_bits(n, tb=12):
    """lz_tile_bits: no tile wider than the next power of two of n, at least 32"""
    while tb > 5 and (1 << (tb - 1)) >= n:
        tb -= 1
    return tb


def _tree(vals, W):
    """heap-ordered min tree over W leaves (padding NONE32): list of 2W values, index 0 unused"""
    t = [NONE32] * (2 * W)
    t[W:W + len(vals)] = [int(v) for v in vals]
    for v in range(W - 1, 0, -1):
        t[v] = min(t[2 * v], t[2 * v + 1])
    return t


def _walk(S, L, leaf, i, half, left, acc):
    """the walk of k_lpf_tile / k_lpf_cross over one heap (S, L) with leaves from `half`: up to the first sibling on
    the chosen side holding an SA value below i, then down to the nearest such node at level `half` (stops there).
    -> (found, node, acc)"""
    v = leaf
    while v > 1:
        sib = v - 1 if left else v + 1
        if (v & 1) == (1 if left else 0):
            if S[sib] < i:
                v = sib
                break
            acc = min(acc, L[sib])
        v >>= 1
    else:
        return False, 0, acc
    while v < half:
        near, far = (2 * v + 1, 2 * v) if left else (2 * v, 2 * v + 1)
        if S[near] < i:
            v = near
        else:
            acc = min(acc, L[near])
            v = far
    return True, v, acc


def gpu_lpf(sa, lcp, tb):
    """k_lpf_tile + k_lpf_top + k_lpf_cross at tile width 2^tb -> (LPF, PREV, number of listed rows)"""
    sa = [int(v) for v in sa]
    lcp = [int(v) for v in lcp]
    n = len(sa)
    W, G = 1 << tb, (1 << tb) >> 5
    nt = -(-n // W)
    P = 1
    while P < nt:
        P <<= 1
    tiles = [(_tree(sa[t * W:(t + 1) * W], W), _tree(lcp[t * W:(t + 1) * W], W)) for t in range(nt)]
    topS = _tree([tiles[t][0][1] for t in range(nt)], P)
    topL = _tree([tiles[t][1][1] for t in range(nt)], P)
    lpf = np.zeros(n, dtype=np.int64)
    prev = np.full(n, -1, dtype=np.int64)
    listed = 0

    def put(i, a, sl, b, sg):
        if a >= b:
            lpf[i], prev[i] = a, (sl if a else -1)
        else:
            lpf[i], prev[i] = b, sg

    for r in range(n):
        t, q = divmod(r, W)
        S, L = tiles[t]
        i = sa[r]
        fl, vl, a = _walk(S, L, W + q, i, W, True, L[W + q])
        fr, vr, b = _walk(S, L, W + q, i, W, False, NONE32)
        if fr:
            b = min(b, L[vr])
        if i == 0 or (fl and fr):
            put(i, a if fl else 0, S[vl] if fl else 0, b if fr else 0, S[vr] if fr else 0)
            continue
        listed += 1
        res = []
        for left, found, acc, node in ((True, fl, a, vl), (False, fr, b, vr)):
            if found:
                res.append((acc, S[node]))
                continue
            ok, v, acc = _walk(topS, topL, P + t, i, P, left, min(acc, n))
            if not ok:
                res.append((0, 0))
                continue
            tt = v - P
            TS, TL = tiles[tt]
            u = 1
            while u < G:
                near, far = (2 * u + 1, 2 * u) if left else (2 * u, 2 * u + 1)
                if TS[near] < i:
                    u = near
                else:
                    acc = min(acc, TL[near])
                    u = far
            # the warp's 32-row group: last (first) row with SA < i
            base = tt * W + (u - G) * 32
            rows = [(sa[k], lcp[k]) for k in range(base, min(base + 32, n))]
            hits = [k for k, (s, _) in enumerate(rows) if s < i]
            h = hits[-1] if left else hits[0]
            span = rows[h + 1:] if left else rows[:h + 1]
            acc = min([acc] + [l for _, l in span])
            res.append((acc, rows[h][0]))
        put(i, res[0][0], res[0][1], res[1][0], res[1][1])
    return lpf.astype(np.int32), prev.astype(np.int32), listed


def gpu_parse(x, lpf, prev, tb):
    """k_lz_exit1, k_lz_jump, k_lz_top, k_lz_down and k_lz_chunk at chunk width 2^tb -> (int32 [z, 2], levels)"""
    n = len(x)
    W = 1 << tb
    lpf = [int(v) for v in lpf]
    nxt = [p + max(1, lpf[p]) for p in range(n)]
    # X_1 by tb rounds of pointer jumping inside each chunk
    X = [list(nxt)]
    for c in range(0, n, W):
        end = min(n, c + W)
        for _ in range(tb):
            X[0][c:end] = [X[0][y] if y < end else y for y in X[0][c:end]]
    L = 1
    while -(-n // (1 << (L * tb))) > W:
        L += 1
    for lv in range(2, L + 1):
        sb = lv * tb
        src, Y = X[-1], list(X[-1])
        for rnd in range(tb):
            S = src if rnd == 0 else Y
            Y = [S[S[p]] if S[p] < min(n, ((p >> sb) + 1) << sb) else S[p] for p in range(n)]
        X.append(Y)
    ent = {lv: [None] * -(-n // (1 << (lv * tb))) for lv in range(1, L + 1)}
    p = 0
    while p < n:   # at most W top-level hops
        ent[L][p >> (L * tb)] = p
        p = X[L - 1][p]
    for lv in range(L, 1, -1):
        for b, e in enumerate(ent[lv]):
            if e is None:
                continue
            end = min(n, (b + 1) << (lv * tb))
            hops = 0
            while e < end:
                ent[lv - 1][e >> ((lv - 1) * tb)] = e
                e = X[lv - 2][e]
                hops += 1
            assert hops <= W
    out = []
    for c, e in enumerate(ent[1]):
        if e is None:
            continue
        end = min(n, (c + 1) * W)
        while e < end:
            out.append((int(prev[e]), lpf[e]) if lpf[e] else (x[e], 0))
            e += max(1, lpf[e])
    return np.array(out, dtype=np.int32).reshape(-1, 2), L


def fibonacci_factor_lengths(n):
    """the closed form of the Fibonacci word's parse: 1, 1, 1, 3, 5, 8, 13, ..., the last one cut at n"""
    out, a, b = [1, 1, 1], 2, 3
    while sum(out) < n:
        out.append(b)
        a, b = b, a + b
    out = out[:]
    while sum(out) > n:
        extra = sum(out) - n
        if out[-1] > extra:
            out[-1] -= extra
        else:
            out.pop()
    return out

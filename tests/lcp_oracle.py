"""Checkers of the suffix array and LCP array (include/bwts_b200.h, bwts_b200_sa_lcp): the C oracle
oracle/liblcp_oracle.so (oracle/lcp_oracle.c: SA-IS plus Kasai, built on demand with gcc), the brute-force
definition, and a numpy restatement of the GPU's irreducible-LCP algorithm (bijective-bwt_b200/csrc/lcp.cuh),
its executable specification.  Nothing in the product imports this module."""
import ctypes
import subprocess

import numpy as np

import helpers

SO = helpers.ORACLE_DIR / "liblcp_oracle.so"


def build():
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-I", str(helpers.ORACLE_DIR), "-o", str(SO),
                           str(helpers.ORACLE_DIR / "lcp_oracle.c"), str(helpers.ORACLE_DIR / "sais.c")])


class LcpOracle:
    def __init__(self):
        if not SO.exists():
            build()
        self.lib = ctypes.CDLL(str(SO))
        vp = ctypes.c_void_p
        self.lib.oracle_sa_lcp.argtypes = [vp, vp, vp, ctypes.c_long]
        self.lib.oracle_sa_lcp.restype = ctypes.c_int
        self.lib.oracle_kasai.argtypes = [vp, vp, vp, ctypes.c_long]
        self.lib.oracle_kasai.restype = ctypes.c_int

    def sa_lcp(self, data):
        """-> (SA, LCP), int32 numpy arrays"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        sa = np.empty(len(src), dtype=np.int32)
        lcp = np.empty(len(src), dtype=np.int32)
        rc = self.lib.oracle_sa_lcp(src.ctypes.data, sa.ctypes.data, lcp.ctypes.data, len(src))
        if rc != 0:
            raise RuntimeError(f"oracle_sa_lcp returned {rc}")
        return sa, lcp

    def kasai(self, data, sa):
        """Kasai's LCP of `data` from a given suffix array"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        sa = np.ascontiguousarray(sa, dtype=np.int32)
        lcp = np.empty(len(src), dtype=np.int32)
        rc = self.lib.oracle_kasai(src.ctypes.data, sa.ctypes.data, lcp.ctypes.data, len(src))
        if rc != 0:
            raise RuntimeError(f"oracle_kasai returned {rc}")
        return lcp


def common_prefix(a, b):
    k = 0
    while k < len(a) and k < len(b) and a[k] == b[k]:
        k += 1
    return k


def brute_sa_lcp(x):
    """sorted suffixes (the end of text below every byte: a proper prefix sorts first) and their common prefixes"""
    x = bytes(x)
    sa = sorted(range(len(x)), key=lambda s: x[s:])
    lcp = [0] + [common_prefix(x[sa[r - 1]:], x[sa[r]:]) for r in range(1, len(x))]
    return np.array(sa, dtype=np.int32), np.array(lcp, dtype=np.int32)


def irreducible_rows(x, sa):
    """step 1 of lcp.cuh, in rank order: row r is irreducible when r == 0, SA[r] == 0, SA[r-1] == 0 or
    B[r] != B[r-1], B[r] = T[SA[r]-1]; -> boolean array over the rows"""
    t = np.frombuffer(bytes(x), dtype=np.uint8).astype(np.int32)
    sa = np.asarray(sa, dtype=np.int64)
    b = np.where(sa > 0, t[np.maximum(sa - 1, 0)], 256)
    irr = np.ones(len(sa), dtype=bool)
    irr[1:] = (b[1:] != b[:-1]) | (b[1:] == 256) | (b[:-1] == 256)
    return irr


def phi(sa):
    """Phi(SA[r]) = SA[r-1]; Phi(SA[0]) = -1"""
    sa = np.asarray(sa, dtype=np.int64)
    out = np.empty(len(sa), dtype=np.int64)
    out[sa[0]] = -1
    out[sa[1:]] = sa[:-1]
    return out


def irreducible_positions(x, sa):
    """by the definition in text order: i is irreducible unless i > 0, Phi(i) > 0 and T[i-1] == T[Phi(i)-1]
    (the row of SA[0] has no Phi and is irreducible)"""
    t = np.frombuffer(bytes(x), dtype=np.uint8)
    f = phi(sa)
    i = np.arange(len(t))
    red = (i > 0) & (f > 0)
    red[red] = t[i[red] - 1] == t[f[red] - 1]
    return ~red


def irreducible_lcp(x, sa):
    """the GPU's algorithm: compare the irreducible pairs only, write PLCP[j] + j at those j into a zeroed
    text-order array, inclusive max-scan, PLCP[i] = scan[i] - i, LCP[r] = PLCP[SA[r]].
    -> (LCP, PLCP, mask of irreducible positions, sum of the irreducible values)"""
    x = bytes(x)
    n = len(x)
    sa = np.asarray(sa, dtype=np.int64)
    irr = irreducible_rows(x, sa)
    P = np.zeros(n, dtype=np.int64)
    total = 0
    for r in np.nonzero(irr)[0]:
        s = int(sa[r])
        v = 0 if r == 0 else common_prefix(x[s:], x[int(sa[r - 1]):])
        P[s] = v + s
        total += v
    plcp = np.maximum.accumulate(P) - np.arange(n)
    mask = np.zeros(n, dtype=bool)
    mask[sa[irr]] = True
    return plcp[sa].astype(np.int32), plcp, mask, total

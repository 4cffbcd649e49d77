"""Checkers of libdivsufsort's end-of-text BWT (include/bwts_b200.h, bwts_b200_divbwt,
bwts_b200_inverse_bw_transform): the C oracle oracle/libdivbwt_oracle.so (oracle/divbwt_oracle.c, built on
demand with gcc) and brute-force statements of the definitions.  Nothing in the product imports this module."""
import ctypes
import subprocess

import numpy as np

import helpers
from bwt_oracle import lf_map

SO = helpers.ORACLE_DIR / "libdivbwt_oracle.so"


def build():
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-I", str(helpers.ORACLE_DIR), "-o", str(SO),
                           str(helpers.ORACLE_DIR / "divbwt_oracle.c"), str(helpers.ORACLE_DIR / "sais.c")])


class DivbwtOracle:
    def __init__(self):
        if not SO.exists():
            build()
        self.lib = ctypes.CDLL(str(SO))
        self.lib.oracle_divbwt.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p]
        self.lib.oracle_divbwt.restype = ctypes.c_int
        self.lib.oracle_inverse_bw_transform.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_long]
        self.lib.oracle_inverse_bw_transform.restype = ctypes.c_int

    def divbwt(self, data):
        """libdivsufsort's divbwt -> (bytes, primary)"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty(len(src), dtype=np.uint8)
        primary = ctypes.c_long(-1)
        rc = self.lib.oracle_divbwt(src.ctypes.data, out.ctypes.data, len(src), ctypes.byref(primary))
        if rc != 0:
            raise RuntimeError(f"oracle_divbwt returned {rc}")
        return out.tobytes(), primary.value

    def inverse_bw_transform(self, data, primary):
        """libdivsufsort's inverse_bw_transform; None for a pair its walk is not defined on (not made by the forward)"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty(len(src), dtype=np.uint8)
        rc = self.lib.oracle_inverse_bw_transform(src.ctypes.data, out.ctypes.data, len(src), primary)
        if rc == -4:
            return None
        if rc != 0:
            raise RuntimeError(f"oracle_inverse_bw_transform returned {rc}")
        return out.tobytes()


def brute_divbwt(x):
    """the BWT of x$ ($ below every byte) from its sorted suffixes, with the $ taken out; primary = its row"""
    x = bytes(x)
    order = sorted(range(len(x) + 1), key=lambda s: x[s:])   # suffixes of x$: the empty one is $ alone
    last = [x[s - 1] if s > 0 else None for s in order]      # None = the $
    primary = last.index(None)
    return bytes(c for c in last if c is not None), primary


def divbwt_prev(u, primary):
    """prev_s of the contract: p = 1 + LF(i), prev_s(i) = 0 if p == primary else p - (p > primary)"""
    p = lf_map(u) + 1
    return np.where(p == primary, 0, p - (p > primary))


def divbwt_inverse_formula(u, primary):
    """out[n-1-j] = u[prev_s^j(0)], defined for every u and every primary in [1, n]"""
    u = bytes(u)
    ps = divbwt_prev(u, primary)
    out = bytearray(len(u))
    q = 0
    for j in range(len(u)):
        out[len(u) - 1 - j] = u[q]
        q = int(ps[q])
    return bytes(out)

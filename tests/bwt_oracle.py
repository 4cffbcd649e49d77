"""Checkers of the classic Burrows-Wheeler transform with a primary index (include/bwts_b200.h,
bwts_b200_bwt_*): the C oracle oracle/libbwt_oracle.so (oracle/bwt_oracle.c, built on demand with gcc)
and a brute-force statement of the definition.  Nothing in the product imports this module."""
import ctypes
import subprocess

import numpy as np

import helpers

SO = helpers.ORACLE_DIR / "libbwt_oracle.so"


def build():
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-I", str(helpers.ORACLE_DIR), "-o", str(SO),
                           str(helpers.ORACLE_DIR / "bwt_oracle.c"), str(helpers.ORACLE_DIR / "sais.c")])


class BwtOracle:
    def __init__(self):
        if not SO.exists():
            build()
        self.lib = ctypes.CDLL(str(SO))
        self.lib.oracle_bwt_forward.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p, ctypes.c_void_p]
        self.lib.oracle_bwt_forward.restype = ctypes.c_int
        self.lib.oracle_bwt_inverse.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_void_p]
        self.lib.oracle_bwt_inverse.restype = ctypes.c_int

    def forward(self, data):
        """-> (bytes, primary index)"""
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty(len(src), dtype=np.uint8)
        primary = ctypes.c_long(-1)
        rc = self.lib.oracle_bwt_forward(src.ctypes.data, len(src), out.ctypes.data, ctypes.byref(primary))
        if rc != 0:
            raise RuntimeError(f"oracle_bwt_forward returned {rc}")
        return out.tobytes(), primary.value

    def inverse(self, data, primary):
        src = np.frombuffer(bytes(data), dtype=np.uint8)
        out = np.empty(len(src), dtype=np.uint8)
        rc = self.lib.oracle_bwt_inverse(src.ctypes.data, len(src), primary, out.ctypes.data)
        if rc != 0:
            raise RuntimeError(f"oracle_bwt_inverse returned {rc}")
        return out.tobytes()


def rows(x):
    """start positions of the sorted rotations; tied rotations by start position"""
    x = bytes(x)
    return sorted(range(len(x)), key=lambda s: (x[s:] + x[:s], s))


def brute_forward(x):
    x = bytes(x)
    r = rows(x)
    return bytes(x[s - 1] for s in r), r.index(0)   # x[-1] is x[n-1]


def lf_map(y):
    """stable LF map: C[c] + occ(c, i)"""
    y = np.frombuffer(bytes(y), dtype=np.uint8)
    order = np.argsort(y, kind="stable")
    lf = np.empty(len(y), dtype=np.int64)
    lf[order] = np.arange(len(y))
    return lf


def brute_inverse(y, primary):
    y = bytes(y)
    lf = lf_map(y)
    out = bytearray(len(y))
    q = primary
    for j in range(len(y)):
        out[len(y) - 1 - j] = y[q]
        q = int(lf[q])
    return bytes(out)

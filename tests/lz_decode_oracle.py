"""Checkers of LZ77 decoding (include/bwts_b200.h, bwts_b200_lz77_decode_*): the C oracle oracle/liblz_decode_oracle.so
(oracle/lz_decode_oracle.c: the content rules, then the sequential byte-by-byte copy; built on demand with gcc), a
pure-Python decode, a numpy restatement of the GPU's chunk and global rounds (bijective-bwt_b200/csrc/lzd.cuh) at any
chunk width, and generators of valid factor lists that are not greedy.  Nothing in the product imports this module."""
import ctypes
import subprocess

import numpy as np

import helpers
import lz_oracle

SO = helpers.ORACLE_DIR / "liblz_decode_oracle.so"
RES = 1 << 31


def build():
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-o", str(SO),
                           str(helpers.ORACLE_DIR / "lz_decode_oracle.c")])


class LzDecodeOracle:
    def __init__(self):
        if not SO.exists():
            build()
        self.lib = ctypes.CDLL(str(SO))
        vp, cl = ctypes.c_void_p, ctypes.c_long
        self.lib.oracle_lz77_decode.argtypes = [vp, cl, vp, cl]
        self.lib.oracle_lz77_decode.restype = ctypes.c_int

    def lz77_decode(self, factors, n):
        """int32 [z, 2] -> bytes, or None for a list the decoder must reject"""
        f = np.ascontiguousarray(factors, dtype=np.int32).reshape(-1, 2)
        out = np.zeros(max(n, 1), dtype=np.uint8)
        if self.lib.oracle_lz77_decode(f.ctypes.data, len(f), out.ctypes.data, n) != 0:
            return None
        return out[:n].tobytes()


def py_decode(factors, n):
    """the definition, one byte at a time (no checks)"""
    out = bytearray()
    for a, l in np.asarray(factors, dtype=np.int64).reshape(-1, 2).tolist():
        if l == 0:
            out.append(a)
        else:
            for j in range(l):
                out.append(out[a + j])
    assert len(out) == n
    return bytes(out)


def round_bound(n, tb):
    """ceil(log2 ceil(n / W)) + 1 at the chunk width the GPU uses for n"""
    nc = -(-n // (1 << lz_oracle.tile_bits(n, tb)))
    return (nc - 1).bit_length() + 1


def gpu_decode(factors, n, tb=12):
    """k_lzd_chunk then k_lzd_jump rounds at chunk width 2^tb (narrowed as lz_tile_bits does) -> (bytes, rounds,
    live_sum); the in-chunk rounds synchronous, the global ones synchronous too (the GPU's in-place reads only
    move faster)"""
    tb = lz_oracle.tile_bits(n, tb)
    f = np.asarray(factors, dtype=np.int64).reshape(-1, 2)
    lens = np.maximum(f[:, 1], 1)
    assert int(lens.sum()) == n
    p = np.cumsum(lens) - lens
    k = np.repeat(np.arange(len(f)), lens)
    i = np.arange(n, dtype=np.int64)
    v = np.where(f[k, 1] == 0, RES | f[k, 0], f[k, 0] + (i - p[k]))
    base = (i >> tb) << tb
    for _ in range(tb):
        inside = ((v & RES) == 0) & (v >= base)
        v = np.where(inside, v[np.where(inside, v, 0)], v)
    live = np.nonzero((v & RES) == 0)[0]
    assert (v[live] < base[live]).all(), "a word still points inside its chunk"
    rounds = live_sum = 0
    while live.size:
        live_sum += live.size
        v[live] = v[v[live]]
        rounds += 1
        live = live[(v[live] & RES) == 0]
    return (v & 0xFF).astype(np.uint8).tobytes(), rounds, live_sum


def random_factors(n, seed, max_len=64, lit=0.2, near=None, period=None):
    """a valid, generally non-greedy list for n bytes: literals with probability `lit` (also where a match exists),
    copies of 1 .. max_len bytes from a source `near` positions back at most, exactly `period` back, or anywhere
    before (far)"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, max_len + 1, size=n).astype(np.int64)
    lens[rng.random(n) < lit] = 0
    lens[0] = 0
    eff = np.maximum(lens, 1)
    cum = np.cumsum(eff)
    z = int(np.searchsorted(cum, n)) + 1
    lens, eff = lens[:z], eff[:z]
    p = np.cumsum(eff) - eff
    last = n - int(p[-1])
    if z > 1 and (lens[-1] or last > 1):
        lens[-1] = last
    f = np.zeros((z, 2), dtype=np.int64)
    f[:, 1] = lens
    copy = lens > 0
    pc = p[copy]
    if period is not None:
        src = np.maximum(pc - period, 0)
    elif near is not None:
        src = np.maximum(pc - rng.integers(1, near + 1, size=pc.size), 0)
    else:
        src = (rng.random(pc.size) * pc).astype(np.int64)
    f[copy, 0] = np.minimum(src, pc - 1)
    f[~copy, 0] = rng.integers(0, 256, size=int((~copy).sum()))
    return f.astype(np.int32)


def strided_chain(n, stride, seed=0):
    """stride literals, then single-byte copies from `stride` positions back: every hop of every chain crosses a
    chunk when stride >= the chunk width, and the chains are n / stride long"""
    rng = np.random.default_rng(seed)
    s = min(stride, n)
    f = np.zeros((n, 2), dtype=np.int64)
    f[:s, 0] = rng.integers(0, 256, size=s)
    f[s:, 0] = np.arange(s, n) - stride
    f[s:, 1] = 1
    return f.astype(np.int32)


def a_n(n):
    return np.array([[97, 0]] + ([[0, n - 1]] if n > 1 else []), dtype=np.int32)

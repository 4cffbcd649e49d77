"""ctypes mirror of include/bwts_b200.h (libbwts_b200.so).

The reference (NealB/Bijective-BWT) is three C command-line tools with no Python
surface; this module exists for the test-suite and bench.py.  It is a thin pass-through:
every function forwards to the C ABI and raises BwtsError on a non-zero status.  There is
no fallback of any kind -- if the shared library is missing, or no CUDA device is
present, calls fail loudly.
"""
import ctypes
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libbwts_b200.so"

NCLASS = 16
NPHASE = 8
MAX_LEN = (1 << 31) - 1

EXPORTS = [
    "bwts_b200_forward", "bwts_b200_inverse", "bwts_b200_forward_blocks", "bwts_b200_inverse_blocks",
    "bwts_b200_device_count", "bwts_b200_create", "bwts_b200_destroy", "bwts_b200_reserve",
    "bwts_b200_forward_host", "bwts_b200_inverse_host", "bwts_b200_forward_device",
    "bwts_b200_inverse_device", "bwts_b200_get_stats", "bwts_b200_class_name", "bwts_b200_set_profile",
    "bwts_b200_strerror", "bwts_b200_last_cuda_error", "bwts_b200_version", "bwts_b200_tune",
    "bwts_b200_divsufsort", "bwts_b200_phase_name",
    "bwts_b200_bwt_forward", "bwts_b200_bwt_inverse", "bwts_b200_bwt_forward_host", "bwts_b200_bwt_inverse_host",
    "bwts_b200_bwt_forward_device", "bwts_b200_bwt_inverse_device", "bwts_b200_bwt_forward_blocks",
    "bwts_b200_bwt_inverse_blocks",
    "bwts_b200_divbwt", "bwts_b200_inverse_bw_transform", "bwts_b200_divbwt_forward_host",
    "bwts_b200_divbwt_inverse_host", "bwts_b200_divbwt_forward_device", "bwts_b200_divbwt_inverse_device",
    "bwts_b200_divbwt_forward_blocks", "bwts_b200_divbwt_inverse_blocks",
    "bwts_b200_sa_host", "bwts_b200_sa_device", "bwts_b200_sa_lcp_host", "bwts_b200_sa_lcp_device", "bwts_b200_sa_lcp",
    "bwts_b200_fm_build_host", "bwts_b200_fm_build_device", "bwts_b200_fm_free", "bwts_b200_fm_bytes",
    "bwts_b200_fm_count_host", "bwts_b200_fm_count_device", "bwts_b200_fm_locate_host", "bwts_b200_fm_locate_device",
    "bwts_b200_lpf_host", "bwts_b200_lpf_device", "bwts_b200_lz77_host", "bwts_b200_lz77_device",
]


class BwtsError(RuntimeError):
    def __init__(self, code, what=""):
        self.code = code
        msg = lib().bwts_b200_strerror(code).decode()
        super().__init__(f"{what}: {msg} (code {code})" if what else f"{msg} (code {code})")


class Stats(ctypes.Structure):
    _fields_ = [
        ("len", ctypes.c_long), ("direction", ctypes.c_int), ("factors", ctypes.c_long),
        ("longest_factor", ctypes.c_long), ("alphabet_bits", ctypes.c_int), ("initial_depth", ctypes.c_int),
        ("rounds", ctypes.c_int), ("radix_passes", ctypes.c_int), ("local_rounds", ctypes.c_int),
        ("cta_rounds", ctypes.c_int), ("live_sum", ctypes.c_long),
        ("splitters", ctypes.c_long), ("unreached", ctypes.c_long), ("launches", ctypes.c_long),
        ("total_ms", ctypes.c_double),
        ("class_launches", ctypes.c_long * NCLASS), ("class_ms", ctypes.c_double * NCLASS),
        ("class_bytes", ctypes.c_double * NCLASS),
        ("h2d_ms", ctypes.c_double), ("d2h_ms", ctypes.c_double), ("lyndon_fallback", ctypes.c_int),
        ("phase_ms", ctypes.c_double * NPHASE), ("arena_bytes", ctypes.c_long), ("first_live", ctypes.c_long),
        ("tuple_rounds", ctypes.c_int), ("tuple_live_sum", ctypes.c_long), ("inverse_attempts", ctypes.c_int),
        ("binned_rounds", ctypes.c_int),
    ]


_lib = None


def lib():
    """Load libbwts_b200.so (built by `make -C bijective-bwt_b200` / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                          "(nvcc, sm_100a). There is no CPU fallback.")
    L = ctypes.CDLL(os.environ.get("BWTS_B200_LIB", str(LIB_PATH)))  # override: diagnostic builds (make profile-lib)
    vp, cl, ci = ctypes.c_void_p, ctypes.c_long, ctypes.c_int
    for name in ("bwts_b200_forward", "bwts_b200_inverse"):
        getattr(L, name).argtypes = [vp, cl, vp, ci]
    for name in ("bwts_b200_forward_blocks", "bwts_b200_inverse_blocks"):
        getattr(L, name).argtypes = [vp, cl, cl, vp, ctypes.POINTER(ci), ci]
    L.bwts_b200_create.argtypes = [ci]
    L.bwts_b200_create.restype = vp
    L.bwts_b200_destroy.argtypes = [vp]
    L.bwts_b200_destroy.restype = None
    L.bwts_b200_reserve.argtypes = [vp, cl]
    for name in ("bwts_b200_forward_host", "bwts_b200_inverse_host"):
        getattr(L, name).argtypes = [vp, vp, cl, vp]
    for name in ("bwts_b200_forward_device", "bwts_b200_inverse_device"):
        getattr(L, name).argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_get_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    L.bwts_b200_class_name.argtypes = [ci]
    L.bwts_b200_class_name.restype = ctypes.c_char_p
    L.bwts_b200_phase_name.argtypes = [ci, ci]
    L.bwts_b200_phase_name.restype = ctypes.c_char_p
    L.bwts_b200_set_profile.argtypes = [vp, ci]
    L.bwts_b200_strerror.argtypes = [ci]
    L.bwts_b200_strerror.restype = ctypes.c_char_p
    L.bwts_b200_last_cuda_error.argtypes = [vp]
    L.bwts_b200_version.restype = ctypes.c_char_p
    L.bwts_b200_tune.argtypes = [ci, cl]
    L.bwts_b200_divsufsort.argtypes = [vp, vp, ci, ci]
    L.bwts_b200_bwt_forward.argtypes = [vp, cl, vp, vp, ci]
    L.bwts_b200_bwt_inverse.argtypes = [vp, cl, cl, vp, ci]
    L.bwts_b200_bwt_forward_host.argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_bwt_inverse_host.argtypes = [vp, vp, cl, cl, vp]
    L.bwts_b200_bwt_forward_device.argtypes = [vp, vp, cl, vp, vp, vp]
    L.bwts_b200_bwt_inverse_device.argtypes = [vp, vp, cl, cl, vp, vp]
    L.bwts_b200_bwt_forward_blocks.argtypes = [vp, cl, cl, vp, vp, ctypes.POINTER(ci), ci]
    L.bwts_b200_bwt_inverse_blocks.argtypes = [vp, cl, cl, vp, vp, ctypes.POINTER(ci), ci]
    L.bwts_b200_divbwt.argtypes = [vp, vp, vp, ci, ci]
    L.bwts_b200_inverse_bw_transform.argtypes = [vp, vp, vp, ci, ci, ci]
    L.bwts_b200_divbwt_forward_host.argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_divbwt_inverse_host.argtypes = [vp, vp, cl, cl, vp]
    L.bwts_b200_divbwt_forward_device.argtypes = [vp, vp, cl, vp, vp, vp]
    L.bwts_b200_divbwt_inverse_device.argtypes = [vp, vp, cl, cl, vp, vp]
    L.bwts_b200_divbwt_forward_blocks.argtypes = [vp, cl, cl, vp, vp, ctypes.POINTER(ci), ci]
    L.bwts_b200_divbwt_inverse_blocks.argtypes = [vp, cl, cl, vp, vp, ctypes.POINTER(ci), ci]
    L.bwts_b200_sa_host.argtypes = [vp, vp, cl, vp]
    L.bwts_b200_sa_device.argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_sa_lcp_host.argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_sa_lcp_device.argtypes = [vp, vp, cl, vp, vp, vp]
    L.bwts_b200_sa_lcp.argtypes = [vp, vp, vp, ci, ci]
    L.bwts_b200_fm_build_host.argtypes = [vp, vp, cl, ci, vp]
    L.bwts_b200_fm_build_device.argtypes = [vp, vp, cl, ci, vp, vp]
    L.bwts_b200_fm_free.argtypes = [vp]
    L.bwts_b200_fm_free.restype = None
    L.bwts_b200_fm_bytes.argtypes = [vp]
    L.bwts_b200_fm_bytes.restype = cl
    L.bwts_b200_fm_count_host.argtypes = [vp, vp, vp, cl, vp, cl, vp, vp]
    L.bwts_b200_fm_count_device.argtypes = [vp, vp, vp, cl, vp, cl, vp, vp, vp]
    L.bwts_b200_fm_locate_host.argtypes = [vp, vp, vp, cl, vp, cl, vp]
    L.bwts_b200_fm_locate_device.argtypes = [vp, vp, vp, cl, vp, cl, vp, vp]
    L.bwts_b200_lpf_host.argtypes = [vp, vp, cl, vp, vp]
    L.bwts_b200_lpf_device.argtypes = [vp, vp, cl, vp, vp, vp]
    L.bwts_b200_lz77_host.argtypes = [vp, vp, cl, vp, cl, ctypes.POINTER(cl)]
    L.bwts_b200_lz77_device.argtypes = [vp, vp, cl, vp, cl, ctypes.POINTER(cl), vp]
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise BwtsError(rc, what)


def _as_u8(data):
    if isinstance(data, np.ndarray):
        assert data.dtype == np.uint8 and data.flags.c_contiguous
        return data
    return np.frombuffer(bytes(data), dtype=np.uint8)


def device_count():
    return lib().bwts_b200_device_count()


def version():
    return lib().bwts_b200_version().decode()


def tune(key, value):
    _check(lib().bwts_b200_tune(key, value), "bwts_b200_tune")


def _one_call(fn, what, data, device):
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    _check(fn(src.ctypes.data if len(src) else None, len(src), out.ctypes.data if len(src) else None, device), what)
    return out.tobytes()


def forward(data, device=0):
    """bwts_b200_forward: BWTS of `data` (bytes-like) -> bytes, host buffers."""
    return _one_call(lib().bwts_b200_forward, "bwts_b200_forward", data, device)


def inverse(data, device=0):
    """bwts_b200_inverse: inverse BWTS of `data` -> bytes, host buffers."""
    return _one_call(lib().bwts_b200_inverse, "bwts_b200_inverse", data, device)


def _blocks(fn, what, data, block_len, devices):
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(fn(src.ctypes.data, len(src), block_len, out.ctypes.data, devs, len(devices)), what)
    return out.tobytes()


def forward_blocks(data, block_len, devices=(0,)):
    return _blocks(lib().bwts_b200_forward_blocks, "bwts_b200_forward_blocks", data, block_len, list(devices))


def inverse_blocks(data, block_len, devices=(0,)):
    return _blocks(lib().bwts_b200_inverse_blocks, "bwts_b200_inverse_blocks", data, block_len, list(devices))


def blocks_ptr(direction, in_ptr, length, block_len, out_ptr, devices=(0,)):
    """bwts_b200_{forward,inverse}_blocks on raw host pointers (pinned buffers take the direct-copy path)."""
    fn = lib().bwts_b200_inverse_blocks if direction else lib().bwts_b200_forward_blocks
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(fn(in_ptr, length, block_len, out_ptr, devs, len(devices)), "bwts_b200_*_blocks")


def bwt_forward(data, device=0):
    """bwts_b200_bwt_forward: classic BWT of `data` -> (bytes, primary index), host buffers."""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    primary = ctypes.c_long(-1)
    _check(lib().bwts_b200_bwt_forward(src.ctypes.data if len(src) else None, len(src),
                                       out.ctypes.data if len(src) else None, ctypes.byref(primary), device),
           "bwts_b200_bwt_forward")
    return out.tobytes(), primary.value


def bwt_inverse(data, primary, device=0):
    """bwts_b200_bwt_inverse: inverse classic BWT of (`data`, `primary`) -> bytes, host buffers."""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    _check(lib().bwts_b200_bwt_inverse(src.ctypes.data if len(src) else None, len(src), primary,
                                       out.ctypes.data if len(src) else None, device), "bwts_b200_bwt_inverse")
    return out.tobytes()


def _nblocks(length, block_len):
    return 1 if block_len <= 0 or block_len >= length else -(-length // block_len)


def bwt_forward_blocks(data, block_len, devices=(0,)):
    """bwts_b200_bwt_forward_blocks -> (bytes, [primary index of each block])"""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    primary = np.full(_nblocks(len(src), block_len), -1, dtype=np.int64)
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(lib().bwts_b200_bwt_forward_blocks(src.ctypes.data, len(src), block_len, out.ctypes.data,
                                              primary.ctypes.data, devs, len(devices)), "bwts_b200_bwt_forward_blocks")
    return out.tobytes(), primary.tolist()


def bwt_inverse_blocks(data, block_len, primary, devices=(0,)):
    """bwts_b200_bwt_inverse_blocks: `primary` holds one index per block"""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    idx = np.ascontiguousarray(primary, dtype=np.int64)
    if len(idx) != _nblocks(len(src), block_len):
        raise ValueError(f"{len(idx)} primary indices for {_nblocks(len(src), block_len)} blocks")
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(lib().bwts_b200_bwt_inverse_blocks(src.ctypes.data, len(src), block_len, idx.ctypes.data,
                                              out.ctypes.data, devs, len(devices)), "bwts_b200_bwt_inverse_blocks")
    return out.tobytes()


def bwt_blocks_ptr(direction, in_ptr, length, block_len, out_ptr, primary, devices=(0,)):
    """bwts_b200_bwt_{forward,inverse}_blocks on raw host pointers; `primary`: int64 array, one per block
    (written by the forward, read by the inverse)"""
    fn = lib().bwts_b200_bwt_inverse_blocks if direction else lib().bwts_b200_bwt_forward_blocks
    assert primary.dtype == np.int64 and primary.flags.c_contiguous and len(primary) == _nblocks(length, block_len)
    devs = (ctypes.c_int * len(devices))(*devices)
    if direction:
        rc = fn(in_ptr, length, block_len, primary.ctypes.data, out_ptr, devs, len(devices))
    else:
        rc = fn(in_ptr, length, block_len, out_ptr, primary.ctypes.data, devs, len(devices))
    _check(rc, "bwts_b200_bwt_*_blocks")


def divbwt_forward(data, device=0):
    """bwts_b200_divbwt (libdivsufsort's divbwt): end-of-text BWT of `data` -> (bytes, primary), primary in [1, n]
    (0 for empty data)"""
    src = _as_u8(data)
    if len(src) == 0:
        return b"", 0
    out = np.empty(len(src), dtype=np.uint8)
    rc = lib().bwts_b200_divbwt(src.ctypes.data, out.ctypes.data, None, len(src), device)
    if rc < 0:
        raise BwtsError(rc, "bwts_b200_divbwt")
    return out.tobytes(), rc


def divbwt_inverse(data, primary, device=0):
    """bwts_b200_inverse_bw_transform (libdivsufsort's inverse_bw_transform) of (`data`, `primary`) -> bytes"""
    src = _as_u8(data)
    if len(src) == 0 and primary == 0:
        return b""
    out = np.empty(len(src), dtype=np.uint8)
    _check(lib().bwts_b200_inverse_bw_transform(src.ctypes.data, out.ctypes.data, None, len(src), primary, device),
           "bwts_b200_inverse_bw_transform")
    return out.tobytes()


def divbwt_forward_blocks(data, block_len, devices=(0,)):
    """bwts_b200_divbwt_forward_blocks -> (bytes, [primary of each block])"""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    primary = np.full(_nblocks(len(src), block_len), -1, dtype=np.int64)
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(lib().bwts_b200_divbwt_forward_blocks(src.ctypes.data, len(src), block_len, out.ctypes.data,
                                                 primary.ctypes.data, devs, len(devices)), "bwts_b200_divbwt_forward_blocks")
    return out.tobytes(), primary.tolist()


def divbwt_inverse_blocks(data, block_len, primary, devices=(0,)):
    """bwts_b200_divbwt_inverse_blocks: `primary` holds one index per block"""
    src = _as_u8(data)
    out = np.empty(len(src), dtype=np.uint8)
    idx = np.ascontiguousarray(primary, dtype=np.int64)
    if len(idx) != _nblocks(len(src), block_len):
        raise ValueError(f"{len(idx)} primary indices for {_nblocks(len(src), block_len)} blocks")
    devs = (ctypes.c_int * len(devices))(*devices)
    _check(lib().bwts_b200_divbwt_inverse_blocks(src.ctypes.data, len(src), block_len, idx.ctypes.data,
                                                 out.ctypes.data, devs, len(devices)), "bwts_b200_divbwt_inverse_blocks")
    return out.tobytes()


def suffix_array(data, device=0):
    """bwts_b200_divsufsort: suffix array (int32) of `data`."""
    src = _as_u8(data)
    sa = np.empty(len(src), dtype=np.int32)
    if len(src) == 0:
        return sa
    _check(lib().bwts_b200_divsufsort(src.ctypes.data, sa.ctypes.data, len(src), device), "bwts_b200_divsufsort")
    return sa


def suffix_array_lcp(data, device=0):
    """bwts_b200_sa_lcp: (suffix array, LCP array) of `data`, both int32; LCP[r] = lcp of the suffixes SA[r-1] and
    SA[r], LCP[0] = 0"""
    src = _as_u8(data)
    sa = np.empty(len(src), dtype=np.int32)
    lcp = np.empty(len(src), dtype=np.int32)
    if len(src) == 0:
        return sa, lcp
    _check(lib().bwts_b200_sa_lcp(src.ctypes.data, sa.ctypes.data, lcp.ctypes.data, len(src), device),
           "bwts_b200_sa_lcp")
    return sa, lcp


class FMIndex:
    """bwts_b200_fm: a device-resident FM-index (Context.fm_build_host / fm_build_device).  It owns its device
    memory until close(), outlives the context that built it, and any context on its device may query it."""

    def __init__(self, handle, length, sample):
        self._h = handle
        self.length = length
        self.sample = sample

    @property
    def handle(self):
        """the bwts_b200_fm pointer, for the C calls"""
        return self._h

    @property
    def nbytes(self):
        """device bytes the index holds (bwts_b200_fm_bytes)"""
        return lib().bwts_b200_fm_bytes(self._h)

    def close(self):
        if self._h:
            lib().bwts_b200_fm_free(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def fm_patterns(patterns):
    """list of bytes -> (concatenated uint8 array, int64 offsets of npat + 1 entries)"""
    pats = [bytes(p) for p in patterns]
    off = np.zeros(len(pats) + 1, dtype=np.int64)
    np.cumsum([len(p) for p in pats], out=off[1:])
    return np.frombuffer(b"".join(pats), dtype=np.uint8), off


class Context:
    """bwts_b200_ctx: reusable device workspace (one per device per host thread)."""

    def __init__(self, device=0):
        self._h = lib().bwts_b200_create(device)
        if not self._h:
            raise BwtsError(-3, f"bwts_b200_create({device})")
        self.device = device

    def close(self):
        if self._h:
            lib().bwts_b200_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, max_len):
        _check(lib().bwts_b200_reserve(self._h, max_len), "bwts_b200_reserve")

    def set_profile(self, on):
        _check(lib().bwts_b200_set_profile(self._h, int(on)), "bwts_b200_set_profile")

    # host buffers (addresses of `length` bytes; e.g. pinned torch tensors' data_ptr())
    def forward_host_ptr(self, in_ptr, length, out_ptr):
        _check(lib().bwts_b200_forward_host(self._h, in_ptr, length, out_ptr), "bwts_b200_forward_host")

    def inverse_host_ptr(self, in_ptr, length, out_ptr):
        _check(lib().bwts_b200_inverse_host(self._h, in_ptr, length, out_ptr), "bwts_b200_inverse_host")

    def forward_host(self, data):
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        self.forward_host_ptr(src.ctypes.data, len(src), out.ctypes.data)
        return out.tobytes()

    def inverse_host(self, data):
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        self.inverse_host_ptr(src.ctypes.data, len(src), out.ctypes.data)
        return out.tobytes()

    def bwt_forward_host_ptr(self, in_ptr, length, out_ptr):
        """classic BWT on host addresses; returns the primary index"""
        primary = ctypes.c_long(-1)
        _check(lib().bwts_b200_bwt_forward_host(self._h, in_ptr, length, out_ptr, ctypes.byref(primary)),
               "bwts_b200_bwt_forward_host")
        return primary.value

    def bwt_inverse_host_ptr(self, in_ptr, length, primary, out_ptr):
        _check(lib().bwts_b200_bwt_inverse_host(self._h, in_ptr, length, primary, out_ptr), "bwts_b200_bwt_inverse_host")

    def bwt_forward_host(self, data):
        """-> (bytes, primary index)"""
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        primary = self.bwt_forward_host_ptr(src.ctypes.data, len(src), out.ctypes.data)
        return out.tobytes(), primary

    def bwt_inverse_host(self, data, primary):
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        self.bwt_inverse_host_ptr(src.ctypes.data, len(src), primary, out.ctypes.data)
        return out.tobytes()

    def divbwt_forward_host(self, data):
        """libdivsufsort's divbwt -> (bytes, primary)"""
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        primary = ctypes.c_long(-1)
        _check(lib().bwts_b200_divbwt_forward_host(self._h, src.ctypes.data, len(src), out.ctypes.data,
                                                   ctypes.byref(primary)), "bwts_b200_divbwt_forward_host")
        return out.tobytes(), primary.value

    def divbwt_inverse_host(self, data, primary):
        src = _as_u8(data)
        out = np.empty(len(src), dtype=np.uint8)
        _check(lib().bwts_b200_divbwt_inverse_host(self._h, src.ctypes.data, len(src), primary, out.ctypes.data),
               "bwts_b200_divbwt_inverse_host")
        return out.tobytes()

    def sa_host(self, data):
        """suffix array (int32)"""
        src = _as_u8(data)
        sa = np.empty(len(src), dtype=np.int32)
        _check(lib().bwts_b200_sa_host(self._h, src.ctypes.data, len(src), sa.ctypes.data), "bwts_b200_sa_host")
        return sa

    def sa_lcp_host(self, data):
        """-> (suffix array, LCP array), int32"""
        src = _as_u8(data)
        sa = np.empty(len(src), dtype=np.int32)
        lcp = np.empty(len(src), dtype=np.int32)
        _check(lib().bwts_b200_sa_lcp_host(self._h, src.ctypes.data, len(src), sa.ctypes.data, lcp.ctypes.data),
               "bwts_b200_sa_lcp_host")
        return sa, lcp

    # device-resident buffers (device addresses, e.g. torch cuda tensors' data_ptr())
    def forward_device(self, d_in, length, d_out, stream=None):
        _check(lib().bwts_b200_forward_device(self._h, d_in, length, d_out, stream), "bwts_b200_forward_device")

    def inverse_device(self, d_in, length, d_out, stream=None):
        _check(lib().bwts_b200_inverse_device(self._h, d_in, length, d_out, stream), "bwts_b200_inverse_device")

    def bwt_forward_device(self, d_in, length, d_out, stream=None):
        """classic BWT on device addresses; returns the primary index"""
        primary = ctypes.c_long(-1)
        _check(lib().bwts_b200_bwt_forward_device(self._h, d_in, length, d_out, ctypes.byref(primary), stream),
               "bwts_b200_bwt_forward_device")
        return primary.value

    def bwt_inverse_device(self, d_in, length, primary, d_out, stream=None):
        _check(lib().bwts_b200_bwt_inverse_device(self._h, d_in, length, primary, d_out, stream),
               "bwts_b200_bwt_inverse_device")

    def divbwt_forward_device(self, d_in, length, d_out, stream=None):
        """divbwt on device addresses; returns the primary"""
        primary = ctypes.c_long(-1)
        _check(lib().bwts_b200_divbwt_forward_device(self._h, d_in, length, d_out, ctypes.byref(primary), stream),
               "bwts_b200_divbwt_forward_device")
        return primary.value

    def divbwt_inverse_device(self, d_in, length, primary, d_out, stream=None):
        _check(lib().bwts_b200_divbwt_inverse_device(self._h, d_in, length, primary, d_out, stream),
               "bwts_b200_divbwt_inverse_device")

    def sa_device(self, d_in, length, d_sa, stream=None):
        """suffix array into d_sa (length int32, 4-byte aligned)"""
        _check(lib().bwts_b200_sa_device(self._h, d_in, length, d_sa, stream), "bwts_b200_sa_device")

    def sa_lcp_device(self, d_in, length, d_sa, d_lcp, stream=None):
        """suffix array into d_sa and LCP array into d_lcp (length int32 each, 4-byte aligned)"""
        _check(lib().bwts_b200_sa_lcp_device(self._h, d_in, length, d_sa, d_lcp, stream), "bwts_b200_sa_lcp_device")

    # longest-previous-factor array and LZ77 parse (include/bwts_b200.h, last section)
    def lpf_host(self, data):
        """-> (LPF, PREV), int32, in text order"""
        src = _as_u8(data)
        lpf = np.empty(len(src), dtype=np.int32)
        prev = np.empty(len(src), dtype=np.int32)
        _check(lib().bwts_b200_lpf_host(self._h, src.ctypes.data, len(src), lpf.ctypes.data, prev.ctypes.data),
               "bwts_b200_lpf_host")
        return lpf, prev

    def lz77_host(self, data):
        """-> int32 [z, 2]: the greedy parse's factors (source, length), or (byte, 0) for a literal"""
        src = _as_u8(data)
        out = np.empty((len(src), 2), dtype=np.int32)
        z = ctypes.c_long(-1)
        _check(lib().bwts_b200_lz77_host(self._h, src.ctypes.data, len(src), out.ctypes.data, len(src),
                                         ctypes.byref(z)), "bwts_b200_lz77_host")
        return out[:z.value].copy()

    def lpf_device(self, d_in, length, d_lpf, d_prev, stream=None):
        """LPF into d_lpf and PREV into d_prev (length int32 each, 4-byte aligned)"""
        _check(lib().bwts_b200_lpf_device(self._h, d_in, length, d_lpf, d_prev, stream), "bwts_b200_lpf_device")

    def lz77_device(self, d_in, length, d_factors, cap, stream=None):
        """factor pairs into d_factors (room for cap pairs of int32, 4-byte aligned) -> z"""
        z = ctypes.c_long(-1)
        _check(lib().bwts_b200_lz77_device(self._h, d_in, length, d_factors, cap, ctypes.byref(z), stream),
               "bwts_b200_lz77_device")
        return z.value

    # FM-index (include/bwts_b200.h, section before)
    def fm_build_host(self, data, sample=32):
        """-> FMIndex over `data` (host bytes), SA sampled at text positions that are multiples of `sample`"""
        src = _as_u8(data)
        h = ctypes.c_void_p()
        _check(lib().bwts_b200_fm_build_host(self._h, src.ctypes.data, len(src), sample, ctypes.byref(h)),
               "bwts_b200_fm_build_host")
        return FMIndex(h.value, len(src), sample)

    def fm_build_device(self, d_in, length, sample=32, stream=None):
        """-> FMIndex over `length` device bytes at d_in"""
        h = ctypes.c_void_p()
        _check(lib().bwts_b200_fm_build_device(self._h, d_in, length, sample, ctypes.byref(h), stream),
               "bwts_b200_fm_build_device")
        return FMIndex(h.value, length, sample)

    def fm_count_host(self, fm, patterns):
        """list of bytes -> (lo, hi), int32 arrays: pattern k occurs hi[k] - lo[k] times, at SA[lo[k]:hi[k]]"""
        pat, off = fm_patterns(patterns)
        rng = np.empty(2 * (len(off) - 1), dtype=np.int32)
        total = ctypes.c_long()
        _check(lib().bwts_b200_fm_count_host(self._h, fm.handle, pat.ctypes.data, len(pat), off.ctypes.data,
                                             len(off) - 1, rng.ctypes.data, ctypes.byref(total)),
               "bwts_b200_fm_count_host")
        return rng[0::2].copy(), rng[1::2].copy()

    def fm_locate_host(self, fm, lo, hi):
        """-> (positions int32, offsets int64 of len(lo) + 1): range k's SA[lo[k]:hi[k]] is
        positions[offsets[k]:offsets[k+1]]"""
        lo = np.asarray(lo, dtype=np.int32)
        hi = np.asarray(hi, dtype=np.int32)
        rng = np.empty(2 * len(lo), dtype=np.int32)
        rng[0::2], rng[1::2] = lo, hi
        off = np.zeros(len(lo) + 1, dtype=np.int64)
        np.cumsum(hi.astype(np.int64) - lo, out=off[1:])
        cap = max(int(off[-1]), 0)
        pos = np.empty(max(cap, 1), dtype=np.int32)
        total = ctypes.c_long()
        _check(lib().bwts_b200_fm_locate_host(self._h, fm.handle, rng.ctypes.data, len(lo), pos.ctypes.data, cap,
                                              ctypes.byref(total)), "bwts_b200_fm_locate_host")
        return pos[:total.value], off

    def fm_count_device(self, fm, d_pat, pat_len, d_off, npat, d_range, stream=None):
        """device arrays: patterns, int64 offsets (npat + 1), int32 ranges (2 npat) -> total of hi - lo"""
        total = ctypes.c_long()
        _check(lib().bwts_b200_fm_count_device(self._h, fm.handle, d_pat, pat_len, d_off, npat, d_range,
                                               ctypes.byref(total), stream), "bwts_b200_fm_count_device")
        return total.value

    def fm_locate_device(self, fm, d_range, nrange, d_pos, cap, stream=None):
        """device arrays: int32 ranges (2 nrange), int32 positions (cap) -> number of positions written"""
        total = ctypes.c_long()
        _check(lib().bwts_b200_fm_locate_device(self._h, fm.handle, d_range, nrange, d_pos, cap, ctypes.byref(total),
                                                stream), "bwts_b200_fm_locate_device")
        return total.value

    def stats(self):
        s = Stats()
        _check(lib().bwts_b200_get_stats(self._h, ctypes.byref(s)), "bwts_b200_get_stats")
        out = {f: getattr(s, f) for f, _ in Stats._fields_ if not f.startswith("class_") and f != "phase_ms"}
        out["arena_bytes_per_byte"] = s.arena_bytes / s.len if s.len else None
        phases = {}
        for ph in range(NPHASE):
            name = lib().bwts_b200_phase_name(s.direction, ph)
            if name:
                phases[name.decode()] = s.phase_ms[ph]
        out["phases"] = phases
        classes = {}
        for c in range(NCLASS):
            if s.class_launches[c]:
                classes[lib().bwts_b200_class_name(c).decode()] = {
                    "launches": s.class_launches[c], "ms": s.class_ms[c], "bytes": s.class_bytes[c]}
        out["classes"] = classes
        return out

    def last_cuda_error(self):
        return lib().bwts_b200_last_cuda_error(self._h)

"""FM-index extract (include/bwts_b200.h, bwts_b200_fm_extract_*): the numpy restatement of the GPU path
(tests/fm_extract_model.py) against slices of the text -- random strings at every sample rate, every range of short
texts, lengths around multiples of the sample rate, the $ row at chosen rows -- and the entry points' argument
checks, which come before any device is looked for."""
import ctypes

import numpy as np
import pytest

import fm_extract_model
import fm_oracle
import helpers
from test_fm_oracle import random_inputs

EINVAL, ENODEV = -1, -3
KNOWN = [(b"banana", 0, 6, b"banana"), (b"banana", 1, 4, b"ana"), (b"banana", 5, 6, b"a"), (b"banana", 3, 3, b""),
         (b"banana", 6, 6, b""), (b"mississippi", 2, 6, b"ssis"), (b"aaaa", 1, 3, b"aa")]


def extracts(x, s, a, b):
    o = fm_oracle.FmOracle(x)
    e = fm_extract_model.ExtractModel(fm_oracle.FmModel(x, s, o.sa))
    out, offs = e.extract(a, b)
    want = b"".join(bytes(x[i:j]) for i, j in zip(a, b))
    assert out.tobytes() == want, (x[:20], s)
    assert offs[-1] == len(want)
    return e


def sample_ranges(n, rng, count):
    a = rng.integers(0, n + 1, size=count)
    b = np.minimum(a + rng.integers(0, 2 * n // 3 + 2, size=count), n)
    return a.tolist(), b.tolist()


def test_known_answers():
    for s in fm_oracle.SAMPLES:
        for text in (b"banana", b"mississippi", b"aaaa"):
            cases = [(a, b, want) for x, a, b, want in KNOWN if x == text]
            e = extracts(text, s, [c[0] for c in cases], [c[1] for c in cases])
            out, offs = e.extract([c[0] for c in cases], [c[1] for c in cases])
            assert [out[offs[k]:offs[k + 1]].tobytes() for k in range(len(cases))] == [c[2] for c in cases]


def test_random_strings_at_every_sample():
    rng = np.random.default_rng(21)
    for x in random_inputs(40, 22):
        for s in fm_oracle.SAMPLES:
            extracts(x, s, *sample_ranges(len(x), rng, 12))


def test_every_range_of_short_texts():
    rng = np.random.default_rng(23)
    texts = [b"a", b"ab", b"ba", b"banana", b"mississippi", b"abracadabra", b"aaaaaaa"]
    texts += [rng.integers(0, 3, size=int(k), dtype=np.uint8).tobytes() for k in (9, 17, 33)]
    for x in texts:
        n = len(x)
        a, b = zip(*[(i, j) for i in range(n + 1) for j in range(i, n + 1)])
        for s in (1, 2, 4, 8, 32):
            extracts(x, s, a, b)


def test_lengths_around_the_sample_rate():
    """n < s, n == s and n == k s +- 1: the last segment short, full, or one byte long"""
    rng = np.random.default_rng(25)
    for s in (2, 8, 32):
        for n in sorted({1, s - 1, s, s + 1, 3 * s - 1, 3 * s, 3 * s + 1}):
            if n < 1:
                continue
            x = rng.integers(0, 4, size=n, dtype=np.uint8).tobytes()
            edges = sorted({0, 1, n - 1, n} | {v for k in range(n // s + 2) for v in (k * s - 1, k * s, k * s + 1)
                                              if 0 <= v <= n})
            a, b = zip(*[(i, j) for i in edges for j in edges if i <= j])
            e = extracts(x, s, a, b)
            assert len(e.isa) == (n + s - 1) // s + 1 and e.isa[-1] == 0


def test_dollar_row_text():
    rng = np.random.default_rng(27)
    for k in (0, 1, 254, 255, 256, 257):
        for m in (0, 1, 300):
            x = fm_oracle.dollar_row_text(k, m)
            for s in (1, 2, 32, 1024):
                extracts(x, s, *sample_ranges(len(x), rng, 6))


def test_families_and_table():
    """the table is the inverse of the samples: isa[v / s] is the FM row of position v"""
    rng = np.random.default_rng(29)
    for n in (255, 256, 257, 1000):
        for x in helpers.families(n).values():
            o = fm_oracle.FmOracle(x)
            rank = np.empty(len(x), dtype=np.int64)
            rank[o.sa] = np.arange(len(x))
            for s in (1, 32):
                e = fm_extract_model.ExtractModel(fm_oracle.FmModel(x, s, o.sa))
                assert e.isa[:-1].tolist() == (rank[::s] + 1).tolist()
                a, b = sample_ranges(len(x), rng, 6)
                out, _ = e.extract(a + [0], b + [len(x)])
                assert out.tobytes() == b"".join(bytes(x[i:j]) for i, j in zip(a + [0], b + [len(x)]))


# --------------------------------------------------------------------------- entry points, no device needed

def test_arguments_are_checked_before_the_device(bwts):
    L = bwts.lib()
    rng = np.zeros(8, dtype=np.int32)
    out = np.zeros(8, dtype=np.uint8)
    r, q = rng.ctypes.data, out.ctypes.data
    fake = ctypes.c_void_p(r)       # never dereferenced before the arguments are refused
    total = ctypes.c_long(7)
    for fn in (L.bwts_b200_fm_extract_host, lambda *a: L.bwts_b200_fm_extract_device(*a, None)):
        assert fn(None, fake, r, 1, q, 8, None) == EINVAL
        assert fn(fake, None, r, 1, q, 8, None) == EINVAL
        assert fn(fake, fake, r, -1, q, 8, None) == EINVAL
        assert fn(fake, fake, r, 1, q, -8, None) == EINVAL
        assert fn(fake, fake, None, 1, q, 8, None) == EINVAL
        assert fn(fake, fake, r, 1, None, 8, None) == EINVAL
        total.value = 7
        assert fn(fake, fake, None, 0, None, 0, ctypes.byref(total)) == 0 and total.value == 0   # nrange == 0
    assert L.bwts_b200_fm_extract_device(fake, fake, r + 2, 1, q, 8, None, None) == EINVAL   # ranges 4-aligned


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = bwts.lib()
    rng = np.array([1, 4], dtype=np.int32)
    out = np.zeros(4, dtype=np.uint8)
    fake = ctypes.c_void_p(rng.ctypes.data)
    # arguments that pass every check that needs no index: no device, so ENODEV, whatever the handles
    assert L.bwts_b200_fm_extract_host(fake, fake, rng.ctypes.data, 1, out.ctypes.data, 4, None) == ENODEV
    assert L.bwts_b200_fm_extract_device(fake, fake, rng.ctypes.data, 1, out.ctypes.data + 1, 4, None, None) == ENODEV
    assert (out == 0).all()

"""The FM-index (include/bwts_b200.h, bwts_b200_fm_*): the oracle (suffix array plus bisection) against the
brute-force definition and the contract's known answers, the numpy restatement of the GPU index (tests/fm_oracle.py)
against the oracle at every sample rate, the bwts_b200_fm_bytes formula, and the entry points' argument checks,
which come before any device is looked for."""
import ctypes

import numpy as np
import pytest

import fm_oracle
import helpers

EINVAL, ETOOBIG, ENODEV = -1, -2, -3


def random_inputs(count, seed):
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        sigma = int(rng.choice([1, 2, 4, 256]))
        if t % 3 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 6)), dtype=np.uint8).tobytes()
            out.append(u * int(rng.integers(1, 40)))
        else:
            out.append(rng.integers(0, sigma, size=int(rng.integers(1, 300)), dtype=np.uint8).tobytes())
    return out


def patterns_for(x, rng, count=24):
    """substrings (hits), the same with one byte changed, random strings, absent bytes, too long, empty"""
    n = len(x)
    out = [b"", x, x + b"\x00", bytes([255]) * (n + 1)]
    for _ in range(count):
        a = int(rng.integers(0, n))
        p = bytearray(x[a:a + int(rng.integers(1, 12))])
        out.append(bytes(p))
        p[int(rng.integers(0, len(p)))] ^= int(rng.integers(1, 256))
        out.append(bytes(p))
        out.append(rng.integers(0, 256, size=int(rng.integers(1, 4)), dtype=np.uint8).tobytes())
    return out


def test_known_answers():
    for x, p, lo, hi, loc in fm_oracle.KNOWN:
        assert fm_oracle.brute_count(x, p) == (lo, hi), (x, p)
        o = fm_oracle.FmOracle(x)
        assert o.count(p) == (lo, hi), (x, p)
        assert o.locate([lo], [hi]).tolist() == loc, (x, p)
        assert [fm_oracle.brute_sa(x)[r] for r in range(lo, hi)] == loc


def test_oracle_matches_brute_force():
    rng = np.random.default_rng(5)
    for x in random_inputs(120, 9):
        o = fm_oracle.FmOracle(x)
        assert o.sa.tolist() == fm_oracle.brute_sa(x)
        for p in patterns_for(x, rng, 6):
            assert o.count(p) == fm_oracle.brute_count(x, p), (x, p)


def model_matches(x, rng, samples=fm_oracle.SAMPLES, count=8):
    o = fm_oracle.FmOracle(x)
    pats = patterns_for(x, rng, count)
    lo, hi = o.count_many(pats)
    for s in samples:
        m = fm_oracle.FmModel(x, s, o.sa)
        assert [m.count(p) for p in pats] == list(zip(lo.tolist(), hi.tolist())), (x[:20], s)
        assert np.array_equal(m.locate([0], [len(x)]), o.sa), (x[:20], s)


def test_model_matches_the_oracle_on_random_inputs():
    rng = np.random.default_rng(11)
    for x in random_inputs(60, 12):
        model_matches(x, rng)


def test_model_matches_the_oracle_on_families():
    rng = np.random.default_rng(13)
    for n in (1, 2, 255, 256, 257, 1000):
        for x in helpers.families(n).values():
            model_matches(x, rng, count=4)


def test_model_places_the_dollar_row():
    rng = np.random.default_rng(17)
    for k in (0, 1, 254, 255, 256, 257):
        for m in (0, 1, 300):
            x = fm_oracle.dollar_row_text(k, m)
            model = fm_oracle.FmModel(x, 2)
            assert model.primary == k + 1
            model_matches(x, rng, samples=(1, 32), count=4)


def test_checkpoint_levels_across_superblocks():
    """n around 65536: B restarts at each superblock and S carries the total"""
    rng = np.random.default_rng(19)
    for n in (65535, 65536, 65537):
        x = rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n).tobytes()
        o = fm_oracle.FmOracle(x)
        m = fm_oracle.FmModel(x, 32, o.sa)
        pats = patterns_for(x, rng, 20)
        assert [m.count(p) for p in pats] == list(zip(*[a.tolist() for a in o.count_many(pats)]))
        rows = rng.integers(0, n, size=200)
        assert [m.locate_row(int(r)) for r in rows] == o.sa[rows].tolist()


def test_index_bytes_formula():
    for x in [b"banana", b"a" * 70000, bytes(range(256)) * 300] + random_inputs(20, 3):
        for s in fm_oracle.SAMPLES:
            m = fm_oracle.FmModel(x, s)
            n, sg = len(x), m.sg
            # every array the model holds, at its GPU element size
            arrays = [m.U.size, 4 * m.S.size, 2 * m.B.size, 4 * ((n + 31) // 32), 4 * m.dir.size, 4 * m.samples.size,
                      4 * 257, 256]
            assert m.nbytes() == sum(fm_oracle.r256(a) for a in arrays) == fm_oracle.fm_bytes(n, sg, s)
            assert m.samples.size == (n + s - 1) // s


# --------------------------------------------------------------------------- entry points, no device needed

def test_arguments_are_checked_before_the_device(bwts):
    L = bwts.lib()
    text = np.frombuffer(bytearray(b"banana" * 4), dtype=np.uint8)
    pat = np.frombuffer(bytearray(b"ana"), dtype=np.uint8)
    off = np.array([0, 3], dtype=np.int64)
    bad_off = np.array([0, 2], dtype=np.int64)
    rng = np.zeros(8, dtype=np.int32)
    pos = np.zeros(8, dtype=np.int32)
    t, p, o, r, q = text.ctypes.data, pat.ctypes.data, off.ctypes.data, rng.ctypes.data, pos.ctypes.data
    fake = ctypes.c_void_p(t)       # never dereferenced before the arguments are refused
    out = ctypes.c_void_p(1)
    total = ctypes.c_long(7)
    # build: NULL pointers, lengths, sample rates
    assert L.bwts_b200_fm_build_host(None, t, 24, 32, ctypes.byref(out)) == EINVAL
    assert out.value is None                                         # *fm cleared on every failure
    assert L.bwts_b200_fm_build_host(fake, None, 24, 32, ctypes.byref(out)) == EINVAL
    assert L.bwts_b200_fm_build_host(fake, t, 24, 32, None) == EINVAL
    assert L.bwts_b200_fm_build_device(fake, t, 0, 32, ctypes.byref(out), None) == EINVAL
    assert L.bwts_b200_fm_build_device(fake, t, -1, 32, ctypes.byref(out), None) == EINVAL
    assert L.bwts_b200_fm_build_host(fake, t, 1 << 31, 32, ctypes.byref(out)) == ETOOBIG
    for s in (0, 3, 6, 2048, -4):
        assert L.bwts_b200_fm_build_host(fake, t, 24, s, ctypes.byref(out)) == EINVAL
        assert L.bwts_b200_fm_build_device(fake, t, 24, s, ctypes.byref(out), None) == EINVAL
    # the index handle: NULL is a no-op and holds no bytes
    L.bwts_b200_fm_free(None)
    assert L.bwts_b200_fm_bytes(None) == 0
    # count: NULL ctx / fm, negative sizes, NULL arrays, offsets breaking their rules, device alignment
    assert L.bwts_b200_fm_count_host(None, fake, p, 3, o, 1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, None, p, 3, o, 1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, o, -1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, p, -3, o, 1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, None, 3, o, 1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, None, 1, r, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, o, 1, None, None) == EINVAL
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, bad_off.ctypes.data, 1, r, None) == EINVAL  # off[npat] != len
    dec = np.array([0, 2, 1, 3], dtype=np.int64)
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, dec.ctypes.data, 3, r, None) == EINVAL   # decreasing
    late = np.array([1, 3], dtype=np.int64)
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, late.ctypes.data, 1, r, None) == EINVAL  # off[0] != 0
    assert L.bwts_b200_fm_count_device(fake, fake, p, 3, o + 4, 1, r, None, None) == EINVAL     # offsets 8-aligned
    assert L.bwts_b200_fm_count_device(fake, fake, p, 3, o, 1, r + 2, None, None) == EINVAL     # ranges 4-aligned
    assert L.bwts_b200_fm_count_device(fake, fake, p, 3, None, 1, r, None, None) == EINVAL
    # npat == 0 does no work and reports total 0
    assert L.bwts_b200_fm_count_host(fake, fake, None, 0, o, 0, r, ctypes.byref(total)) == 0 and total.value == 0
    total.value = 7
    assert L.bwts_b200_fm_count_device(fake, fake, None, 0, None, 0, None, ctypes.byref(total), None) == 0
    assert total.value == 0
    # locate: NULL ctx / fm, negative sizes, NULL arrays, device alignment; nrange == 0 does no work
    assert L.bwts_b200_fm_locate_host(None, fake, r, 1, q, 8, None) == EINVAL
    assert L.bwts_b200_fm_locate_host(fake, None, r, 1, q, 8, None) == EINVAL
    assert L.bwts_b200_fm_locate_host(fake, fake, r, -1, q, 8, None) == EINVAL
    assert L.bwts_b200_fm_locate_host(fake, fake, r, 1, q, -8, None) == EINVAL
    assert L.bwts_b200_fm_locate_host(fake, fake, None, 1, q, 8, None) == EINVAL
    assert L.bwts_b200_fm_locate_host(fake, fake, r, 1, None, 8, None) == EINVAL
    assert L.bwts_b200_fm_locate_device(fake, fake, r + 1, 1, q, 8, None, None) == EINVAL
    assert L.bwts_b200_fm_locate_device(fake, fake, r, 1, q + 2, 8, None, None) == EINVAL
    total.value = 7
    assert L.bwts_b200_fm_locate_host(fake, fake, None, 0, None, 0, ctypes.byref(total)) == 0 and total.value == 0


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = bwts.lib()
    text = np.frombuffer(bytearray(b"banana"), dtype=np.uint8)
    pat = np.frombuffer(bytearray(b"ana"), dtype=np.uint8)
    off = np.array([0, 3], dtype=np.int64)
    rng = np.array([1, 3], dtype=np.int32)
    pos = np.zeros(4, dtype=np.int32)
    fake = ctypes.c_void_p(text.ctypes.data)
    out = ctypes.c_void_p()
    t, p, o, r, q = text.ctypes.data, pat.ctypes.data, off.ctypes.data, rng.ctypes.data, pos.ctypes.data
    # arguments that pass every check that needs no index: no device, so ENODEV, whatever the handles
    assert L.bwts_b200_fm_build_host(fake, t, 6, 32, ctypes.byref(out)) == ENODEV
    assert L.bwts_b200_fm_build_device(fake, t, 6, 1, ctypes.byref(out), None) == ENODEV
    assert out.value is None
    assert L.bwts_b200_fm_count_host(fake, fake, p, 3, o, 1, r, None) == ENODEV
    assert L.bwts_b200_fm_count_device(fake, fake, p, 3, o, 1, r, None, None) == ENODEV
    assert L.bwts_b200_fm_locate_host(fake, fake, r, 1, q, 4, None) == ENODEV
    assert L.bwts_b200_fm_locate_device(fake, fake, r, 1, q, 4, None, None) == ENODEV
    with pytest.raises(bwts.BwtsError) as e:
        bwts.Context(0)
    assert e.value.code == ENODEV

"""The LPF array and the greedy LZ77 parse (include/bwts_b200.h, bwts_b200_lpf_* / bwts_b200_lz77_*): the C oracle
(SA-IS, a stack pass for the previous and next smaller values, direct comparison) against the brute-force definition
and the contract's known answers, the restatement of the GPU's two stages (tests/lz_oracle.py) against the oracle at
every tile width, the closed forms of a^n and the Fibonacci word, and the entry points' argument checks, which come
before any device is looked for."""
import ctypes

import numpy as np
import pytest

import helpers
import lcp_oracle
import lz_oracle

EINVAL, ETOOBIG, ENODEV = -1, -2, -3

KNOWN = [(b"banana", [0, 0, 0, 3, 2, 1], [-1, -1, -1, 1, 2, 3], [(98, 0), (97, 0), (110, 0), (1, 3)]),
         (b"abracadabra", [0, 0, 0, 1, 0, 1, 0, 4, 3, 2, 1], [-1, -1, -1, 0, -1, 3, -1, 0, 1, 2, 7],
          [(97, 0), (98, 0), (114, 0), (0, 1), (99, 0), (3, 1), (100, 0), (0, 4)]),
         (b"mississippi", [0, 0, 0, 1, 4, 3, 2, 1, 0, 1, 1], [-1, -1, -1, 2, 1, 2, 3, 4, -1, 8, 7],
          [(109, 0), (105, 0), (115, 0), (2, 1), (1, 4), (112, 0), (8, 1), (7, 1)]),
         (b"aaaa", [0, 3, 2, 1], [-1, 0, 1, 2], [(97, 0), (0, 3)]),
         (b"a", [0], [-1], [(97, 0)])]


@pytest.fixture(scope="module")
def orc():
    return lz_oracle.LzOracle()


@pytest.fixture(scope="module")
def sa_orc():
    return lcp_oracle.LcpOracle()


def random_inputs(count, seed, top=80):
    """inputs of 1..top bytes over alphabets of 1, 2, 3, 4 and 256 letters, a quarter of them periodic (u^k)"""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        sigma = int(rng.choice([1, 2, 3, 4, 256]))
        if t % 4 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 6)), dtype=np.uint8).tobytes()
            out.append((u * top)[:int(rng.integers(1, top + 1))])
        else:
            out.append(rng.integers(0, sigma, size=int(rng.integers(1, top + 1)), dtype=np.uint8).tobytes())
    return out


def test_known_answers(orc):
    for x, lpf, prev, fac in KNOWN:
        got_lpf, got_prev = orc.lpf(x)
        want_lpf, want_prev = lz_oracle.brute_lpf(x)
        assert got_lpf.tolist() == lpf == want_lpf.tolist(), x
        assert got_prev.tolist() == prev == want_prev.tolist(), x
        assert [tuple(f) for f in orc.lz77(x).tolist()] == fac, x
        assert [tuple(f) for f in lz_oracle.parse(x, got_lpf, got_prev).tolist()] == fac, x


def test_oracle_matches_brute_force(orc):
    cases = random_inputs(3000, 25)
    for n in range(1, 70, 11):
        cases.extend(helpers.families(n).values())
    for x in cases:
        lpf, prev = orc.lpf(x)
        want_lpf, want_prev = lz_oracle.brute_lpf(x)
        assert np.array_equal(lpf, want_lpf) and np.array_equal(prev, want_prev), x
        assert np.array_equal(orc.lz77(x), lz_oracle.parse(x, want_lpf, want_prev)), x


@pytest.mark.parametrize("tb", [5, 6, 7, 8, 10, 12])
def test_gpu_model_matches_oracle(orc, sa_orc, tb):
    """both GPU stages, restated at tile / chunk width 2^tb: the cross-tile rows and several parse levels"""
    cases = random_inputs(60, tb, top=700)
    for n in (1, 2, 31, 32, 33, 63, 64, 65, 1023, 1025, 4095, 4097):
        cases.extend(helpers.families(n).values())
    levels = set()
    listed = 0
    for x in cases:
        sa, lcp = sa_orc.sa_lcp(x)
        lpf, prev = orc.lpf(x)
        t = lz_oracle.tile_bits(len(x), tb)
        got_lpf, got_prev, m = lz_oracle.gpu_lpf(sa, lcp, t)
        assert np.array_equal(got_lpf, lpf) and np.array_equal(got_prev, prev), (tb, len(x), x[:16])
        got, L = lz_oracle.gpu_parse(x, lpf, prev, t)
        assert np.array_equal(got, orc.lz77(x)), (tb, len(x), x[:16])
        levels.add(L)
        listed += m
    assert listed > 0
    if tb <= 6:
        assert max(levels) >= 2   # the multi-level parse ran


def test_closed_forms(orc):
    for n in (1, 2, 3, 100, 5000):
        lpf, prev = orc.lpf(b"a" * n)
        assert lpf.tolist() == [0] + list(range(n - 1, 0, -1))
        assert prev.tolist() == [-1] + list(range(n - 1))
        want = [(97, 0)] + ([(0, n - 1)] if n > 1 else [])
        assert [tuple(f) for f in orc.lz77(b"a" * n).tolist()] == want
    for n in (1, 2, 3, 4, 7, 100, 3000, 100_000):
        f = orc.lz77(helpers.fibonacci_word(n))
        assert np.maximum(f[:, 1], 1).tolist() == lz_oracle.fibonacci_factor_lengths(n), n
    # LPF[i] >= LPF[i-1] - 1 on anything
    for x in random_inputs(300, 7, top=400):
        lpf, _ = orc.lpf(x)
        assert (lpf[1:] >= lpf[:-1] - 1).all()


# --------------------------------------------------------------------------- entry points, no device needed

def test_arguments_are_checked_before_the_device(bwts):
    L = bwts.lib()
    text = np.zeros(16, dtype=np.uint8)
    a = np.zeros(16, dtype=np.int32)
    b = np.zeros(16, dtype=np.int32)
    f = np.zeros(32, dtype=np.int32)
    t, pa, pb, pf = text.ctypes.data, a.ctypes.data, b.ctypes.data, f.ctypes.data
    z = ctypes.c_long(-7)
    zp = ctypes.byref(z)
    # a NULL context
    assert L.bwts_b200_lpf_host(None, t, 16, pa, pb) == EINVAL
    assert L.bwts_b200_lpf_device(None, t, 16, pa, pb, None) == EINVAL
    assert L.bwts_b200_lz77_host(None, t, 16, pf, 16, zp) == EINVAL
    assert L.bwts_b200_lz77_device(None, t, 16, pf, 16, zp, None) == EINVAL
    # a context that is not NULL, not dereferenced before the arguments are refused
    fake = ctypes.c_void_p(t)
    for n in (0, -3):
        assert L.bwts_b200_lpf_host(fake, t, n, pa, pb) == EINVAL
        assert L.bwts_b200_lpf_device(fake, t, n, pa, pb, None) == EINVAL
        assert L.bwts_b200_lz77_host(fake, t, n, pf, 16, zp) == EINVAL
        assert L.bwts_b200_lz77_device(fake, t, n, pf, 16, zp, None) == EINVAL
    assert L.bwts_b200_lpf_host(fake, None, 16, pa, pb) == EINVAL
    assert L.bwts_b200_lpf_host(fake, t, 16, None, pb) == EINVAL
    assert L.bwts_b200_lpf_device(fake, t, 16, pa, None, None) == EINVAL
    assert L.bwts_b200_lz77_host(fake, None, 16, pf, 16, zp) == EINVAL
    assert L.bwts_b200_lz77_host(fake, t, 16, None, 16, zp) == EINVAL
    assert L.bwts_b200_lz77_host(fake, t, 16, pf, 16, None) == EINVAL
    assert L.bwts_b200_lz77_device(fake, t, 16, pf, 16, None, None) == EINVAL
    assert L.bwts_b200_lz77_host(fake, t, 16, pf, -1, zp) == EINVAL
    assert L.bwts_b200_lz77_device(fake, t, 16, pf, -1, zp, None) == EINVAL
    assert L.bwts_b200_lpf_host(fake, t, 1 << 31, pa, pb) == ETOOBIG
    assert L.bwts_b200_lpf_device(fake, t, 1 << 31, pa, pb, None) == ETOOBIG
    assert L.bwts_b200_lz77_host(fake, t, 1 << 31, pf, 16, zp) == ETOOBIG
    assert L.bwts_b200_lz77_device(fake, t, 1 << 31, pf, 16, zp, None) == ETOOBIG
    # no two of in, lpf and prev may share a byte, nor in and factors[0 .. 2 cap)
    assert L.bwts_b200_lpf_host(fake, t, 16, t + 12, pb) == EINVAL
    assert L.bwts_b200_lpf_host(fake, t, 16, pa, t) == EINVAL
    assert L.bwts_b200_lpf_host(fake, t, 16, pa, pa + 60) == EINVAL
    assert L.bwts_b200_lpf_device(fake, t, 16, pb, pb, None) == EINVAL
    assert L.bwts_b200_lz77_host(fake, pf + 8, 16, pf, 16, zp) == EINVAL
    assert L.bwts_b200_lz77_device(fake, pf + 64, 16, pf, 16, zp, None) == EINVAL
    # device outputs must be 4-byte aligned
    assert L.bwts_b200_lpf_device(fake, t, 4, pa + 2, pb, None) == EINVAL
    assert L.bwts_b200_lpf_device(fake, t, 4, pa, pb + 1, None) == EINVAL
    assert L.bwts_b200_lz77_device(fake, t, 4, pf + 2, 4, zp, None) == EINVAL
    assert z.value == -7   # no call above ran the parse
    for v in (-1, 1, 4, 13):
        assert L.bwts_b200_tune(25, v) == EINVAL
    for v in (5, 12, 0):
        assert L.bwts_b200_tune(25, v) == 0


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    # the calls need a context, and bwts_b200_create finds no device
    assert bwts.lib().bwts_b200_create(0) is None
    with pytest.raises(bwts.BwtsError) as e:
        bwts.Context(0)
    assert e.value.code == ENODEV

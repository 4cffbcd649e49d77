"""libdivsufsort's end-of-text BWT (include/bwts_b200.h, bwts_b200_divbwt / _inverse_bw_transform): the C
oracle against the brute-force definition and the contract's known answers, its inverse (a restatement of
libdivsufsort's forward walk) against the round trip and the GPU's backward formula, and the entry points'
argument checks, which come before any device is looked for."""
import ctypes

import numpy as np
import pytest

import divbwt_oracle
import helpers

EINVAL, ETOOBIG, ENODEV = -1, -2, -3

KNOWN = [(b"banana", b"annbaa", 4), (b"abracadabra", b"ardrcaaaabb", 3), (b"mississippi", b"ipssmpissii", 5),
         (b"aaaa", b"aaaa", 4), (b"a", b"a", 1)]


@pytest.fixture(scope="module")
def bwt():
    return divbwt_oracle.DivbwtOracle()


def random_inputs(count, seed):
    """inputs of 1..300 bytes over 1..256 letters, a third of them periodic (u^k)"""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        sigma = int(rng.choice([1, 2, 3, 4, 256]))
        if t % 3 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 8)), dtype=np.uint8).tobytes()
            out.append(u * int(rng.integers(1, 40)))
        else:
            out.append(rng.integers(0, sigma, size=int(rng.integers(1, 301)), dtype=np.uint8).tobytes())
    return out


def test_known_answers(bwt):
    for x, u, primary in KNOWN:
        assert bwt.divbwt(x) == (u, primary) == divbwt_oracle.brute_divbwt(x), x
        assert bwt.inverse_bw_transform(u, primary) == x
        assert divbwt_oracle.divbwt_inverse_formula(u, primary) == x


def test_oracle_matches_brute_force_on_families(bwt):
    for n in range(1, 301, 7):
        for name, x in helpers.families(n).items():
            assert bwt.divbwt(x) == divbwt_oracle.brute_divbwt(x), (name, n)


def test_oracle_matches_brute_force_and_round_trips_on_random_inputs(bwt):
    for x in random_inputs(400, 11):
        u, primary = bwt.divbwt(x)
        assert (u, primary) == divbwt_oracle.brute_divbwt(x), x
        assert 1 <= primary <= len(x) and u[0] == x[-1]
        assert bwt.inverse_bw_transform(u, primary) == x
        assert divbwt_oracle.divbwt_inverse_formula(u, primary) == x
        # a pair made by the forward: prev_s is one n-cycle
        ps, q, seen = divbwt_oracle.divbwt_prev(u, primary), 0, 0
        while True:
            q, seen = int(ps[q]), seen + 1
            if q == 0:
                break
        assert seen == len(x), x


def test_prev_s_is_a_permutation_for_arbitrary_pairs(bwt):
    """any bytes and any primary in [1, n]: prev_s is a permutation of [0, n), so the inverse has a defined result
    (the cycle through 0, written repeatedly); libdivsufsort's walk agrees wherever it is defined"""
    rng = np.random.default_rng(5)
    agreed = 0
    for t in range(2000):
        n = int(rng.integers(1, 120))
        u = rng.integers(0, int(rng.choice([1, 2, 3, 256])), size=n, dtype=np.uint8).tobytes()
        primary = int(rng.integers(1, n + 1))
        ps = divbwt_oracle.divbwt_prev(u, primary)
        assert np.array_equal(np.sort(ps), np.arange(n)), (u, primary)
        got = divbwt_oracle.divbwt_inverse_formula(u, primary)
        cyc, q = [], 0
        while True:
            cyc.append(u[q])
            q = int(ps[q])
            if q == 0:
                break
        assert got[::-1] == bytes(cyc[j % len(cyc)] for j in range(n))
        lib = bwt.inverse_bw_transform(u, primary)
        if lib is not None:
            assert lib == got, (u, primary)
            agreed += 1
    assert agreed > 50


def test_the_oracles_inverse_refuses_pairs_its_walk_leaves(bwt):
    """(ab, 1) is no divbwt output: prev_s = [0, 1], the cycle through 0 is u[0] alone, while libdivsufsort's walk
    would step to row -1"""
    assert bwt.inverse_bw_transform(b"ab", 1) is None
    assert divbwt_oracle.divbwt_inverse_formula(b"ab", 1) == b"aa"
    assert bwt.inverse_bw_transform(b"ba", 1) == b"ab" == divbwt_oracle.divbwt_inverse_formula(b"ba", 1)


def _lib(bwts):
    return bwts.lib()


def test_arguments_are_checked_before_the_device(bwts):
    L = _lib(bwts)
    buf = np.zeros(16, dtype=np.uint8)
    b = buf.ctypes.data
    prim = ctypes.c_long(0)
    pp = ctypes.byref(prim)
    # libdivsufsort's rules for the one-call functions
    assert L.bwts_b200_divbwt(None, b, None, 16, 0) == EINVAL
    assert L.bwts_b200_divbwt(b, None, None, 16, 0) == EINVAL
    assert L.bwts_b200_divbwt(b, b, None, -1, 0) == EINVAL
    assert L.bwts_b200_divbwt(b, b, None, 0, 0) == 0
    for n, idx in ((16, -1), (16, 17), (16, 0), (0, 1), (-1, 0)):
        assert L.bwts_b200_inverse_bw_transform(b, b, None, n, idx, 0) == EINVAL, (n, idx)
    assert L.bwts_b200_inverse_bw_transform(None, b, None, 16, 1, 0) == EINVAL
    assert L.bwts_b200_inverse_bw_transform(b, None, None, 16, 1, 0) == EINVAL
    assert L.bwts_b200_inverse_bw_transform(b, b, None, 0, 0, 0) == 0
    # the context and block calls: primary in [1, len]
    for bad in (0, 17):
        assert L.bwts_b200_divbwt_inverse_host(None, b, 16, bad, b) == EINVAL
    assert L.bwts_b200_divbwt_forward_host(None, b, 16, b, pp) == EINVAL
    assert L.bwts_b200_divbwt_forward_device(None, b, 16, b, pp, None) == EINVAL
    assert L.bwts_b200_divbwt_inverse_device(None, b, 16, 1, b, None) == EINVAL
    devs = (ctypes.c_int * 1)(0)
    idx = np.array([1, 1, 1], dtype=np.int64)   # blocks of 6, 6 and 4 bytes
    assert L.bwts_b200_divbwt_forward_blocks(b, 16, 6, b, None, devs, 1) == EINVAL
    assert L.bwts_b200_divbwt_inverse_blocks(b, 16, 6, None, b, devs, 1) == EINVAL
    assert L.bwts_b200_divbwt_forward_blocks(b, 1 << 31, 1 << 31, b, idx.ctypes.data, devs, 1) == ETOOBIG
    for blk, bad in ((0, 0), (1, 7), (2, 5), (2, 0)):
        idx[:] = 1
        idx[blk] = bad
        assert L.bwts_b200_divbwt_inverse_blocks(b, 16, 6, idx.ctypes.data, b, devs, 1) == EINVAL, (blk, bad)


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = _lib(bwts)
    buf = np.frombuffer(bytearray(b"annbaa" * 3), dtype=np.uint8)
    b = buf.ctypes.data
    prim = ctypes.c_long(0)
    devs = (ctypes.c_int * 1)(0)
    idx = np.array([1, 1], dtype=np.int64)
    for n in (1, 18):   # n == 1 too: there is no host path of any length
        assert L.bwts_b200_divbwt(b, b, None, n, 0) == ENODEV
        assert L.bwts_b200_inverse_bw_transform(b, b, None, n, 1, 0) == ENODEV
    assert L.bwts_b200_divbwt_forward_blocks(b, 18, 9, b, idx.ctypes.data, devs, 1) == ENODEV
    assert L.bwts_b200_divbwt_inverse_blocks(b, 18, 9, idx.ctypes.data, b, devs, 1) == ENODEV
    for call in (lambda: bwts.divbwt_forward(b"banana"), lambda: bwts.divbwt_inverse(b"annbaa", 4),
                 lambda: bwts.divbwt_forward_blocks(b"banana" * 10, 16),
                 lambda: bwts.divbwt_inverse_blocks(b"banana" * 10, 16, [1, 1, 1, 1])):
        with pytest.raises(bwts.BwtsError) as e:
            call()
        assert e.value.code == ENODEV
    # the context calls need a context, and bwts_b200_create finds no device
    assert L.bwts_b200_create(0) is None
    assert L.bwts_b200_divbwt_forward_host(None, b, 18, b, ctypes.byref(prim)) == EINVAL

"""The classic BWT's checkers agree with each other and with the identities the contract states
(include/bwts_b200.h), and the entry points reject bad arguments before they look for a device."""
import ctypes

import numpy as np
import pytest

import bwt_oracle
import helpers

EINVAL, ETOOBIG, ENODEV = -1, -2, -3


@pytest.fixture(scope="module")
def bwt():
    return bwt_oracle.BwtOracle()


def random_inputs(count, seed):
    """short inputs over 1..256 letters, a third of them periodic (u^k)"""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        sigma = int(rng.choice([1, 2, 3, 4, 256]))
        if t % 3 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 8)), dtype=np.uint8).tobytes()
            out.append(u * int(rng.integers(1, 12)))
        else:
            out.append(rng.integers(0, sigma, size=int(rng.integers(1, 200)), dtype=np.uint8).tobytes())
    return out


def test_oracle_matches_brute_force_on_families(bwt):
    for n in range(1, 301):
        for name, x in helpers.families(n).items():
            assert bwt.forward(x) == bwt_oracle.brute_forward(x), (name, n)


def test_oracle_matches_brute_force_on_random_inputs(bwt):
    rng = np.random.default_rng(7)
    for x in random_inputs(300, 1):
        y, p = bwt.forward(x)
        assert (y, p) == bwt_oracle.brute_forward(x), x
        assert bwt.inverse(y, p) == x
        # any pair (L, idx), valid BWT or not, against the n-step walk
        idx = int(rng.integers(0, len(x)))
        z = rng.permutation(np.frombuffer(x, dtype=np.uint8)).tobytes()
        assert bwt.inverse(z, idx) == bwt_oracle.brute_inverse(z, idx)


def test_lyndon_word_gives_the_bwts_with_primary_zero(bwt, oracle):
    rng = np.random.default_rng(3)
    words = [b"a", b"ab", b"aab", b"abb", b"aabab", b"abcabd"[:5] + b"e"]
    words += [bytes([0]) + rng.integers(1, 256, size=int(m), dtype=np.uint8).tobytes() for m in rng.integers(1, 400, 50)]
    for w in words:
        assert len(oracle.lyndon_starts(w)) == 1, w
        y, p = bwt.forward(w)
        assert p == 0 and y == oracle.forward(w), w


def test_rotations_share_the_output_and_the_primary_row_holds_the_last_byte(bwt):
    for x in random_inputs(60, 2) + [b"banana", b"abab" * 5, b"a" * 9]:
        y, p = bwt.forward(x)
        assert y[p] == x[-1]
        for s in range(len(x)):
            ys, ps = bwt.forward(x[s:] + x[:s])
            assert ys == y, (x, s)
            assert ys[ps] == x[s - 1]


def test_inverse_from_every_row_is_that_rows_rotation(bwt):
    for x in random_inputs(60, 4) + [b"mississippi", b"abcabc", b"zz"]:
        y, _ = bwt.forward(x)
        for r, s in enumerate(bwt_oracle.rows(x)):
            assert bwt.inverse(y, r) == x[s:] + x[:s], (x, r)


def test_inverse_of_arbitrary_pairs_repeats_the_cycle_of_the_index(bwt):
    """a pair that is no BWT: the output is the LF cycle through idx, written repeatedly"""
    z = b"bbaaccab" * 3 + b"cab"
    lf = bwt_oracle.lf_map(z)
    for idx in range(len(z)):
        got = bwt.inverse(z, idx)
        assert got == bwt_oracle.brute_inverse(z, idx)
        cyc, q = [], idx
        while True:
            cyc.append(z[q])
            q = int(lf[q])
            if q == idx:
                break
        assert got[::-1] == bytes(cyc[j % len(cyc)] for j in range(len(z)))


def _lib(bwts):
    return bwts.lib()


def test_arguments_are_checked_before_the_device(bwts):
    L = _lib(bwts)
    buf = np.zeros(16, dtype=np.uint8)
    b = buf.ctypes.data
    prim = ctypes.c_long(0)
    pp = ctypes.byref(prim)
    assert L.bwts_b200_bwt_forward(b, 16, b, None, 0) == EINVAL
    assert L.bwts_b200_bwt_forward(b, 0, b, pp, 0) == EINVAL
    assert L.bwts_b200_bwt_forward(b, -3, b, pp, 0) == EINVAL
    assert L.bwts_b200_bwt_forward(None, 16, b, pp, 0) == EINVAL
    assert L.bwts_b200_bwt_forward(b, 1 << 31, b, pp, 0) == ETOOBIG
    for bad in (-1, 16):
        assert L.bwts_b200_bwt_inverse(b, 16, bad, b, 0) == EINVAL
        assert L.bwts_b200_bwt_inverse_host(None, b, 16, bad, b) == EINVAL
    assert L.bwts_b200_bwt_inverse(b, 0, 0, b, 0) == EINVAL
    assert L.bwts_b200_bwt_inverse(b, 1 << 31, 0, b, 0) == ETOOBIG
    assert L.bwts_b200_bwt_forward_host(None, b, 16, b, pp) == EINVAL
    assert L.bwts_b200_bwt_forward_device(None, b, 16, b, pp, None) == EINVAL
    assert L.bwts_b200_bwt_inverse_device(None, b, 16, 0, b, None) == EINVAL
    devs = (ctypes.c_int * 1)(0)
    idx = np.array([0, 0, 0], dtype=np.int64)   # blocks of 6, 6 and 4 bytes
    assert L.bwts_b200_bwt_forward_blocks(b, 16, 6, b, None, devs, 1) == EINVAL
    assert L.bwts_b200_bwt_inverse_blocks(b, 16, 6, None, b, devs, 1) == EINVAL
    for blk, bad in ((0, -1), (1, 6), (2, 4)):
        idx[:] = 0
        idx[blk] = bad
        assert L.bwts_b200_bwt_inverse_blocks(b, 16, 6, idx.ctypes.data, b, devs, 1) == EINVAL, (blk, bad)


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    for call in (lambda: bwts.bwt_forward(b"banana"), lambda: bwts.bwt_inverse(b"annbaa", 2),
                 lambda: bwts.bwt_forward_blocks(b"banana" * 10, 16),
                 lambda: bwts.bwt_inverse_blocks(b"banana" * 10, 16, [0, 0, 0, 0])):
        with pytest.raises(bwts.BwtsError) as e:
            call()
        assert e.value.code == ENODEV

"""The suffix array and LCP array (include/bwts_b200.h, bwts_b200_sa_lcp and the bwts_b200_sa_* calls): the C
oracle (SA-IS plus Kasai) against the brute-force definition and the contract's known answers, the numpy
restatement of the GPU's irreducible-LCP algorithm (tests/lcp_oracle.py) against Kasai together with the facts it
rests on, and the entry points' argument checks, which come before any device is looked for."""
import ctypes
import math

import numpy as np
import pytest

import helpers
import lcp_oracle

EINVAL, ETOOBIG, ENODEV = -1, -2, -3

KNOWN = [(b"banana", [5, 3, 1, 0, 4, 2], [0, 1, 3, 0, 0, 2]),
         (b"mississippi", [10, 7, 4, 1, 0, 9, 8, 6, 3, 5, 2], [0, 1, 1, 4, 0, 0, 1, 0, 2, 1, 3]),
         (b"abracadabra", [10, 7, 0, 3, 5, 8, 1, 4, 6, 9, 2], [0, 1, 4, 1, 1, 0, 3, 0, 0, 0, 2]),
         (b"aaaa", [3, 2, 1, 0], [0, 1, 2, 3]), (b"a", [0], [0])]


@pytest.fixture(scope="module")
def orc():
    return lcp_oracle.LcpOracle()


def random_inputs(count, seed):
    """inputs of 1..300 bytes over alphabets of 1, 2, 4 and 256 letters, a third of them periodic (u^k)"""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(count):
        sigma = int(rng.choice([1, 2, 4, 256]))
        if t % 3 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 8)), dtype=np.uint8).tobytes()
            out.append(u * int(rng.integers(1, 40)))
        else:
            out.append(rng.integers(0, sigma, size=int(rng.integers(1, 301)), dtype=np.uint8).tobytes())
    return out


def all_inputs():
    out = [x for x, _, _ in KNOWN]
    for n in range(1, 301, 13):
        out.extend(helpers.families(n).values())
    return out + random_inputs(400, 24)


def test_known_answers(orc):
    for x, sa, lcp in KNOWN:
        got_sa, got_lcp = orc.sa_lcp(x)
        want_sa, want_lcp = lcp_oracle.brute_sa_lcp(x)
        assert got_sa.tolist() == sa == want_sa.tolist(), x
        assert got_lcp.tolist() == lcp == want_lcp.tolist(), x
        assert lcp_oracle.irreducible_lcp(x, got_sa)[0].tolist() == lcp, x
    for n in (1, 2, 5, 77):   # a^n: SA[r] = n-1-r, LCP[r] = r
        sa, lcp = orc.sa_lcp(b"a" * n)
        assert sa.tolist() == list(range(n - 1, -1, -1)) and lcp.tolist() == list(range(n))


def test_kasai_matches_brute_force(orc):
    for x in all_inputs():
        sa, lcp = orc.sa_lcp(x)
        want_sa, want_lcp = lcp_oracle.brute_sa_lcp(x)
        assert np.array_equal(sa, want_sa) and np.array_equal(lcp, want_lcp), x


def test_irreducible_algorithm_matches_kasai(orc):
    for x in all_inputs():
        sa, lcp = orc.sa_lcp(x)
        got, _, _, _ = lcp_oracle.irreducible_lcp(x, sa)
        assert np.array_equal(got, lcp), x


def test_rank_order_rule_marks_exactly_the_irreducible_positions(orc):
    """step 1 of lcp.cuh (run boundaries of the BWT, rows of suffix 0, row 0) in rank order marks the positions
    i with i == 0, Phi(i) == 0, no Phi(i), or T[i-1] != T[Phi(i)-1] -- and nothing else"""
    for x in all_inputs():
        sa, _ = orc.sa_lcp(x)
        rows = lcp_oracle.irreducible_rows(x, sa)
        by_position = np.zeros(len(x), dtype=bool)
        by_position[sa] = rows
        assert np.array_equal(by_position, lcp_oracle.irreducible_positions(x, sa)), x
        assert by_position[0] and rows[0]


def test_reducible_positions_follow_their_predecessor(orc):
    for x in all_inputs():
        sa, lcp = orc.sa_lcp(x)
        plcp = np.empty(len(x), dtype=np.int64)
        plcp[sa] = lcp
        irr = lcp_oracle.irreducible_positions(x, sa)
        i = np.nonzero(~irr)[0]
        assert (i > 0).all()
        assert np.array_equal(plcp[i], plcp[i - 1] - 1), x
        # and so PLCP[i] + i never decreases: the max-scan of the irreducible values fills everything
        assert (np.diff(plcp + np.arange(len(x))) >= 0).all(), x


def test_irreducible_sum_within_2_n_log_n(orc):
    rng = np.random.default_rng(3)
    cases = all_inputs() + [helpers.fibonacci_word(5000), helpers.thue_morse(4096), b"ab" * 2000, b"a" * 3000,
                            rng.integers(0, 2, size=5000, dtype=np.uint8).tobytes()]
    for x in cases:
        sa, _ = orc.sa_lcp(x)
        _, _, _, total = lcp_oracle.irreducible_lcp(x, sa)
        n = len(x)
        assert total <= 2 * n * max(1.0, math.log2(n)), (n, total)


# --------------------------------------------------------------------------- entry points, no device needed

def test_arguments_are_checked_before_the_device(bwts):
    L = bwts.lib()
    text = np.zeros(16, dtype=np.uint8)
    sa = np.zeros(16, dtype=np.int32)
    lcp = np.zeros(16, dtype=np.int32)
    t, s, c = text.ctypes.data, sa.ctypes.data, lcp.ctypes.data
    # the one-call form: libdivsufsort's rules
    assert L.bwts_b200_sa_lcp(None, s, c, 16, 0) == EINVAL
    assert L.bwts_b200_sa_lcp(t, None, c, 16, 0) == EINVAL
    assert L.bwts_b200_sa_lcp(t, s, None, 16, 0) == EINVAL
    assert L.bwts_b200_sa_lcp(t, s, c, -1, 0) == EINVAL
    assert L.bwts_b200_sa_lcp(t, s, c, 0, 0) == 0
    assert L.bwts_b200_sa_lcp(t, t, c, 16, 0) == EINVAL              # aliasing
    assert L.bwts_b200_sa_lcp(t, s, s + 8, 16, 0) == EINVAL
    assert L.bwts_b200_divsufsort(None, s, 16, 0) == EINVAL
    assert L.bwts_b200_divsufsort(t, s, 0, 0) == 0
    # the context calls: a NULL context, NULL buffers, len <= 0, len > MAX_LEN
    assert L.bwts_b200_sa_host(None, t, 16, s) == EINVAL
    assert L.bwts_b200_sa_lcp_host(None, t, 16, s, c) == EINVAL
    assert L.bwts_b200_sa_device(None, t, 16, s, None) == EINVAL
    assert L.bwts_b200_sa_lcp_device(None, t, 16, s, c, None) == EINVAL
    # a context that is not NULL, not dereferenced before the arguments are refused
    fake = ctypes.c_void_p(t)
    for n in (0, -3):
        assert L.bwts_b200_sa_host(fake, t, n, s) == EINVAL
        assert L.bwts_b200_sa_lcp_host(fake, t, n, s, c) == EINVAL
        assert L.bwts_b200_sa_device(fake, t, n, s, None) == EINVAL
        assert L.bwts_b200_sa_lcp_device(fake, t, n, s, c, None) == EINVAL
    assert L.bwts_b200_sa_host(fake, None, 16, s) == EINVAL
    assert L.bwts_b200_sa_host(fake, t, 16, None) == EINVAL
    assert L.bwts_b200_sa_lcp_host(fake, t, 16, s, None) == EINVAL
    assert L.bwts_b200_sa_lcp_device(fake, t, 16, None, c, None) == EINVAL
    assert L.bwts_b200_sa_lcp_device(fake, t, 16, s, None, None) == EINVAL
    assert L.bwts_b200_sa_host(fake, t, 1 << 31, s) == ETOOBIG
    assert L.bwts_b200_sa_lcp_host(fake, t, 1 << 31, s, c) == ETOOBIG
    assert L.bwts_b200_sa_device(fake, t, 1 << 31, s, None) == ETOOBIG
    assert L.bwts_b200_sa_lcp_device(fake, t, 1 << 31, s, c, None) == ETOOBIG
    # no two of in, sa and lcp may share a byte
    assert L.bwts_b200_sa_host(fake, t, 16, t + 12) == EINVAL
    assert L.bwts_b200_sa_lcp_host(fake, t, 16, s, s + 60) == EINVAL
    assert L.bwts_b200_sa_lcp_host(fake, t, 16, s, t) == EINVAL
    assert L.bwts_b200_sa_lcp_device(fake, t, 16, s, s, None) == EINVAL
    assert L.bwts_b200_sa_device(fake, s + 60, 16, s, None) == EINVAL
    # device outputs must be 4-byte aligned
    assert L.bwts_b200_sa_device(fake, t, 4, s + 2, None) == EINVAL
    assert L.bwts_b200_sa_lcp_device(fake, t, 4, s, c + 1, None) == EINVAL
    assert L.bwts_b200_tune(24, 3) == EINVAL and L.bwts_b200_tune(24, -1) == EINVAL
    assert L.bwts_b200_tune(24, 0) == 0


def test_no_cpu_fallback(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = bwts.lib()
    text = np.frombuffer(bytearray(b"banana" * 3), dtype=np.uint8)
    sa = np.zeros(18, dtype=np.int32)
    lcp = np.zeros(18, dtype=np.int32)
    for n in (1, 18):   # n == 1 too: there is no host path of any length
        assert L.bwts_b200_sa_lcp(text.ctypes.data, sa.ctypes.data, lcp.ctypes.data, n, 0) == ENODEV
        assert L.bwts_b200_divsufsort(text.ctypes.data, sa.ctypes.data, n, 0) == ENODEV
    for call in (lambda: bwts.suffix_array_lcp(b"banana"), lambda: bwts.suffix_array(b"banana")):
        with pytest.raises(bwts.BwtsError) as e:
            call()
        assert e.value.code == ENODEV
    # the context and device calls need a context, and bwts_b200_create finds no device
    assert L.bwts_b200_create(0) is None
    with pytest.raises(bwts.BwtsError) as e:
        bwts.Context(0)
    assert e.value.code == ENODEV

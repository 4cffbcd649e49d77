"""LZ77 decoding (include/bwts_b200.h, bwts_b200_lz77_decode_*) on the CPU: the C oracle (oracle/lz_decode_oracle.c)
inverts the parse oracle and agrees with a pure-Python decode on non-greedy lists; the restatement of the GPU's chunk
and global rounds (tests/lz_decode_oracle.py) matches it at every chunk width within the stated round bound; and the
entry points' argument checks come before any device is looked for."""
import ctypes

import numpy as np
import pytest

import helpers
import lz_decode_oracle as lzd
import lz_oracle

EINVAL, ETOOBIG, ENODEV = -1, -2, -3

KNOWN = [(b"banana", [(98, 0), (97, 0), (110, 0), (1, 3)]),
         (b"abracadabra", [(97, 0), (98, 0), (114, 0), (0, 1), (99, 0), (3, 1), (100, 0), (0, 4)]),
         (b"mississippi", [(109, 0), (105, 0), (115, 0), (2, 1), (1, 4), (112, 0), (8, 1), (7, 1)]),
         (b"aaaa", [(97, 0), (0, 3)])]


@pytest.fixture(scope="module")
def dec():
    return lzd.LzDecodeOracle()


@pytest.fixture(scope="module")
def orc():
    return lz_oracle.LzOracle()


def test_known_answers(dec):
    for x, f in KNOWN:
        assert dec.lz77_decode(f, len(x)) == x == lzd.py_decode(f, len(x))
    for n in (1, 2, 3, 100, 4097):
        assert dec.lz77_decode(lzd.a_n(n), n) == b"a" * n


def test_inverts_the_parse(dec, orc):
    rng = np.random.default_rng(11)
    for t in range(3000):
        sigma = int(rng.choice([1, 2, 3, 4, 256]))
        n = int(rng.integers(1, 81))
        if t % 4 == 0:
            u = rng.integers(0, sigma, size=int(rng.integers(1, 6)), dtype=np.uint8).tobytes()
            x = (u * n)[:n]
        else:
            x = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
        assert dec.lz77_decode(orc.lz77(x), n) == x, x


def non_greedy_lists():
    out = []
    for seed, n in enumerate((1, 2, 7, 100, 1000, 5000)):
        out.append((f"lit_far_{n}", lzd.random_factors(n, seed, lit=0.5), n))
        out.append((f"near_{n}", lzd.random_factors(n, seed + 100, near=8), n))
        out.append((f"single_chain_{n}", lzd.random_factors(n, seed + 200, max_len=1, lit=0.01, near=1), n))
    for period in (1, 2, 3, 17, 64):
        out.append((f"period_{period}", lzd.random_factors(3000, period, max_len=200, lit=0.05, period=period), 3000))
    out.append(("strided_33", lzd.strided_chain(3000, 33), 3000))
    out.append(("fibonacci", lz_oracle.LzOracle().lz77(helpers.fibonacci_word(3000)), 3000))
    return out


def test_non_greedy_lists(dec):
    for name, f, n in non_greedy_lists():
        got = dec.lz77_decode(f, n)
        assert got is not None and got == lzd.py_decode(f, n), name


@pytest.mark.parametrize("tb", [5, 6, 8, 10, 12])
def test_gpu_model_matches_oracle(dec, tb):
    """widths 32 .. 4096: the chunk rounds leave every word resolved or pointing into an earlier chunk, and the
    global rounds stay within ceil(log2 ceil(n / W)) + 1"""
    cases = non_greedy_lists() + [("a_n", lzd.a_n(20_000), 20_000), ("strided_W", lzd.strided_chain(20_000, 1 << tb),
                                                                       20_000)]
    for name, f, n in cases:
        got, rounds, _ = lzd.gpu_decode(f, n, tb)
        assert got == dec.lz77_decode(f, n), (name, tb)
        assert rounds <= lzd.round_bound(n, tb), (name, tb, rounds)


def test_bad_lists_are_rejected(dec):
    n = 6
    good = [[98, 0], [97, 0], [110, 0], [1, 3]]
    assert dec.lz77_decode(good, n) == b"banana"
    for bad in ([[256, 0], [97, 0], [110, 0], [1, 3]],    # literal byte above 255
                [[-1, 0], [97, 0], [110, 0], [1, 3]],     # and below 0
                [[98, 0], [97, 0], [110, 0], [1, -3]],    # negative length
                [[98, 0], [0, 1], [110, 0], [3, 3]],      # source at p_k
                [[98, 0], [97, 0], [110, 0], [-1, 3]],    # negative source
                [[98, 0], [97, 0], [110, 0], [1, 2]],     # the lengths sum to 5
                [[98, 0], [97, 0], [110, 0], [1, 4]]):    # and to 7
        assert dec.lz77_decode(bad, n) is None, bad


# --------------------------------------------------------------------------- entry points, no device needed

def test_arguments_are_checked_before_the_device(bwts):
    L = bwts.lib()
    f = np.array([[98, 0], [97, 0], [110, 0], [1, 3]], dtype=np.int32)
    out = np.zeros(64, dtype=np.uint8)
    pf, po = f.ctypes.data, out.ctypes.data
    assert L.bwts_b200_lz77_decode_host(None, pf, 4, po, 6) == EINVAL
    assert L.bwts_b200_lz77_decode_device(None, pf, 4, po, 6, None) == EINVAL
    fake = ctypes.c_void_p(po)   # not dereferenced before the arguments are refused
    host = lambda *a: L.bwts_b200_lz77_decode_host(fake, *a)          # noqa: E731
    device = lambda *a: L.bwts_b200_lz77_decode_device(fake, *a, None)  # noqa: E731
    for call in (host, device):
        assert call(None, 4, po, 6) == EINVAL
        assert call(pf, 4, None, 6) == EINVAL
        for z in (0, -1):
            assert call(pf, z, po, 6) == EINVAL
        for n in (0, -6):
            assert call(pf, 4, po, n) == EINVAL
        assert call(pf, 7, po, 6) == EINVAL              # z > len
        assert call(pf, 4, po, 1 << 31) == ETOOBIG
        assert call(pf, 4, pf + 31, 6) == EINVAL         # out on the last byte of the pairs
        assert call(pf, 4, pf - 5, 6) == EINVAL          # on the first
    assert device(pf + 2, 1, po, 6) == EINVAL            # device pairs must be 4-byte aligned
    for v in (-1, 4, 13):
        assert L.bwts_b200_tune(25, v) == EINVAL


def test_no_device(bwts):
    if bwts.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L = bwts.lib()
    f = np.array([[98, 0], [97, 0], [110, 0], [1, 3]], dtype=np.int32)
    out = np.full(6, 7, dtype=np.uint8)
    fake = ctypes.c_void_p(out.ctypes.data + 4096)
    assert L.bwts_b200_lz77_decode_host(fake, f.ctypes.data, 4, out.ctypes.data, 6) == ENODEV
    assert L.bwts_b200_lz77_decode_device(fake, f.ctypes.data, 4, out.ctypes.data + 1, 5, None) == ENODEV
    assert (out == 7).all()

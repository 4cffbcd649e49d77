"""GPU tests of libdivsufsort's end-of-text BWT (bwts_b200_divbwt, bwts_b200_inverse_bw_transform and the
bwts_b200_divbwt_* context and block calls): output bytes and primary against the CPU oracle
(oracle/divbwt_oracle.c) under every forward tune key that acts in linear mode, the inverse against the oracle on
pairs the forward made and against the contract's formula on arbitrary pairs under every inverse path, host /
device / block entry points, aliasing, and full sizes up to 2^31 - 1 bytes.  Run on a B200."""
import ctypes
import json
from pathlib import Path

import numpy as np
import pytest

import divbwt_oracle
import helpers
from test_gpu_dispatch_edges import cycle_labels, equal_factors, lyndon_word
from test_gpu_parity import GOLDEN, golden_input

pytestmark = pytest.mark.gpu

DIVBWT_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "divbwt_fullsize.json").read_text())
TUNE_KEYS = (0, 1, 2, 3, 6, 7, 8, 9, 12, 13, 14, 15, 16, 18, 20, 21, 22, 23)


@pytest.fixture(scope="module")
def bwt():
    return divbwt_oracle.DivbwtOracle()


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def tuned(bwts):
    for k in TUNE_KEYS:
        bwts.tune(k, 0)
    yield
    for k in TUNE_KEYS:
        bwts.tune(k, 0)


def forward_checked(ctx, x, want):
    y, p = ctx.divbwt_forward_host(x)
    assert (y, p) == want, (len(x), bytes(x[:32]))
    st = ctx.stats()
    assert (st["factors"], st["longest_factor"], st["lyndon_fallback"], st["direction"]) == (1, len(x), 0, 0)
    return y, p


# --------------------------------------------------------------------------- forward

def forward_cases(gen):
    """name -> input: families at tile edges, periodic inputs, runs of one byte, generated text and DNA"""
    out = {}
    for n in (1, 2, 3, 255, 257, 2049, 4095, 4609, 8193, 65537):
        out.update({f"{k}_{n}": x for k, x in helpers.families(n).items()})
    for u, k in ((b"ba", 50), (b"cab", 1400), (b"abcabd", 3), (b"\x00\xff", 2048), (b"abacabb", 4097)):
        out[f"({u.hex()})^{k}"] = u * k
    for n in (1, 2, 4097, 100_003):
        out[f"all_{n}"] = b"a" * n
    out["all_00"] = b"\x00" * 5000
    out["all_ff"] = b"\xff" * 5000
    out["text1m"] = gen.make("text", 41, (1 << 20) + 7)
    out["dna1m"] = gen.make("dna", 42, 1 << 20)
    return out


@pytest.fixture(scope="module")
def fwd_wants(bwt, gen):
    return {name: (x, bwt.divbwt(x)) for name, x in forward_cases(gen).items()}


def test_known_answers(ctx, bwts):
    for x, want in ((b"banana", (b"annbaa", 4)), (b"abracadabra", (b"ardrcaaaabb", 3)),
                    (b"mississippi", (b"ipssmpissii", 5)), (b"aaaa", (b"aaaa", 4)), (b"a", (b"a", 1))):
        assert ctx.divbwt_forward_host(x) == want
        assert bwts.divbwt_forward(x) == want
        assert ctx.divbwt_inverse_host(*want) == x
        assert bwts.divbwt_inverse(*want) == x


def test_forward_golden_vector_inputs(ctx, bwt, gen):
    for v in GOLDEN:
        x = golden_input(v, gen)
        forward_checked(ctx, x, bwt.divbwt(x))


def test_forward_families_periodic_and_runs(ctx, fwd_wants):
    for name, (x, want) in fwd_wants.items():
        forward_checked(ctx, x, want)


# (key, value) of every forward tune key that acts on the linear sort and the byte emit
FWD_SETTINGS = [(2, 1), (2, 3), (3, 1), (6, 16), (7, 2), (7, 4), (8, 1), (9, 1), (9, 2), (9, 3), (14, 1), (14, 2),
                (18, 1), (20, 1), (21, 1), (22, 1), (23, 16)]


@pytest.fixture(scope="module")
def tune_wants(bwt, gen):
    cases = {f"{k}_{n}": x for n in (257, 4609) for k, x in helpers.families(n).items()}
    cases.update({"u7^4097": equal_factors(b"abacabb", 4097), "(cab)^1400": b"cab" * 1400, "all_70k": b"a" * 70_000,
                  "text1m": gen.make("text", 41, (1 << 20) + 7), "copies": b"xyz" * 9 + gen.make("dna", 43, 300_000) * 3})
    cases["text17m"] = gen.make("text", 44, (17 << 20) + 3)   # more than one 16 MiB emit window
    return {name: (x, bwt.divbwt(x)) for name, x in cases.items()}


@pytest.mark.parametrize("key,value", FWD_SETTINGS, ids=[f"tune{k}={v}" for k, v in FWD_SETTINGS])
def test_forward_under_tune_keys(bwts, ctx, tune_wants, key, value):
    bwts.tune(key, value)
    for name, (x, want) in tune_wants.items():
        if name == "text17m" and key not in (9, 23):
            continue
        y, p = forward_checked(ctx, x, want)
        assert ctx.divbwt_inverse_host(y, p) == x, name


# --------------------------------------------------------------------------- inverse

def inverse_pairs(bwt, oracle, gen):
    """(name, U, primary, want, cycles of prev_s): pairs the forward made (want = the oracle's libdivsufsort walk) and arbitrary
    pairs (want = the contract's formula), with the primary at both ends and in between"""
    rng = np.random.default_rng(600)
    out = []
    for name, x in (("text", gen.make("text", 51, 200_003)), ("dna", gen.make("dna", 52, 300_000)),
                    ("all_a", b"a" * 65_537), ("(cab)^1400", b"cab" * 1400), ("fib", helpers.fibonacci_word(50_000))):
        y, p = bwt.divbwt(x)
        assert bwt.inverse_bw_transform(y, p) == x
        out.append((name, y, p, x, 1))
    arbitrary = {f"equal{L}x{g}": oracle.forward(equal_factors(lyndon_word(L, rng), g))
                 for L, g in ((1, 3000), (32, 2000), (129, 400))}
    for sigma, n in ((256, 100_000), (4, 77_777), (2, 50_001)):
        arbitrary[f"bytes{sigma}"] = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
    for name, y in arbitrary.items():
        n = len(y)
        for p in (1, n, int(rng.integers(1, n + 1))):
            cycles = len(np.unique(cycle_labels(divbwt_oracle.divbwt_prev(y, p))))
            out.append((name, y, p, divbwt_oracle.divbwt_inverse_formula(y, p), cycles))
    return out


@pytest.fixture(scope="module")
def inv_cases(bwt, oracle, gen):
    return inverse_pairs(bwt, oracle, gen)


# (tune 12 two read-only walks, 13 sublists per warp, 15 mark mode, 1 splitter shift)
INV_SETTINGS = [(0, 0, 0, 0), (1, 0, 0, 0), (0, 1, 0, 29), (0, 0, 1, 0), (0, 0, 2, 0), (1, 0, 0, 29), (0, 5, 2, 29)]


@pytest.mark.parametrize("setting", INV_SETTINGS, ids=[f"t12={a},t13={b},t15={c},t1={d}" for a, b, c, d in INV_SETTINGS])
def test_inverse_of_valid_and_arbitrary_pairs(bwts, ctx, inv_cases, setting):
    two_walk, q, marks, shift = setting
    bwts.tune(12, two_walk)
    bwts.tune(13, q)
    bwts.tune(15, marks)
    bwts.tune(1, shift)
    for name, y, p, want, cycles in inv_cases:
        assert ctx.divbwt_inverse_host(y, p) == want, (name, p)
        st = ctx.stats()
        assert st["factors"] == cycles, (name, p)
        assert st["direction"] == 1 and st["phases"]["Place bytes"] >= 0


def test_inverse_restarts(bwts, ctx, bwt, oracle):
    """with primary 1, prev_s is the LF map itself: one splitter per 4096 elements leaves 138 of the 150 cycles of
    300 without one, and a step budget of 1024 makes the first attempts give up (12.4 M fallback steps); primary
    12345 leaves two cycles of 15 M steps without a splitter"""
    rng = np.random.default_rng(77)
    y = oracle.forward(equal_factors(lyndon_word(300, rng), 150))
    bwts.tune(1, 20)
    bwts.tune(16, 1024)
    for p in (1, 12345):
        assert ctx.divbwt_inverse_host(y, p) == divbwt_oracle.divbwt_inverse_formula(y, p), p
        assert ctx.stats()["inverse_attempts"] > 1, p
    x = b"abracadabra" * 3000   # the same context and settings on a pair the forward made: no restart needed
    yx, px = bwt.divbwt(x)
    assert ctx.divbwt_inverse_host(yx, px) == x
    assert ctx.stats()["inverse_attempts"] == 1


def test_round_trip_of_forward_cases(ctx, fwd_wants):
    for name, (x, (y, p)) in fwd_wants.items():
        assert ctx.divbwt_inverse_host(y, p) == x, name
        assert ctx.stats()["factors"] == 1, name


def test_shortest_inputs(bwts, ctx, bwt):
    for x in (b"\x00", b"a", b"\xff", b"aa", b"ab", b"ba", b"\x00\xff", b"\xff\x00"):
        y, p = bwt.divbwt(x)
        assert ctx.divbwt_forward_host(x) == (y, p) == bwts.divbwt_forward(x), x
        assert ctx.divbwt_inverse_host(y, p) == x == bwts.divbwt_inverse(y, p), x
    for u in (b"ab", b"ba", b"aa"):   # every pair of length 2, whether the forward made it or not
        for p in (1, 2):
            assert ctx.divbwt_inverse_host(u, p) == divbwt_oracle.divbwt_inverse_formula(u, p), (u, p)


# --------------------------------------------------------------------------- entry points

def test_one_call_entry_points_and_aliasing(bwts, bwt):
    L = bwts.lib()
    x = b"abracadabra" * 1000
    want_y, want_p = bwt.divbwt(x)
    buf = np.frombuffer(bytearray(x), dtype=np.uint8)
    scratch = np.full(len(x), 7, dtype=np.int32)
    # U == T, and libdivsufsort's A accepted and left alone
    assert L.bwts_b200_divbwt(buf.ctypes.data, buf.ctypes.data, scratch.ctypes.data, len(x), 0) == want_p
    assert buf.tobytes() == want_y and (scratch == 7).all()
    assert L.bwts_b200_inverse_bw_transform(buf.ctypes.data, buf.ctypes.data, None, len(x), want_p, 0) == 0
    assert buf.tobytes() == x
    assert bwts.divbwt_forward(b"") == (b"", 0)
    assert bwts.divbwt_inverse(b"", 0) == b""
    with pytest.raises(bwts.BwtsError) as e:
        bwts.divbwt_inverse(want_y, 0)
    assert e.value.code == -1
    with pytest.raises(bwts.BwtsError) as e:
        bwts.divbwt_inverse(want_y, len(want_y) + 1)
    assert e.value.code == -1
    with pytest.raises(bwts.BwtsError):
        bwts.divbwt_forward(x, device=999)


def test_device_resident_calls_at_unaligned_offsets_on_a_caller_stream(ctx, bwt, gen):
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("dna", 45, 300_001)
    want_y, want_p = bwt.divbwt(x)
    big = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    out = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream(dev)
    for off in (1, 3, 7, 8, 13, 15):
        view = big[off:off + len(x)]
        view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
        torch.cuda.synchronize()
        o = out[(off * 7) % 16:(off * 7) % 16 + len(x)]
        p = ctx.divbwt_forward_device(view.data_ptr(), len(x), o.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert p == want_p and bytes(o.cpu().numpy()) == want_y, off
        view.copy_(o)
        torch.cuda.synchronize()
        ctx.divbwt_inverse_device(view.data_ptr(), len(x), p, o.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert bytes(o.cpu().numpy()) == x, off


def test_workspace_is_that_of_the_bwts(bwts, gen):
    x = gen.make("dna", 46, 3_000_000)
    with bwts.Context(0) as a, bwts.Context(0) as b:
        a.forward_host(x)
        a.inverse_host(x)
        y, p = b.divbwt_forward_host(x)
        b.divbwt_inverse_host(y, p)
        assert b.stats()["arena_bytes"] <= a.stats()["arena_bytes"]


def test_blocks_ragged_tail_one_and_all_devices(bwts, bwt, gen):
    x = gen.make("text", 47, 3_000_000) + b"a" * 500_000 + gen.make("dna", 48, 1_234_567)
    b = 700_001
    want = [bwt.divbwt(x[o:o + b]) for o in range(0, len(x), b)]
    for devs in ([0], list(range(bwts.device_count()))):
        y, prim = bwts.divbwt_forward_blocks(x, b, devs)
        assert y == b"".join(w[0] for w in want) and prim == [w[1] for w in want], devs
        assert bwts.divbwt_inverse_blocks(y, b, prim, devs) == x, devs


def test_blocks_reject_a_bad_index_before_any_work(bwts, bwt):
    """the last block is 3 bytes long: its index 4 is refused, and no block's output is written"""
    L = bwts.lib()
    x = b"mississippi" * 3   # 33 bytes: blocks of 10, 10, 10 and 3
    y, prim = bwts.divbwt_forward_blocks(x, 10)
    devs = (ctypes.c_int * 1)(0)
    out = np.full(len(x), 0x5A, dtype=np.uint8)
    src = np.frombuffer(y, dtype=np.uint8)
    for bad in ([prim[0], prim[1], prim[2], 4], [0, prim[1], prim[2], prim[3]], [prim[0], 11, prim[2], prim[3]]):
        idx = np.array(bad, dtype=np.int64)
        assert L.bwts_b200_divbwt_inverse_blocks(src.ctypes.data, len(x), 10, idx.ctypes.data, out.ctypes.data,
                                                 devs, 1) == -1, bad
        assert (out == 0x5A).all(), bad
    assert bwts.divbwt_inverse_blocks(y, 10, prim) == x


# --------------------------------------------------------------------------- full size

@pytest.mark.parametrize("name", ["C2", "C3", "C3F"])
def test_full_size_against_the_oracle(bwts, gen, name):
    gold = DIVBWT_FULLSIZE[name]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        y, p = c.divbwt_forward_host(x)
        assert p == gold["primary"] and helpers.sha256(y) == gold["divbwt_sha256"]
        assert c.divbwt_inverse_host(y, p) == x
        assert c.stats()["factors"] == 1


def full_size_properties(c, x):
    xa = np.frombuffer(x, np.uint8)
    y, p = c.divbwt_forward_host(x)
    ya = np.frombuffer(y, np.uint8)
    assert 1 <= p <= len(x) and ya[0] == xa[-1]
    assert np.array_equal(np.bincount(xa, minlength=256), np.bincount(ya, minlength=256))
    back = c.divbwt_inverse_host(y, p)
    assert np.array_equal(np.frombuffer(back, np.uint8), xa)


def test_full_size_c4(bwts, gen):
    with bwts.Context(0) as c:
        full_size_properties(c, gen.make("dna", 4, 1 << 30))


def test_largest_length(bwts, gen):
    import torch
    n = (1 << 31) - 1
    if torch.cuda.mem_get_info(0)[0] < 73 * n + (1 << 28):
        pytest.skip("needs 157 GB of free device memory")
    with bwts.Context(0) as c:
        full_size_properties(c, gen.make("dna", 7, n))

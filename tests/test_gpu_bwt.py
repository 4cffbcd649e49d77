"""GPU tests of the classic Burrows-Wheeler transform with a primary index (bwts_b200_bwt_*): output bytes
and primary index against the CPU oracle (oracle/bwt_oracle.c) under every forward tune key the suite
forces, the inverse against the oracle's LF walk on arbitrary (L, idx) pairs under every inverse path,
host / device / block entry points, and full sizes up to 2^31 - 1 bytes.  Run on a B200."""
import json
import os
from pathlib import Path

import numpy as np
import pytest

import bwt_oracle
import helpers
from test_gpu_dispatch_edges import (cycle_labels, default_shift, equal_factors, factorization, lyndon_word,
                                     splitter_mask, steps_to_splitter)
from test_gpu_parity import GOLDEN, golden_input

pytestmark = pytest.mark.gpu

BWT_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "bwt_fullsize.json").read_text())
TUNE_KEYS = (0, 1, 2, 3, 6, 7, 8, 9, 12, 13, 14, 15, 16, 18, 20, 21, 22, 23)


@pytest.fixture(scope="module")
def bwt():
    return bwt_oracle.BwtOracle()


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
    y, p = ctx.bwt_forward_host(x)
    assert (y, p) == want, (len(x), bytes(x[:32]))
    st = ctx.stats()
    assert (st["factors"], st["longest_factor"], st["lyndon_fallback"], st["direction"]) == (1, len(x), 0, 0)
    return y, p


# --------------------------------------------------------------------------- forward

def lyndon_like_inputs():
    """name -> input whose classic BWT equals its BWTS with primary 0: Lyndon words, u^k and w w for a
    Lyndon word u / w, and runs of one byte"""
    rng = np.random.default_rng(21)
    out = {}
    for m in (1, 2, 31, 4096, 70_000):
        out[f"lyndon{m}"] = lyndon_word(m, rng)
    for m, k in ((1, 5000), (3, 1000), (7, 4097), (64, 300), (1000, 7)):
        out[f"u{m}^{k}"] = equal_factors(lyndon_word(m, rng), k)
    w = lyndon_word(30_000, rng)
    out["ww"] = w + w
    for n in (1, 2, 4097, 100_003):
        out[f"all_{n}"] = b"\x61" * n
    out["all_ff"] = b"\xff" * 5000
    return out


def forward_cases(gen):
    """name -> input: families at tile edges, periodic inputs that are not powers of a Lyndon word, every
    rotation of a short text, generated text"""
    out = {}
    for n in (1, 2, 3, 255, 257, 2049, 4095, 4609, 8193, 65537):
        out.update({f"{k}_{n}": x for k, x in helpers.families(n).items()})
    for u, k in ((b"ba", 50), (b"cab", 1400), (b"abcabd", 3), (b"\x00\xff", 2048)):
        out[f"({u.hex()})^{k}"] = u * k
    t = b"mississippi banana abracadabra"
    out.update({f"rot{s}": t[s:] + t[:s] for s in range(len(t))})
    out["text1m"] = gen.make("text", 41, (1 << 20) + 7)
    out["dna1m"] = gen.make("dna", 42, 1 << 20)
    return out


@pytest.fixture(scope="module")
def fwd_wants(bwt, gen):
    cases = forward_cases(gen)
    return {name: (x, bwt.forward(x)) for name, x in cases.items()}


def test_forward_golden_vector_inputs(ctx, bwt, gen):
    for v in GOLDEN:
        x = golden_input(v, gen)
        forward_checked(ctx, x, bwt.forward(x))


def test_forward_families_periodic_and_rotations(ctx, fwd_wants):
    for name, (x, want) in fwd_wants.items():
        forward_checked(ctx, x, want)
    rot = {fwd_wants[f"rot{s}"][1][0] for s in range(30)}
    assert len(rot) == 1, "every rotation of a text has the same BWT"


def test_forward_of_lyndon_words_and_their_powers_is_the_bwts(ctx, bwt):
    for name, x in lyndon_like_inputs().items():
        y, p = forward_checked(ctx, x, bwt.forward(x))
        assert p == 0 and y == ctx.forward_host(x), name


# (key, value) of every forward tune key the suite forces elsewhere
FWD_SETTINGS = [(2, 1), (2, 3), (3, 1), (6, 16), (7, 2), (7, 4), (8, 1), (9, 1), (9, 2), (9, 3), (14, 1), (14, 2),
                (18, 1), (20, 1), (21, 1), (22, 1), (23, 16)]


@pytest.fixture(scope="module")
def tune_wants(bwt, gen):
    cases = {f"{k}_{n}": x for n in (257, 4609) for k, x in helpers.families(n).items()}
    cases.update({"u7^4097": equal_factors(b"abacabb", 4097), "(cab)^1400": b"cab" * 1400, "all_70k": b"a" * 70_000,
                  "text1m": gen.make("text", 41, (1 << 20) + 7), "copies": b"xyz" * 9 + gen.make("dna", 43, 300_000) * 3})
    cases["text17m"] = gen.make("text", 44, (17 << 20) + 3)   # more than one 16 MiB emit window
    return {name: (x, bwt.forward(x)) for name, x in cases.items()}


@pytest.mark.parametrize("key,value", FWD_SETTINGS, ids=[f"tune{k}={v}" for k, v in FWD_SETTINGS])
def test_forward_under_tune_keys(bwts, ctx, tune_wants, key, value):
    bwts.tune(key, value)
    for name, (x, want) in tune_wants.items():
        if name == "text17m" and key not in (9, 23):
            continue
        forward_checked(ctx, x, want)


# --------------------------------------------------------------------------- inverse

def inverse_inputs_with_indices(bwt, oracle, shift):
    """(name, L, idx, what) with idx at random rows, in a cycle without splitters, and far from the next
    splitter (splitters of the first attempt with splitter shift `shift`)"""
    rng = np.random.default_rng(500 + shift)
    pairs = {}
    for L, g in ((1, 3000), (32, 2000), (129, 400)):
        pairs[f"equal{L}x{g}"] = oracle.forward(equal_factors(lyndon_word(L, rng), g))
    pairs["mixed"] = oracle.forward(factorization(rng.choice(np.array([1, 2, 31, 64, 65, 300, 4097]), size=300).tolist(), 501))
    for sigma, n in ((256, 100_000), (4, 77_777), (2, 50_001)):
        pairs[f"bytes{sigma}"] = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
    pairs["all_a"] = b"a" * 65_537
    out = []
    for name, y in pairs.items():
        n = len(y)
        lf = bwt_oracle.lf_map(y)
        lab = cycle_labels(lf)
        spl = splitter_mask(n, shift)
        has = np.bincount(lab, weights=spl, minlength=n) > 0
        for r in rng.integers(0, n, size=3):
            out.append((name, y, int(r), "random"))
        lone = np.flatnonzero(~has[lab])
        if len(lone):
            out.append((name, y, int(lone[len(lone) // 2]), "cycle without splitters"))
        far = np.where(has[lab], steps_to_splitter(lf, spl), -1)
        out.append((name, y, int(np.argmax(far)), f"{int(far.max())} steps to a splitter"))
    return out


@pytest.fixture(scope="module")
def inv_cases(bwt, oracle):
    cases = {}
    for shift in (default_shift(1 << 20), 29):
        cases[shift] = [(name, y, idx, what, bwt.inverse(y, idx)) for name, y, idx, what in
                        inverse_inputs_with_indices(bwt, oracle, shift)]
    return cases


# (tune 12 two read-only walks, 13 sublists per warp, 15 mark mode, 1 splitter shift)
INV_SETTINGS = [(0, 0, 0, 0), (1, 0, 0, 0), (0, 1, 0, 29), (0, 0, 1, 0), (0, 0, 2, 0), (1, 0, 0, 29), (0, 5, 2, 29)]


@pytest.mark.parametrize("setting", INV_SETTINGS, ids=[f"t12={a},t13={b},t15={c},t1={d}" for a, b, c, d in INV_SETTINGS])
def test_inverse_of_arbitrary_pairs(bwts, ctx, inv_cases, setting):
    two_walk, q, marks, shift = setting
    bwts.tune(12, two_walk)
    bwts.tune(13, q)
    bwts.tune(15, marks)
    bwts.tune(1, shift)
    seen = set()
    for name, y, idx, what, want in inv_cases[shift or default_shift(1 << 20)]:
        assert ctx.bwt_inverse_host(y, idx) == want, (name, idx, what)
        st = ctx.stats()
        if name not in seen:
            seen.add(name)
            assert st["factors"] == len(np.unique(cycle_labels(bwt_oracle.lf_map(y)))), name
        assert st["direction"] == 1 and st["phases"]["Place bytes"] >= 0


def test_inverse_restarts_with_the_scratch_layout(bwts, ctx, bwt, oracle):
    """one splitter per 4096 elements leaves 138 of 150 cycles of 300 without one, and a fallback step budget
    of 1024 makes the attempt give up on them (11586 units of 1024 steps, inverse_prediction); each attempt
    lays out its own scratch copy and the successful one rotates it into the output"""
    rng = np.random.default_rng(77)
    y = oracle.forward(equal_factors(lyndon_word(300, rng), 150))
    bwts.tune(1, 20)
    bwts.tune(16, 1024)
    for idx in (0, 12345, len(y) - 1):
        assert ctx.bwt_inverse_host(y, idx) == bwt.inverse(y, idx), idx
        assert ctx.stats()["inverse_attempts"] > 1


def test_round_trip_of_forward_cases(ctx, fwd_wants):
    for name, (x, (y, p)) in fwd_wants.items():
        assert ctx.bwt_inverse_host(y, p) == x, name


def test_inverse_from_every_row_of_a_short_text(ctx, bwt):
    x = b"abracadabra, mississippi"
    y, _ = bwt.forward(x)
    for r, s in enumerate(bwt_oracle.rows(x)):
        assert ctx.bwt_inverse_host(y, r) == x[s:] + x[:s], r


# --------------------------------------------------------------------------- entry points

def test_one_call_entry_points(bwts, bwt):
    x = b"abracadabra" * 1000
    y, p = bwts.bwt_forward(x)
    assert (y, p) == bwt.forward(x)
    assert bwts.bwt_inverse(y, p) == x
    with pytest.raises(bwts.BwtsError) as e:
        bwts.bwt_inverse(y, len(y))
    assert e.value.code == -1
    with pytest.raises(bwts.BwtsError):
        bwts.bwt_forward(x, device=999)


def test_device_resident_calls_at_unaligned_offsets_on_a_caller_stream(ctx, bwt, gen):
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("text", 45, 300_001)
    want_y, want_p = bwt.forward(x)
    big = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    out = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream(dev)
    for off in range(1, 16):
        view = big[off:off + len(x)]
        view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
        torch.cuda.synchronize()
        o = out[(off * 7) % 16:(off * 7) % 16 + len(x)]
        p = ctx.bwt_forward_device(view.data_ptr(), len(x), o.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert p == want_p and bytes(o.cpu().numpy()) == want_y, off
        view.copy_(o)
        torch.cuda.synchronize()
        ctx.bwt_inverse_device(view.data_ptr(), len(x), p, o.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert bytes(o.cpu().numpy()) == x, off


def test_workspace_is_that_of_the_bwts(bwts, gen):
    x = gen.make("dna", 46, 3_000_000)
    with bwts.Context(0) as a, bwts.Context(0) as b:
        a.forward_host(x)
        a.inverse_host(x)
        y, p = b.bwt_forward_host(x)
        b.bwt_inverse_host(y, p)
        assert b.stats()["arena_bytes"] <= a.stats()["arena_bytes"]


def test_blocks_pageable_one_and_all_devices(bwts, bwt, gen):
    x = gen.make("text", 47, 3_000_000) + b"a" * 500_000 + gen.make("dna", 48, 1_234_567)
    b = 700_001
    want = [bwt.forward(x[o:o + b]) for o in range(0, len(x), b)]
    for devs in ([0], list(range(bwts.device_count()))):
        y, prim = bwts.bwt_forward_blocks(x, b, devs)
        assert y == b"".join(w[0] for w in want) and prim == [w[1] for w in want], devs
        assert bwts.bwt_inverse_blocks(y, b, prim, devs) == x, devs
    with bwts.Context(0) as c:   # each block equals the one-call result
        for o, (wy, wp) in zip(range(0, len(x), b), want):
            assert c.bwt_forward_host(x[o:o + b]) == (wy, wp)


def test_blocks_pinned_buffers(bwts, bwt, gen):
    import torch
    x = gen.make("text", 49, 5_000_000)
    b = 700_001
    src = torch.frombuffer(bytearray(x), dtype=torch.uint8).pin_memory()
    mid = torch.empty_like(src).pin_memory()
    back = torch.empty_like(src).pin_memory()
    prim = np.full(-(-len(x) // b), -1, dtype=np.int64)
    bwts.bwt_blocks_ptr(0, src.data_ptr(), len(x), b, mid.data_ptr(), prim, devices=[0])
    want = [bwt.forward(x[o:o + b]) for o in range(0, len(x), b)]
    assert bytes(mid.numpy()) == b"".join(w[0] for w in want)
    assert prim.tolist() == [w[1] for w in want]
    bwts.bwt_blocks_ptr(1, mid.data_ptr(), len(x), b, back.data_ptr(), prim, devices=[0])
    assert bytes(back.numpy()) == x


# --------------------------------------------------------------------------- full size

@pytest.mark.parametrize("name", ["C2", "C3"])
def test_full_size_against_the_oracle(bwts, gen, name):
    gold = BWT_FULLSIZE[name]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        y, p = c.bwt_forward_host(x)
        assert p == gold["primary"] and helpers.sha256(y) == gold["bwt_sha256"]
        assert c.bwt_inverse_host(y, p) == x


def full_size_properties(c, x):
    xa = np.frombuffer(x, np.uint8)
    y, p = c.bwt_forward_host(x)
    ya = np.frombuffer(y, np.uint8)
    assert ya[p] == xa[-1]
    assert np.array_equal(np.bincount(xa, minlength=256), np.bincount(ya, minlength=256))
    back = c.bwt_inverse_host(y, p)
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

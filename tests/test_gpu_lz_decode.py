"""GPU tests of LZ77 decoding (bwts_b200_lz77_decode_*): the known answers; decode(lz77(x)) == x on families around
32, 4096 and 4096^2 bytes at the smallest and the default chunk width (tune key 25); non-greedy lists against the
CPU oracle (oracle/lz_decode_oracle.c), a^n and the Fibonacci word at chunk-edge sizes, strided chains that cross a
chunk at every hop, a self-overlapping factor over many chunks; the round bound after every call; every argument and
content rule, with the output left untouched; the device form with torch tensors on a caller stream; one context
across parse, decode and BWTS; the parses of C2, C3 and C3F against their input hashes, C4 and 2^31 - 1 bytes
compared on the device.  Run on a B200."""
import ctypes
import gc
import json
from pathlib import Path

import numpy as np
import pytest

import helpers
import lz_decode_oracle as lzd
import lz_oracle

pytestmark = pytest.mark.gpu

EINVAL = -1
LZ_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "lz_fullsize.json").read_text())
KNOWN = [(b"banana", [[98, 0], [97, 0], [110, 0], [1, 3]]),
         (b"abracadabra", [[97, 0], [98, 0], [114, 0], [0, 1], [99, 0], [3, 1], [100, 0], [0, 4]]),
         (b"mississippi", [[109, 0], [105, 0], [115, 0], [2, 1], [1, 4], [112, 0], [8, 1], [7, 1]]),
         (b"aaaa", [[97, 0], [0, 3]])]
BIG = (1 << 31) - 1


@pytest.fixture(scope="module")
def dec():
    return lzd.LzDecodeOracle()


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def tuned(bwts):
    bwts.tune(25, 0)
    yield
    bwts.tune(25, 0)


def decoded(ctx, f, n, tb=12):
    """the host form, then the statistics every call must show"""
    f = np.ascontiguousarray(f, dtype=np.int32).reshape(-1, 2)
    out = ctx.lz77_decode_host(f, n)
    st = ctx.stats()
    assert (st["direction"], st["len"], st["factors"]) == (1, n, len(f))
    assert st["rounds"] <= lzd.round_bound(n, tb), (n, tb, st["rounds"])
    return out


def test_known_answers(ctx):
    for x, f in KNOWN:
        assert decoded(ctx, f, len(x)) == x
    for n in (1, 2, 3, 4096, 4097, 100_000):
        assert decoded(ctx, lzd.a_n(n), n) == b"a" * n


def family_cases():
    out = {}
    for n in (31, 32, 33, 4095, 4096, 4097):
        out.update({f"{k}_{n}": x for k, x in helpers.families(n).items()})
    n = 4096 * 4096 + 1
    fam = helpers.families(n)
    out.update({f"{k}_{n}": fam[k] for k in ("all_a", "descending", "fibonacci", "de_bruijn", "random4", "random256",
                                              "runs")})
    return out


@pytest.mark.parametrize("tb", [5, 0], ids=["chunk32", "chunk4096"])
def test_round_trip_families(bwts, ctx, tb):
    bwts.tune(25, tb)
    for name, x in family_cases().items():
        assert decoded(ctx, ctx.lz77_host(x), len(x), tb or 12) == x, name


def non_greedy_cases(W):
    fib = lz_oracle.LzOracle()
    out = []
    for n in (W - 1, W, W + 1, W * W - 1, W * W + 1):
        out.append((f"a_{n}", lzd.a_n(n), n))
        out.append((f"fib_{n}", fib.lz77(helpers.fibonacci_word(n)), n))
    n = 3 * min(W * W, 1 << 20) + 7
    for seed, kw in enumerate(({"lit": 0.5}, {"near": 8}, {"max_len": 1, "lit": 0.01, "near": 1},
                               {"max_len": 300, "lit": 0.05, "period": 17}, {"max_len": 4 * W, "lit": 0.01})):
        out.append((f"random_{seed}", lzd.random_factors(n, seed, **kw), n))
    for stride in (W - 1, W, W + 1, 2 * W + 3):
        out.append((f"strided_{stride}", lzd.strided_chain(n, stride, stride), n))
    # one factor overlapping itself across every chunk after the first
    head = lzd.random_factors(100, 5, lit=1.0)
    out.append(("overlap", np.concatenate([head, [[63, n - 100]]]).astype(np.int32), n))
    return out


@pytest.mark.parametrize("tb", [5, 0], ids=["chunk32", "chunk4096"])
def test_non_greedy_lists_against_the_oracle(bwts, ctx, dec, tb):
    bwts.tune(25, tb)
    W = 1 << (tb or 12)
    for name, f, n in non_greedy_cases(W):
        want = dec.lz77_decode(f, n)
        assert want is not None, name
        assert decoded(ctx, f, n, tb or 12) == want, name


def test_rounds_reach_their_bound(bwts, ctx):
    """a^n: every chunk waits on the one before, so chunk c resolves in the round r with 2^r >= c + 1: ceil(log2 nc)
    rounds in all, fewer only where in-place reads run ahead"""
    bwts.tune(25, 5)
    n = 32 * 1025
    assert decoded(ctx, lzd.a_n(n), n, 5) == b"a" * n
    st = ctx.stats()
    assert 1 <= st["rounds"] <= 11 and st["live_sum"] >= n - 32
    assert {"inv_scan", "inv_walk", "inv_jump", "inv_place"} <= set(st["classes"])


def bad_lists():
    """(name, factors, len): each breaks one content rule; the three-factor cases wrap a u32 sum to len"""
    big = BIG
    return [("byte_256", [[256, 0], [97, 0], [110, 0], [1, 3]], 6),
            ("byte_neg", [[98, 0], [-1, 0], [110, 0], [1, 3]], 6),
            ("len_neg", [[98, 0], [97, 0], [110, 0], [1, -3]], 6),
            ("src_at_p", [[98, 0], [97, 0], [110, 0], [3, 3]], 6),
            ("src_neg", [[98, 0], [97, 0], [110, 0], [-2, 3]], 6),
            ("first_copy", [[0, 1], [97, 0]], 2),
            ("sum_short", [[98, 0], [97, 0], [110, 0], [1, 2]], 6),
            ("sum_long", [[98, 0], [97, 0], [110, 0], [1, 4]], 6),
            ("three_big", [[97, 0], [0, big], [0, big], [0, big]], 16),
            ("wrap_to_len", [[97, 0], [0, big], [0, big], [0, 11]], 10)]


def test_bad_lists_leave_the_output_untouched(bwts, ctx):
    import torch
    L = bwts.lib()
    dev = torch.device("cuda:0")
    for name, f, n in bad_lists():
        f = np.array(f, dtype=np.int32)
        h = np.full(n, 0x5A, dtype=np.uint8)
        assert L.bwts_b200_lz77_decode_host(ctx._h, f.ctypes.data, len(f), h.ctypes.data, n) == EINVAL, name
        assert (h == 0x5A).all(), name
        d_f = torch.from_numpy(f).to(dev)
        d_o = torch.full((n + 1,), 0x5A, dtype=torch.uint8, device=dev)
        assert L.bwts_b200_lz77_decode_device(ctx._h, d_f.data_ptr(), len(f), d_o.data_ptr() + 1, n, None) == EINVAL
        torch.cuda.synchronize()
        assert bool((d_o == 0x5A).all()), name
    # argument rules on real buffers
    f = torch.tensor(KNOWN[0][1], dtype=torch.int32, device=dev)
    buf = torch.full((256,), 0x5A, dtype=torch.uint8, device=dev)
    p = buf.data_ptr()
    assert L.bwts_b200_lz77_decode_device(ctx._h, f.data_ptr(), 4, p, 3, None) == EINVAL            # z > len
    buf[:32].copy_(f.view(torch.uint8).reshape(-1))
    assert L.bwts_b200_lz77_decode_device(ctx._h, p, 4, p + 31, 6, None) == EINVAL                  # overlap
    assert L.bwts_b200_lz77_decode_device(ctx._h, p + 64 + 2, 4, p + 128, 6, None) == EINVAL        # misaligned
    torch.cuda.synchronize()
    assert bool((buf[32:] == 0x5A).all())
    # just apart is fine, and the context still decodes
    assert L.bwts_b200_lz77_decode_device(ctx._h, p, 4, p + 32, 6, None) == 0
    torch.cuda.synchronize()
    assert bytes(buf[32:38].cpu().numpy()) == b"banana"
    assert decoded(ctx, KNOWN[1][1], 11) == b"abracadabra"


def test_device_form_on_a_caller_stream(ctx, dec, gen):
    import torch
    dev = torch.device("cuda:0")
    s = torch.cuda.Stream(dev)
    for n, f in ((6, np.array(KNOWN[0][1], dtype=np.int32)), (4097, ctx.lz77_host(gen.make("text", 91, 4097))),
                 (300_001, lzd.random_factors(300_001, 92, near=1000))):
        want = dec.lz77_decode(f, n)
        raw = torch.zeros(8 * len(f) + 8, dtype=torch.uint8, device=dev)
        raw[4:4 + 8 * len(f)].copy_(torch.from_numpy(f.view(np.uint8).reshape(-1)))   # pairs at a 4-byte offset
        out = torch.full((n + 64,), 0x5A, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            ctx.lz77_decode_device(raw.data_ptr() + 4, len(f), n, out.data_ptr() + 3, s.cuda_stream)
        s.synchronize()
        got = out.cpu().numpy()
        assert got[3:3 + n].tobytes() == want
        assert (got[:3] == 0x5A).all() and (got[3 + n:] == 0x5A).all()
        st = ctx.stats()
        assert st["factors"] == len(f) and st["rounds"] <= lzd.round_bound(n, 12)


def test_one_context_across_transforms(ctx, gen, oracle):
    for x in (gen.make("text", 93, 100_000), b"banana" * 999, gen.make("dna", 94, 300_007), b"zz"):
        f = ctx.lz77_host(x)
        assert np.array_equal(f, lz_oracle.LzOracle().lz77(x))
        assert decoded(ctx, f, len(x)) == x
        assert ctx.forward_host(x) == oracle.forward(x)
        assert decoded(ctx, f, len(x)) == x
        y = x[: max(1, len(x) // 3)]
        assert decoded(ctx, ctx.lz77_host(y), len(y)) == y


def release_device_memory():
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def parse_and_decode(bwts, x, n, cap=None):
    """lz77_device then lz77_decode_device on one context -> (decoded tensor, z, rounds)"""
    import torch
    dev = x.device
    fac = torch.empty((cap or n // 2 + 64, 2), dtype=torch.int32, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    with bwts.Context(0) as c:
        z = c.lz77_device(x.data_ptr(), n, fac.data_ptr(), fac.shape[0])
        c.lz77_decode_device(fac.data_ptr(), z, n, out.data_ptr())
        torch.cuda.synchronize()
        rounds = c.stats()["rounds"]
    del fac
    return out, z, rounds


@pytest.mark.parametrize("name", ["C2", "C3", "C3F"])
def test_full_size_round_trip(bwts, gen, name):
    import torch
    gold = LZ_FULLSIZE[name]
    x = torch.frombuffer(bytearray(gen.make(gold["kind"], gold["seed"], gold["n"])), dtype=torch.uint8).to("cuda:0")
    out, z, rounds = parse_and_decode(bwts, x, gold["n"])
    assert z == gold["z"] and rounds <= lzd.round_bound(gold["n"], 12)
    assert helpers.sha256(out.cpu().numpy()) == gold["input_sha256"]
    del x, out
    release_device_memory()


def test_full_size_c4(bwts, gen):
    import torch
    release_device_memory()
    n = 1 << 30
    x = torch.frombuffer(bytearray(gen.make("dna", 4, n)), dtype=torch.uint8).to("cuda:0")
    out, z, rounds = parse_and_decode(bwts, x, n)
    assert rounds <= lzd.round_bound(n, 12)
    assert torch.equal(out, x)
    del x, out
    release_device_memory()


def test_largest_length(bwts, gen):
    """2^31 - 1 bytes: (97,0) (0,n-1) against a^n, and the Fibonacci word's own parse against the word"""
    import torch
    n = BIG
    release_device_memory()
    if torch.cuda.mem_get_info(0)[0] < 74 * n + (1 << 28):
        pytest.skip("needs 160 GB of free device memory")
    dev = torch.device("cuda:0")
    f = torch.tensor(lzd.a_n(n), device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    with bwts.Context(0) as c:
        c.lz77_decode_device(f.data_ptr(), 2, n, out.data_ptr())
        torch.cuda.synchronize()
        st = c.stats()
    assert st["rounds"] <= lzd.round_bound(n, 12) and st["factors"] == 2
    assert bool((out == 97).all())
    del out, f
    release_device_memory()
    x = torch.frombuffer(bytearray(gen.make("fibonacci", 0, n)), dtype=torch.uint8).to(dev)
    out, z, rounds = parse_and_decode(bwts, x, n, cap=128)
    assert z == len(lz_oracle.fibonacci_factor_lengths(n)) and rounds <= lzd.round_bound(n, 12)
    assert torch.equal(out, x)
    del x, out
    release_device_memory()

"""GPU tests of FM-index extract (bwts_b200_fm_extract_*): ranges of the text read back from its index and compared
with slices of the text -- the known answers, the shortest inputs, sizes at the checkpoint layout's edges on DNA,
text and all-byte alphabets with ranges on and around segment edges, the $ row at chosen rows, the one-byte
alphabet, count -> locate -> extract of every hit, malformed ranges and a total above cap in both forms, the device
form on a caller stream with the output at an odd address, lifetimes and threads, interleaving with the other
calls, the arena of a build, a total above 2^32 bytes, and the whole text at 64 MiB, 1 GiB and 2^31 - 1 bytes.
Run on a B200."""
import gc
import threading

import numpy as np
import pytest

import fm_oracle
import helpers
from test_fm_extract_oracle import KNOWN
from test_gpu_fm import pattern_set

pytestmark = pytest.mark.gpu
EINVAL = -1


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


def _release():
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def edge_ranges(n, s, rng, count=64):
    """ranges from and to multiples of s and +-1 from them, empty ranges, the last byte, [0, n), random ones"""
    pts = sorted({v for k in rng.integers(0, n // s + 1, size=count).tolist() for v in (k * s - 1, k * s, k * s + 1)
                  if 0 <= v <= n} | {0, 1, n - 1, n})
    pick = rng.choice(pts, size=(count, 2))
    a, b = pick.min(axis=1).tolist(), pick.max(axis=1).tolist()
    a += [0, n - 1, n, 0, n // 2]
    b += [n, n, n, 0, n // 2]
    r = rng.integers(0, n, size=count)
    a += r.tolist()
    b += np.minimum(r + rng.integers(1, 3 * s + 2, size=count), n).tolist()
    return a, b


def check(ctx, x, samples, a, b):
    want = b"".join(x[i:j] for i, j in zip(a, b))
    for s in samples:
        with ctx.fm_build_host(x, s) as fm:
            out, off = ctx.fm_extract_host(fm, a, b)
            assert out.tobytes() == want, (len(x), s)
            assert off[-1] == len(want)
            st = ctx.stats()
            assert st["direction"] == 1 and st["len"] == len(x)
            if want:
                assert {"inv_scan", "inv_walk"} <= set(st["classes"])


def test_known_answers(ctx):
    for s in fm_oracle.SAMPLES:
        for text in (b"banana", b"mississippi", b"aaaa"):
            cases = [(a, b, w) for x, a, b, w in KNOWN if x == text]
            with ctx.fm_build_host(text, s) as fm:
                out, off = ctx.fm_extract_host(fm, [c[0] for c in cases], [c[1] for c in cases])
                assert [out[off[k]:off[k + 1]].tobytes() for k in range(len(cases))] == [c[2] for c in cases]


def test_shortest_inputs(ctx):
    for x in (b"\x00", b"\xff", b"a", b"ab", b"ba", b"aa", b"\x00\xff", b"\xff\x00", b"abc"):
        n = len(x)
        a, b = zip(*[(i, j) for i in range(n + 1) for j in range(i, n + 1)])
        check(ctx, x, fm_oracle.SAMPLES, a, b)


@pytest.mark.parametrize("n", [255, 256, 257, 65535, 65536, 65537, 200_003])
def test_sizes_at_the_layout_edges(ctx, gen, n):
    rng = np.random.default_rng(n)
    inputs = [gen.make("dna", 4, n), gen.make("text", 2, n), rng.integers(0, 256, size=n, dtype=np.uint8).tobytes()]
    for x in inputs:
        for s in (1, 32, 1024) if n < 70_000 else (32,):
            check(ctx, x, (s,), *edge_ranges(n, s, rng))


@pytest.mark.parametrize("k", [0, 1, 255, 256, 65535, 65536])
def test_dollar_row_at_chosen_rows(ctx, k):
    rng = np.random.default_rng(k)
    for m in (0, 1, 300):
        x = fm_oracle.dollar_row_text(k, m)
        for s in (1, 2, 32, 1024) if k < 300 else (2, 1024):
            check(ctx, x, (s,), *edge_ranges(len(x), s, rng, 16))


def test_one_byte_alphabet(ctx):
    rng = np.random.default_rng(3)
    for n in (1000, 65537):
        check(ctx, b"a" * n, fm_oracle.SAMPLES, *edge_ranges(n, 32, rng, 16))


def test_count_locate_extract_returns_every_hit(ctx, gen):
    x = gen.make("text", 6, 300_001)
    pats = [p for p in pattern_set(x, 4, count=30, longest=200) if p]
    with ctx.fm_build_host(x, 16) as fm:
        lo, hi = ctx.fm_count_host(fm, pats)
        pos, off = ctx.fm_locate_host(fm, lo, hi)
        assert len(pos) > 0
        owner = np.repeat(np.arange(len(pats)), np.diff(off))
        m = np.array([len(p) for p in pats], dtype=np.int64)[owner]
        out, eoff = ctx.fm_extract_host(fm, pos, pos + m)
        assert np.array_equal(np.diff(eoff), m)
        assert out.tobytes() == b"".join(pats[k] for k in owner)


def test_bad_ranges_and_cap(bwts, ctx):
    import torch
    dev = torch.device("cuda:0")
    x = b"mississippi" * 100
    n = len(x)
    with ctx.fm_build_host(x, 4) as fm:
        out = torch.full((64,), 0x5a, dtype=torch.uint8, device=dev)
        host = np.full(64, 0x5a, dtype=np.uint8)
        for bad in ([5, 4], [-1, 2], [0, n + 1], [n + 1, n + 1]):
            r = torch.tensor([0, 1] + bad, dtype=torch.int32, device=dev)
            with pytest.raises(bwts.BwtsError) as e:
                ctx.fm_extract_device(fm, r.data_ptr(), 2, out.data_ptr(), 64)
            assert e.value.code == EINVAL, bad
            rh = np.array([0, 1] + bad, dtype=np.int32)
            assert bwts.lib().bwts_b200_fm_extract_host(ctx._h, fm.handle, rh.ctypes.data, 2, host.ctypes.data, 64,
                                                        None) == EINVAL, bad
        r = torch.tensor([0, 40, 100, 130], dtype=torch.int32, device=dev)    # 70 bytes, cap 64
        with pytest.raises(bwts.BwtsError) as e:
            ctx.fm_extract_device(fm, r.data_ptr(), 2, out.data_ptr(), 64)
        assert e.value.code == EINVAL
        rh = r.cpu().numpy()
        assert bwts.lib().bwts_b200_fm_extract_host(ctx._h, fm.handle, rh.ctypes.data, 2, host.ctypes.data, 64,
                                                    None) == EINVAL
        assert (out.cpu() == 0x5a).all() and (host == 0x5a).all()        # nothing written
        for lo, hi in (([5], [4]), ([-1], [2]), ([0], [n + 1])):
            with pytest.raises(bwts.BwtsError) as e:
                ctx.fm_extract_host(fm, lo, hi)
            assert e.value.code == EINVAL


def test_device_form_torch_stream_odd_address(ctx, gen):
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("dna", 5, 300_001)
    n = len(x)
    rng = np.random.default_rng(8)
    a, b = edge_ranges(n, 8, rng, 200)
    want = b"".join(x[i:j] for i, j in zip(a, b))
    s = torch.cuda.Stream(dev)
    d_rng = torch.tensor(np.stack([a, b], 1).reshape(-1), dtype=torch.int32, device=dev)
    big = torch.full((len(want) + 16,), 7, dtype=torch.uint8, device=dev)
    view = big[3:3 + len(want) + 5]                              # output at an odd address
    tx = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        fm = ctx.fm_build_device(tx.data_ptr(), n, 8, stream=s.cuda_stream)
        total = ctx.fm_extract_device(fm, d_rng.data_ptr(), len(a), view.data_ptr(), len(want) + 5,
                                      stream=s.cuda_stream)
        s.synchronize()
    assert total == len(want)
    got = big.cpu().numpy()
    assert got[3:3 + total].tobytes() == want
    assert (got[:3] == 7).all() and (got[3 + total:] == 7).all()
    fm.close()


def test_lifetimes_and_threads(bwts, gen):
    x = gen.make("text", 9, 100_000)
    rng = np.random.default_rng(10)
    a, b = edge_ranges(len(x), 16, rng, 100)
    want = b"".join(x[i:j] for i, j in zip(a, b))
    with bwts.Context(0) as c:
        fm = c.fm_build_host(x, 16)
    errors = []

    def worker():
        try:
            with bwts.Context(0) as c:
                for _ in range(5):
                    assert c.fm_extract_host(fm, a, b)[0].tobytes() == want
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    threads = [threading.Thread(target=worker) for _ in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    fm.close()


def test_interleaved_with_other_calls(bwts, oracle, gen):
    x = gen.make("text", 11, 200_000)
    o = fm_oracle.FmOracle(x)
    pats = pattern_set(x, 12)
    rng = np.random.default_rng(13)
    a, b = edge_ranges(len(x), 32, rng, 50)
    want = b"".join(x[i:j] for i, j in zip(a, b))
    with bwts.Context(0) as c, c.fm_build_host(x, 32) as fm:
        for _ in range(2):
            lo, hi = c.fm_count_host(fm, pats)
            assert np.array_equal(lo, o.count_many(pats)[0])
            assert c.fm_extract_host(fm, a, b)[0].tobytes() == want
            assert np.array_equal(c.fm_locate_host(fm, lo, hi)[0], o.locate(lo, hi))
            y = c.forward_host(x[:50_000])
            assert y == oracle.forward(x[:50_000])
            assert c.fm_extract_host(fm, [0], [len(x)])[0].tobytes() == x


def test_build_arena_is_enough(bwts, gen):
    x = gen.make("dna", 14, 1 << 20)
    with bwts.Context(0) as c, c.fm_build_host(x, 1) as fm:
        before = c.stats()["arena_bytes"]
        out, _ = c.fm_extract_host(fm, [0, 5], [len(x), 1000])
        assert out.tobytes() == x + x[5:1000]
        assert c.stats()["arena_bytes"] == before


def test_total_above_four_gib(bwts, gen):
    """257 copies of [0, n) over 16 MiB: 4.2 GB of output, offsets past 2^32, compared on the device"""
    import torch
    n = 16 << 20
    dev = torch.device("cuda:0")
    tx = torch.frombuffer(bytearray(gen.make("text", 15, n)), dtype=torch.uint8).to(dev)
    copies = 257
    d_rng = torch.tensor([0, n] * copies, dtype=torch.int32, device=dev)
    out = torch.empty(copies * n, dtype=torch.uint8, device=dev)
    try:
        with bwts.Context(0) as c, c.fm_build_device(tx.data_ptr(), n, 32) as fm:
            assert c.fm_extract_device(fm, d_rng.data_ptr(), copies, out.data_ptr(), copies * n) == copies * n
        assert torch.equal(out.view(copies, n), tx.expand(copies, n))
    finally:
        del out, tx
        _release()


@pytest.mark.parametrize("name,kind,seed,n", [("C2", "text", 2, 64 << 20), ("C4", "dna", 4, 1 << 30)])
def test_whole_text_at_full_size(bwts, gen, name, kind, seed, n):
    """the self-index property: extract [0, n) equals the input"""
    import torch
    dev = torch.device("cuda:0")
    tx = torch.frombuffer(bytearray(gen.make(kind, seed, n)), dtype=torch.uint8).to(dev)
    d_rng = torch.tensor([0, n], dtype=torch.int32, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    try:
        for s in (32, 1024):
            with bwts.Context(0) as c:
                fm = c.fm_build_device(tx.data_ptr(), n, s)
            with fm, bwts.Context(0) as c:
                out.fill_(0)
                assert c.fm_extract_device(fm, d_rng.data_ptr(), 1, out.data_ptr(), n) == n
                assert torch.equal(out, tx), (name, s)
    finally:
        del out, tx
        _release()


def closed_form(i):
    """T[i] = 'ACGT'[a 32-bit hash of i]: the expected bytes of any range without the text on the host"""
    v = (i.astype(np.uint64) * np.uint64(0x9E3779B1)) & np.uint64(0xffffffff)
    v ^= v >> np.uint64(15)
    v = (v * np.uint64(0x2C1B3C6D)) & np.uint64(0xffffffff)
    v ^= v >> np.uint64(12)
    return np.frombuffer(b"ACGT", dtype=np.uint8)[((v >> np.uint64(8)) & np.uint64(3)).astype(np.int64)]


def test_largest_length(bwts):
    """2^31 - 1 bytes of a closed-form text: sampled ranges, the end of the text included.  The build's context is
    destroyed before the extract, so that its workspace is free again."""
    import torch
    n = (1 << 31) - 1
    _release()
    if torch.cuda.mem_get_info(0)[0] < 80 * n + (1 << 28):
        pytest.skip("needs ~170 GB of free device memory")
    dev = torch.device("cuda:0")
    tx = torch.empty(n, dtype=torch.uint8, device=dev)
    step = 1 << 26
    for p in range(0, n, step):
        q = min(p + step, n)
        tx[p:q] = torch.from_numpy(closed_form(np.arange(p, q, dtype=np.int64))).to(dev)
    with bwts.Context(0) as c:
        fm = c.fm_build_device(tx.data_ptr(), n, 32)
    del tx
    _release()
    rng = np.random.default_rng(31)
    starts = np.concatenate([rng.integers(0, n - 100, size=4000), [0, n - 100, n - 1, n]])
    ends = np.minimum(starts + rng.integers(0, 100, size=len(starts)), n)
    ends[-3:] = n
    try:
        with bwts.Context(0) as c:
            out, off = c.fm_extract_host(fm, starts, ends)
        want = np.concatenate([closed_form(np.arange(a, b, dtype=np.int64)) for a, b in zip(starts, ends)])
        assert np.array_equal(out, want)
    finally:
        fm.close()
        _release()

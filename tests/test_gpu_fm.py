"""GPU tests of the FM-index (bwts_b200_fm_*): count and locate against the CPU oracle (the suffix array of
oracle/lcp_oracle.c plus bisection, tests/fm_oracle.py) on the known answers, the shortest inputs, sizes at the
checkpoint layout's edges, the $ row at chosen rows, one-byte / DNA / text / all-byte alphabets, hits, near misses,
absent bytes, patterns longer than the text and the empty pattern, at every sample rate; host and device calls
(torch tensors, a caller stream, patterns at an odd address); lifetimes (two indexes, an index outliving its context,
two threads querying one index); malformed device arrays; golden hashes at 64 and 256 MiB; and properties checked on
the GPU at 1 GiB and 2^31 - 1 bytes.  Run on a B200."""
import gc
import json
import threading
from pathlib import Path

import numpy as np
import pytest

import fm_oracle
import helpers

pytestmark = pytest.mark.gpu

FM_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "fm_fullsize.json").read_text())
EINVAL = -1


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


def pattern_set(x, seed, count=40, longest=1000):
    """hits (substrings of 1..longest bytes), near misses (one byte changed at the start, middle or end), random
    strings, absent bytes first / middle / last, longer than the text, and the empty pattern"""
    rng = np.random.default_rng(seed)
    n = len(x)
    present = set(x)
    absent = next((b for b in (0x00, 0xff, 0x7f, ord("z")) if b not in present), None)
    out = [b"", x, x + x[:1], bytes(x[:1]) * (n + 1)]
    for k in range(count):
        a = int(rng.integers(0, n))
        length = int(rng.integers(1, longest + 1)) if k % 2 else int(rng.integers(1, 17))
        p = x[a:a + length]
        out.append(p)
        q = bytearray(p)
        q[[0, len(q) // 2, len(q) - 1][k % 3]] ^= int(rng.integers(1, 256))
        out.append(bytes(q))
        out.append(rng.integers(0, 256, size=int(rng.integers(1, 9)), dtype=np.uint8).tobytes())
        if absent is not None and len(p) >= 3:
            for j in (0, len(p) // 2, len(p) - 1):
                r = bytearray(p)
                r[j] = absent
                out.append(bytes(r))
    return out


def check(ctx, x, samples=(32,), pats=None, seed=0, o=None):
    o = o or fm_oracle.FmOracle(x)
    pats = pattern_set(x, seed) if pats is None else pats
    want_lo, want_hi = o.count_many(pats)
    for s in samples:
        with ctx.fm_build_host(x, s) as fm:
            st = ctx.stats()
            assert (st["direction"], st["factors"], st["longest_factor"]) == (0, 1, len(x))
            assert fm.nbytes == fm_oracle.fm_bytes(len(x), len(set(x)), s)
            lo, hi = ctx.fm_count_host(fm, pats)
            bad = np.nonzero((lo != want_lo) | (hi != want_hi))[0]
            assert not len(bad), (len(x), s, [(pats[k][:16], lo[k], hi[k], want_lo[k], want_hi[k]) for k in bad[:4]])
            st = ctx.stats()
            assert st["direction"] == 1 and "inv_walk" in st["classes"]
            pos, off = ctx.fm_locate_host(fm, lo, hi)
            assert np.array_equal(pos, o.locate(lo, hi)), (len(x), s)
            assert off[-1] == len(pos)
    return o


def test_known_answers(ctx):
    for s in fm_oracle.SAMPLES:
        for text in (b"banana", b"mississippi", b"aaaa"):
            cases = [(p, lo, hi, loc) for x, p, lo, hi, loc in fm_oracle.KNOWN if x == text]
            with ctx.fm_build_host(text, s) as fm:
                lo, hi = ctx.fm_count_host(fm, [c[0] for c in cases])
                assert list(zip(lo.tolist(), hi.tolist())) == [(c[1], c[2]) for c in cases], (text, s)
                pos, off = ctx.fm_locate_host(fm, lo, hi)
                assert [pos[off[k]:off[k + 1]].tolist() for k in range(len(cases))] == [c[3] for c in cases]


def test_shortest_inputs(ctx):
    for x in (b"\x00", b"\xff", b"a", b"ab", b"ba", b"aa", b"\x00\xff", b"\xff\x00"):
        pats = [b"", b"\x00", b"\xff", b"a", b"b", b"ab", b"ba", b"aa", b"\x00\xff", b"\xff\x00", x, x + x]
        check(ctx, x, fm_oracle.SAMPLES, pats)


@pytest.mark.parametrize("n", [255, 256, 257, 65535, 65536, 65537, 200_003])
def test_sizes_at_the_layout_edges(ctx, gen, n):
    rng = np.random.default_rng(n)
    inputs = {"dna": gen.make("dna", 4, n), "text": gen.make("text", 2, n),
              "all256": rng.integers(0, 256, size=n, dtype=np.uint8).tobytes()}
    for i, x in enumerate(inputs.values()):
        check(ctx, x, (1, 32) if n < 70_000 else (32,), seed=i)


def test_one_byte_alphabet_longest_walks(ctx):
    for n in (1000, 65537):
        x = b"a" * n
        pats = [b"", b"a", b"a" * 7, b"a" * (n - 1), b"a" * n, b"a" * (n + 1), b"b", b"ab", b"\x00a"]
        check(ctx, x, fm_oracle.SAMPLES, pats)


@pytest.mark.parametrize("k", [0, 1, 254, 255, 256, 257, 65534, 65535, 65536, 65537])
def test_dollar_row_at_chosen_rows(ctx, k):
    for m in (0, 1, 300 + k % 7):
        x = fm_oracle.dollar_row_text(k, m)
        o = fm_oracle.FmOracle(x)
        assert o.sa[k] == 0
        pats = [b"", b"b", b"ba", b"a", b"ac", b"c", b"bc", x[:50], x[-50:], b"a" * (k + 1), b"d", b"\x00"]
        check(ctx, x, (1, 2, 32, 1024) if k < 300 else (2, 1024), pats, o=o)


def test_sample_rates_rejected(ctx, bwts):
    for s in (0, 3, 6, 2048, -1):
        with pytest.raises(bwts.BwtsError) as e:
            ctx.fm_build_host(b"banana", s)
        assert e.value.code == EINVAL


def _dna_counts(x, pats):
    """count by sorted fixed-length keys of the suffixes: byte + 1 in base 257, 0 past the end of text"""
    t = np.frombuffer(x, dtype=np.uint8).astype(np.uint64) + 1
    n = len(t)
    lo = np.empty(len(pats), dtype=np.int64)
    hi = np.empty(len(pats), dtype=np.int64)
    lens = np.array([len(p) for p in pats])
    for m in np.unique(lens):
        m = int(m)
        key = np.zeros(n, dtype=np.uint64)
        for j in range(m):
            col = np.zeros(n, dtype=np.uint64)
            col[:n - j] = t[j:]
            key = key * np.uint64(257) + col
        key.sort()
        idx = np.nonzero(lens == m)[0]
        pk = np.zeros(len(idx), dtype=np.uint64)
        for j in range(m):
            pk = pk * np.uint64(257) + np.array([pats[i][j] + 1 for i in idx], dtype=np.uint64)
        lo[idx] = np.searchsorted(key, pk, "left")
        hi[idx] = np.searchsorted(key, pk, "right")
    return lo, hi


def test_million_patterns_in_one_call(ctx, gen):
    n = 1 << 20
    x = gen.make("dna", 4, n)
    rng = np.random.default_rng(7)
    starts = rng.integers(0, n, size=1 << 20)
    lens = rng.integers(1, 8, size=1 << 20)
    alphabet = np.frombuffer(b"ACGTN", dtype=np.uint8)
    pats = []
    for k, (a, m) in enumerate(zip(starts.tolist(), lens.tolist())):
        pats.append(x[a:a + m] if k % 2 else bytes(rng.choice(alphabet, size=m)))
    want_lo, want_hi = _dna_counts(x, pats)
    with ctx.fm_build_host(x, 32) as fm:
        lo, hi = ctx.fm_count_host(fm, pats)
        assert np.array_equal(lo, want_lo) and np.array_equal(hi, want_hi)
        lo0, hi0 = ctx.fm_count_host(fm, [])
        assert len(lo0) == len(hi0) == 0


def test_device_calls_torch_stream_odd_address(bwts, ctx, gen):
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("text", 5, 300_001)
    o = fm_oracle.FmOracle(x)
    pats = pattern_set(x, 3)
    want_lo, want_hi = o.count_many(pats)
    cat, off = bwts.fm_patterns(pats)
    s = torch.cuda.Stream(dev)
    big = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    view = big[3:3 + len(x)]                                   # text at an odd address
    view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
    pbuf = torch.zeros(len(cat) + 16, dtype=torch.uint8, device=dev)
    pview = pbuf[1:1 + len(cat)]                                # patterns at an odd address
    pview.copy_(torch.from_numpy(cat.copy()))
    d_off = torch.from_numpy(off).to(dev)
    d_rng = torch.full((2 * len(pats),), -7, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        fm = ctx.fm_build_device(view.data_ptr(), len(x), 8, stream=s.cuda_stream)
        total = ctx.fm_count_device(fm, pview.data_ptr(), len(cat), d_off.data_ptr(), len(pats), d_rng.data_ptr(),
                                    stream=s.cuda_stream)
        s.synchronize()
    rng = d_rng.cpu().numpy()
    assert np.array_equal(rng[0::2], want_lo) and np.array_equal(rng[1::2], want_hi)
    assert total == int((want_hi.astype(np.int64) - want_lo).sum())
    pos = torch.full((total + 5,), -9, dtype=torch.int32, device=dev)
    with torch.cuda.stream(s):
        got = ctx.fm_locate_device(fm, d_rng.data_ptr(), len(pats), pos.data_ptr(), total + 5, stream=s.cuda_stream)
        s.synchronize()
    assert got == total
    p = pos.cpu().numpy()
    assert np.array_equal(p[:total], o.locate(want_lo, want_hi)) and (p[total:] == -9).all()
    # the host forms agree with the device forms on the same index
    lo, hi = ctx.fm_count_host(fm, pats)
    assert np.array_equal(lo, want_lo) and np.array_equal(hi, want_hi)
    fm.close()


def test_lifetimes(bwts, gen):
    x1, x2 = gen.make("dna", 8, 100_000), gen.make("text", 9, 100_000)
    o1, o2 = fm_oracle.FmOracle(x1), fm_oracle.FmOracle(x2)
    p1, p2 = pattern_set(x1, 1), pattern_set(x2, 2)
    with bwts.Context(0) as c:                        # two indexes on one context
        fm1, fm2 = c.fm_build_host(x1, 16), c.fm_build_host(x2, 4)
        assert c.fm_count_host(fm1, p1)[1].tolist() == o1.count_many(p1)[1].tolist()
        assert c.fm_count_host(fm2, p2)[1].tolist() == o2.count_many(p2)[1].tolist()
    # the building context is gone; other contexts query the index, two threads at once
    errors = []

    def worker(fm, pats, o, rounds):
        try:
            with bwts.Context(0) as c:
                want = o.count_many(pats)
                for _ in range(rounds):
                    lo, hi = c.fm_count_host(fm, pats)
                    assert np.array_equal(lo, want[0]) and np.array_equal(hi, want[1])
                    pos, _ = c.fm_locate_host(fm, lo, hi)
                    assert np.array_equal(pos, o.locate(lo, hi))
        except Exception as e:  # noqa: BLE001 -- reported below
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(fm1, p1, o1, 5)) for _ in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    fm1.close()
    fm2.close()
    fm2.close()                                       # closing twice is a no-op


def test_malformed_device_arrays(bwts, ctx):
    """only values a missing check would turn into a wrong return code: every access stays inside the buffers"""
    import torch
    dev = torch.device("cuda:0")
    x = b"mississippi" * 100
    with ctx.fm_build_host(x, 4) as fm:
        pat = torch.frombuffer(bytearray(b"ssiissippi"), dtype=torch.uint8).to(dev)
        rng = torch.full((6,), -5, dtype=torch.int32, device=dev)
        for off in ([0, 5, 3, 10], [1, 3, 6, 10], [0, 3, 6, 9], [0, 3, 6, 11]):  # decreasing, off[0], off[npat]
            d_off = torch.tensor(off, dtype=torch.int64, device=dev)
            with pytest.raises(bwts.BwtsError) as e:
                ctx.fm_count_device(fm, pat.data_ptr(), 10, d_off.data_ptr(), 3, rng.data_ptr())
            assert e.value.code == EINVAL, off
        assert (rng.cpu() == -5).all()                 # nothing written
        d_off = torch.tensor([0, 3, 6, 10], dtype=torch.int64, device=dev)
        assert ctx.fm_count_device(fm, pat.data_ptr(), 10, d_off.data_ptr(), 3, rng.data_ptr()) >= 0
        pos = torch.full((64,), -3, dtype=torch.int32, device=dev)
        n = len(x)
        for bad in ([5, 4], [-1, 2], [0, n + 1], [n + 1, n + 1]):
            r = torch.tensor([0, 1] + bad, dtype=torch.int32, device=dev)
            with pytest.raises(bwts.BwtsError) as e:
                ctx.fm_locate_device(fm, r.data_ptr(), 2, pos.data_ptr(), 64)
            assert e.value.code == EINVAL, bad
        r = torch.tensor([0, 40, 100, 130], dtype=torch.int32, device=dev)   # 70 positions, cap 64
        with pytest.raises(bwts.BwtsError) as e:
            ctx.fm_locate_device(fm, r.data_ptr(), 2, pos.data_ptr(), 64)
        assert e.value.code == EINVAL
        assert (pos.cpu() == -3).all()
        # the host forms check the same rules on the host
        for lo, hi in (([5], [4]), ([-1], [2]), ([0], [n + 1])):
            with pytest.raises(bwts.BwtsError) as e:
                ctx.fm_locate_host(fm, lo, hi)
            assert e.value.code == EINVAL


@pytest.mark.parametrize("name", ["C2", "C3", "C3F"])
def test_full_size_against_the_oracle(bwts, gen, name):
    gold = FM_FULLSIZE[name]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    pats = fm_oracle.golden_patterns(x, gold["pattern_seed"])
    with bwts.Context(0) as c, c.fm_build_host(x, 32) as fm:
        lo, hi = c.fm_count_host(fm, pats)
        llo, lhi = fm_oracle.golden_locate_ranges(lo, hi)
        pos, _ = c.fm_locate_host(fm, llo, lhi)
        h = fm_oracle.golden_hashes(lo, hi, pos)
    for key in ("ranges_sha256", "positions_sha256", "hits", "located"):
        assert h[key] == gold[key], key


def _release():
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def sampled_substring_property(c, fm, tx, n, count=1 << 20, length=24, seed=5):
    """for `count` substrings P = T[s:s+length]: every located position of [lo, hi) starts with P, s is among them,
    and the rows lo - 1 and hi, located on their own, do not start with P"""
    import torch
    dev = tx.device
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    s = torch.randint(0, n - length, (count,), device=dev, generator=g)
    j = torch.arange(length, device=dev)
    P = tx[s[:, None] + j].contiguous()                                # (count, length)
    off = torch.arange(count + 1, dtype=torch.int64, device=dev) * length
    rng = torch.empty(2 * count, dtype=torch.int32, device=dev)
    total = c.fm_count_device(fm, P.data_ptr(), count * length, off.data_ptr(), count, rng.data_ptr())
    lo, hi = rng[0::2].long(), rng[1::2].long()
    assert bool((hi > lo).all()) and total == int((hi - lo).sum())

    def starts_with(pos, pats):
        idx = pos[:, None] + j
        return ((tx[idx.clamp(max=n - 1)] == pats) & (idx < n)).all(dim=1)

    pos = torch.empty(total, dtype=torch.int32, device=dev)
    assert c.fm_locate_device(fm, rng.data_ptr(), count, pos.data_ptr(), total) == total
    owner = torch.repeat_interleave(torch.arange(count, device=dev), hi - lo)
    assert bool(starts_with(pos.long(), P[owner]).all())
    hit = torch.zeros(count, dtype=torch.int32, device=dev)
    hit.index_add_(0, owner, (pos.long() == s[owner]).to(torch.int32))
    assert bool((hit == 1).all())
    del pos, owner
    # the rows just outside each range
    below, above = torch.nonzero(lo > 0)[:, 0], torch.nonzero(hi < n)[:, 0]
    rows = torch.cat([lo[below] - 1, hi[above]])
    owners = torch.cat([below, above])
    edge = torch.stack([rows, rows + 1], 1).to(torch.int32).reshape(-1).contiguous()
    epos = torch.empty(len(rows), dtype=torch.int32, device=dev)
    assert c.fm_locate_device(fm, edge.data_ptr(), len(rows), epos.data_ptr(), len(rows)) == len(rows)
    assert not bool(starts_with(epos.long(), P[owners]).any())
    return total


def byte_histogram_property(c, fm, tx):
    import torch
    pats = torch.arange(256, dtype=torch.uint8, device=tx.device)
    off = torch.arange(257, dtype=torch.int64, device=tx.device)
    rng = torch.empty(512, dtype=torch.int32, device=tx.device)
    c.fm_count_device(fm, pats.data_ptr(), 256, off.data_ptr(), 256, rng.data_ptr())
    hist = torch.bincount(tx.long(), minlength=256)
    assert torch.equal((rng[1::2] - rng[0::2]).long(), hist)


def test_full_size_c4(bwts, gen):
    """1 GiB DNA: locate of the empty pattern equals the suffix array (every sample walk), the sampled-substring
    property, and the single-byte counts equal the byte histogram"""
    import torch
    n = 1 << 30
    dev = torch.device("cuda:0")
    tx = torch.frombuffer(bytearray(gen.make("dna", 4, n)), dtype=torch.uint8).to(dev)
    sa = torch.empty(n, dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:
        c.sa_device(tx.data_ptr(), n, sa.data_ptr())
        fm = c.fm_build_device(tx.data_ptr(), n, 16)
    try:
        with bwts.Context(0) as c:
            rng = torch.tensor([0, n], dtype=torch.int32, device=dev)
            pos = torch.empty(n, dtype=torch.int32, device=dev)
            assert c.fm_locate_device(fm, rng.data_ptr(), 1, pos.data_ptr(), n) == n
            assert torch.equal(pos, sa)
            del pos
            sampled_substring_property(c, fm, tx, n)
            byte_histogram_property(c, fm, tx)
    finally:
        fm.close()
        del sa, tx
        _release()


def test_largest_length(bwts, gen):
    """2^31 - 1 bytes of DNA: build, the sampled-substring property through locate, the byte histogram"""
    import torch
    n = (1 << 31) - 1
    _release()
    if torch.cuda.mem_get_info(0)[0] < 80 * n + (1 << 28):
        pytest.skip("needs ~170 GB of free device memory")
    dev = torch.device("cuda:0")
    tx = torch.frombuffer(bytearray(gen.make("dna", 7, n)), dtype=torch.uint8).to(dev)
    with bwts.Context(0) as c:
        fm = c.fm_build_device(tx.data_ptr(), n, 32)
        st = c.stats()
        assert (st["factors"], st["longest_factor"]) == (1, n)
    _release()
    try:
        with bwts.Context(0) as c:
            sampled_substring_property(c, fm, tx, n, count=1 << 18)
            byte_histogram_property(c, fm, tx)
    finally:
        fm.close()
        del tx
        _release()

"""GPU tests of the longest-previous-factor array and the greedy LZ77 parse (bwts_b200_lpf_*, bwts_b200_lz77_*): both
against the CPU oracle (oracle/lz_oracle.c) on the known answers and on families around 32, 4096 and 4096^2 bytes
under the smallest and the default tile width (tune key 25), after each forced tier of the LCP stage (tune key 24);
host and device forms (torch tensors, unaligned input, a caller stream); cap overflow and overlap rejection; one
context reused across transforms; golden hashes at 64 and 256 MiB; properties checked on the GPU at 1 GiB and the
closed forms of a^n and the Fibonacci word at 2^31 - 1 bytes.  Run on a B200."""
import ctypes
import gc
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

import helpers
import lcp_oracle
import lz_oracle

pytestmark = pytest.mark.gpu

EINVAL = -1
LZ_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "lz_fullsize.json").read_text())
TUNE_KEYS = (24, 25)
KNOWN = [(b"banana", [0, 0, 0, 3, 2, 1], [-1, -1, -1, 1, 2, 3], [[98, 0], [97, 0], [110, 0], [1, 3]]),
         (b"abracadabra", [0, 0, 0, 1, 0, 1, 0, 4, 3, 2, 1], [-1, -1, -1, 0, -1, 3, -1, 0, 1, 2, 7],
          [[97, 0], [98, 0], [114, 0], [0, 1], [99, 0], [3, 1], [100, 0], [0, 4]]),
         (b"mississippi", [0, 0, 0, 1, 4, 3, 2, 1, 0, 1, 1], [-1, -1, -1, 2, 1, 2, 3, 4, -1, 8, 7],
          [[109, 0], [105, 0], [115, 0], [2, 1], [1, 4], [112, 0], [8, 1], [7, 1]]),
         (b"aaaa", [0, 3, 2, 1], [-1, 0, 1, 2], [[97, 0], [0, 3]]),
         (b"a", [0], [-1], [[97, 0]])]


@pytest.fixture(scope="module")
def orc():
    return lz_oracle.LzOracle()


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


def checked(ctx, orc, x):
    want_lpf, want_prev = orc.lpf(x)
    lpf, prev = ctx.lpf_host(x)
    where = (len(x), bytes(x[:24]))
    assert np.array_equal(lpf, want_lpf), where + (int(np.argmax(lpf != want_lpf)),)
    assert np.array_equal(prev, want_prev), where + (int(np.argmax(prev != want_prev)),)
    st = ctx.stats()
    assert (st["factors"], st["longest_factor"], st["direction"]) == (1, len(x), 0)
    f = ctx.lz77_host(x)
    assert np.array_equal(f, orc.lz77(x)), where
    assert "emit" in ctx.stats()["classes"]


def test_known_answers(ctx, orc):
    for x, lpf, prev, fac in KNOWN:
        got = ctx.lpf_host(x)
        assert (got[0].tolist(), got[1].tolist()) == (lpf, prev), x
        assert ctx.lz77_host(x).tolist() == fac, x
    for x in (b"\x00", b"\xff", b"aa", b"ab", b"ba", b"\x00\x00", b"\xff\x00"):
        checked(ctx, orc, x)


def family_cases(big):
    out = {}
    for n in (31, 32, 33, 4095, 4096, 4097):
        out.update({f"{k}_{n}": x for k, x in helpers.families(n).items()})
    if big:
        n = 4096 * 4096 + 1
        fam = helpers.families(n)
        out.update({f"{k}_{n}": fam[k] for k in ("all_a", "descending", "fibonacci", "de_bruijn", "random4",
                                                   "random256", "runs")})
    return out


@pytest.mark.parametrize("tb", [5, 0], ids=["tile32", "tile4096"])
def test_families_against_the_oracle(bwts, ctx, orc, tb):
    """tile / chunk width 32 sends most rows across tiles and runs the parse on up to four levels"""
    bwts.tune(25, tb)
    for name, x in family_cases(big=True).items():
        checked(ctx, orc, x)


@pytest.mark.parametrize("tier", [1, 2], ids=["warp_tier", "multi_cta_tier"])
def test_after_each_lcp_tier(bwts, ctx, orc, gen, tier):
    """the stages run after each scratch layout of the LCP stage (tune key 24)"""
    bwts.tune(24, tier)
    bwts.tune(25, 6)
    cases = list(helpers.families(4609).values()) + [b"a" * 70_000, helpers.fibonacci_word(50_000),
                                                     b"q" + gen.make("text", 62, 90_000) * 2]
    for x in cases:
        checked(ctx, orc, x)


def test_device_forms_unaligned_on_a_caller_stream(ctx, orc, gen):
    import torch
    dev = torch.device("cuda:0")
    s = torch.cuda.Stream(dev)
    for n, x in ((5, b"abaab"), (4097, gen.make("text", 71, 4097)), (300_001, gen.make("dna", 72, 300_001))):
        want_lpf, want_prev = orc.lpf(x)
        want_f = orc.lz77(x)
        for off in (0, 3, 16):
            big = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
            view = big[off:off + n]
            view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
            lpf = torch.full((n,), -9, dtype=torch.int32, device=dev)
            prev = torch.full((n,), -9, dtype=torch.int32, device=dev)
            fac = torch.full((n + 1, 2), -9, dtype=torch.int32, device=dev)
            torch.cuda.synchronize()
            with torch.cuda.stream(s):
                ctx.lpf_device(view.data_ptr(), n, lpf.data_ptr(), prev.data_ptr(), s.cuda_stream)
                z = ctx.lz77_device(view.data_ptr(), n, fac.data_ptr(), n + 1, s.cuda_stream)
            s.synchronize()
            assert np.array_equal(lpf.cpu().numpy(), want_lpf) and np.array_equal(prev.cpu().numpy(), want_prev)
            assert z == len(want_f)
            got = fac.cpu().numpy()
            assert np.array_equal(got[:z], want_f)
            assert (got[z:] == -9).all()   # nothing past the z pairs
        # the default stream (NULL: the context's own)
        z = ctx.lz77_device(view.data_ptr(), n, fac.data_ptr(), n)
        torch.cuda.synchronize()
        assert z == len(want_f) and np.array_equal(fac.cpu().numpy()[:z], want_f)


def test_cap_overflow_leaves_the_buffer_untouched(bwts, ctx, orc, gen):
    import torch
    L = bwts.lib()
    x = gen.make("text", 73, 20_000)
    want = orc.lz77(x)
    zw = len(want)
    dev = torch.device("cuda:0")
    d_x = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
    fac = torch.full((zw, 2), -9, dtype=torch.int32, device=dev)
    z = ctypes.c_long(-1)
    assert L.bwts_b200_lz77_device(ctx._h, d_x.data_ptr(), len(x), fac.data_ptr(), zw - 1, ctypes.byref(z), None) == EINVAL
    torch.cuda.synchronize()
    assert z.value == zw and bool((fac == -9).all())
    z.value = -1
    assert L.bwts_b200_lz77_device(ctx._h, d_x.data_ptr(), len(x), fac.data_ptr(), 0, ctypes.byref(z), None) == EINVAL
    assert z.value == zw
    h = np.full((zw, 2), -9, dtype=np.int32)
    z.value = -1
    assert L.bwts_b200_lz77_host(ctx._h, x, len(x), h.ctypes.data, zw - 1, ctypes.byref(z)) == EINVAL
    assert z.value == zw and (h == -9).all()
    # exactly z fits
    assert L.bwts_b200_lz77_host(ctx._h, x, len(x), h.ctypes.data, zw, ctypes.byref(z)) == 0
    assert z.value == zw and np.array_equal(h, want)
    # and the context still works
    checked(ctx, orc, b"abracadabra")


def test_overlap_rejection(bwts, ctx):
    import torch
    L = bwts.lib()
    dev = torch.device("cuda:0")
    buf = torch.zeros(1 << 16, dtype=torch.uint8, device=dev)
    p = buf.data_ptr()
    n = 1000
    z = ctypes.c_long(-1)
    assert L.bwts_b200_lpf_device(ctx._h, p, n, p + 512, p + 8192, None) == EINVAL       # in / lpf
    assert L.bwts_b200_lpf_device(ctx._h, p, n, p + 4096, p + 4096 + 3996, None) == EINVAL   # lpf / prev
    assert L.bwts_b200_lpf_device(ctx._h, p + 20000, n, p + 4096, p + 17000, None) == EINVAL  # prev / in
    assert L.bwts_b200_lz77_device(ctx._h, p + 4096 + 8 * 99, n, p + 4096, 100, ctypes.byref(z), None) == EINVAL
    assert z.value == -1
    # just apart is fine
    assert L.bwts_b200_lz77_device(ctx._h, p + 4096 + 8 * 100, n, p + 4096, 100, ctypes.byref(z), None) == 0
    torch.cuda.synchronize()
    assert z.value == 2


def test_one_context_across_transforms(ctx, orc, gen, oracle):
    sa_orc = lcp_oracle.LcpOracle()
    for x in (gen.make("text", 81, 100_000), b"banana" * 999, gen.make("dna", 82, 300_007), b"zz"):
        assert ctx.forward_host(x) == oracle.forward(x)
        sa, lcp = ctx.sa_lcp_host(x)
        want = sa_orc.sa_lcp(x)
        assert np.array_equal(sa, want[0]) and np.array_equal(lcp, want[1])
        checked(ctx, orc, x)
        y = x[: max(1, len(x) // 3)]
        checked(ctx, orc, y)


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<i4").tobytes()).hexdigest()


@pytest.mark.parametrize("name", ["C2", "C3", "C3F"])
def test_full_size_against_the_oracle(bwts, gen, name):
    gold = LZ_FULLSIZE[name]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        lpf, prev = c.lpf_host(x)
        assert int(lpf.max()) == gold["lpf_max"]
        assert _sha(lpf) == gold["lpf_sha256"] and _sha(prev) == gold["prev_sha256"]
        f = c.lz77_host(x)
        assert len(f) == gold["z"] and _sha(f) == gold["factors_sha256"]
    if name == "C3F":   # the closed form used at 2^31 - 1, confirmed at 256 MiB
        assert np.maximum(f[:, 1], 1).tolist() == lz_oracle.fibonacci_factor_lengths(gold["n"])


def release_device_memory():
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def check_parse_on_gpu(x, lpf, prev, fac):
    """torch on the GPU: the parse is the chain of LPF / PREV from 0; every factor's bytes equal its source's"""
    import torch
    n = x.numel()
    lens = fac[:, 1].long().clamp(min=1)
    assert int(lens.sum()) == n
    p = torch.cumsum(lens, 0) - lens
    assert torch.equal(fac[:, 1], lpf[p])
    lit = fac[:, 1] == 0
    assert torch.equal(fac[:, 0][~lit], prev[p][~lit])
    assert torch.equal(fac[:, 0][lit].long(), x[p[lit]].long())
    # each position of a copied factor against its source position
    shift = torch.repeat_interleave(torch.where(lit, 0, fac[:, 0].long() - p), lens)
    del p, lens, lit
    pos = torch.arange(n, device=x.device)
    src = pos + shift
    del shift
    assert bool((src <= pos).all())
    assert torch.equal(x[src], x)
    del src, pos


def check_lpf_on_gpu(x, lpf, prev, samples=1 << 16):
    """LPF[0] = 0, LPF[i] >= LPF[i-1] - 1, PREV[i] < i exactly where LPF[i] > 0, and sampled sources match"""
    import torch
    n = x.numel()
    assert int(lpf[0]) == 0 and int(prev[0]) == -1
    assert bool((lpf[1:] >= lpf[:-1] - 1).all())
    assert torch.equal(lpf == 0, prev == -1)
    g = torch.Generator(device=x.device)
    g.manual_seed(9)
    i = torch.randint(1, n, (samples,), device=x.device, generator=g)
    l, s = lpf[i].long(), prev[i].long()
    assert bool((s < i).all()) and bool((l <= n - i).all())
    for k0 in range(0, int(l.max()) + 1, 256):
        j = torch.arange(k0, k0 + 256, device=x.device)
        inside = j[None, :] < l[:, None]
        a = x[(i[:, None] + j).clamp(max=n - 1)]
        b = x[(s[:, None] + j).clamp(min=0, max=n - 1)]
        assert bool(((a == b) | ~inside).all())


def test_full_size_c4(bwts, gen):
    """1 GiB DNA: LPF / PREV and the parse checked on the GPU"""
    import torch
    release_device_memory()
    dev = torch.device("cuda:0")
    n = 1 << 30
    x = torch.frombuffer(bytearray(gen.make("dna", 4, n)), dtype=torch.uint8).to(dev)
    lpf = torch.empty(n, dtype=torch.int32, device=dev)
    prev = torch.empty(n, dtype=torch.int32, device=dev)
    fac = torch.empty((n // 4, 2), dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:
        c.lpf_device(x.data_ptr(), n, lpf.data_ptr(), prev.data_ptr())
        z = c.lz77_device(x.data_ptr(), n, fac.data_ptr(), n // 4)
        torch.cuda.synchronize()
    release_device_memory()
    check_lpf_on_gpu(x, lpf, prev)
    check_parse_on_gpu(x, lpf, prev, fac[:z])
    del x, lpf, prev, fac
    release_device_memory()


def test_largest_length_closed_forms(bwts, gen):
    """2^31 - 1 bytes: a^n against LPF[i] = n - i, PREV[i] = i - 1 and (97,0) (0,n-1); the Fibonacci word's parse
    against 1, 1, 1, 3, 5, 8, ... and its LPF against the properties"""
    import torch
    n = (1 << 31) - 1
    release_device_memory()
    if torch.cuda.mem_get_info(0)[0] < 80 * n + (1 << 28):
        pytest.skip("needs 172 GB of free device memory")
    dev = torch.device("cuda:0")
    x = torch.full((n,), ord("a"), dtype=torch.uint8, device=dev)
    lpf = torch.empty(n, dtype=torch.int32, device=dev)
    prev = torch.empty(n, dtype=torch.int32, device=dev)
    fac = torch.full((128, 2), -9, dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:   # closed before checking: the workspace leaves no room beside it
        c.lpf_device(x.data_ptr(), n, lpf.data_ptr(), prev.data_ptr())
        z = c.lz77_device(x.data_ptr(), n, fac.data_ptr(), 128)
        torch.cuda.synchronize()
    release_device_memory()
    assert z == 2 and fac[:2].tolist() == [[97, 0], [0, n - 1]]
    r = torch.arange(n, dtype=torch.int32, device=dev)
    assert torch.equal(lpf[1:], n - r[1:]) and torch.equal(prev[1:], r[:-1]) and int(lpf[0]) == 0
    del r
    release_device_memory()
    x.copy_(torch.frombuffer(bytearray(gen.make("fibonacci", 0, n)), dtype=torch.uint8))
    with bwts.Context(0) as c:
        c.lpf_device(x.data_ptr(), n, lpf.data_ptr(), prev.data_ptr())
        z = c.lz77_device(x.data_ptr(), n, fac.data_ptr(), 128)
        torch.cuda.synchronize()
    release_device_memory()
    want = lz_oracle.fibonacci_factor_lengths(n)
    assert z == len(want) and fac[:z, 1].clamp(min=1).tolist() == want
    check_lpf_on_gpu(x, lpf, prev)
    p = torch.cumsum(fac[:z, 1].long().clamp(min=1), 0) - fac[:z, 1].long().clamp(min=1)
    assert torch.equal(fac[:z, 1], lpf[p]) and torch.equal(fac[3:z, 0], prev[p[3:]])
    del x, lpf, prev, fac, p
    release_device_memory()

"""GPU tests of the suffix array and LCP array (bwts_b200_sa_lcp, bwts_b200_sa_* context and device calls): both
arrays against the CPU oracle (oracle/lcp_oracle.c: SA-IS plus Kasai) on families at tile edges, under each forced
tier of the LCP stage (tune key 24) and under every forward tune key that acts on the linear sort; host, device
(torch tensors, unaligned input, a caller stream) and one-call entry points; a^n against the closed form; golden
hashes at 64 and 256 MiB; and properties checked on the GPU at 1 GiB and 2^31 - 1 bytes.  Run on a B200."""
import gc
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

import helpers
import lcp_oracle
from test_gpu_dispatch_edges import equal_factors

pytestmark = pytest.mark.gpu

SA_LCP_FULLSIZE = json.loads((Path(__file__).parent / "golden" / "sa_lcp_fullsize.json").read_text())
TUNE_KEYS = (0, 1, 2, 3, 6, 7, 8, 9, 12, 13, 14, 15, 16, 18, 20, 21, 22, 23, 24)
KNOWN = [(b"banana", [5, 3, 1, 0, 4, 2], [0, 1, 3, 0, 0, 2]),
         (b"mississippi", [10, 7, 4, 1, 0, 9, 8, 6, 3, 5, 2], [0, 1, 1, 4, 0, 0, 1, 0, 2, 1, 3]),
         (b"abracadabra", [10, 7, 0, 3, 5, 8, 1, 4, 6, 9, 2], [0, 1, 4, 1, 1, 0, 3, 0, 0, 0, 2]),
         (b"aaaa", [3, 2, 1, 0], [0, 1, 2, 3]), (b"a", [0], [0])]


@pytest.fixture(scope="module")
def orc():
    return lcp_oracle.LcpOracle()


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


def checked(ctx, x, want):
    sa, lcp = ctx.sa_lcp_host(x)
    assert np.array_equal(sa, want[0]), (len(x), bytes(x[:32]))
    assert np.array_equal(lcp, want[1]), (len(x), bytes(x[:32]), int(np.argmax(lcp != want[1])))
    st = ctx.stats()
    assert (st["factors"], st["longest_factor"], st["direction"]) == (1, len(x), 0)
    return st


def test_known_answers(ctx, bwts):
    for x, sa, lcp in KNOWN:
        got = ctx.sa_lcp_host(x)
        assert (got[0].tolist(), got[1].tolist()) == (sa, lcp), x
        got = bwts.suffix_array_lcp(x)
        assert (got[0].tolist(), got[1].tolist()) == (sa, lcp), x
        assert ctx.sa_host(x).tolist() == sa == bwts.suffix_array(x).tolist(), x
    sa, lcp = bwts.suffix_array_lcp(b"")
    assert len(sa) == len(lcp) == 0


def test_shortest_inputs(ctx, bwts, orc):
    for x in (b"\x00", b"a", b"\xff", b"aa", b"ab", b"ba", b"\x00\xff", b"\xff\x00", b"\x00\x00"):
        want = orc.sa_lcp(x)
        checked(ctx, x, want)
        got = bwts.suffix_array_lcp(x)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), x


def family_cases(gen):
    """name -> input: families at tile edges, periodic inputs, runs of one byte, generated text and DNA"""
    out = {}
    for n in (3, 255, 257, 2049, 4095, 4097, 4609, 8193, 65537):
        out.update({f"{k}_{n}": x for k, x in helpers.families(n).items()})
    for u, k in ((b"ba", 50), (b"cab", 1400), (b"abcabd", 3), (b"\x00\xff", 2048), (b"abacabb", 4097)):
        out[f"({u.hex()})^{k}"] = u * k
    for n in (4097, 100_003):
        out[f"all_{n}"] = b"a" * n
    out["all_00"] = b"\x00" * 5000
    out["text1m"] = gen.make("text", 41, (1 << 20) + 7)
    out["dna1m"] = gen.make("dna", 42, 1 << 20)
    out["copies"] = b"xyz" * 9 + gen.make("dna", 43, 300_000) * 3   # pairs of 300 KB: the multi-CTA tier
    return out


@pytest.fixture(scope="module")
def family_wants(orc, gen):
    return {name: (x, orc.sa_lcp(x)) for name, x in family_cases(gen).items()}


def test_families_against_the_oracle(ctx, family_wants):
    for name, (x, want) in family_wants.items():
        st = checked(ctx, x, want)
        assert "emit" in st["classes"], name


@pytest.fixture(scope="module")
def tier_wants(orc, gen):
    cases = {f"{k}_4609": x for k, x in helpers.families(4609).items()}
    cases.update({"all_70k": b"a" * 70_000, "(cab)^1400": b"cab" * 1400, "fib50k": helpers.fibonacci_word(50_000),
                  "u7^4097": equal_factors(b"abacabb", 4097), "dna200k": gen.make("dna", 61, 200_000),
                  "copies": b"q" + gen.make("text", 62, 90_000) * 2})
    return {name: (x, orc.sa_lcp(x)) for name, x in cases.items()}


@pytest.mark.parametrize("tier", [0, 1, 2], ids=["by_length", "warp_tier", "multi_cta_tier"])
def test_each_lcp_tier(bwts, ctx, tier_wants, tier):
    """tune key 24: 1 sends every irreducible pair through the warp tier, 2 through the multi-CTA tier"""
    bwts.tune(24, tier)
    for name, (x, want) in tier_wants.items():
        checked(ctx, x, want)


# (key, value) of every forward tune key that acts on the linear sort, as tests/test_gpu_divbwt.py sweeps them
FWD_SETTINGS = [(2, 1), (2, 3), (3, 1), (6, 16), (7, 2), (7, 4), (8, 1), (9, 1), (9, 2), (9, 3), (14, 1), (14, 2),
                (18, 1), (20, 1), (21, 1), (22, 1), (23, 16)]


@pytest.fixture(scope="module")
def tune_input(orc, gen):
    x = b"xyz" * 9 + gen.make("text", 63, 200_000) * 2 + gen.make("dna", 64, 300_001)
    return x, orc.sa_lcp(x)


@pytest.mark.parametrize("key,value", FWD_SETTINGS, ids=[f"tune{k}={v}" for k, v in FWD_SETTINGS])
def test_under_forward_tune_keys(bwts, ctx, tune_input, key, value):
    bwts.tune(key, value)
    checked(ctx, *tune_input)


# --------------------------------------------------------------------------- entry points

def test_device_calls_at_unaligned_offsets_on_a_caller_stream(ctx, orc, gen):
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("text", 65, 300_001) + b"abc" * 40_000
    want_sa, want_lcp = orc.sa_lcp(x)
    n = len(x)
    big = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
    sa = torch.zeros(n + 16, dtype=torch.int32, device=dev)
    lcp = torch.zeros(n + 16, dtype=torch.int32, device=dev)
    s = torch.cuda.Stream(dev)
    for off in (0, 1, 3, 8, 13):
        view = big[off:off + n]
        view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
        torch.cuda.synchronize()
        o = off % 5   # int32 views: 4-byte aligned at any element offset
        sa_v, lcp_v = sa[o:o + n], lcp[o + 1:o + 1 + n]
        ctx.sa_lcp_device(view.data_ptr(), n, sa_v.data_ptr(), lcp_v.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert np.array_equal(sa_v.cpu().numpy(), want_sa) and np.array_equal(lcp_v.cpu().numpy(), want_lcp), off
        sa_v.zero_()
        torch.cuda.synchronize()
        ctx.sa_device(view.data_ptr(), n, sa_v.data_ptr(), s.cuda_stream)
        s.synchronize()
        assert np.array_equal(sa_v.cpu().numpy(), want_sa), off
    with pytest.raises(RuntimeError) as e:   # a device output that is not 4-byte aligned
        ctx.sa_lcp_device(big.data_ptr(), n, sa.data_ptr() + 2, lcp.data_ptr(), s.cuda_stream)
    assert e.value.code == -1


def test_one_call_and_the_divsufsort_seam_agree(bwts, ctx, orc, gen):
    L = bwts.lib()
    x = gen.make("dna", 66, 500_000)
    want_sa, want_lcp = orc.sa_lcp(x)
    src = np.frombuffer(x, dtype=np.uint8)
    sa = np.full(len(x), -7, dtype=np.int32)
    lcp = np.full(len(x), -7, dtype=np.int32)
    assert L.bwts_b200_sa_lcp(src.ctypes.data, sa.ctypes.data, lcp.ctypes.data, len(x), 0) == 0
    assert np.array_equal(sa, want_sa) and np.array_equal(lcp, want_lcp)
    assert np.array_equal(bwts.suffix_array(x), want_sa)
    assert np.array_equal(ctx.sa_host(x), want_sa)
    assert L.bwts_b200_sa_lcp(src.ctypes.data, sa.ctypes.data, sa.ctypes.data, len(x), 0) == -1
    with pytest.raises(bwts.BwtsError):
        bwts.suffix_array_lcp(x, device=999)


def test_workspace_is_that_of_the_bwts(bwts, gen):
    x = gen.make("dna", 67, 3_000_000)
    with bwts.Context(0) as a, bwts.Context(0) as b:
        a.forward_host(x)
        b.sa_lcp_host(x)
        # the BWTS host call holds 2 bytes per byte of I/O, the SA + LCP host call 9
        assert b.stats()["arena_bytes"] <= a.stats()["arena_bytes"] + 7 * len(x) + (1 << 20)


# --------------------------------------------------------------------------- sizes

@pytest.mark.parametrize("n", [1 << 20, 256 << 20], ids=["1MiB", "256MiB"])
def test_all_one_byte_closed_form(bwts, n):
    """a^n: SA[r] = n-1-r, LCP[r] = r; one irreducible pair of length n-1 (the multi-CTA tier's whole GPU)"""
    import torch
    dev = torch.device("cuda:0")
    x = torch.full((n,), ord("a"), dtype=torch.uint8, device=dev)
    sa = torch.empty(n, dtype=torch.int32, device=dev)
    lcp = torch.empty(n, dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:
        c.sa_lcp_device(x.data_ptr(), n, sa.data_ptr(), lcp.data_ptr())
        torch.cuda.synchronize()
    r = torch.arange(n, dtype=torch.int32, device=dev)
    assert torch.equal(lcp, r)
    assert torch.equal(sa, n - 1 - r)


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype="<i4").tobytes()).hexdigest()


@pytest.mark.parametrize("name", ["C2", "C3", "C3F"])
def test_full_size_against_the_oracle(bwts, gen, name):
    gold = SA_LCP_FULLSIZE[name]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        sa, lcp = c.sa_lcp_host(x)
        assert _sha(sa) == gold["sa_sha256"]
        assert (int(lcp.max()), int(lcp.astype(np.int64).sum())) == (gold["lcp_max"], gold["lcp_sum"])
        assert _sha(lcp) == gold["lcp_sha256"]
        assert c.stats()["factors"] == 1


def check_on_gpu(x, sa, lcp, samples=1 << 16):
    """torch on the GPU: PLCP[i] >= PLCP[i-1] - 1 for every i, LCP[0] = 0, and for sampled rows r the suffixes
    SA[r-1] and SA[r] agree on LCP[r] bytes and the next byte orders them (or the smaller one has ended)"""
    import torch
    n = x.numel()
    dev = x.device
    assert int(lcp[0]) == 0 and int(lcp.min()) >= 0
    plcp = torch.empty_like(lcp)
    plcp[sa.long()] = lcp
    assert bool((plcp[1:] >= plcp[:-1] - 1).all())
    del plcp
    g = torch.Generator(device=dev)
    g.manual_seed(8)
    r = torch.randint(1, n, (samples,), device=dev, generator=g)
    a, b, l = sa[r - 1].long(), sa[r].long(), lcp[r].long()
    assert bool((l <= n - torch.maximum(a, b)).all())
    K = int(l.max()) + 1
    for k0 in range(0, K, 256):   # windows of 256 bytes of every sampled pair
        j = torch.arange(k0, min(K, k0 + 256), device=dev)
        pa, pb = a[:, None] + j, b[:, None] + j
        inside = j[None, :] < l[:, None]
        xa = x[pa.clamp(max=n - 1)]
        xb = x[pb.clamp(max=n - 1)]
        assert bool(((xa == xb) | ~inside).all())
    end_a, end_b = a + l, b + l
    ca = x[end_a.clamp(max=n - 1)].long()
    cb = x[end_b.clamp(max=n - 1)].long()
    assert bool(((end_a == n) | ((end_b < n) & (ca < cb))).all())


def test_full_size_c4(bwts, gen):
    """1 GiB DNA: the SA equals bwts_b200_sa_device's, the LCP array passes check_on_gpu"""
    import torch
    dev = torch.device("cuda:0")
    n = 1 << 30
    x = torch.frombuffer(bytearray(gen.make("dna", 4, n)), dtype=torch.uint8).to(dev)
    sa = torch.empty(n, dtype=torch.int32, device=dev)
    lcp = torch.empty(n, dtype=torch.int32, device=dev)
    sa2 = torch.empty(n, dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:
        c.sa_lcp_device(x.data_ptr(), n, sa.data_ptr(), lcp.data_ptr())
        c.sa_device(x.data_ptr(), n, sa2.data_ptr())
        torch.cuda.synchronize()
    assert torch.equal(sa, sa2)
    del sa2
    check_on_gpu(x, sa, lcp)
    del x, sa, lcp
    release_device_memory()


def release_device_memory():
    """hand torch's cached blocks back to the driver, so that the next test's memory gate sees them free"""
    import torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def test_largest_length(bwts, gen):
    """2^31 - 1 bytes: a second SA does not fit beside the workspace, so the SA is checked to be a permutation"""
    import torch
    n = (1 << 31) - 1
    release_device_memory()
    if torch.cuda.mem_get_info(0)[0] < 80 * n + (1 << 28):
        pytest.skip("needs 172 GB of free device memory")
    dev = torch.device("cuda:0")
    x = torch.frombuffer(bytearray(gen.make("dna", 7, n)), dtype=torch.uint8).to(dev)
    sa = torch.empty(n, dtype=torch.int32, device=dev)
    lcp = torch.empty(n, dtype=torch.int32, device=dev)
    with bwts.Context(0) as c:
        c.sa_lcp_device(x.data_ptr(), n, sa.data_ptr(), lcp.data_ptr())
        torch.cuda.synchronize()
    assert int(sa.min()) == 0
    seen = torch.zeros(n, dtype=torch.bool, device=dev)
    seen[sa.long()] = True
    assert bool(seen.all())
    del seen
    torch.cuda.empty_cache()
    check_on_gpu(x, sa, lcp)
    del x, sa, lcp
    release_device_memory()

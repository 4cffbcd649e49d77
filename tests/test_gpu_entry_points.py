"""GPU test of what every entry point reports in bwts_b200_stats: each host form on a 1 MiB text times its
transform (total_ms, launches) apart from its staging copies (h2d_ms, and d2h_ms wherever it copies something
back), and each device form, on a caller stream, reports no copies.  Run on a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N = 1 << 20


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def inputs(ctx, gen):
    """the text and what the inverse, decoding and FM query forms take as input"""
    x = gen.make("text", 7, N)
    bwts_out = ctx.forward_host(x)
    bwt_out, bwt_primary = ctx.bwt_forward_host(x)
    div_out, div_primary = ctx.divbwt_forward_host(x)
    factors = ctx.lz77_host(x)
    fm = ctx.fm_build_host(x)
    pats = [x[k:k + 8] for k in range(0, N, N // 64)]
    lo, hi = ctx.fm_count_host(fm, pats)
    yield dict(x=x, bwts=bwts_out, bwt=(bwt_out, bwt_primary), div=(div_out, div_primary), factors=factors, fm=fm,
               pats=pats, lo=lo, hi=hi)
    fm.close()


# host form -> (call, copies something back)
HOST = {
    "forward": (lambda c, i: c.forward_host(i["x"]), True),
    "inverse": (lambda c, i: c.inverse_host(i["bwts"]), True),
    "bwt_forward": (lambda c, i: c.bwt_forward_host(i["x"]), True),
    "bwt_inverse": (lambda c, i: c.bwt_inverse_host(*i["bwt"]), True),
    "divbwt_forward": (lambda c, i: c.divbwt_forward_host(i["x"]), True),
    "divbwt_inverse": (lambda c, i: c.divbwt_inverse_host(*i["div"]), True),
    "sa": (lambda c, i: c.sa_host(i["x"]), True),
    "sa_lcp": (lambda c, i: c.sa_lcp_host(i["x"]), True),
    "lpf": (lambda c, i: c.lpf_host(i["x"]), True),
    "lz77": (lambda c, i: c.lz77_host(i["x"]), True),
    "lz77_decode": (lambda c, i: c.lz77_decode_host(i["factors"], N), True),
    "fm_build": (lambda c, i: c.fm_build_host(i["x"]).close(), False),
    "fm_count": (lambda c, i: c.fm_count_host(i["fm"], i["pats"]), True),
    "fm_locate": (lambda c, i: c.fm_locate_host(i["fm"], i["lo"], i["hi"]), True),
}


@pytest.mark.parametrize("name", list(HOST))
def test_host_form_times_its_copies_apart(ctx, inputs, name):
    call, copies_back = HOST[name]
    call(ctx, inputs)
    st = ctx.stats()
    assert st["total_ms"] > 0 and st["launches"] > 0, st
    assert st["h2d_ms"] > 0, st
    if copies_back:
        assert st["d2h_ms"] > 0, st
    else:
        assert st["d2h_ms"] == 0, st


def _device_calls(torch, keep):
    """device form -> call(ctx, inputs, stream); every tensor a call uses is held in keep until it is done"""
    def t(a):
        keep.append(torch.tensor(np.asarray(a), device="cuda"))
        return keep[-1].data_ptr()
    u8 = lambda b: t(np.frombuffer(b, dtype=np.uint8).copy())
    out8 = lambda: t(np.empty(N, dtype=np.uint8))
    out32 = lambda: t(np.empty(N, dtype=np.int32))

    def fm_count(c, i, s):
        pat = np.frombuffer(b"".join(i["pats"]), dtype=np.uint8).copy()
        off = np.zeros(len(i["pats"]) + 1, dtype=np.int64)
        np.cumsum([len(p) for p in i["pats"]], out=off[1:])
        c.fm_count_device(i["fm"], t(pat), len(pat), t(off), len(i["pats"]), t(np.empty(2 * len(i["pats"]), np.int32)), s)

    def fm_locate(c, i, s):
        rng = np.empty(2 * len(i["lo"]), dtype=np.int32)
        rng[0::2], rng[1::2] = i["lo"], i["hi"]
        cap = int((i["hi"].astype(np.int64) - i["lo"]).sum())
        c.fm_locate_device(i["fm"], t(rng), len(i["lo"]), t(np.empty(max(cap, 1), np.int32)), cap, s)

    return {
        "forward": lambda c, i, s: c.forward_device(u8(i["x"]), N, out8(), s),
        # at an odd address: the text is copied into the arena first
        "forward_unaligned": lambda c, i, s: c.forward_device(u8(b"\0" + i["x"]) + 1, N, out8(), s),
        "inverse": lambda c, i, s: c.inverse_device(u8(i["bwts"]), N, out8(), s),
        "bwt_forward": lambda c, i, s: c.bwt_forward_device(u8(i["x"]), N, out8(), s),
        "bwt_inverse": lambda c, i, s: c.bwt_inverse_device(u8(i["bwt"][0]), N, i["bwt"][1], out8(), s),
        "divbwt_forward": lambda c, i, s: c.divbwt_forward_device(u8(i["x"]), N, out8(), s),
        "divbwt_inverse": lambda c, i, s: c.divbwt_inverse_device(u8(i["div"][0]), N, i["div"][1], out8(), s),
        "sa": lambda c, i, s: c.sa_device(u8(i["x"]), N, out32(), s),
        "sa_lcp": lambda c, i, s: c.sa_lcp_device(u8(i["x"]), N, out32(), out32(), s),
        "lpf": lambda c, i, s: c.lpf_device(u8(i["x"]), N, out32(), out32(), s),
        "lz77": lambda c, i, s: c.lz77_device(u8(i["x"]), N, t(np.empty((N, 2), np.int32)), N, s),
        "lz77_decode": lambda c, i, s: c.lz77_decode_device(t(i["factors"]), len(i["factors"]), N, out8(), s),
        "fm_build": lambda c, i, s: c.fm_build_device(u8(i["x"]), N, 32, s).close(),
        "fm_count": fm_count,
        "fm_locate": fm_locate,
    }


DEVICE = ["forward", "forward_unaligned", "inverse", "bwt_forward", "bwt_inverse", "divbwt_forward", "divbwt_inverse",
          "sa", "sa_lcp", "lpf", "lz77", "lz77_decode", "fm_build", "fm_count", "fm_locate"]


@pytest.mark.parametrize("name", DEVICE)
def test_device_form_reports_no_copies(ctx, inputs, name):
    torch = pytest.importorskip("torch")
    keep = []
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):  # the inputs' copies, the call and its outputs all on the caller's stream
        _device_calls(torch, keep)[name](ctx, inputs, s.cuda_stream)
    s.synchronize()
    st = ctx.stats()
    assert st["total_ms"] > 0 and st["launches"] > 0, st
    assert st["h2d_ms"] == 0 and st["d2h_ms"] == 0, st

"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle and the
golden vectors made by the unmodified reference.  Bit-exact (bytes and 32-bit indices;
there is no floating point on this path).  Run on a B200: python -m pytest tests -m gpu
"""
import json
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

import helpers

pytestmark = pytest.mark.gpu

GOLDEN = json.loads((Path(__file__).parent / "golden" / "vectors.json").read_text())
# SHA-256 of the unmodified reference's forward output at the full BASELINE sizes (make_fullsize_golden.py)
FULLSIZE = json.loads((Path(__file__).parent / "golden" / "fullsize.json").read_text())


def golden_input(v, gen):
    if "input" in v:
        return bytes.fromhex(v["input"])
    spec = v["spec"]
    if "kind" in spec:
        data = gen.make(spec["kind"], spec["seed"], spec["n"])
    else:
        data = helpers.families(spec["n"])[spec["family"]]
    assert helpers.sha256(data) == v["input_sha256"]
    return data


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def default_tuning(bwts):
    bwts.tune(0, 0)
    bwts.tune(1, 0)
    yield
    bwts.tune(0, 0)
    bwts.tune(1, 0)


def test_golden_vectors_forward_and_inverse(bwts, ctx, gen):
    """every vector produced by the reference's own mk_bwts / unbwts binaries"""
    for v in GOLDEN:
        x = golden_input(v, gen)
        fwd = ctx.forward_host(x)
        inv = ctx.inverse_host(x)
        if "fwd" in v:
            assert fwd == bytes.fromhex(v["fwd"]), v["name"]
            assert inv == bytes.fromhex(v["inv"]), v["name"]
        else:
            assert helpers.sha256(fwd) == v["fwd_sha256"], v["name"]
            assert helpers.sha256(inv) == v["inv_sha256"], v["name"]


@pytest.mark.parametrize("chunk,shift", [(1, 31), (7, 30), (64, 28), (0, 0)])
def test_golden_small_with_tiny_chunks(bwts, ctx, gen, chunk, shift):
    """same vectors with the Lyndon chunk and splitter density forced small, so that inputs
    of a few bytes already cross chunk / sublist boundaries"""
    bwts.tune(0, chunk)
    bwts.tune(1, shift)
    for v in GOLDEN:
        if v["n"] > 70_000:
            continue
        x = golden_input(v, gen)
        fwd = ctx.forward_host(x)
        inv = ctx.inverse_host(x)
        if "fwd" in v:
            assert fwd == bytes.fromhex(v["fwd"]), v["name"]
            assert inv == bytes.fromhex(v["inv"]), v["name"]
        else:
            assert helpers.sha256(fwd) == v["fwd_sha256"], v["name"]
            assert helpers.sha256(inv) == v["inv_sha256"], v["name"]


@pytest.mark.parametrize("n", [1, 2, 3, 255, 256, 257, 2047, 2048, 2049, 4095, 4096, 4097, 4607, 4608, 4609,
                               8191, 8192, 8193, 9216, 65535, 65536, 65537, 14 * 4608])  # 4608 = onesweep tile
def test_families_at_tile_edges(bwts, ctx, oracle, n):
    bwts.tune(0, 512)
    bwts.tune(1, 29)
    for name, x in helpers.families(n).items():
        assert ctx.forward_host(x) == oracle.forward(x), (name, n)
        assert ctx.inverse_host(x) == oracle.inverse(x), (name, n)


def test_random_small_against_oracle(bwts, ctx, oracle):
    rng = np.random.default_rng(123)
    bwts.tune(0, 16)
    bwts.tune(1, 30)
    for _ in range(300):
        n = int(rng.integers(1, 3000))
        sigma = int(rng.choice([1, 2, 3, 4, 16, 256]))
        x = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
        assert ctx.forward_host(x) == oracle.forward(x), x[:64]
        assert ctx.inverse_host(x) == oracle.inverse(x), x[:64]


@pytest.mark.parametrize("kind,seed,n", [("random", 11, 1 << 20), ("text", 12, (1 << 22) + 12345),
                                         ("tiled", 13, 5 << 20), ("dna", 14, (1 << 23) - 1),
                                         ("fibonacci", 0, 3_000_001)])
def test_generated_medium_against_oracle(ctx, oracle, gen, kind, seed, n):
    x = gen.make(kind, seed, n)
    y = ctx.forward_host(x)
    assert y == oracle.forward(x)
    assert ctx.inverse_host(y) == x
    assert ctx.inverse_host(x) == oracle.inverse(x)


def test_adversarial_one_mib(bwts, ctx, oracle):
    n = 1 << 20
    for name, x in helpers.families(n).items():
        y = ctx.forward_host(x)
        assert y == oracle.forward(x), name
        assert ctx.inverse_host(y) == x, name


def test_full_size_properties_64mib(ctx, gen):
    """BASELINE configs[1] at full size: size-independent properties (the oracle comparison
    at this size lives in bench.py's cpu_baseline sample)"""
    n = 64 << 20
    x = gen.make("text", 2, n)
    assert helpers.sha256(x) == FULLSIZE["C2"]["input_sha256"]
    y = ctx.forward_host(x)
    assert helpers.sha256(y) == FULLSIZE["C2"]["fwd_sha256"], "differs from the reference's mk_bwts output"
    assert len(y) == n and y[0] == x[-1]
    assert np.array_equal(np.bincount(np.frombuffer(x, np.uint8), minlength=256),
                          np.bincount(np.frombuffer(y, np.uint8), minlength=256))
    assert ctx.inverse_host(y) == x
    # bijectivity the other way round: forward(inverse(x)) == x for an arbitrary string
    assert ctx.forward_host(ctx.inverse_host(x)) == x


@pytest.mark.parametrize("kind,seed,n", [("tiled", 3, 256 << 20), ("dna", 4, 1 << 30)])
def test_full_size_properties_c3_c4(bwts, gen, kind, seed, n):
    """BASELINE configs[2] and configs[3] at full size (256 MiB tiled text, 1 GiB DNA): SHA-256 of the
    forward output equals the unmodified reference's (tests/golden/fullsize.json), round trip,
    out[0] == x[-1], byte histogram; 1 GiB also runs the binned emit"""
    x = gen.make(kind, seed, n)
    gold = FULLSIZE["C3" if kind == "tiled" else "C4"]
    assert gold["n"] == n and helpers.sha256(x) == gold["input_sha256"]
    xa = np.frombuffer(x, np.uint8)
    with bwts.Context(0) as c:
        y = c.forward_host(x)
        st = c.stats()
        assert helpers.sha256(y) == gold["fwd_sha256"], "differs from the reference's mk_bwts output"
        assert len(y) == n and y[0] == x[-1]
        ya = np.frombuffer(y, np.uint8)
        assert np.array_equal(np.bincount(xa, minlength=256), np.bincount(ya, minlength=256))
        assert st["rounds"] >= 5 and st["factors"] >= 1
        assert st["binned_rounds"] >= 4, "later re-ranks that move most of their ranks go through the bin pass"
        back = c.inverse_host(y)
        assert np.array_equal(np.frombuffer(back, np.uint8), xa)
        del back, y


def test_largest_length_the_reference_accepts(gen):
    """len = 2^31 - 1, the top of the reference's range (`int` / `saidx_t`): forward through the tools, SHA-256
    against the unmodified reference's output where tests/golden/fullsize.json has it (C7: 16 minutes and 21 GB
    of host memory for the reference), inverse back to the exact input.  157 GB of device workspace."""
    import hashlib
    import shutil
    import tempfile
    import torch
    n = (1 << 31) - 1
    if torch.cuda.mem_get_info(0)[0] < 73 * n + (1 << 28):
        pytest.skip("needs 157 GB of free device memory")
    gold = FULLSIZE.get("C7")
    bindir = helpers.PKG / "bin"
    td = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        src, mid, back = (os.path.join(td, f) for f in ("in", "mid", "back"))
        x = gen.make("dna", 7, n)
        if gold:
            assert gold["n"] == n and helpers.sha256(x) == gold["input_sha256"]
        with open(src, "wb") as f:
            f.write(x)
        p = subprocess.run([str(bindir / "mk_bwts"), src, mid], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        assert os.path.getsize(mid) == n
        if gold:
            h = hashlib.sha256()
            with open(mid, "rb") as f:
                for blk in iter(lambda: f.read(1 << 24), b""):
                    h.update(blk)
            assert h.hexdigest() == gold["fwd_sha256"], "differs from the reference's mk_bwts output"
        p = subprocess.run([str(bindir / "unbwts"), mid, back], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        with open(back, "rb") as f:
            assert f.read() == x
    finally:
        shutil.rmtree(td, ignore_errors=True)


def test_full_size_c6_above_2_30_through_the_tools(gen):
    """the reference accepts any len < 2^31 (mk_bwts_sa.c:26-27, unbwts.c:12-13): a 1.5 GiB DNA file goes through
    the drop-in tools, `bin/mk_bwts in out` then `bin/unbwts out back`; the forward file's SHA-256 equals
    the unmodified reference's (tests/golden/fullsize.json, 748 s of one host core), the round trip is exact,
    and the diagnostics line reports the workspace per input byte"""
    import hashlib
    import re
    import shutil
    import tempfile
    if "C6" not in FULLSIZE:
        pytest.skip("tests/golden/fullsize.json has no C6 entry")
    gold = FULLSIZE["C6"]
    bindir = helpers.PKG / "bin"
    td = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        src, mid, back = (os.path.join(td, f) for f in ("in", "mid", "back"))
        x = gen.make(gold["kind"], gold["seed"], gold["n"])
        assert helpers.sha256(x) == gold["input_sha256"]
        with open(src, "wb") as f:
            f.write(x)
        env = dict(os.environ, BWTS_B200_TIMINGS="1")
        p = subprocess.run([str(bindir / "mk_bwts"), src, mid], capture_output=True, text=True, env=env)
        assert p.returncode == 0, p.stderr
        m = re.search(r"workspace bytes/byte: ([0-9.]+)", p.stderr)
        assert m and 60.0 <= float(m.group(1)) <= 75.0, p.stderr
        h = hashlib.sha256()
        with open(mid, "rb") as f:
            for blk in iter(lambda: f.read(1 << 24), b""):
                h.update(blk)
        assert h.hexdigest() == gold["fwd_sha256"], "differs from the reference's mk_bwts output"
        p = subprocess.run([str(bindir / "unbwts"), mid, back], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        with open(back, "rb") as f:
            assert f.read() == x
    finally:
        shutil.rmtree(td, ignore_errors=True)


def test_oracle_sample_16mib(ctx, oracle, gen):
    x = gen.make("text", 2, 16 << 20)
    assert ctx.forward_host(x) == oracle.forward(x)


def test_blocks_equal_concatenated_single_blocks(bwts, oracle, gen):
    """the in-process dealer (run_blocks: one host thread, context and pipeline per device) over ALL
    devices of the box, ragged last block, against the per-block oracle output"""
    x = gen.make("text", 21, 3_000_000)
    b = 1 << 20
    want = b"".join(oracle.forward(x[o:o + b]) for o in range(0, len(x), b))
    ndev = bwts.device_count()
    devs = list(range(ndev))
    got = bwts.forward_blocks(x, b, devices=devs)
    assert got == want, f"forward_blocks over {ndev} device(s)"
    assert bwts.inverse_blocks(got, b, devices=devs) == x, f"inverse_blocks over {ndev} device(s)"
    # block_len <= 0 means the reference's behaviour: one block
    assert bwts.forward_blocks(x, 0) == oracle.forward(x)


def test_dealer_needs_two_devices(bwts, oracle, gen):
    """the multi-device path proper: more blocks than devices, ragged tail, every device used, device
    lists in both orders.  Skipped (explicitly, not silently narrowed) on a one-GPU box."""
    ndev = bwts.device_count()
    if ndev < 2:
        pytest.skip(f"needs >= 2 CUDA devices, this box has {ndev}")
    x = gen.make("dna", 22, 7 * (1 << 20) + 4321)
    b = 1 << 20
    want = b"".join(oracle.forward(x[o:o + b]) for o in range(0, len(x), b))
    for devs in (list(range(ndev)), list(range(ndev))[::-1], [1, 0]):
        got = bwts.forward_blocks(x, b, devices=devs)
        assert got == want, f"forward_blocks, devices {devs}"
        assert bwts.inverse_blocks(got, b, devices=devs) == x, f"inverse_blocks, devices {devs}"


@pytest.mark.parametrize("block", range(8))
def test_full_size_c5_blocks(bwts, gen, block):
    """BASELINE configs[4]: each of the eight 256 MiB blocks of the multi-block file (seeds 50..57),
    SHA-256 of the forward output == the unmodified reference's, and the round trip"""
    gold = FULLSIZE[f"C5_{block}"]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        y = c.forward_host(x)
        assert helpers.sha256(y) == gold["fwd_sha256"], "differs from the reference's mk_bwts output"
        assert c.inverse_host(y) == x


def test_full_size_fibonacci_256mib(bwts, gen):
    """SURVEY 8(d)'s stress variant of configs[2]: the 256 MiB Fibonacci word"""
    if "C3F" not in FULLSIZE:
        pytest.skip("tests/golden/fullsize.json has no C3F entry (the reference run did not finish)")
    gold = FULLSIZE["C3F"]
    x = gen.make(gold["kind"], gold["seed"], gold["n"])
    assert helpers.sha256(x) == gold["input_sha256"]
    with bwts.Context(0) as c:
        y = c.forward_host(x)
        assert helpers.sha256(y) == gold["fwd_sha256"], "differs from the reference's mk_bwts output"
        assert c.inverse_host(y) == x


def test_onesweep_tile_shapes(bwts, ctx, oracle, gen):
    """every compiled shape of the onesweep kernel (tune 2: 0 = 384x12 with a 2-word look-back
    window, 1 = 512x8, 2 = 256x16, 3 / 4 = 384x12 with 8 / 4 words) sorts identically"""
    cases = [gen.make("text", 95, 1_300_000), gen.make("random", 96, 300_000), helpers.families(70_001)["ww"],
             helpers.families(4608 * 3)["random4"]]
    try:
        for shape in (1, 2, 3, 4, 0):
            bwts.tune(2, shape)
            bwts.tune(8, 1)   # keep the large-group set on the radix path so that every round sorts
            for x in cases:
                assert ctx.forward_host(x) == oracle.forward(x), (shape, len(x))
    finally:
        bwts.tune(2, 0)
        bwts.tune(8, 0)


def test_binned_rank_scatter_forced_on_small_inputs(bwts, ctx, oracle, gen):
    """first re-rank: ranks binned by text region with one u32 onesweep pass, then scattered
    (default for >= 4 Mi bytes); forced here so that few-byte inputs cross the bin edges"""
    bwts.tune(7, 2)
    try:
        for n in (256, 257, 1000, 3072, 3073, 70_001, 1 << 20):
            for name, x in helpers.families(n).items():
                assert ctx.forward_host(x) == oracle.forward(x), (name, n)
        x = gen.make("text", 25, 3_000_001)
        assert ctx.forward_host(x) == oracle.forward(x)
        assert np.array_equal(bwts.suffix_array(x[:500_000]), oracle.suffix_array(x[:500_000]))
    finally:
        bwts.tune(7, 0)
    bwts.tune(7, 1)
    try:
        x = gen.make("dna", 26, 5_000_000)
        assert ctx.forward_host(x) == oracle.forward(x)
    finally:
        bwts.tune(7, 0)


def test_initial_sort_histograms_from_window_counts(bwts, ctx, oracle, gen):
    """the digit histograms of the initial sort come from one histogram of the leading symbols of the keys
    (k_init_keys + k_digit_hists) for alphabets of 1-4, 6 and 8 bits per symbol, from k_radix_hist otherwise
    (tune 21 = 1: always); the bits the whole symbols leave free in the key hold the top of one more symbol
    (tune 22 = 1: off); every alphabet width, many short factors (the rotation wraps inside the key), narrow
    keys (tune 6)"""
    rng = np.random.default_rng(21)
    cases = []
    for sigma in (1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65, 128, 129, 256):
        for n in (1, 5, 4097, 300_001):
            cases.append((f"iid{sigma}", rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()))
    cases.append(("descending", bytes(sorted(rng.integers(0, 256, size=200_000, dtype=np.uint8).tobytes(), reverse=True))))
    cases.append(("descending4", bytes(sorted(rng.integers(97, 101, size=100_000, dtype=np.uint8).tobytes(), reverse=True))))
    cases.append(("short factors", b"".join(bytes([255 - (i % 200)]) + b"ab" * (i % 7) for i in range(20_000))))
    cases.append(("dna", gen.make("dna", 33, 3_000_000)))
    cases.append(("text", gen.make("text", 34, 2_500_000)))
    want = {name + str(len(x)): oracle.forward(x) for name, x in cases}
    try:
        for hist, partial in ((0, 0), (1, 0), (0, 1), (1, 1)):
            for keybits in (0, 40, 17):
                bwts.tune(21, hist)
                bwts.tune(22, partial)
                bwts.tune(6, keybits)
                for name, x in cases:
                    if (keybits or partial) and len(x) > 400_000:
                        continue
                    assert ctx.forward_host(x) == want[name + str(len(x))], (name, len(x), hist, partial, keybits)
    finally:
        bwts.tune(21, 0)
        bwts.tune(22, 0)
        bwts.tune(6, 0)


def test_window_histogram_packed_counts_do_not_overflow(bwts, ctx):
    """7-bit alphabets count the leading symbol pairs in 16-bit halves of shared-memory words, flushed every 31
    tiles: 48 MiB in which 99 % of the bytes are one symbol put ~62 k counts per flush on a single bin.  Checked
    against the path without the window histogram (tune 21 = 1) and by the round trip."""
    rng = np.random.default_rng(77)
    n = 48 << 20
    x = np.full(n, 120, dtype=np.uint8)
    hits = rng.integers(0, n, size=n // 100)
    x[hits] = rng.integers(40, 110, size=len(hits), dtype=np.uint8)   # 70 other symbols: 71 distinct bytes, 7 bits
    x = x.tobytes()
    got = ctx.forward_host(x)
    assert ctx.stats()["alphabet_bits"] == 7
    bwts.tune(21, 1)
    try:
        assert ctx.forward_host(x) == got
    finally:
        bwts.tune(21, 0)
    assert ctx.inverse_host(got) == x


def test_binned_rank_scatter_in_later_rounds(bwts, ctx, oracle, gen):
    """re-ranks after the first one also send their ranks through the bin pass when a third of the set's ranks moved
    in the round before (inputs of 128 Mi bytes and more; both the large-group and the small-group set); tune 7 = 4
    forces it for every re-rank so that small and sparse sets cross the counted-bin path too, 3 keeps it to the
    first re-rank"""
    fam = helpers.families(70_001)
    cases = [gen.make("tiled", 90, 6_000_000), helpers.fibonacci_word(5_000_000), gen.make("dna", 91, 4_500_000),
             gen.make("text", 92, 4_200_000), fam["ww"], fam["runs"], fam["thue_morse"], fam["random2"],
             (b"abcab" * 50_000) + b"b", bytes(1000), b"ab" * 130]
    want = [oracle.forward(x) for x in cases]
    try:
        for mode in (4, 3, 0):
            bwts.tune(7, mode)
            later = 0
            for x, w in zip(cases, want):
                assert ctx.forward_host(x) == w, (mode, len(x))
                later += max(0, ctx.stats()["binned_rounds"] - 1)
            if mode == 4:
                assert later >= 10, "forced: the later re-ranks must have used the bin pass"
            if mode == 3:
                assert later == 0
            if mode == 0:
                assert later == 0, "below 128 Mi bytes only the first re-rank is binned (the 256 MiB / 1 GiB tests see the rest)"
        # linear mode (suffix array) through the same path
        bwts.tune(7, 4)
        x = cases[0][:1_500_000]
        assert np.array_equal(bwts.suffix_array(x), oracle.suffix_array(x))
    finally:
        bwts.tune(7, 0)


def test_cta_local_sort_path_and_radix_path_agree(bwts, ctx, oracle, gen):
    """rounds whose large-group set fits the CTA-local bitonic sort (default) and the global radix
    path for them (tune 8 = 1) must both equal the oracle; with the warp-local path off (tune 3)
    every live group goes through the CTA-local sort"""
    fam = helpers.families(300_000)
    cases = [gen.make("tiled", 80, 2_500_000), gen.make("dna", 81, 1_500_000), gen.make("text", 82, 1_000_000),
             fam["ww"], fam["runs"], fam["thue_morse"], fam["de_bruijn"], fam["random2"], helpers.fibonacci_word(200_000)]
    used = 0
    for x in cases:
        want = oracle.forward(x)
        for local_off in (0, 1):
            bwts.tune(3, local_off)
            bwts.tune(8, 0)
            a = ctx.forward_host(x)          # CTA-local sort = radix in shared memory (default)
            used += ctx.stats()["cta_rounds"]
            bwts.tune(18, 1)
            a2 = ctx.forward_host(x)         # CTA-local sort = the bitonic network
            bwts.tune(18, 0)
            bwts.tune(8, 1)
            b = ctx.forward_host(x)
            assert ctx.stats()["cta_rounds"] == 0
            bwts.tune(8, 0)
            bwts.tune(3, 0)
            assert a == want and a2 == want and b == want
    assert used > 0, "the CTA-local sort never ran"
    # suffix-array mode (linear successor) through the same kernel
    y = gen.make("tiled", 83, 700_000)
    assert np.array_equal(bwts.suffix_array(y), oracle.suffix_array(y))


def test_binned_emit_forced_on_small_inputs(bwts, ctx, oracle, gen):
    """emit binned by rank region (default from 512 Mi bytes), forced here: as one packed word per element
    (tune 9 = 2: in-bin rank bits | byte, the bin pass reads the text itself) and as (rank, byte) pairs in two
    u32 streams (3: round 1); rank windows (1) as the sibling"""
    try:
        for mode in (2, 3, 1):
            bwts.tune(9, mode)
            for n in (256, 257, 1000, 3073, 4608, 4609, 70_001):
                for name, x in helpers.families(n).items():
                    assert ctx.forward_host(x) == oracle.forward(x), (name, n, mode)
            for kind, seed, n in (("text", 27, 3_000_001), ("dna", 28, 2_000_003), ("tiled", 29, 1_500_000)):
                x = gen.make(kind, seed, n)
                assert ctx.forward_host(x) == oracle.forward(x), (kind, mode)
    finally:
        bwts.tune(9, 0)


def test_block_pipeline_many_ragged_blocks(bwts, oracle, gen):
    """per device: loader / compute / drainer overlap over many blocks (SURVEY 8f.1); pageable buffers
    go through the pinned chunk rings (blocks larger than one 8 MiB chunk and much smaller ones)"""
    x = gen.make("text", 22, 1_234_567)
    for b in (100_003, 65_536, 1_234_566):
        want = b"".join(oracle.forward(x[o:o + b]) for o in range(0, len(x), b))
        got = bwts.forward_blocks(x, b, devices=[0])
        assert got == want, b
        assert bwts.inverse_blocks(got, b, devices=[0]) == x, b
    # overlap off (one block at a time) gives the same bytes
    bwts.tune(5, 1)
    try:
        b = 100_003
        assert bwts.forward_blocks(x, b, devices=[0]) == b"".join(
            oracle.forward(x[o:o + b]) for o in range(0, len(x), b))
    finally:
        bwts.tune(5, 0)
    # blocks that span several ring chunks
    y = gen.make("dna", 23, 40_000_000)
    b = 17_000_000
    got = bwts.forward_blocks(y, b, devices=[0])
    assert got == b"".join(oracle.forward(y[o:o + b]) for o in range(0, len(y), b))
    assert bwts.inverse_blocks(got, b, devices=[0]) == y


def test_block_pipeline_pinned_buffers(bwts, oracle, gen):
    """pinned caller buffers are copied directly (no chunk ring)"""
    import torch
    x = gen.make("text", 24, 5_000_000)
    b = 700_001
    src = torch.frombuffer(bytearray(x), dtype=torch.uint8).pin_memory()
    mid = torch.empty_like(src).pin_memory()
    back = torch.empty_like(src).pin_memory()
    bwts.blocks_ptr(0, src.data_ptr(), len(x), b, mid.data_ptr(), devices=[0])
    assert bytes(mid.numpy()) == b"".join(oracle.forward(x[o:o + b]) for o in range(0, len(x), b))
    bwts.blocks_ptr(1, mid.data_ptr(), len(x), b, back.data_ptr(), devices=[0])
    assert bytes(back.numpy()) == x


def test_one_call_entry_points_and_errors(bwts, oracle):
    x = b"abracadabra" * 1000
    assert bwts.forward(x) == oracle.forward(x)
    assert bwts.inverse(x) == oracle.inverse(x)
    L = bwts.lib()
    buf = np.zeros(8, dtype=np.uint8)
    assert L.bwts_b200_forward(None, 8, buf.ctypes.data, 0) == -1
    assert L.bwts_b200_forward(buf.ctypes.data, 0, buf.ctypes.data, 0) == -1
    assert L.bwts_b200_forward(buf.ctypes.data, 8, buf.ctypes.data, 999) == -1
    assert L.bwts_b200_inverse(buf.ctypes.data, 1 << 31, buf.ctypes.data, 0) == -2


def test_device_resident_api_with_torch(bwts, ctx, oracle, gen):
    import torch
    x = gen.make("dna", 31, 2_000_000)
    dev = torch.device("cuda:0")
    d_in = torch.frombuffer(bytearray(x), dtype=torch.uint8).to(dev)
    d_out = torch.empty_like(d_in)
    d_back = torch.empty_like(d_in)
    stream = torch.cuda.current_stream(dev).cuda_stream
    ctx.forward_device(d_in.data_ptr(), len(x), d_out.data_ptr(), stream)
    ctx.inverse_device(d_out.data_ptr(), len(x), d_back.data_ptr(), stream)
    torch.cuda.synchronize()
    assert bytes(d_out.cpu().numpy()) == oracle.forward(x)
    assert bytes(d_back.cpu().numpy()) == x
    st = ctx.stats()
    assert st["launches"] > 0 and st["direction"] == 1


def test_device_api_accepts_unaligned_input(bwts, ctx, oracle, gen):
    """d_in at every offset 1..15 from a 16-byte boundary (a slice of a larger tensor): the text kernels
    read 16-byte vectors, the library must realign instead of faulting"""
    import torch
    dev = torch.device("cuda:0")
    x = gen.make("text", 33, 300_001)
    big = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    out = torch.zeros(len(x) + 64, dtype=torch.uint8, device=dev)
    want_f, want_i = oracle.forward(x), oracle.inverse(x)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for off in (1, 2, 3, 5, 8, 13, 15):
        view = big[off:off + len(x)]
        view.copy_(torch.frombuffer(bytearray(x), dtype=torch.uint8))
        o = out[(off * 7) % 16:(off * 7) % 16 + len(x)]
        ctx.forward_device(view.data_ptr(), len(x), o.data_ptr(), stream)
        torch.cuda.synchronize()
        assert bytes(o.cpu().numpy()) == want_f, off
        ctx.inverse_device(view.data_ptr(), len(x), o.data_ptr(), stream)
        torch.cuda.synchronize()
        assert bytes(o.cpu().numpy()) == want_i, off


def test_inverse_mark_modes_and_many_short_cycles(bwts, ctx, oracle, gen):
    """the staged walk marks reached elements with one count per 128 (default) or one bit each (tune 15 = 1);
    unreached elements are found from the short counts (few deficient blocks: candidates are tested one by
    one) or, when very many blocks are short (a^n: every element is its own cycle), by an exact marking walk"""
    rng = np.random.default_rng(13)
    cases = [b"a" * 100_000, b"ab" * 60_000, bytes(rng.integers(0, 2, size=200_000, dtype=np.uint8)),
             gen.make("text", 91, 1_000_000), gen.make("dna", 92, 1_500_000), helpers.fibonacci_word(120_000),
             bytes(np.repeat(rng.integers(0, 256, size=3000, dtype=np.uint8), 40))]
    try:
        for x in cases:
            want = oracle.inverse(x)
            for mark in (2, 1):
                bwts.tune(15, mark)
                for shift in (0, 22, 29):
                    bwts.tune(1, shift)
                    assert ctx.inverse_host(x) == want, (len(x), mark, shift)
    finally:
        bwts.tune(15, 0)
        bwts.tune(1, 0)


def test_inverse_fallback_budget_restarts_with_another_hash(bwts, ctx, oracle):
    """a cycle without splitters is walked by each of its members (L^2 steps): the fallback has a step budget,
    and when it runs out the inverse starts again with another hash multiplier and denser splitters.
    Input: 200 Lyndon factors of 8192 bytes each (first letter strictly smallest, decreasing from word to
    word); with splitter density 2^-12 about 13 % of the 8192-cycles hold no splitter."""
    rng = np.random.default_rng(5)
    L = 8192
    x = b"".join(bytes([c]) + bytes(rng.integers(c + 1, 256, size=L - 1, dtype=np.uint8)) for c in range(200, 0, -1))
    y = ctx.forward_host(x)
    assert y == oracle.forward(x) and ctx.stats()["factors"] == 200
    try:
        bwts.tune(1, 20)
        bwts.tune(16, 1 << 20)
        back = ctx.inverse_host(y)
        st = ctx.stats()
        assert back == x
        assert st["inverse_attempts"] >= 2 and st["factors"] == 200
        bwts.tune(16, 0)      # the default budget (32 n steps) lets the same input through without a restart
        bwts.tune(1, 24)
        assert ctx.inverse_host(y) == x and ctx.stats()["inverse_attempts"] == 1
    finally:
        bwts.tune(1, 0)
        bwts.tune(16, 0)


def test_two_contexts_share_one_gpu_concurrently(bwts, oracle, gen):
    """the C ABI allows one context per host thread on the same device: two threads, each with its own context
    and stream, run transforms at the same time -- forward against inverse, then forward against forward (two
    sets of look-back chains in flight, which only assume that each kernel's own CTAs start in index order)"""
    import threading
    xs = [gen.make("text", 61, 3_000_000), gen.make("dna", 62, 4_000_000)]
    fw = [oracle.forward(x) for x in xs]
    errors = []

    def worker(which, direction, rounds):
        try:
            with bwts.Context(0) as c:
                for _ in range(rounds):
                    if direction == 0:
                        assert c.forward_host(xs[which]) == fw[which], ("forward", which)
                    else:
                        assert c.inverse_host(fw[which]) == xs[which], ("inverse", which)
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    for plan in (((0, 0, 6), (1, 1, 6)), ((0, 0, 5), (1, 0, 5)), ((0, 1, 5), (1, 1, 5))):
        threads = [threading.Thread(target=worker, args=a) for a in plan]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors, errors


def test_suffix_array_seam(bwts, oracle, gen):
    for x in (b"banana", b"mississippi", b"a" * 1000, gen.make("text", 5, 200_000), gen.make("dna", 6, 300_000),
              helpers.fibonacci_word(50_000)):
        assert np.array_equal(bwts.suffix_array(x), oracle.suffix_array(x))


def test_cli_tools_match_reference_layout(oracle, gen, tmp_path):
    bindir = helpers.PKG / "bin"
    x = gen.make("text", 41, 500_000)
    src = tmp_path / "in.txt"
    src.write_bytes(x)
    out = subprocess.run([str(bindir / "mk_bwts"), str(src)], capture_output=True, check=True).stdout
    assert out == oracle.forward(x)  # stdout default
    dst = tmp_path / "out.bwts"
    subprocess.run([str(bindir / "mbwt_new"), str(src), str(dst)], check=True)
    assert dst.read_bytes() == oracle.forward(x)
    back = tmp_path / "back.txt"
    subprocess.run([str(bindir / "unbwts"), str(dst), str(back)], check=True)
    assert back.read_bytes() == x
    r = subprocess.run([str(bindir / "unbwts"), str(dst)], capture_output=True, check=True, cwd=tmp_path)
    assert r.stdout.startswith(b"Writing to ")
    name = r.stdout.decode().split("Writing to ", 1)[1].strip()
    assert name.startswith(str(dst) + "_") and Path(name).read_bytes() == x
    env = dict(os.environ, BWTS_B200_BLOCK="131072")
    out = subprocess.run([str(bindir / "mk_bwts"), str(src)], capture_output=True, check=True, env=env).stdout
    assert out == b"".join(oracle.forward(x[o:o + 131072]) for o in range(0, len(x), 131072))


def test_timings_use_the_reference_phase_labels(gen, tmp_path):
    """SURVEY 8f row 3: BWTS_B200_TIMINGS=1 prints the reference's `<label> time <seconds>` lines
    (-DSHOW_TIMINGS, /root/reference/mk_bwts_sa.c:13-22,50,62,124,168,190) with the reference's labels in the
    reference's order -- compared with what the unmodified timed reference binary prints for the same
    file -- then one line of per-transform diagnostics (mk_bwts_new_algo.c:127's counterpart)."""
    import re
    bindir = helpers.PKG / "bin"
    x = gen.make("dna", 77, 700_000)
    src, dst = tmp_path / "in", tmp_path / "out"
    src.write_bytes(x)
    env = dict(os.environ, BWTS_B200_TIMINGS="1")
    p = subprocess.run([str(bindir / "mk_bwts"), str(src), str(dst)], capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    pat = re.compile(r"^([A-Z][A-Za-z ]+) time (\d+\.\d{3})$")
    labels = [m.group(1) for m in (pat.match(ln) for ln in p.stderr.splitlines()) if m]
    stored = json.loads((Path(__file__).parent / "golden" / "reference_checks.json").read_text())["timed"]
    assert (stored["kind"], stored["seed"], stored["n"]) == ("dna", 77, len(x)) and helpers.sha256(x) == stored["input_sha256"]
    want = stored["labels"]
    assert helpers.sha256(dst.read_bytes()) == stored["fwd_sha256"], "differs from the reference's output"
    ref_timed = helpers.REF_DIR / "mk_bwts_timed"
    if ref_timed.exists():
        r = subprocess.run([str(ref_timed), str(src), str(tmp_path / "ref_out")], capture_output=True, text=True)
        assert r.returncode == 0
        ref_labels = [m.group(1) for m in (pat.match(ln) for ln in r.stderr.splitlines()) if m]
        assert ref_labels == want, "the reference's own marks"
        assert (tmp_path / "ref_out").read_bytes() == dst.read_bytes()
    assert [l for l in labels if l in want] == want, p.stderr
    diag = [ln for ln in p.stderr.splitlines() if ln.startswith("Factors:")]
    assert len(diag) == 1
    m = re.match(r"Factors:\s+(\d+); longest:\s+(\d+); alphabet bits: (\d+); initial depth: (\d+); "
                 r"live after initial sort:\s+(\d+); doubling rounds: (\d+) \(warp-local (\d+), CTA-local (\d+), tuple set (\d+)\); "
                 r"radix passes: (\d+); live sum: (\d+); workspace bytes/byte: ([0-9.]+)$", diag[0])
    assert m, diag[0]
    factors, longest, bits, depth, live0, rounds = (int(m.group(i)) for i in range(1, 7))
    assert factors >= 1 and 1 <= longest <= len(x) and bits == 2 and depth == 32 and rounds >= 1 and live0 <= len(x)
    assert int(m.group(11)) >= live0 > 0
    # the inverse tool: additive labels, same format
    p = subprocess.run([str(bindir / "unbwts"), str(dst), str(tmp_path / "back")], capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    labels = [m.group(1) for m in (pat.match(ln) for ln in p.stderr.splitlines()) if m]
    assert [l for l in labels if l != "Transform"] == ["Count bytes", "LF map", "Walk sublists", "Rank sublists", "Place bytes", "Write text"], p.stderr
    assert re.search(r"^Cycles:\s+%d; sublists:\s+\d+; unreached:\s+\d+;" % factors, p.stderr, re.M), p.stderr
    assert (tmp_path / "back").read_bytes() == x


def test_context_reuse_across_sizes(ctx, oracle, gen):
    """one context, large and small inputs interleaved: the workspace is re-laid-out per call
    and must not depend on what an earlier transform left behind (regression: stale keys in
    the look-back status region were read as live status words)"""
    seq = [("text", 2, 300_000), ("dna", 4, 100_000), ("random", 3, 700_001), ("dna", 4, 100_000),
           ("text", 8, 50_000), ("tiled", 3, 1_200_000), ("dna", 9, 33_333), ("text", 2, 300_000)]
    for kind, seed, n in seq:
        x = gen.make(kind, seed, n)
        y = ctx.forward_host(x)
        assert y == oracle.forward(x), (kind, seed, n)
        assert ctx.inverse_host(y) == x, (kind, seed, n)


def test_local_sort_path_and_radix_only_path_agree(bwts, ctx, oracle, gen):
    """forward with the warp-local sort of small groups (default) and with the global radix
    path only (tune 3 = 1) must both equal the oracle"""
    cases = [gen.make("dna", 77, 1_500_000), gen.make("text", 78, 1_000_000), gen.make("tiled", 79, 1_300_000),
             helpers.families(70_000)["ww"], helpers.families(70_000)["runs"], helpers.fibonacci_word(200_000)]
    for x in cases:
        want = oracle.forward(x)
        bwts.tune(3, 1)
        a = ctx.forward_host(x)
        ra = ctx.stats()["local_rounds"]
        bwts.tune(3, 0)
        b = ctx.forward_host(x)
        assert a == want and b == want
        assert ra == 0


def test_tuple_set_sizes_agree(bwts, ctx, oracle, gen):
    """the text-ordered tuple set (rings by text position, k_tuple_round / k_tuple_apply) switched off
    (tune 14 = 1), taking pairs only (2), its default (8) and everything the small-group set would take
    (32): all equal the oracle; suffix arrays (linear successor) through the same paths"""
    rng = np.random.default_rng(11)
    base = bytes(rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=40_000))
    copies = base + b"T" + base[5_000:30_000] + b"G" + base + base[100:20_000] + b"A" + base[5_000:30_000]
    cases = [gen.make("dna", 81, 2_500_000), gen.make("text", 82, 1_200_000), gen.make("tiled", 83, 1_100_000), copies,
             helpers.families(60_000)["ww"], helpers.families(60_000)["runs"], helpers.families(4097)["abab"],
             helpers.fibonacci_word(150_000), b"a" * 5000, gen.make("dna", 84, 4609)]
    try:
        for x in cases:
            want = oracle.forward(x)
            for tmode in (0, 1):   # one thread per member / one thread per group (rings marked with a head)
                bwts.tune(20, tmode)
                seen = {}
                for tmax in (1, 2, 8, 32):
                    bwts.tune(14, tmax)
                    assert ctx.forward_host(x) == want, (len(x), tmode, tmax)
                    seen[tmax] = ctx.stats()["tuple_rounds"]
                assert seen[1] == 0
        bwts.tune(20, 0)
        bwts.tune(14, 0)
        ctx.forward_host(cases[0])
        st = ctx.stats()
        assert st["tuple_rounds"] >= 3 and st["tuple_live_sum"] > len(cases[0]), "the DNA input must use the tuple set"
        for tmax in (1, 2, 32):
            bwts.tune(14, tmax)
            for x in (cases[3], cases[0][:300_000], helpers.fibonacci_word(50_000)):
                assert np.array_equal(bwts.suffix_array(x), oracle.suffix_array(x)), tmax
    finally:
        bwts.tune(14, 0)
        bwts.tune(20, 0)


def test_lyndon_suffix_sort_fallback(bwts, ctx, oracle, gen):
    """factor starts taken from the strict prefix minima of a GPU-built inverse suffix array
    (the reference's own criterion, mk_bwts_sa.c:126-129) -- the route periodic inputs take
    when the chunk kernels run out of budget -- forced here on every kind of input"""
    bwts.tune(4, 1)
    try:
        for v in GOLDEN:
            if v["n"] > 70_000 or "input" not in v:
                continue
            x = bytes.fromhex(v["input"])
            assert ctx.forward_host(x) == bytes.fromhex(v["fwd"]), v["name"]
            assert ctx.stats()["lyndon_fallback"] == 1
        for kind, seed, n in (("text", 3, 300_000), ("dna", 4, 200_000), ("tiled", 5, 500_000)):
            x = gen.make(kind, seed, n)
            assert ctx.forward_host(x) == oracle.forward(x), kind
        for name, x in helpers.families(65_537).items():
            assert ctx.forward_host(x) == oracle.forward(x), name
    finally:
        bwts.tune(4, 0)


def test_lyndon_scan_variants_agree(bwts, ctx, oracle, gen):
    """the chunk-minimum prefix scan: hierarchical with CTA-wide comparisons (default) and the Hillis-Steele
    levels of round 1 (tune 17 = 1), on inputs with short and with very long common prefixes between chunk
    minima (tiled text), with small chunks so that several levels exist"""
    cases = [gen.make("tiled", 85, 3_000_000), gen.make("text", 86, 2_000_000), gen.make("dna", 87, 2_000_000),
             helpers.fibonacci_word(300_000), helpers.families(200_000)["ww"], helpers.families(200_000)["descending"]]
    try:
        for x in cases:
            want = oracle.forward(x)
            for chunk in (0, 64, 16):
                bwts.tune(0, chunk)
                for scan in (0, 1, 2):
                    bwts.tune(17, scan)
                    assert ctx.forward_host(x) == want, (len(x), chunk, scan)
    finally:
        bwts.tune(17, 0)
        bwts.tune(0, 0)


def test_periodic_inputs_trigger_the_fallback_by_budget(bwts, ctx, oracle):
    """a^n and a short-period text at 8 MiB exhaust the chunk kernels' budget on their own"""
    n = 8 << 20
    for x in (b"a" * n, (b"abcabd" * (n // 6 + 1))[:n]):
        y = ctx.forward_host(x)
        assert ctx.stats()["lyndon_fallback"] == 1
        assert y == oracle.forward(x)
        assert ctx.inverse_host(y) == x

"""Decisions that depend on the data rather than on the length or a tune key, driven to their edges
on purpose and checked against a CPU reference of the same operation.

Forward: which set sorts a tied group in a doubling round (k_rerank, forward.cuh: the text-ordered
tuple set takes groups of at most tmax members, the warp-local sort groups of at most 32 that sit in
one re-rank tile, the large-group set everything else), whether k_ls_probe lets the large-group set be
sorted CTA-locally (no CTA owns more than LS_CAP = 8192 slots) or sends it to the onesweep passes, and
the finalize branch of each set when equal Lyndon factors leave ties that never split.
`round_structure` predicts the per-round counters and the probe verdict of every round exactly.

Inverse: splitters from the public hash, the cycles that hold none (their members are the unreached
elements), and with one count mark per 128 elements the number of short blocks, which chooses between
k_inv_verify_candidates (at most `cap` of them) and k_inv_walk_mark.  `inverse_prediction` computes
all of it from the LF map.

Inputs: `copies` (groups of exactly g members at every depth), `equal_factors` (w^g: g equal factors,
groups of g that never split, g cycles of |w|) and `factorization` (factor starts and cycle lengths
chosen by the caller).  The CPU tests check the reference against the oracle and each constructor's
premise; the GPU tests check the bytes and the path counters.
"""
import numpy as np
import pytest

import helpers
from model_gpu_algorithms import owned_ranges

LS_T = 4096          # live slots per CTA of k_local_sort_cta / k_local_sort_cta_radix
LS_CAP = 2 * LS_T    # most slots one CTA may own (k_ls_probe)
SPL_MUL = 0x9E3779B1  # splitter hash of the inverse's first attempt (inverse_core)


# --------------------------------------------------------------------------- CPU reference: forward

def key_layout(sigma):
    """bits per symbol code, whole symbols in the initial key (k0), top bits of the next symbol behind them"""
    bits = max(1, (sigma - 1).bit_length())
    k0 = 64 // bits
    return bits, k0, min(bits - 1, 64 - k0 * bits)


def round_structure(x, starts):
    """Prefix doubling with exact ranks on the rotations inside the Lyndon factors `starts`, stopped by the
    rules of forward_core: nothing live, a round that split no group, or k >= 2 * lmax.

    Returns rounds / first_live / live_sum as the stats count them, `layouts` (per round: the sizes of the
    tied groups in rank order, i.e. the live array of a set that holds every group), `verdicts` (per round:
    k_ls_probe accepts that layout) and `rank` (final rank of every position, ties broken by position)."""
    T = np.frombuffer(bytes(x), dtype=np.uint8)
    n = len(T)
    FS = np.append(np.asarray(starts, dtype=np.int64), n)
    pos = np.arange(n, dtype=np.int64)
    fid = np.searchsorted(FS, pos, side="right") - 1
    fs, fl = FS[fid], FS[fid + 1] - FS[fid]
    lmax = int(fl.max())
    present = np.zeros(256, dtype=bool)
    present[T] = True
    code = (np.cumsum(present) - 1).astype(np.uint64)
    bits, k0, extra = key_layout(int(present.sum()))

    def succ(k):
        return fs + (pos - fs + k) % fl

    key = np.zeros(n, dtype=np.uint64)
    for t in range(k0):
        key = (key << np.uint64(bits)) | code[T[succ(t)]]
    if extra:
        key = (key << np.uint64(extra)) | (code[T[succ(k0)]] >> np.uint64(bits - extra))
    cls = np.unique(key, return_inverse=True)[1].reshape(-1).astype(np.int64)

    rounds = first_live = live_sum = 0
    layouts, verdicts = [], []
    classes_before, k = 1, k0   # before the first re-rank the whole text is one group
    while True:
        sizes = np.bincount(cls)  # class ids are ranks: the sizes come in rank order
        split = len(sizes) != classes_before
        classes_before = len(sizes)
        tied = sizes[sizes >= 2]
        live = int(tied.sum())
        if live == 0 or not split or k >= 2 * lmax:
            break
        rounds += 1
        first_live = first_live or live
        live_sum += live
        layouts.append(tied)
        gst = np.repeat(np.cumsum(tied) - tied, tied)
        verdicts.append(all(hi - lo <= LS_CAP for lo, hi in owned_ranges(gst, LS_T)))
        pair = cls * len(sizes) + cls[succ(k)]
        cls = np.unique(pair, return_inverse=True)[1].reshape(-1).astype(np.int64)
        k *= 2
    rank = np.empty(n, dtype=np.int64)
    rank[np.lexsort((pos, cls))] = np.arange(n)
    return dict(rounds=rounds, first_live=first_live, live_sum=live_sum, layouts=layouts, verdicts=verdicts,
                rank=rank, factors=len(starts), longest_factor=lmax, bits=bits, k0=k0, extra=extra)


def emit(x, starts, rank):
    """out[rank[i]] = the byte before i in its factor (cyclically)"""
    T = np.frombuffer(bytes(x), dtype=np.uint8)
    n = len(T)
    FS = np.append(np.asarray(starts, dtype=np.int64), n)
    prev = np.arange(n, dtype=np.int64) - 1
    prev[FS[:-1]] = FS[1:] - 1
    out = np.empty(n, dtype=np.uint8)
    out[rank] = T[prev]
    return out.tobytes()


# --------------------------------------------------------------------------- CPU reference: inverse

def cycle_labels(lf):
    """smallest member of each element's cycle under lf (pointer jumping)"""
    lab = np.arange(len(lf), dtype=np.int64)
    p = lf.astype(np.int64)
    for _ in range(max(1, len(lf)).bit_length() + 1):
        lab = np.minimum(lab, lab[p])
        p = p[p]
    return lab


def splitter_mask(n, shift, mul=SPL_MUL):
    i = np.arange(n, dtype=np.uint64)
    return ((i * np.uint64(mul)) & np.uint64(0xFFFFFFFF)) >> np.uint64(shift) == 0


def steps_to_splitter(lf, spl):
    """steps k_inv_verify_candidates takes from each element to the first splitter on its prev chain
    (meaningless on cycles without one)"""
    idx = np.arange(len(lf), dtype=np.int64)
    f = np.where(spl, idx, lf.astype(np.int64))
    w = (~spl).astype(np.int64)
    for _ in range(max(1, len(lf)).bit_length() + 1):
        w = w + w[f]
        f = f[f]
    return w


def inverse_prediction(y, lf, lab, shift, count_marks):
    """What the inverse's first attempt reports for input y with splitter shift `shift`, and whether its
    fallback walks run out of their step budget (32 n steps) so that the inverse starts again.

    The budget counts whole units of 1024 steps per thread, and the attempt gives up once more units than
    (32 n) >> 10 are counted.  k_inv_self_walk runs one thread per 32-element word over the unreached
    elements, L - 1 steps each; with count marks and at most `cap` short blocks k_inv_verify_candidates runs
    first, one thread per element of a short block: L - 1 steps on a cycle without splitters, otherwise
    the steps to the first splitter on its chain."""
    n = len(y)
    spl = splitter_mask(n, shift)
    length = np.bincount(lab, minlength=n)
    has = np.bincount(lab, weights=spl, minlength=n) > 0
    unreached = ~has[lab]
    cyc_len = length[lab]
    blocks = np.unique(np.flatnonzero(unreached) >> 7)
    cap = max(4096, n >> 13)
    walk = np.bincount(np.arange(n) >> 5, weights=np.where(unreached, cyc_len - 1, 0))
    units = int((walk.astype(np.int64) >> 10).sum())
    if count_marks and 0 < len(blocks) <= cap:
        cand = (blocks[:, None] * 128 + np.arange(128)[None, :]).reshape(-1)
        cand = cand[cand < n]
        steps = np.where(unreached[cand], cyc_len[cand] - 1, steps_to_splitter(lf, spl)[cand])
        units += int((steps >> 10).sum())
    budget_k = max(1, min((32 * n) >> 10, 0xFFFFFFFE))
    return dict(splitters=int(spl.sum()), unreached=int(unreached.sum()), factors=int((length > 0).sum()),
                short_blocks=len(blocks), cap=cap, units=units, restart=units > budget_k)


def default_shift(n):
    return 25 if n >= (1 << 28) else 26


# --------------------------------------------------------------------------- constructors

def lyndon_word(length, rng, first=0):
    """`first`, then bytes drawn above it: every proper rotation starts higher, so the word is Lyndon"""
    assert length == 1 or first <= 254
    return bytes([first]) + rng.integers(first + 1, 256, size=length - 1, dtype=np.uint8).tobytes()


def copies(g, m, seed):
    """0x00 (the whole input is one Lyndon factor), then random filler over 1..255 holding g copies of one
    random block of m bytes; for g <= 255 every copy has its own preceding and its own following byte, so
    at every depth a tie group has exactly g members (the same offset in every copy) or one.  The filler
    ends with every byte value once: 8-bit codes, so the initial key holds 8 whole symbols and no partial
    one.  Gaps of 2..5 filler bytes keep g <= 33 copies under one re-rank tile (2048 slots) in the first
    re-rank, so that the route of a group never depends on where a tile border falls."""
    rng = np.random.default_rng(seed)
    block = rng.integers(1, 256, size=m, dtype=np.uint8).tobytes()
    pre, post = rng.permutation(np.arange(1, 256)), rng.permutation(np.arange(1, 256))
    parts = [b"\x00"]
    for c in range(g):
        parts.append(rng.integers(1, 256, size=int(rng.integers(2, 6)), dtype=np.uint8).tobytes())
        parts.append(bytes([pre[c % 255]]) + block + bytes([post[c % 255]]))
    parts.append(rng.permutation(np.arange(1, 256)).astype(np.uint8).tobytes())
    return b"".join(parts)


def equal_factors(w, g):
    """w^g for a Lyndon word w: g equal factors"""
    return bytes(w) * g


def factorization(lengths, seed):
    """Random Lyndon words of the given lengths, concatenated in non-increasing order: by the uniqueness of
    the Lyndon factorization these words are the factors.  Built from the last word back: a word keeps the
    first byte of the word after it when it can still be at least that word, otherwise the byte goes up."""
    rng = np.random.default_rng(seed)
    words = [b""] * len(lengths)
    after = b""  # sorts below every word
    for j in range(len(lengths) - 1, -1, -1):
        L = int(lengths[j])
        c = after[0] if after else 1
        while True:
            if c > (255 if L == 1 else 254):
                raise ValueError("the alphabet cannot hold this many non-increasing factors")
            w = bytearray(lyndon_word(L, rng, c))
            if bytes(w) >= after:
                break
            if L > 1 and len(after) > 1 and after[0] == c and after[1] < 255:
                w[1] = after[1] + 1   # same first byte, larger second byte: above `after`, still Lyndon
                break
            c += 1
        words[j] = after = bytes(w)
    return b"".join(words)


def starts_of(lengths):
    return np.concatenate(([0], np.cumsum(lengths)[:-1])).astype(np.int64)


def lengths_for_starts(starts, n):
    s = sorted(set(int(v) for v in starts if 0 < v < n) | {0})
    return np.diff(s + [n]).tolist()


def edge_starts(step, count):
    """factor starts at step*c - 1, step*c and step*c + 1"""
    return [step * c + d for c in range(1, count + 1) for d in (-1, 0, 1)]


# --------------------------------------------------------------------------- the cases

TMAX_G = (2, 7, 8, 9, 31, 32, 33, 64, 255)      # around tmax 2 / 8 / 32 and the warp-local limit of 32
COPIES_M = 40                                      # depths 8, 16, 32 tie; 64 resolves: three rounds
SPAN_G = (4095, 4096, 4097, 8191, 8192, 8193)      # group sizes around LS_T and LS_CAP
SPAN_W = 300                                       # |w| for w^g: > 128 byte values, 8-bit codes, k0 = 8
SPAN_COPIES_G = (4096, 6000, 8192, 8193)           # > 255 copies: mixed group sizes, both verdicts
SMALL_EQUAL_G = (2, 8, 9, 32, 33)
CYCLE_LENGTHS = (1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 4095, 4096, 4097)
CHUNKS = (1, 7, 64, 512)
# one-byte factors before 200 factors of 64 bytes: the 1-cycles take the top ranks in one run that starts on
# a 128-block edge (200 x 64 = 100 blocks), and 128 of them make one short block (a block holds about 2
# splitters); the 64-cycles short some of the 100 blocks below.  So 3995 + (0..100) <= 4096 short blocks,
# then 4097 + (0..100) > 4096: under and over cap = max(4096, n >> 13) at every splitter density
CAP_ONES = (3995 * 128, 4097 * 128)


def boundary_inputs():
    """factor starts at chunk edges (for the chunk sizes of CHUNKS) and at +-1 around the 4096-byte
    blocks of the coarse factor index (COARSE_BITS = 12)"""
    out = {}
    for step, count in ((7, 200), (64, 150), (512, 150)):
        lengths = lengths_for_starts(edge_starts(step, count), step * count + 5)
        out[f"chunk{step}"] = (factorization(lengths, 100 + step), lengths)
    lengths = lengths_for_starts([4096 * c + d for c in range(1, 25) for d in (-1, 1)], 4096 * 25 + 3)
    out["coarse4096"] = (factorization(lengths, 200), lengths)
    return out


def inverse_inputs():
    """name -> (input of the inverse, expected output)"""
    rng = np.random.default_rng(400)
    out = {}
    for L in CYCLE_LENGTHS:
        out[f"uniform{L}"] = factorization([L] * (40_000 // L if L < 4000 else 19), 300 + L)
    mixed = rng.choice(np.array(CYCLE_LENGTHS[:-3]), size=900).tolist() + [4095, 4096, 4097, 4096]
    rng.shuffle(mixed)
    out["mixed"] = factorization(mixed, 301)
    # a one-byte factor after a longer one needs a larger byte: the 1-cycles go last, in one run
    out["mixed_short"] = factorization(rng.choice(np.array([2, 31, 32, 33]), size=3000).tolist() + [1] * 500, 302)
    for L, g in ((32, 2000), (64, 700), (129, 400), (300, 150), (4097, 9)):
        out[f"equal{L}x{g}"] = equal_factors(lyndon_word(L, rng), g)
    cases = {name: (None, x) for name, x in out.items()}   # the fixture computes the forward of x
    for sigma, n in ((256, 100_000), (4, 77_777), (2, 50_001)):
        cases[f"bytes{sigma}"] = (rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes(), None)
    fam = helpers.families(65_537)
    for name in ("all_a", "abab", "fibonacci", "runs"):
        cases[name] = (fam[name], None)
    return cases


def cap_input(ones):
    return factorization([1] * ones + [64] * 200, 500)


# --------------------------------------------------------------------------- CPU tests

def test_round_structure_emits_the_oracle_transform(oracle):
    """the reference's final ranks give the oracle's BWTS: its round predictions come from a correct
    transform (families of several lengths, and 300 small random inputs over 1..256 symbols)"""
    for n in (1, 2, 3, 17, 64, 255, 1000, 4097):
        for name, x in helpers.families(n).items():
            starts = oracle.lyndon_starts(x)
            assert emit(x, starts, round_structure(x, starts)["rank"]) == oracle.forward(x), (name, n)
    rng = np.random.default_rng(1)
    for _ in range(300):
        n = int(rng.integers(1, 1500))
        sigma = int(rng.choice([1, 2, 3, 5, 16, 200, 256]))
        x = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
        starts = oracle.lyndon_starts(x)
        assert emit(x, starts, round_structure(x, starts)["rank"]) == oracle.forward(x), x[:32]


def test_round_structure_key_layout_matches_the_driver():
    """k0 whole codes and the top `extra` bits of the next one fill 64 bits (forward_core)"""
    assert key_layout(1) == (1, 64, 0)
    assert key_layout(4) == (2, 32, 0)
    assert key_layout(5) == (3, 21, 1)
    assert key_layout(33) == (6, 10, 4)
    assert key_layout(256) == (8, 8, 0)


@pytest.mark.parametrize("g", TMAX_G)
def test_copies_give_groups_of_exactly_g(oracle, g):
    x = copies(g, COPIES_M, g)
    starts = oracle.lyndon_starts(x)
    assert list(starts) == [0]
    assert g > 33 or len(x) <= 2048
    rs = round_structure(x, starts)
    assert rs["rounds"] == 3 and rs["first_live"] == g * (COPIES_M - 7)
    for sizes in rs["layouts"]:
        assert set(sizes.tolist()) == {g}


def test_equal_factors_give_g_factors_and_g_cycles(oracle):
    rng = np.random.default_rng(2)
    for L, g in ((SPAN_W, 2), (SPAN_W, 9), (SPAN_W, 33), (5, 7), (64, 40), (1, 6)):
        w = lyndon_word(L, rng)
        x = equal_factors(w, g)
        assert list(oracle.lyndon_starts(x)) == [L * j for j in range(g)]
        lab = cycle_labels(oracle.lf_map(oracle.forward(x)))
        assert sorted(np.bincount(lab)[np.unique(lab)].tolist()) == [L] * g


@pytest.mark.parametrize("g", SPAN_G)
def test_equal_factors_span_edges_predicted(oracle, span_cases, g):
    """one doubling round over groups of exactly g, then final ties; k_ls_probe accepts up to g = 8192"""
    x, rs = span_cases[g]
    assert rs["rounds"] == 1 and rs["first_live"] == rs["live_sum"] == len(x)
    assert set(rs["layouts"][0].tolist()) == {g}
    assert rs["verdicts"] == [g <= LS_CAP]
    assert (rs["bits"], rs["k0"]) == (8, 8)


def test_copies_span_sweep_holds_both_verdicts(span_copies):
    seen = [v for _, rs in span_copies.values() for v in rs["verdicts"]]
    assert True in seen and False in seen


def test_factorization_starts_and_cycles(oracle):
    rng = np.random.default_rng(3)
    cases = [[1], [5], [1, 1, 1], [3, 1, 1, 2, 1], rng.integers(1, 40, size=300).tolist(),
             rng.choice(np.array(CYCLE_LENGTHS), size=60).tolist()]
    cases += [lengths_for_starts(edge_starts(7, 30), 215), [1] * 1000 + [64] * 10]
    for lengths in cases:
        x = factorization(lengths, len(lengths))
        assert np.array_equal(oracle.lyndon_starts(x), starts_of(lengths)), lengths[:20]
        lab = cycle_labels(oracle.lf_map(oracle.forward(x)))
        assert sorted(np.bincount(lab)[np.unique(lab)].tolist()) == sorted(lengths)
    for name, (x, lengths) in boundary_inputs().items():
        assert np.array_equal(oracle.lyndon_starts(x), starts_of(lengths)), name


def test_inverse_prediction_against_a_plain_walk(oracle):
    """the vectorised prediction equals a cycle-by-cycle walk on small inputs"""
    rng = np.random.default_rng(4)
    for n, sigma, shift in ((1, 2, 26), (700, 2, 29), (3000, 4, 27), (5000, 256, 26), (4096, 1, 30)):
        y = rng.integers(0, sigma, size=n, dtype=np.uint8)
        lf = oracle.lf_map(y.tobytes())
        spl = [((i * SPL_MUL) & 0xFFFFFFFF) >> shift == 0 for i in range(n)]
        seen = [False] * n
        cycles = unreached = 0
        for s in range(n):
            if seen[s]:
                continue
            members, i = [], s
            while not seen[i]:
                seen[i] = True
                members.append(i)
                i = int(lf[i])
            cycles += 1
            if not any(spl[i] for i in members):
                unreached += len(members)
        p = inverse_prediction(y, lf, cycle_labels(lf), shift, False)
        assert (p["splitters"], p["factors"], p["unreached"]) == (sum(spl), cycles, unreached)
        assert spl[0]


def test_cap_inputs_straddle_the_short_block_cap(oracle, cap_cases):
    """one case under cap (k_inv_verify_candidates), one over it (k_inv_walk_mark)"""
    sides = []
    for ones, (x, y, lf, lab) in cap_cases.items():
        p = inverse_prediction(y, lf, lab, default_shift(len(y)), True)
        assert p["cap"] == 4096 and not p["restart"]
        sides.append(p["short_blocks"] > p["cap"])
    assert sides == [False, True]


# --------------------------------------------------------------------------- fixtures

@pytest.fixture(scope="module")
def span_cases(oracle):
    rng = np.random.default_rng(7)
    w = lyndon_word(SPAN_W, rng)
    out = {}
    for g in SPAN_G:
        x = equal_factors(w, g)
        out[g] = (x, round_structure(x, oracle.lyndon_starts(x)))
    return out


@pytest.fixture(scope="module")
def span_copies(oracle):
    out = {}
    for g in SPAN_COPIES_G:
        x = copies(g, 24, g)
        out[g] = (x, round_structure(x, oracle.lyndon_starts(x)))
    return out


@pytest.fixture(scope="module")
def cap_cases(oracle):
    out = {}
    for ones in CAP_ONES:
        x = cap_input(ones)
        y = oracle.forward(x)
        lf = oracle.lf_map(y)
        out[ones] = (x, y, lf, cycle_labels(lf))
    return out


# --------------------------------------------------------------------------- GPU tests

TUNE_KEYS = (0, 1, 3, 8, 9, 12, 13, 14, 15, 18, 20, 23)


@pytest.fixture(scope="module")
def ctx(bwts):
    assert bwts.device_count() >= 1, "no CUDA device: the product has no CPU path"
    c = bwts.Context(0)
    yield c
    c.close()


@pytest.fixture
def tuned(bwts):
    """tuned({key: value}) sets bwts_b200_tune keys; every key goes back to its default afterwards"""
    def apply(settings):
        for key in TUNE_KEYS:
            bwts.tune(key, settings.get(key, 0))
    yield apply
    for key in TUNE_KEYS:
        bwts.tune(key, 0)


def forward_checked(ctx, x, want, starts):
    y = ctx.forward_host(x)
    st = ctx.stats()
    assert y == want
    lens = np.diff(np.append(starts, len(x)))
    assert st["factors"] == len(starts) and st["longest_factor"] == int(lens.max())
    return st


def assert_rounds(st, rs, what):
    got = (st["rounds"], st["first_live"], st["live_sum"])
    assert got == (rs["rounds"], rs["first_live"], rs["live_sum"]), what


@pytest.fixture(scope="module")
def routing_cases(oracle):
    out = {}
    for g in TMAX_G:
        x = copies(g, COPIES_M, g)
        starts = oracle.lyndon_starts(x)
        out[g] = (x, oracle.forward(x), starts, round_structure(x, starts), oracle.suffix_array(x))
    return out


ROUTING_SETTINGS = {
    "default": {},
    "tmax2": {14: 2, 20: 0},
    "tmax8": {14: 8, 20: 0},
    "tmax32_heads": {14: 32, 20: 1},
    "no_local": {3: 1},
    "no_cta": {8: 1},
    "no_local_no_cta": {3: 1, 8: 1},
    "bitonic": {18: 1},
}


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(ROUTING_SETTINGS))
def test_group_routing_at_tmax_and_warp_limits(bwts, ctx, tuned, routing_cases, setting):
    """groups of exactly g members: the tuple set takes g <= tmax, the warp-local sort tmax < g <= 32, the
    large-group set g >= 33; the round counters equal the CPU reference in every setting"""
    s = ROUTING_SETTINGS[setting]
    tuned(s)
    for g, (x, want, starts, rs, sa) in routing_cases.items():
        st = forward_checked(ctx, x, want, starts)
        what = (setting, g)
        assert_rounds(st, rs, what)
        if s.get(14, 0) >= 2:
            tmax = s[14]
            assert (st["tuple_rounds"] >= 1) == (g <= tmax), what
            assert (st["local_rounds"] >= 1) == (tmax < g <= 32), what
        if s.get(3):
            assert st["local_rounds"] == st["tuple_rounds"] == 0, what
            assert st["cta_rounds"] == (0 if s.get(8) else sum(rs["verdicts"])), what
        if s.get(8):
            assert st["cta_rounds"] == 0, what
        assert np.array_equal(bwts.suffix_array(x), sa), what


@pytest.fixture(scope="module")
def span_wants(oracle, span_cases):
    return {g: oracle.forward(x) for g, (x, _) in span_cases.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("bitonic", (0, 1))
@pytest.mark.parametrize("no_local", (0, 1))
def test_cta_span_edges_of_equal_factors(ctx, tuned, oracle, span_cases, span_wants, bitonic, no_local):
    """w^g: one round over groups of g, CTA spans of 0 or g; CTA-local up to g = 8192, radix passes above
    (tune 0 = n: one Duval chunk, so that the periodic input stays off the suffix-sort fallback)"""
    for g, (x, rs) in span_cases.items():
        tuned({0: len(x), 18: bitonic, 3: no_local})
        st = forward_checked(ctx, x, span_wants[g], oracle.lyndon_starts(x))
        what = (g, bitonic, no_local)
        assert st["lyndon_fallback"] == 0, what
        assert_rounds(st, rs, what)
        assert st["rounds"] == 1, what
        accepted = g <= LS_CAP
        assert rs["verdicts"] == [accepted]
        assert st["cta_rounds"] == int(accepted), what
        p0 = -(-(rs["k0"] * rs["bits"] + rs["extra"]) // 8)   # passes of the initial sort
        assert (st["radix_passes"] > p0) == (not accepted), what


@pytest.mark.gpu
@pytest.mark.parametrize("bitonic", (0, 1))
def test_cta_span_sweep_of_copies(ctx, tuned, oracle, span_copies, bitonic):
    """more than 255 copies: groups of g next to groups of about g / 255; with routing off every group is in
    the large-group set and cta_rounds counts the rounds k_ls_probe accepts"""
    tuned({3: 1, 18: bitonic})
    for g, (x, rs) in span_copies.items():
        st = forward_checked(ctx, x, oracle.forward(x), oracle.lyndon_starts(x))
        assert_rounds(st, rs, g)
        assert st["cta_rounds"] == sum(rs["verdicts"]), (g, rs["verdicts"])


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ("default", "tmax8", "no_local"))
def test_final_ties_of_small_groups_of_equal_factors(ctx, tuned, oracle, setting):
    """w^g with g in {2, 8, 9, 32, 33}: the ties never split and end in the finalize branch of the tuple
    set (g <= 8 with tmax 8), of the warp-local set (9..32) or of the large-group set"""
    rng = np.random.default_rng(8)
    w = lyndon_word(SPAN_W, rng)
    for g in SMALL_EQUAL_G:
        x = equal_factors(w, g)
        starts = oracle.lyndon_starts(x)
        rs = round_structure(x, starts)
        s = dict(ROUTING_SETTINGS[setting])
        s[0] = len(x)
        tuned(s)
        st = forward_checked(ctx, x, oracle.forward(x), starts)
        what = (setting, g)
        assert st["lyndon_fallback"] == 0 and st["factors"] == g, what
        assert_rounds(st, rs, what)
        assert st["rounds"] == 1, what
        if setting == "tmax8":
            assert (st["tuple_rounds"] >= 1) == (g <= 8), what
            assert (st["local_rounds"] >= 1) == (8 < g <= 32), what
        if setting == "no_local":
            assert st["local_rounds"] == st["tuple_rounds"] == 0, what


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", CHUNKS)
def test_factor_starts_at_chunk_and_block_edges(ctx, tuned, oracle, chunk):
    tuned({0: chunk})
    for name, (x, _) in boundary_inputs().items():
        forward_checked(ctx, x, oracle.forward(x), oracle.lyndon_starts(x))


@pytest.mark.gpu
def test_emit_windows_of_16_mib(ctx, tuned, oracle, gen):
    """k_emit through rank windows of 16 MiB (tune 23) at n = 16 MiB - 1, 16 MiB, 16 MiB + 1 and
    32 MiB + 1 equals the default single window and the binned emit (tune 9 = 2)"""
    for n in ((16 << 20) - 1, 16 << 20, (16 << 20) + 1, (32 << 20) + 1):
        x = gen.make("text", 60, n)
        tuned({})
        base = ctx.forward_host(x)
        tuned({23: 16})
        assert ctx.forward_host(x) == base, n
        tuned({9: 2})
        assert ctx.forward_host(x) == base, n
        if n == (16 << 20) + 1:
            assert base == oracle.forward(x)


@pytest.fixture(scope="module")
def inv_cases(oracle):
    out = {}
    for name, (y, x) in inverse_inputs().items():
        if y is None:
            y = oracle.forward(x)
        else:
            x = oracle.inverse(y)
        lf = oracle.lf_map(y)
        out[name] = (np.frombuffer(y, np.uint8), x, lf, cycle_labels(lf))
    return out


INV_SETTINGS = [  # (tune 12 two read-only walks, 13 sublists per warp, 15 mark mode, 1 splitter shift)
    (0, 0, 0, 0), (0, 1, 2, 20), (0, 3, 1, 24), (0, 32, 2, 26), (0, 1 << 20, 0, 29), (0, 0, 2, 31),
    (0, 3, 2, 29), (0, 32, 1, 31), (0, 1, 0, 26), (0, 1 << 20, 2, 24), (0, 0, 1, 20), (0, 0, 2, 0),
    (1, 0, 0, 20), (1, 0, 0, 26), (1, 0, 0, 31), (1, 0, 0, 0),
]


def check_inverse(ctx, y, x, lf, lab, shift, count_marks, what):
    got = ctx.inverse_host(y.tobytes())
    st = ctx.stats()
    assert got == x, what
    p = inverse_prediction(y, lf, lab, shift or default_shift(len(y)), count_marks)
    assert (st["inverse_attempts"] > 1) == p["restart"], (what, p)
    if not p["restart"]:   # a restart hashes with another multiplier: only the bytes are predicted then
        assert (st["splitters"], st["unreached"], st["factors"]) == (p["splitters"], p["unreached"], p["factors"]), (what, p)
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("setting", INV_SETTINGS, ids=lambda s: "t12_%d-t13_%d-t15_%d-t1_%d" % s)
def test_inverse_cycle_accounting(ctx, tuned, inv_cases, setting):
    """bytes, splitters, unreached elements and cycles against the CPU prediction for cycle lengths around
    32, 64, 128 and 4096 (uniform, mixed, equal factors) and arbitrary byte strings"""
    t12, t13, t15, t1 = setting
    tuned({12: t12, 13: t13, 15: t15, 1: t1})
    fallback = 0
    for name, (y, x, lf, lab) in inv_cases.items():
        p = check_inverse(ctx, y, x, lf, lab, t1, t12 == 0 and t15 == 2, (setting, name))
        fallback += p["unreached"] > 0 and not p["restart"]
    assert fallback >= 1, "some input must leave cycles without splitters to the fallback"


@pytest.mark.gpu
@pytest.mark.parametrize("shift", (0, 29))
def test_inverse_short_block_cap(ctx, tuned, cap_cases, shift):
    """count marks (tune 15 = 2) on inputs whose one-byte factors leave just under and just over
    cap = 4096 short blocks: both k_inv_verify_candidates and k_inv_walk_mark must place every byte"""
    tuned({15: 2, 1: shift})
    sides = set()
    for ones, (x, y, lf, lab) in cap_cases.items():
        p = check_inverse(ctx, np.frombuffer(y, np.uint8), x, lf, lab, shift, True, (ones, shift))
        assert not p["restart"] and p["unreached"] >= ones // 2
        sides.add(p["short_blocks"] > p["cap"])
    assert sides == {False, True}

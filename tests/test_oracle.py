"""CPU tests: the oracle restatement against (1) the golden vectors produced by the
unmodified reference binaries, (2) the brute-force BWTS definition, (3) round trips.
"""
import json
from pathlib import Path

import numpy as np
import pytest

import bwts_definition as defn
import helpers

GOLDEN = json.loads((Path(__file__).parent / "golden" / "vectors.json").read_text())

KAT = {  # SURVEY.md section 0 (probe: unmodified reference output)
    b"banana": b"annbaa", b"^BANANA|": b"|NNBAA^A", b"abracadabra": b"ardrcaaaabb",
    b"mississippi": b"ipssmpissii", b"a": b"a", b"aaaa": b"aaaa", b"abab": b"bbaa", b"ba": b"ab",
    b"cbacbacba": b"abbccbaac", b"zyxwv": b"vwxyz", b"abcabcabd": b"dccaaabbb",
    bytes.fromhex("00ff00ff80"): bytes.fromhex("80ffff0000"), b"bananabanana": b"annbnnabaaaa",
}


def golden_input(v, gen):
    if "input" in v:
        return bytes.fromhex(v["input"])
    spec = v["spec"]
    if "kind" in spec:
        data = gen.make(spec["kind"], spec["seed"], spec["n"])
    else:
        data = helpers.families(spec["n"])[spec["family"]]
    assert helpers.sha256(data) == v["input_sha256"], f"generator drifted for {v['name']}"
    return data


def test_kat_table(oracle):
    for x, y in KAT.items():
        assert oracle.forward(x) == y
        assert oracle.inverse(y) == x
        assert defn.forward(x) == y
        assert defn.inverse(y) == x


def test_golden_table_agrees_with_kat():
    by_input = {bytes.fromhex(v["input"]): bytes.fromhex(v["fwd"]) for v in GOLDEN if "input" in v}
    for x, y in KAT.items():
        assert by_input[x] == y


@pytest.mark.parametrize("v", GOLDEN, ids=[v["name"] for v in GOLDEN])
def test_oracle_matches_reference_golden(v, oracle, gen):
    data = golden_input(v, gen)
    fwd = oracle.forward(data)
    inv = oracle.inverse(data)
    if "fwd" in v:
        assert fwd == bytes.fromhex(v["fwd"])
        assert inv == bytes.fromhex(v["inv"])
    else:
        assert helpers.sha256(fwd) == v["fwd_sha256"]
        assert helpers.sha256(inv) == v["inv_sha256"]
    assert oracle.inverse(fwd) == data
    assert oracle.forward(inv) == data


def test_oracle_matches_definition_random_small(oracle):
    rng = np.random.default_rng(7)
    for trial in range(300):
        n = int(rng.integers(1, 120))
        sigma = int(rng.choice([1, 2, 3, 4, 256]))
        x = rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes()
        assert oracle.forward(x) == defn.forward(x), x
        assert oracle.inverse(x) == defn.inverse(x), x


def test_oracle_matches_definition_families(oracle):
    for n in (1, 2, 5, 31, 64, 150):
        for name, x in helpers.families(n).items():
            assert oracle.forward(x) == defn.forward(x), (name, n)


def test_suffix_array_against_naive(oracle):
    rng = np.random.default_rng(11)
    cases = [b"a", b"aa", b"ab", b"ba", b"banana", b"mississippi", b"abab" * 50, b"\xff\x00" * 33]
    for _ in range(100):
        n = int(rng.integers(1, 300))
        sigma = int(rng.choice([1, 2, 3, 256]))
        cases.append(rng.integers(0, sigma, size=n, dtype=np.uint8).tobytes())
    for x in cases:
        sa = oracle.suffix_array(x).tolist()
        assert sa == sorted(range(len(x)), key=lambda i: x[i:]), x


def test_lyndon_starts_are_isa_prefix_minima(oracle):
    # the reference's criterion (mk_bwts_sa.c:126-129) == Duval
    rng = np.random.default_rng(5)
    for _ in range(100):
        n = int(rng.integers(1, 400))
        x = rng.integers(0, int(rng.choice([2, 3, 256])), size=n, dtype=np.uint8).tobytes()
        sa = oracle.suffix_array(x)
        isa = np.empty(n, dtype=np.int64)
        isa[sa] = np.arange(n)
        mins = np.minimum.accumulate(isa)
        starts = [0] + [i for i in range(1, n) if isa[i] < mins[i - 1]]
        assert oracle.lyndon_starts(x).tolist() == starts
        assert defn.duval(x) == starts


def test_invariants_medium(oracle, gen):
    for kind, seed, n in (("random", 9, 50_000), ("text", 9, 50_000), ("dna", 9, 50_000), ("tiled", 9, 150_000)):
        x = gen.make(kind, seed, n)
        y = oracle.forward(x)
        assert y[0] == x[-1]
        assert np.array_equal(np.bincount(np.frombuffer(x, np.uint8), minlength=256),
                              np.bincount(np.frombuffer(y, np.uint8), minlength=256))
        assert oracle.inverse(y) == x


def test_live_reference_binaries_agree(oracle):
    """the oracle against the reference's output for ten seeded inputs, stored in
    golden/reference_checks.json; where oracle/_ref is built, the binaries themselves as well"""
    stored = json.loads((Path(__file__).parent / "golden" / "reference_checks.json").read_text())["random"]
    rng = np.random.default_rng(3)
    assert len(stored) == 10
    for v in stored:
        n = int(rng.integers(1, 5000))
        x = rng.integers(0, int(rng.choice([2, 4, 256])), size=n, dtype=np.uint8).tobytes()
        assert x == bytes.fromhex(v["input"])
        fwd, inv = bytes.fromhex(v["fwd"]), bytes.fromhex(v["inv"])
        assert oracle.forward(x) == fwd
        assert oracle.inverse(x) == inv
        if helpers.ref_available():
            assert helpers.ref_run("mk_bwts", x) == fwd
            assert helpers.ref_run("mbwt_new", x) == fwd
            assert helpers.ref_run("unbwts", x) == inv

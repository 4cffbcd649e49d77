"""Full-size golden values of the FM-index (bwts_b200_fm_*): for the seeded pattern set of
fm_oracle.golden_patterns, SHA-256 of the count ranges (lo, hi interleaved, int32 little-endian) and of the
located positions of those ranges cut to 4096 rows each (fm_oracle.golden_locate_ranges), at C2 (64 MiB text),
C3 (256 MiB tiled text) and C3F (the 256 MiB Fibonacci word), from the CPU oracle: the suffix array of
oracle/lcp_oracle.c and bisection on the text.  tests/test_gpu_fm.py compares the GPU with them.

    python tests/golden/make_fm_golden.py
"""
import hashlib
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import fm_oracle  # noqa: E402
import helpers  # noqa: E402

CASES = [("C2", "text", 2, 64 << 20), ("C3", "tiled", 3, 256 << 20), ("C3F", "fibonacci", 0, 256 << 20)]
OUT = Path(__file__).parent / "fm_fullsize.json"
PATTERN_SEED = 41


def main():
    gen = helpers.Generator()
    out = {}
    for name, kind, seed, n in CASES:
        x = gen.make(kind, seed, n)
        t = time.time()
        o = fm_oracle.FmOracle(x)
        pats = fm_oracle.golden_patterns(x, PATTERN_SEED)
        lo, hi = o.count_many(pats)
        llo, lhi = fm_oracle.golden_locate_ranges(lo, hi)
        h = fm_oracle.golden_hashes(lo, hi, o.locate(llo, lhi))
        out[name] = {"kind": kind, "seed": seed, "n": n, "input_sha256": hashlib.sha256(x).hexdigest(),
                     "pattern_seed": PATTERN_SEED, "patterns": len(pats), **h,
                     "oracle_seconds": round(time.time() - t, 1)}
        print(name, out[name], flush=True)
    OUT.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

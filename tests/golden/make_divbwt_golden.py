"""Full-size golden values of libdivsufsort's end-of-text BWT (bwts_b200_divbwt): SHA-256 of the output
and the primary at C2 (64 MiB text), C3 (256 MiB tiled text) and C3F (the 256 MiB Fibonacci word), from
the CPU oracle oracle/divbwt_oracle.c (SA-IS over T, then libdivsufsort's copy rule; every output is also
inverted by the oracle's restatement of libdivsufsort's walk).  C3 and C3F take a few minutes each.
tests/test_gpu_divbwt.py compares the GPU forward with them.

    python tests/golden/make_divbwt_golden.py
"""
import hashlib
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import divbwt_oracle  # noqa: E402
import helpers  # noqa: E402

CASES = [("C2", "text", 2, 64 << 20), ("C3", "tiled", 3, 256 << 20), ("C3F", "fibonacci", 0, 256 << 20)]
OUT = Path(__file__).parent / "divbwt_fullsize.json"


def main():
    gen, orc = helpers.Generator(), divbwt_oracle.DivbwtOracle()
    out = {}
    for name, kind, seed, n in CASES:
        x = gen.make(kind, seed, n)
        t = time.time()
        y, primary = orc.divbwt(x)
        assert orc.inverse_bw_transform(y, primary) == x
        out[name] = {"kind": kind, "seed": seed, "n": n, "input_sha256": hashlib.sha256(x).hexdigest(),
                     "divbwt_sha256": hashlib.sha256(y).hexdigest(), "primary": primary,
                     "oracle_seconds": round(time.time() - t, 1)}
        print(name, out[name], flush=True)
    OUT.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

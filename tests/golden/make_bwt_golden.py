"""Full-size golden values of the classic BWT: SHA-256 of the output and the primary index at the C2
(64 MiB text) and C3 (256 MiB tiled text) sizes, from the CPU oracle oracle/bwt_oracle.c (SA-IS over
T.T; C3 needs ~3 GiB of RAM and a few minutes).  tests/test_gpu_bwt.py compares the GPU forward with them.

    python tests/golden/make_bwt_golden.py
"""
import hashlib
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bwt_oracle  # noqa: E402
import helpers  # noqa: E402

CASES = [("C2", "text", 2, 64 << 20), ("C3", "tiled", 3, 256 << 20)]
OUT = Path(__file__).parent / "bwt_fullsize.json"


def main():
    gen, orc = helpers.Generator(), bwt_oracle.BwtOracle()
    out = {}
    for name, kind, seed, n in CASES:
        x = gen.make(kind, seed, n)
        t = time.time()
        y, primary = orc.forward(x)
        assert orc.inverse(y, primary) == x
        out[name] = {"kind": kind, "seed": seed, "n": n, "input_sha256": hashlib.sha256(x).hexdigest(),
                     "bwt_sha256": hashlib.sha256(y).hexdigest(), "primary": primary,
                     "oracle_seconds": round(time.time() - t, 1)}
        print(name, out[name], flush=True)
    OUT.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

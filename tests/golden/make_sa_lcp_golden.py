"""Full-size golden values of the suffix array and LCP array (bwts_b200_sa_lcp): SHA-256 of the SA and LCP
bytes (int32, little-endian), the largest LCP value and the LCP sum at C2 (64 MiB text), C3 (256 MiB tiled
text) and C3F (the 256 MiB Fibonacci word), from the CPU oracle oracle/lcp_oracle.c (SA-IS, then Kasai).
C3 and C3F take a few minutes each.  tests/test_gpu_sa_lcp.py compares the GPU with them.

    python tests/golden/make_sa_lcp_golden.py
"""
import hashlib
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import helpers  # noqa: E402
import lcp_oracle  # noqa: E402

CASES = [("C2", "text", 2, 64 << 20), ("C3", "tiled", 3, 256 << 20), ("C3F", "fibonacci", 0, 256 << 20)]
OUT = Path(__file__).parent / "sa_lcp_fullsize.json"


def main():
    gen, orc = helpers.Generator(), lcp_oracle.LcpOracle()
    out = {}
    for name, kind, seed, n in CASES:
        x = gen.make(kind, seed, n)
        t = time.time()
        sa, lcp = orc.sa_lcp(x)
        out[name] = {"kind": kind, "seed": seed, "n": n, "input_sha256": hashlib.sha256(x).hexdigest(),
                     "sa_sha256": hashlib.sha256(sa.astype("<i4").tobytes()).hexdigest(),
                     "lcp_sha256": hashlib.sha256(lcp.astype("<i4").tobytes()).hexdigest(),
                     "lcp_max": int(lcp.max()), "lcp_sum": int(lcp.astype("int64").sum()),
                     "oracle_seconds": round(time.time() - t, 1)}
        print(name, out[name], flush=True)
    OUT.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

"""Full-size golden values of the LPF array and the LZ77 parse (bwts_b200_lpf_*, bwts_b200_lz77_*): SHA-256 of the
LPF, PREV and factor-pair bytes (int32, little-endian), the number of factors z and the largest LPF value at C2
(64 MiB text), C3 (256 MiB tiled text) and C3F (the 256 MiB Fibonacci word), from the CPU oracle
oracle/lz_oracle.c (SA-IS, the previous and next smaller values, direct comparison).  tests/test_gpu_lz.py
compares the GPU with them.

    python tests/golden/make_lz_golden.py
"""
import hashlib
import json
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import helpers  # noqa: E402
import lz_oracle  # noqa: E402

CASES = [("C2", "text", 2, 64 << 20), ("C3", "tiled", 3, 256 << 20), ("C3F", "fibonacci", 0, 256 << 20)]
OUT = Path(__file__).parent / "lz_fullsize.json"


def main():
    gen, orc = helpers.Generator(), lz_oracle.LzOracle()
    out = {}
    for name, kind, seed, n in CASES:
        x = gen.make(kind, seed, n)
        t = time.time()
        lpf, prev = orc.lpf(x)
        f = orc.lz77(x)
        out[name] = {"kind": kind, "seed": seed, "n": n, "input_sha256": hashlib.sha256(x).hexdigest(),
                     "lpf_sha256": hashlib.sha256(lpf.astype("<i4").tobytes()).hexdigest(),
                     "prev_sha256": hashlib.sha256(prev.astype("<i4").tobytes()).hexdigest(),
                     "factors_sha256": hashlib.sha256(f.astype("<i4").tobytes()).hexdigest(),
                     "z": int(len(f)), "lpf_max": int(lpf.max()),
                     "oracle_seconds": round(time.time() - t, 1)}
        print(name, out[name], flush=True)
    OUT.write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

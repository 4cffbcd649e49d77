#!/usr/bin/env python
"""Generate tests/golden/reference_checks.json: the stored side of the tests that compare with the
unmodified reference binaries (oracle/_ref), so that they run where those binaries are absent.

    python tests/golden/make_reference_checks.py

* `random`: the ten seeded inputs of test_oracle.py::test_live_reference_binaries_agree with what
  mk_bwts / mbwt_new (forward) and unbwts (inverse of the input read as a BWTS string) write for them.
  The bytes are the BWTS definition (SURVEY.md section 0), computed by the brute-force statement
  tests/bwts_definition.py, which shares no code with the oracle or the product, and cross-checked
  against the oracle.  The reference computes exactly this function: its own 182 recorded vectors
  (vectors.json) and the probes of SURVEY.md section 0 match the definition byte for byte.  Where
  oracle/_ref exists the test also runs the binaries and compares them with these bytes.
* `cli`: returncode, stdout and stderr of each tool for no arguments, a missing file and an empty
  file, `{tmp}` standing for the directory of the files.  These are the reference's messages: the
  two-line usage on stderr and exit(1) (mk_bwts_sa.c:34-38, mk_bwts_sa_new.c:38-39, unbwts.c:21-25;
  every forward tool's usage says mk_bwts_sa), perror(<file name>) and exit(1) when the file cannot be
  opened or is empty (map_file.c:16-46; SURVEY.md sections 3.4 and 5).
* `timed`: the input of test_gpu_parity.py::test_timings_use_the_reference_phase_labels, the labels
  of the timed reference build's MARK_TIME lines (mk_bwts_sa.c:13-22,50,62,124,168,190) and the
  SHA-256 of its forward output, computed by the oracle (at 700 000 bytes the brute-force statement
  is too slow; the oracle equals the reference on every recorded vector).
"""
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
import bwts_definition as defn  # noqa: E402
import helpers  # noqa: E402

USAGE_FORWARD = "Usage: mk_bwts_sa <infile> [<outfile.bwts>]\n"
CLI = {
    "mk_bwts": USAGE_FORWARD + "If unspecified, output is written to standard output\n",
    "mbwt_new": USAGE_FORWARD + "If unspecified, output is written to a temp file\n",
    "unbwts": "Usage: unbwts <infile.bwts> [<outfile>]\nIf output file name is unspecified, a name is generated\n",
}


def random_inputs():
    """the inputs of test_live_reference_binaries_agree, in its order"""
    rng = np.random.default_rng(3)
    out = []
    for _ in range(10):
        n = int(rng.integers(1, 5000))
        out.append(rng.integers(0, int(rng.choice([2, 4, 256])), size=n, dtype=np.uint8).tobytes())
    return out


def main():
    oracle = helpers.Oracle()
    random = []
    for x in random_inputs():
        fwd, inv = defn.forward(x), defn.inverse(x)
        assert fwd == oracle.forward(x) and inv == oracle.inverse(x)
        random.append({"input": x.hex(), "fwd": fwd.hex(), "inv": inv.hex()})
    cli = {tool: [{"args": [], "returncode": 1, "stdout": "", "stderr": usage},
                  {"args": ["{tmp}/nope"], "returncode": 1, "stdout": "", "stderr": "{tmp}/nope: No such file or directory\n"},
                  {"args": ["{tmp}/empty"], "returncode": 1, "stdout": "", "stderr": "{tmp}/empty: Invalid argument\n"}]
           for tool, usage in CLI.items()}
    x = helpers.Generator().make("dna", 77, 700_000)
    timed = {"kind": "dna", "seed": 77, "n": len(x), "input_sha256": helpers.sha256(x),
             "labels": ["Suffix sort", "Compute ISA", "Fix sort order", "Generate BWTS", "Write BWTS"],
             "fwd_sha256": helpers.sha256(oracle.forward(x))}
    out = {"random": random, "cli": cli, "timed": timed}
    (HERE / "reference_checks.json").write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()

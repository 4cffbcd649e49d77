"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol the
header declares, fails loudly without a device, and the host tools keep the reference's CLI."""
import json
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import helpers

HEADER = helpers.REPO / "include" / "bwts_b200.h"
BIN = helpers.PKG / "bin"


def _have_gpu(bwts):
    return bwts.device_count() > 0


def test_header_symbols_are_exported(bwts):
    text = HEADER.read_text()
    declared = set(re.findall(r"\b(bwts_b200_[a-z_0-9]+)\s*\(", text))
    declared -= {"bwts_b200_ctx", "bwts_b200_stats"}
    assert declared == set(bwts.EXPORTS), declared ^ set(bwts.EXPORTS)
    L = bwts.lib()
    for name in sorted(declared):
        assert hasattr(L, name), name


def test_header_cites_the_reference_seams():
    text = HEADER.read_text()
    for cite in ("mk_bwts_sa.c:47-52", "mk_bwts_sa_new.c:50-55", "unbwts.c:31-86"):
        assert cite in text


def test_version_and_error_strings(bwts):
    assert "sm_100a" in bwts.version()
    L = bwts.lib()
    for code in range(0, -7, -1):
        assert L.bwts_b200_strerror(code)
    assert L.bwts_b200_class_name(4) == b"onesweep_pass"
    assert L.bwts_b200_class_name(99) is None


def test_argument_validation_needs_no_device(bwts):
    L = bwts.lib()
    buf = np.zeros(16, dtype=np.uint8)
    assert L.bwts_b200_forward(None, 16, buf.ctypes.data, 0) == -1
    assert L.bwts_b200_inverse(buf.ctypes.data, -5, buf.ctypes.data, 0) == -1
    assert L.bwts_b200_forward(buf.ctypes.data, 1 << 31, buf.ctypes.data, 0) == -2
    assert L.bwts_b200_tune(99, 1) == -1
    assert L.bwts_b200_tune(1, 5) == -1


def test_no_cpu_fallback(bwts):
    """on a box without a GPU every transform must fail loudly, not compute on the host"""
    if _have_gpu(bwts):
        pytest.skip("a CUDA device is present")
    with pytest.raises(bwts.BwtsError) as e:
        bwts.forward(b"banana")
    assert e.value.code == -3
    with pytest.raises(bwts.BwtsError):
        bwts.inverse(b"annbaa")
    with pytest.raises(bwts.BwtsError):
        bwts.forward_blocks(b"banana" * 10, 16)
    with pytest.raises(bwts.BwtsError):
        bwts.Context(0)


def test_product_does_not_reference_the_oracle():
    for p in list((helpers.PKG / "csrc").glob("*")) + list((helpers.PKG / "host").glob("*")) + [helpers.PKG / "bwts_b200.py"]:
        text = p.read_text()
        assert "liboracle" not in text and "oracle_bwts" not in text and "sais" not in text, p


@pytest.mark.parametrize("tool,second", [("mk_bwts", "If unspecified, output is written to standard output"),
                                         ("mbwt_new", "If unspecified, output is written to a temp file"),
                                         ("unbwts", "If output file name is unspecified, a name is generated")])
def test_cli_usage_text_and_exit_code(tool, second):
    r = subprocess.run([str(BIN / tool)], capture_output=True)
    assert r.returncode == 1 and r.stdout == b""
    lines = r.stderr.decode().splitlines()
    first = "Usage: unbwts <infile.bwts> [<outfile>]" if tool == "unbwts" else "Usage: mk_bwts_sa <infile> [<outfile.bwts>]"
    assert lines == [first, second]


@pytest.mark.parametrize("tool", ["mk_bwts", "mbwt_new", "unbwts"])
def test_cli_missing_and_empty_input(tool, tmp_path):
    r = subprocess.run([str(BIN / tool), str(tmp_path / "nope")], capture_output=True)
    assert r.returncode == 1 and b"No such file or directory" in r.stderr
    empty = tmp_path / "empty"
    empty.write_bytes(b"")
    r = subprocess.run([str(BIN / tool), str(empty)], capture_output=True)
    assert r.returncode == 1 and r.stderr.decode().strip() == f"{empty}: Invalid argument"


@pytest.mark.parametrize("tool,ref", [("mk_bwts", "mk_bwts"), ("mbwt_new", "mbwt_new"), ("unbwts", "unbwts")])
def test_cli_error_behaviour_equals_reference_binaries(tool, ref, tmp_path):
    """returncode, stdout and stderr for no arguments, a missing file and an empty file equal the reference's,
    stored in golden/reference_checks.json; where oracle/_ref is built, the binaries' own as well"""
    stored = json.loads((Path(__file__).parent / "golden" / "reference_checks.json").read_text())["cli"][tool]
    empty = tmp_path / "empty"
    empty.write_bytes(b"")
    assert len(stored) == 3
    for want in stored:
        args = [a.replace("{tmp}", str(tmp_path)) for a in want["args"]]
        a = subprocess.run([str(BIN / tool)] + args, capture_output=True)
        expected = (want["returncode"], want["stdout"].replace("{tmp}", str(tmp_path)).encode(),
                    want["stderr"].replace("{tmp}", str(tmp_path)).encode())
        assert (a.returncode, a.stdout, a.stderr) == expected, args
        if helpers.ref_available():
            b = subprocess.run([str(helpers.REF_DIR / ref)] + args, capture_output=True)
            assert (b.returncode, b.stdout, b.stderr) == expected, args


def test_stats_struct_layout_matches_the_header(tmp_path):
    """the ctypes mirror of bwts_b200_stats has the size the C compiler gives the header's struct"""
    import ctypes
    import subprocess
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "bwts_b200.h"\n'
                   'int main(void){printf("%zu\\n", sizeof(bwts_b200_stats));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-I", str(helpers.REPO / "include"), "-o", str(exe), str(src)])
    csize = int(subprocess.check_output([str(exe)]).decode())
    bwts = helpers.load_product()
    assert csize == ctypes.sizeof(bwts.Stats)


def test_phase_names_are_the_reference_marks(bwts):
    """bwts_b200_phase_name: forward phases carry the labels of the reference's MARK_TIME calls
    (/root/reference/mk_bwts_sa.c:50,124,168,190) in the reference's order"""
    L = bwts.lib()
    fwd = [L.bwts_b200_phase_name(0, i) for i in range(bwts.NPHASE)]
    assert [f.decode() for f in fwd if f] == ["Suffix sort", "Compute ISA", "Fix sort order", "Generate BWTS"]
    inv = [L.bwts_b200_phase_name(1, i) for i in range(bwts.NPHASE)]
    assert [f.decode() for f in inv if f] == ["Count bytes", "LF map", "Walk sublists", "Rank sublists", "Place bytes"]
    assert L.bwts_b200_phase_name(0, -1) is None and L.bwts_b200_phase_name(1, 99) is None

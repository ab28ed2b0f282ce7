"""The library reads the process environment only for the switches the GPU tests use
to force a layout or get a bitwise reference that default plans do not reach.  Any
other switch would let a stray variable change what a launch computes; measurement
variants are built with ``build.py -D... --out=...`` and loaded through
``SOUNDML_B200_LIB`` instead."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "soundml_b200", "csrc")

TEST_SWITCHES = {
    "SMB_ROWS_SPLIT",     # row-form resampler: split or unsplit main shift
    "SMB_ROWS_SMEM_A",    # row-form resampler: A tiles in shared memory
    "SMB_ROWS_TMEM_A",    # row-form resampler: A tiles in tensor memory
    "SMB_GEMM_WINDOWS",   # tensor-core resampler stages in the window form
    "SMB_NO_CARRY",       # bin-major write-out without the sector carry (bitwise reference)
}


def _sources():
    return sorted(p for ext in ("cu", "cuh", "cpp", "h") for p in glob.glob(os.path.join(CSRC, "*." + ext)))


def _getenv_calls():
    """(file, line, argument text) of every getenv call in the library sources."""
    calls = []
    for path in _sources():
        with open(path, encoding="utf-8") as f:
            text = f.read()
        for m in re.finditer(r"\bgetenv\s*\(([^)]*)\)", text):
            calls.append((os.path.basename(path), text.count("\n", 0, m.start()) + 1, m.group(1).strip()))
    return calls


def test_library_reads_only_the_test_switches():
    calls = _getenv_calls()
    assert _sources() and calls
    not_literal = [c for c in calls if not re.fullmatch(r'"[A-Za-z0-9_]+"', c[2])]
    assert not not_literal, f"getenv with a computed name: {not_literal}"
    names = {c[2].strip('"') for c in calls}
    assert names == TEST_SWITCHES, (f"unexpected: {sorted(names - TEST_SWITCHES)}, "
                                    f"no longer read: {sorted(TEST_SWITCHES - names)}")


def test_every_switch_is_used_by_a_test():
    here = os.path.abspath(__file__)
    texts = []
    for path in glob.glob(os.path.join(ROOT, "tests", "**", "*.py"), recursive=True):
        if os.path.abspath(path) != here:
            with open(path, encoding="utf-8") as f:
                texts.append(f.read())
    unused = sorted(name for name in TEST_SWITCHES if not any(name in t for t in texts))
    assert not unused, f"switches no test sets: {unused}"

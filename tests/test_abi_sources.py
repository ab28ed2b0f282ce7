"""The C ABI states each shared precondition and the memory-kind rule once, in one helper
that every entry point calls.  A fix to a message or to the rule then reaches every entry
point; a copy left behind would answer the same input in two ways."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
API = os.path.join(ROOT, "soundml_b200", "csrc", "api.cu")

SINGLE_HOME_LITERALS = [
    "soundml_b200: unknown memory kind",
    "the overlap-added squared window must stay above 1e-10",
    "the two configurations must agree on fft_size",
    "reference must be finite and positive",
    "no such stage",
]


def _api_source():
    with open(API, encoding="utf-8") as f:
        return re.sub(r"//[^\n]*", "", f.read())


def test_each_shared_message_is_written_once():
    text = _api_source()
    for literal in SINGLE_HOME_LITERALS:
        assert text.count(literal) == 1, f"{literal!r} appears {text.count(literal)} times in api.cu"

"""Every CUDA resource the library allocates is owned by a ``std::unique_ptr`` whose
deleter is the one place that releases that kind of resource.  A plan, handle or call
that freed its own members would repeat its member list in a destructor or cleanup
block, and the paths that fail halfway would leak or keep half-built state.  The only
other release calls are the ABI's own ``smb_device_free`` and ``smb_host_free_pinned``."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "soundml_b200", "csrc")

RELEASE_CALLS = {
    "cudaFree": 2,            # the device-memory deleter, smb_device_free
    "cudaFreeHost": 2,        # the pinned-memory deleter, smb_host_free_pinned
    "cudaFreeAsync": 1,       # the stream-ordered scratch deleter
    "cudaStreamDestroy": 1,   # the stream deleter
    "cudaEventDestroy": 1,    # the event deleter
}


def _sources():
    return sorted(p for ext in ("cu", "cuh", "cpp", "h") for p in glob.glob(os.path.join(CSRC, "*." + ext)))


def test_each_kind_of_resource_is_released_in_one_place():
    assert _sources()
    found = {name: [] for name in RELEASE_CALLS}
    for path in _sources():
        with open(path, encoding="utf-8") as f:
            text = f.read()
        for name in RELEASE_CALLS:
            for m in re.finditer(r"\b" + name + r"\s*\(", text):
                found[name].append(f"{os.path.basename(path)}:{text.count(chr(10), 0, m.start()) + 1}")
    wrong = {name: sites for name, sites in found.items() if len(sites) != RELEASE_CALLS[name]}
    assert not wrong, f"release calls outside the owners' deleters: {wrong}"

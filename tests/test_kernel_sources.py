"""The kernels share one copy of each device helper: the PTX wrappers of the mbarrier,
bulk-copy and tcgen05 pipelines (sm100.cuh), the reference's boundary rule and the
cp.async fetch of a tile's samples (stft_stage.cuh), and the FFT pieces (fft32.cuh).
A fix to one of them -- the spin-wait every TMA and MMA pipeline waits in, or the
padding rule the parity tests hold the kernels to -- then reaches every kernel."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "soundml_b200", "csrc")

SHARED_HELPERS = {
    "sm100.cuh": ["named_sync", "smem_u32", "mbar_init", "mbar_expect_tx", "mbar_arrive", "mbar_wait",
                  "bulk_g2s", "tmem_alloc", "tmem_dealloc", "umma_commit", "tmem_ld16", "tmem_ld_wait",
                  "tmem_st16"],
    "stft_stage.cuh": ["src_index", "copy_real_samples"],
    "fft32.cuh": ["kW64C", "kW64S", "fft1024", "pk_add", "pk_sub", "pk_mul"],
}

# PTX that only the shared wrappers issue
SINGLE_HOME_ASM = ["mbarrier.try_wait", "cp.async.bulk.shared::cluster", "tcgen05.alloc", "tcgen05.commit"]


def _sources():
    """File name -> text without // comments (which may name a helper or an instruction)."""
    paths = sorted(p for ext in ("cu", "cuh", "cpp", "h") for p in glob.glob(os.path.join(CSRC, "*." + ext)))
    out = {}
    for path in paths:
        with open(path, encoding="utf-8") as f:
            out[os.path.basename(path)] = re.sub(r"//[^\n]*", "", f.read())
    return out


def _definitions(name, sources):
    """Files that define device function or constant table `name`."""
    pattern = re.compile(r"__device__\b[^;{}()]*\b" + re.escape(name) + r"\s*[(\[]")
    return sorted(f for f, text in sources.items() if pattern.search(text))


def test_each_shared_helper_is_defined_once():
    sources = _sources()
    for home, names in SHARED_HELPERS.items():
        assert home in sources
        for name in names:
            assert _definitions(name, sources) == [home], f"{name}: defined in {_definitions(name, sources)}"


def test_pipeline_ptx_has_one_home():
    sources = _sources()
    for asm in SINGLE_HOME_ASM:
        files = sorted(f for f, text in sources.items() if asm in text)
        assert files == ["sm100.cuh"], f"{asm!r} appears in {files}"


def test_every_included_file_is_a_build_dependency():
    """build.py rebuilds when a file in CUDA_SOURCES, HOST_SOURCES or HEADERS is newer than
    the library: a header it does not list (max_key.cuh once) could change without a rebuild."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("soundml_b200_build", os.path.join(ROOT, "soundml_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    listed = {os.path.normpath(os.path.join(CSRC, f)) for f in b.CUDA_SOURCES + b.HOST_SOURCES + b.HEADERS}
    for name, text in _sources().items():
        for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', text, re.M):
            path = os.path.normpath(os.path.join(CSRC, inc))
            assert os.path.exists(path), f"{name} includes {inc}, which does not exist"
            assert path in listed, f"{name} includes {inc}, which build.py does not list"
    for f in listed:
        assert os.path.exists(f), f"build.py lists {f}, which does not exist"


def test_kernel_tables_make_no_cuda_runtime_calls():
    """kernel_tables.{h,cpp} decide and fill the kernels' tables on the host; api.cu uploads
    and owns them.  A CUDA runtime call there would make a layout query need a device."""
    sources = _sources()
    for name in ("kernel_tables.h", "kernel_tables.cpp"):
        calls = sorted(set(re.findall(r"\bcuda[A-Z]\w*\s*\(", sources[name])))
        assert not calls, f"{name} calls {calls}"

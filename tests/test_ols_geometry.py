"""Which overlap-save kernel and branch each planned stage and FIR runs (CPU only).

``Config.ols_geometry(i)`` and ``Fir.ols_geometry()`` report the plan the library's
overlap-save executor launches, computed on the host from the same rules the executor
uses (``ols_plan_for_stage`` / ``ols_plan_for_fir`` in csrc/host_design.cpp and
``ols2048_supports`` in csrc/ols2048.cu).  The table below gives one row per kernel
branch; tests/test_gpu_ols_bounds.py runs the single-stage rows and the FIRs on the GPU.

Branches:
  * ``ols2048_kernel`` (one warp per block, N = 2048): plain (FIR), /2 (every other
    sample of the full-length inverse), any other /M (through the transpose buffer), and
    xL as its L polyphase branches at the input rate;
  * ``ols_kernel`` (one CTA per block, Stockham, power-of-two N): plain, /M alias fold
    onto W = N / M bins, xL periodic extension onto W = N L bins.
"""
import ctypes

import pytest

# (kind, arguments, stage, summary of ols_geometry).  "rs" rows are Resample.Config.create
# (sample_rate, target, quality); "fir" rows Fir.lowpass(k=...).
ROWS = [
    # ols2048, /2: the store branch that keeps v.x of every complex output
    ("rs", (44100, 22050, "high"), 0, "ols2048 /2 N=2048 B=1668 delta=0 W=2048 K=190"),
    # ols2048, general M through the transpose buffer; the planner priced N = 3072 for the CPU
    ("rs", (24000, 8000, "high"), 0, "ols2048 /3 N=2048 B=1479 delta=0 W=2048 K=284"),
    # ... M = 4 with delta != 0
    ("rs", (32000, 8000, ("custom", 80.0, 0.95)), 0, "ols2048 /4 N=2048 B=1244 delta=2 W=2048 K=402"),
    # ols2048 polyphase, L = 2, 3, 4
    ("rs", (22050, 44100, "high"), 0, "ols2048 polyphase x2 N=2048 B=1858 delta=0 W=2048 K=95"),
    ("rs", (8000, 24000, "high"), 0, "ols2048 polyphase x3 N=2048 B=1858 delta=0 W=2048 K=95"),
    ("rs", (8000, 32000, "high"), 0, "ols2048 polyphase x4 N=2048 B=1858 delta=0 W=2048 K=95"),
    # inside cascades: stage 0 of an interpolating pair, stage 1 of a decimating one
    ("rs", (8000, 48000, "high"), 0, "ols2048 polyphase x2 N=2048 B=1848 delta=0 W=2048 K=100"),
    ("rs", (48000, 8000, "high"), 1, "ols2048 /2 N=2048 B=1650 delta=1 W=2048 K=199"),
    # ols_kernel /M alias fold, W = 4096; at 60 dB the folded terms are 1e-3 of the output
    ("rs", (88200, 44100, ("custom", 200.0, 0.95)), 0, "ols /2 fold N=8192 B=7120 delta=0 W=4096 K=536"),
    ("rs", (88200, 44100, ("custom", 60.0, 0.99)), 0, "ols /2 fold N=8192 B=6740 delta=0 W=4096 K=726"),
    # ... W = 2048 with delta != 0
    ("rs", (88200, 22050, "best"), 0, "ols /4 fold N=8192 B=7120 delta=3 W=2048 K=535"),
    # ols_kernel xL periodic extension, W = 16384: 196 KB of shared memory, under the
    # launcher's 200 KB cap
    ("rs", (88200, 24000, ("custom", 160.0, 0.95)), 0, "ols x2 extend N=8192 B=6572 delta=0 W=16384 K=810"),
    ("rs", (96000, 192000, ("custom", 100.0, 0.99)), 0, "ols x2 extend N=8192 B=6908 delta=0 W=16384 K=642"),
    # ... the lowest attenuation at which a single x2 stage still needs it (K = 516 > 511)
    ("rs", (96000, 192000, ("custom", 82.0, 0.99)), 0, "ols x2 extend N=8192 B=7160 delta=0 W=16384 K=516"),
    # Tagged "ols" by the planner with N = 6144, which is not a power of two: finish_ols
    # gives up and the direct kernel runs the stage.  Pinned as it behaves today; whether
    # this stage should run overlap-save at another N is a separate question.
    ("rs", (48000, 16000, ("custom", 140.0, 0.95)), 0, "direct"),
    # FIR: N = 2048 up to K = 512 (odd K shifts by delta = 1 so stores pair up) ...
    ("fir", 300, None, "ols2048 plain N=2048 B=1448 delta=0 W=2048 K=300"),
    ("fir", 301, None, "ols2048 plain N=2048 B=1446 delta=1 W=2048 K=301"),
    ("fir", 512, None, "ols2048 plain N=2048 B=1024 delta=0 W=2048 K=512"),
    # ... then the smallest power of two >= 10 K on ols_kernel, capped at 16384 ...
    ("fir", 513, None, "ols plain N=8192 B=7166 delta=0 W=8192 K=513"),
    ("fir", 600, None, "ols plain N=8192 B=6992 delta=0 W=8192 K=600"),
    ("fir", 1638, None, "ols plain N=16384 B=13108 delta=0 W=16384 K=1638"),
    ("fir", 1639, None, "ols plain N=16384 B=13106 delta=0 W=16384 K=1639"),
    # ... while the hop B = N - 2K is at least N / 4
    ("fir", 6144, None, "ols plain N=16384 B=4096 delta=0 W=16384 K=6144"),
    ("fir", 6145, None, "direct"),
]


def row_id(r):
    kind, args, stage, _ = r
    if kind == "fir":
        return f"fir-k{args}"
    q = args[2] if isinstance(args[2], str) else "custom%g-%g" % args[2][1:]
    return f"{args[0]}-{args[1]}-{q}-stage{stage}"


def summary(g):
    """ols_geometry in the table's notation."""
    if g["kernel"] == "direct":
        return "direct"
    if g["polyphase"]:
        branch = f"polyphase x{g['l']}"
    elif g["l"] > 1:
        branch = f"x{g['l']} extend"
    elif g["m"] > 1:
        branch = f"/{g['m']}" + ("" if g["full_inverse"] else " fold")
    else:
        branch = "plain"
    return (f"{g['kernel']} {branch} N={g['n']} B={g['b']} delta={g['delta']} "
            f"W={g['w']} K={g['k']}")


def geometry_of(lib, row):
    kind, args, stage, _ = row
    if kind == "fir":
        return lib.Resample.Fir.lowpass(k=args, cutoff=0.5).ols_geometry()
    sr, target, quality = args
    cfg = lib.Resample.Config.create(sample_rate=sr, target=target, quality=quality)
    st = cfg.stages()[stage]
    g = cfg.ols_geometry(stage)
    assert st["exec"] == "ols", (row, st)
    assert (g["kernel"] == "direct") or (g["l"], g["m"], g["k"]) == (st["l"], st["m"], st["k"])
    return g


@pytest.mark.parametrize("row", ROWS, ids=[row_id(r) for r in ROWS])
def test_row_reports_its_kernel_and_branch(lib, row):
    assert summary(geometry_of(lib, row)) == row[3]


def test_table_reaches_every_branch(lib):
    gs = [geometry_of(lib, r) for r in ROWS]
    on2048 = [g for g in gs if g["kernel"] == "ols2048"]
    onstock = [g for g in gs if g["kernel"] == "ols"]
    want = {
        "ols2048 plain": any(g["l"] == g["m"] == 1 for g in on2048),
        "ols2048 M = 2": any(g["m"] == 2 for g in on2048),
        "ols2048 general M = 3": any(g["m"] == 3 for g in on2048),
        "ols2048 general M = 4": any(g["m"] == 4 for g in on2048),
        "ols plain": any(g["l"] == g["m"] == 1 for g in onstock),
        "ols /M fold": any(g["m"] > 1 and g["w"] == g["n"] // g["m"] for g in onstock),
        "ols xL extension": any(g["l"] > 1 and g["w"] == g["n"] * g["l"] for g in onstock),
        "ols2048 delta != 0": any(g["delta"] for g in on2048),
        "ols delta != 0": any(g["delta"] for g in onstock),
        "a tagged stage on the direct kernel": any(r[0] == "rs" and g["kernel"] == "direct"
                                                   for r, g in zip(ROWS, gs)),
    }
    for l in (2, 3, 4):
        want[f"ols2048 polyphase L = {l}"] = any(g["polyphase"] and g["l"] == l for g in on2048)
    firs = {r[1]: g for r, g in zip(ROWS, gs) if r[0] == "fir"}
    want["FIR k = 1638 below the N cap"] = firs[1638]["n"] == 16384 and 10 * 1638 <= 16384
    want["FIR k = 1639 on the N cap"] = firs[1639]["n"] == 16384 and 10 * 1639 > 16384
    want["FIR k = 6144 allowed"] = firs[6144]["kernel"] == "ols"
    want["FIR k = 6145 refused"] = firs[6145]["kernel"] == "direct"
    missing = [k for k, ok in want.items() if not ok]
    assert not missing, missing


def hi(g, b):
    """Last output block b completes (resample.ml:1313-1315)."""
    if g["l"] > 1:
        return g["l"] * (b * g["b"] + g["n"] - 3 * g["k"]) - 1
    num = b * g["b"] + g["n"] - 3 * g["k"] - g["delta"] - 1
    return num // g["m"] if num >= 0 else -1


@pytest.mark.parametrize("row", [r for r in ROWS if r[3] != "direct"],
                         ids=[row_id(r) for r in ROWS if r[3] != "direct"])
def test_blocks_for_is_the_fewest_covering_blocks(lib, row):
    g = geometry_of(lib, row)
    for n_out in (1, 2, g["b"] - 1, g["b"], 3 * g["b"] + 1, 123457):
        blocks = g["blocks_for"](n_out)
        assert hi(g, blocks - 1) >= n_out - 1, (n_out, blocks)
        assert blocks == 1 or hi(g, blocks - 2) < n_out - 1, (n_out, blocks)
    assert g["blocks_for"](0) == 0


def test_no_geometry_for_stages_off_overlap_save_and_bad_input(lib):
    cfg = lib.Resample.Config.create(sample_rate=44100, target=16000, quality="high")
    assert cfg.stages()[0]["exec"] == "gemm"
    g = cfg.ols_geometry(0)
    assert summary(g) == "direct" and g["n"] == g["b"] == g["w"] == 0
    with pytest.raises(ValueError, match="not an overlap-save geometry"):
        g["blocks_for"](10)
    with pytest.raises(ValueError, match="stage_ols: no such stage"):
        cfg.ols_geometry(1)
    # hand-made geometries the executor never runs are refused, not divided by
    good = lib.Resample.Config.create(sample_rate=44100, target=22050, quality="high").ols_geometry(0)
    for field, value in [("m", 0), ("l", 0), ("l", -1), ("b", 0)]:
        bad = _lib_geometry(lib, good, **{field: value})
        assert lib._lib.lib.smb_ols_blocks(ctypes.byref(bad), 100) == -1, field
    bad = _lib_geometry(lib, good, l=2, m=2)
    assert lib._lib.lib.smb_ols_blocks(ctypes.byref(bad), 100) == -1
    assert lib._lib.lib.smb_ols_blocks(ctypes.byref(_lib_geometry(lib, good)), 100) == good["blocks_for"](100)


def _lib_geometry(lib, g, **changes):
    """An smb_ols_geometry holding g's fields, some of them changed."""
    fields = {name: g[name] for name, _ in lib._lib.OlsGeometry._fields_ if name != "kernel"}
    fields.update(changes)
    out = lib._lib.OlsGeometry(kernel=1, **{k: int(v) for k, v in fields.items()})
    return out

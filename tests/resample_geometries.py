"""The tensor-core resampler's geometry table, shared by the host-only layout tests
(test_resample_layouts.py) and the GPU bounds tests (test_gpu_resample_bounds.py): rows of
(sample_rate, target, quality, expected layout) that together reach every branch of the
row-form planner in csrc/kernel_tables.cpp, and the environment switches that force the
other layouts."""
import pytest

SWITCHES = ("SMB_ROWS_SPLIT", "SMB_ROWS_SMEM_A", "SMB_ROWS_TMEM_A", "SMB_GEMM_WINDOWS")


# (sample_rate, target, quality, the layout Config.layout(0) reports under the default switches,
# one entry per column group).  tools/resample_layouts.py sweeps ~1600 gemm-tagged
# plans; these rows reach every branch of the planner (test_table_covers_every_layout_branch).
GEOMETRIES = [
    # configs[3]: one group, split main shift (14 chunks >= 8), shared-memory A at (3, 2)
    # (the stage's 53 KB B stages leave no room for (2, 3)), runs split by the split
    (44100, 16000, "high",
     "row 160 split smem-A 3/2 shifts 3 chunks 14 slices 42"),
    # split wanted but its extra accumulator does not fit: the fall back to unsplit; (2, 2)
    (44100, 16000, "best",
     "row 160 unsplit smem-A 2/2 shifts 3 chunks 14 slices 28"),
    # one group with A in tensor memory, B at 3 stages; L mod 4 = 0
    (44100, 48000, "high",
     "row 160 unsplit tmem-A 2/3 shifts 3 chunks 5 slices 5"),
    # L mod 4 = 3 (the epilogue's transposed stores)
    (48000, 44100, "high",
     "row 147 unsplit tmem-A 2/3 shifts 3 chunks 5 slices 5"),
    # no row layout fits (five shifts): a gemm stage on the window form
    (48000, 44100, "best",
     "window 147 chunks 15"),
    # two column groups, split, (2, 3)
    (44100, 32000, "high",
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 27 | "
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 27"),
    # three groups, L mod 4 = 1, (2, 2) and (3, 2) in one stage, runs split at gaps (6 and 7
    # slices over 5 chunks, unsplit)
    (16000, 44100, "high",
     "row 160 unsplit smem-A 2/2 shifts 2 chunks 5 slices 6 | "
     "row 160 unsplit smem-A 2/2 shifts 2 chunks 5 slices 7 | "
     "row 121 unsplit smem-A 3/2 shifts 3 chunks 5 slices 5"),
    # four groups, split
    (11025, 16000, "high",
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 18 | "
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 18 | "
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 18 | "
     "row 160 split smem-A 2/3 shifts 2 chunks 14 slices 18"),
    # 10 chunks wants split, which does not fit with A in tensor memory: unsplit, tensor-memory A
    (48000, 22050, "high",
     "row 147 unsplit tmem-A 2/3 shifts 3 chunks 10 slices 10"),
    # a standard pair on the window form (row layout fails), three window groups
    (8000, 44100, "high",
     "window 160 chunks 7 | window 160 chunks 8 | window 121 chunks 8"),
    # L mod 4 = 2, four shifts, 3 chunks, tensor-memory A at (2, 2), a run split
    (6500, 9800, "fast",
     "row 98 unsplit tmem-A 2/2 shifts 4 chunks 3 slices 6"),
    # 3 chunks with tensor-memory A: the B stages capped at 3 (with 4, the B loader never took
    # back the stage lent to the epilogue and overwrote it: wrong outputs on misaligned clips)
    (6500, 6400, ("custom", 80.0, 0.8),
     "row 64 unsplit tmem-A 2/3 shifts 2 chunks 3 slices 3"),
    # a column group whose taps stay inside one shift
    (9700, 44100, ("custom", 80.0, 0.8),
     "row 160 unsplit smem-A 2/3 shifts 1 chunks 4 slices 3 | "
     "row 160 unsplit smem-A 2/3 shifts 2 chunks 4 slices 4 | "
     "row 121 unsplit smem-A 2/3 shifts 2 chunks 4 slices 4"),
    # M = 20 < 32: window form
    (12000, 88200, ("custom", 80.0, 0.8),
     "window 147 chunks 3"),
    # M = 40: two K-chunks per row, below the row form's three: window form
    (12000, 44100, ("custom", 80.0, 0.8),
     "window 147 chunks 3"),
    # split with A in tensor memory (four B stages), L mod 4 = 3
    (25600, 12700, ("custom", 80.0, 0.8),
     "row 127 split tmem-A 2/4 shifts 3 chunks 8 slices 20"),
    # gemm-tagged but L = 1280 > 1024: no tcgen05 tables, the direct kernel
    (11025, 96000, ("custom", 80.0, 0.8),
     "direct 1280"),
]
GEOM_IDS = [f"{g[0]}-{g[1]}-{g[2] if isinstance(g[2], str) else 'custom%g-%g' % g[2][1:]}" for g in GEOMETRIES]


def geometry(sr, target, quality="high"):
    return next(g for g in GEOMETRIES if g[:3] == (sr, target, quality))


@pytest.fixture
def env(monkeypatch):
    """The layout switches cleared; a test sets the ones it forces.  They are read when a
    plan's tables are built (its first layout() or apply), SMB_GEMM_WINDOWS at every
    layout() and apply."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def plan(sb, geom, executor="planned"):
    """A fresh Config with its tables built now, under the current switches (host-only)."""
    sr, target, quality = geom[:3]
    cfg = sb.Resample.Config.create(sample_rate=sr, target=target, quality=quality)
    st = cfg.stages()
    assert len(st) == 1 and st[0]["exec"] == "gemm", cfg.pp()
    cfg.set_executor(executor)
    return cfg, st[0], cfg.layout(0), cfg.stage_prototype(0)


def summary(layout):
    """Config.layout as one line per column group, the table's notation."""
    parts = []
    for g in layout:
        if g["form"] != "row":
            parts.append(f'{g["form"]} {g["columns"]}' + (f' chunks {g["chunks"]}' if g["form"] == "window" else ""))
        else:
            parts.append(f'row {g["columns"]} {"split" if g["two_issuers"] else "unsplit"} '
                         f'{"tmem" if g["a_tmem"] else "smem"}-A {g["a_stages"]}/{g["b_stages"]} '
                         f'shifts {g["shifts"]} chunks {g["chunks"]} slices {g["slices"]}')
    return " | ".join(parts)


# (switch, value or the executor, geometry): each switch on geometries where it changes the layout
FORCED = [
    ("SMB_ROWS_SMEM_A", "1", (44100, 48000, "high")),          # tensor-memory A -> shared (3, 2)
    ("SMB_ROWS_SMEM_A", "1", (6500, 9800, "fast")),            # ... no shared-memory staging fits: window form
    ("SMB_ROWS_TMEM_A", "1", (16000, 44100, "high")),          # three groups, shared -> tensor-memory A
    ("SMB_ROWS_SPLIT", "0", (44100, 16000, "high")),           # split -> unsplit (tensor-memory A)
    ("SMB_ROWS_SPLIT", "0", (44100, 32000, "high")),
    ("SMB_ROWS_SPLIT", "1", (16000, 44100, "high")),           # unsplit -> split, five chunks
    ("SMB_ROWS_SPLIT", "1", (6500, 6400, ("custom", 80.0, 0.8))),   # ... three chunks
    ("SMB_GEMM_WINDOWS", "1", (44100, 16000, "high")),         # row -> window form
    ("SMB_GEMM_WINDOWS", "1", (16000, 44100, "high")),
    ("executor", "direct", (44100, 16000, "high")),            # the blocked direct float32 kernel
    ("executor", "direct", (48000, 44100, "high")),
]

"""The tensor-core resampler's layouts are host tables: ``Config.layout`` reports them
without a GPU, so the planner's branches and the layout switches are checked here (the
audio each layout computes is held to its bounds in test_gpu_resample_bounds.py)."""
import json
import os
import subprocess
import sys

import pytest

from resample_geometries import FORCED, GEOMETRIES, env, geometry, plan, summary  # noqa: F401 (env)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def sb(lib):
    return lib


def test_table_covers_every_layout_branch(sb, env):
    """Each row still builds the layout its comment describes, and together the rows reach
    every branch of the row-form planner and its fall backs."""
    layouts = []
    for g in GEOMETRIES:
        cfg, s, layout, _ = plan(sb, g)
        assert summary(layout) == g[3], (g[:3], summary(layout))
        layouts += [(s, x) for x in layout]
    rows = [(s, x) for s, x in layouts if x["form"] == "row"]
    want = {
        "row form, one column group": any(x["groups"] == 1 for _, x in rows),
        "row form, several column groups": any(x["groups"] > 1 for _, x in rows),
        "split main shift (two issuers)": any(x["two_issuers"] for _, x in rows),
        "unsplit": any(not x["two_issuers"] for _, x in rows),
        "A tiles in tensor memory": any(x["a_tmem"] for _, x in rows),
        "A tiles in shared memory": any(not x["a_tmem"] for _, x in rows),
        "one K-chunk count of 3": any(x["chunks"] == 3 for _, x in rows),
        "14 or more K-chunks": any(x["chunks"] >= 14 for _, x in rows),
        "a run split (slices > chunks, unsplit)": any(not x["two_issuers"] and x["slices"] > x["chunks"]
                                                      for _, x in rows),
        "a gemm stage on the window form": any(x["form"] == "window" for _, x in layouts),
        "a gemm stage on the direct kernel (L > 1024)": any(x["form"] == "direct" for _, x in layouts),
    }
    # every staging depth the planner can pick: tensor-memory A at B = 4, 3, 2, shared-memory
    # A at (2, 3), (3, 2), (2, 2)
    for tmem, a_st, b_st in [(True, 2, 4), (True, 2, 3), (True, 2, 2), (False, 2, 3), (False, 3, 2), (False, 2, 2)]:
        want[f"{'tensor' if tmem else 'shared'}-memory A, stages ({a_st}, {b_st})"] = any(
            x["a_tmem"] == tmem and (x["a_stages"], x["b_stages"]) == (a_st, b_st) for _, x in rows)
    for q in range(1, 5):
        want[f"{q} shifts"] = any(x["shifts"] == q for _, x in rows)
    for r in range(4):
        want[f"L mod 4 = {r}"] = any(s["l"] % 4 == r for s, _ in rows)
    missing = [k for k, ok in want.items() if not ok]
    assert not missing, missing


@pytest.mark.parametrize("switch,value,geom", [f for f in FORCED if f[0] != "executor"],
                         ids=[f"{a}={b}-{g[0]}-{g[1]}" for a, b, g in FORCED if a != "executor"])
def test_forced_switch_changes_the_layout(sb, env, switch, value, geom):
    """Each environment switch of the GPU bounds test moves its geometry off the default
    layout (the switches are read when a fresh Config builds its tables)."""
    env.setenv(switch, value)
    _, _, layout, _ = plan(sb, geom)
    assert summary(layout) != geometry(*geom)[3], (switch, summary(layout))


def test_layout_answers_without_a_device():
    """With every CUDA device hidden, layout() still reports the planned layouts: it reads
    host tables only and never needs a device."""
    code = (
        "import json, sys\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import soundml_b200 as sb\n"
        "out = []\n"
        f"for sr, target, q in {[g[:3] for g in GEOMETRIES[:3]]!r}:\n"
        "    out.append(sb.Resample.Config.create(sample_rate=sr, target=target, quality=q).layout(0))\n"
        "print(json.dumps(out))\n")
    clean = {k: v for k, v in os.environ.items() if not k.startswith("SMB_")}
    res = subprocess.run([sys.executable, "-s", "-c", code], capture_output=True, text=True, timeout=600,
                         env=dict(clean, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 0, res.stderr[-2000:]
    layouts = json.loads(res.stdout.strip().splitlines()[-1])
    assert [summary(x) for x in layouts] == [g[3] for g in GEOMETRIES[:3]]

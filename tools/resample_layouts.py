"""Which tcgen05 layout the resampler's device plan builds, over a sweep of rate pairs
and qualities (needs a GPU: the layout is decided when the device tables are built).

    python tools/resample_layouts.py [out.jsonl]

One JSON line per plan whose single stage the planner tags "gemm": the stage's L, M, K
and ``Config.layout(0)`` under the default switches and under each of SMB_ROWS_SPLIT=0/1,
SMB_ROWS_SMEM_A=1, SMB_ROWS_TMEM_A=1.  tests/test_gpu_resample_bounds.py picks its
geometry table from this output."""
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import soundml_b200 as sb  # noqa: E402

RATES = [8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000, 88200, 96000, 192000]
# synthetic ratios L/M (rates L * 100 and M * 100): every L mod 4, M from one K-chunk up
LS = [64, 65, 66, 67, 98, 99, 101, 127, 128, 147, 160, 161, 200, 320, 441, 640, 1000]
MS = [20, 49, 65, 80, 97, 100, 147, 160, 200, 256, 300, 441, 500, 700, 1000]
QUALITIES = ["fast", "high", "best", ("custom", 80.0, 0.8), ("custom", 100.0, 0.9),
             ("custom", 126.0, 0.95), ("custom", 160.0, 0.9), ("custom", 160.0, 0.97),
             ("custom", 200.0, 0.99)]
SWITCHES = {"split0": {"SMB_ROWS_SPLIT": "0"}, "split1": {"SMB_ROWS_SPLIT": "1"},
            "smem_a": {"SMB_ROWS_SMEM_A": "1"}, "tmem_a": {"SMB_ROWS_TMEM_A": "1"}}


def layout(sr, target, quality, env):
    for k in ("SMB_ROWS_SPLIT", "SMB_ROWS_SMEM_A", "SMB_ROWS_TMEM_A", "SMB_GEMM_WINDOWS"):
        os.environ.pop(k, None)
    os.environ.update(env)
    cfg = sb.Resample.Config.create(sample_rate=sr, target=target, quality=quality)
    st = cfg.stages()
    if len(st) != 1 or st[0]["exec"] != "gemm":
        return None, None
    return st[0], cfg.layout(0)


def main():
    pairs = [(a, b) for a in RATES for b in RATES if a != b]
    pairs += [(m * 100, l * 100) for l in LS for m in MS if math.gcd(l, m) == 1]
    out = open(sys.argv[1], "w") if len(sys.argv) > 1 else sys.stdout
    for sr, target in pairs:
        for q in QUALITIES:
            try:
                st, lay = layout(sr, target, q, {})
            except ValueError:
                continue
            if st is None:
                continue
            rec = dict(sr=sr, target=target, quality=q, l=st["l"], m=st["m"], k=st["k"], default=lay)
            for name, env in SWITCHES.items():
                rec[name] = layout(sr, target, q, env)[1]
            out.write(json.dumps(rec) + "\n")
            out.flush()


if __name__ == "__main__":
    main()

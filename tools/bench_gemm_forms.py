"""Window form against row form of the tensor-core resampler stage (one GPU, device
resident): 44.1 -> 16 kHz at BASELINE configs[3]'s per-GPU share (512 clips x 30 s),
and the 44.1 <-> 48 kHz pair.  SMB_GEMM_WINDOWS=1 selects the window form.
python tools/bench_gemm_forms.py"""
import json
import os
import sys

import torch

sys.path.insert(0, ".")
import soundml_b200 as sb  # noqa: E402
from bench import peak_hbm  # noqa: E402


def run(cfg, x, out, reps=5):
    sb.Resample.apply(cfg, x, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        sb.Resample.apply(cfg, x, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    peak, _ = peak_hbm()
    for sr, target, clips in [(44100, 16000, 512), (44100, 48000, 128), (48000, 44100, 128), (44100, 32000, 128), (16000, 44100, 128)]:
        n = 30 * sr
        x = torch.rand((clips, n), device="cuda") * 2 - 1
        cfg = sb.Resample.Config.create(sample_rate=sr, target=target)
        out = torch.empty((clips, cfg.output_frames(n)), device="cuda")
        os.environ.pop("SMB_GEMM_WINDOWS", None)
        rows_ms = run(cfg, x, out)
        got = out.clone()
        os.environ["SMB_GEMM_WINDOWS"] = "1"
        win_ms = run(cfg, x, out)
        os.environ.pop("SMB_GEMM_WINDOWS", None)
        diff = float((got - out).abs().max() / out.abs().max())
        gb = (x.numel() + out.numel()) * 4 / 1e9
        print(json.dumps({"pair": f"{sr}->{target}", "clips": clips, "plan": cfg.pp(),
                          "rows_ms": round(rows_ms, 3), "windows_ms": round(win_ms, 3),
                          "rows_hbm_frac": round(gb / (rows_ms * 1e-3) / peak, 3),
                          "windows_hbm_frac": round(gb / (win_ms * 1e-3) / peak, 3),
                          "max_diff_of_peak": diff}), flush=True)
        del x, out, got


if __name__ == "__main__":
    main()

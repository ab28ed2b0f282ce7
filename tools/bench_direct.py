"""The direct-form polyphase kernel on the cases VERDICT r1 names: short FIRs, the
48 <-> 8 kHz cascades (their short stages run on the direct kernel), float64 against
float32, each against the HBM bound (input + output once).  Ratios the blocked kernel
takes (L, M <= 4) run on it; the others on the one-output-per-thread kernel.
    python tools/bench_direct.py"""
import json
import sys

import torch

sys.path.insert(0, ".")
import soundml_b200 as sb  # noqa: E402
from bench import peak_hbm  # noqa: E402


def timed(fn, steps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    peak, _ = peak_hbm()

    def measure(name, fn, nbytes):
        ms = timed(fn)
        print(json.dumps({"case": name, "ms": round(ms, 3),
                          "hbm_frac": round(nbytes / (ms * 1e-3) / 1e9 / peak, 3)}), flush=True)

    lines, n = 128, 60 * 48000
    x = torch.rand((lines, n), device="cuda") * 2 - 1
    y = torch.empty_like(x)
    for k in (7, 25, 255):
        fir = sb.Fir.lowpass(k=k, cutoff=0.25)
        measure(f"fir_{2 * k + 1}_taps_direct_f32", lambda: fir.apply(x, method="direct", out=y), 2 * x.numel() * 4)
    del x, y
    for sr, target in ((48000, 8000), (8000, 48000), (48000, 16000), (16000, 48000), (32000, 16000)):
        for dtype in (torch.float32, torch.float64):
            n = 30 * sr
            x = (torch.rand((128, n), device="cuda", dtype=dtype) * 2 - 1)
            cfg = sb.Resample.Config.create(sample_rate=sr, target=target)
            if dtype == torch.float32:
                cfg.set_executor("direct")       # float64 always runs the direct kernel
            out = torch.empty((128, cfg.output_frames(n)), device="cuda", dtype=dtype)
            measure(f"{sr}->{target} direct {str(dtype)[6:]} [{cfg.pp()}]",
                    lambda: sb.Resample.apply(cfg, x, out=out), (x.numel() + out.numel()) * x.element_size())
            del x, out


if __name__ == "__main__":
    main()

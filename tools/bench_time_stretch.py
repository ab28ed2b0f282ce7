"""time_stretch on one GPU: per-stage CUDA-event times and the vocoder's HBM fraction.

    python tools/bench_time_stretch.py [--clips 1024] [--seconds 10] [--rates 0.8,1,1.25]
                                       [--repeat 5] [--out FILE]

A batch of float32 clips (22050 Hz, fft 2048 / hop 512, the fused path) is stretched at
each rate.  Reported per rate, medians over --repeat timed passes after a warm-up:

* transform / vocoder / invert: the three stages as separate calls, each between two
  CUDA events (transform and vocoder write into preallocated outputs, so their times are
  the kernels'; invert allocates its zero-filled output as a user's call does);
* time_stretch: the one-call form (transform -> vocoder -> invert on one stream, output
  allocation included);
* the vocoder's HBM traffic, 8 (T + T') bytes per (clip, bin) row for complex64, over its
  time, and that rate as a fraction of the B200's 7.7 TB/s data-sheet bandwidth;
* kernel launches per time_stretch call (kernel_launch_count).

The card's name, power limit and maximum SM clock are read in the same run.  The
spectra (3.6 GB for the default batch) are far larger than the 126 MB L2, so every pass
reads HBM.  JSON lines go to stdout and, with --out, to FILE.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12      # HGX B200 data sheet, one GPU


def card():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power, clock = [v.strip() for v in q.stdout.strip().split(",")]
        info.update(power_limit=power, max_sm_clock=clock)
    except Exception as e:                              # report, do not guess
        info.update(power_limit=f"unavailable ({type(e).__name__})", max_sm_clock=None)
    return info


def timed(fn, repeat):
    import torch
    times = []
    for _ in range(repeat):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    return times[len(times) // 2]


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--rates", default="0.8,1,1.25")
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_time_stretch: needs a CUDA device (nothing is measured on the CPU)")
    import soundml_b200 as sb

    sr, fft, hop = 22050, 2048, 512
    n = int(round(args.seconds * sr))
    c = sb.Stft.Config.create(fft_size=fft, hop=hop)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(args.clips, n, device="cuda", generator=g) * 0.1
    z = sb.Stft.transform(c, x)
    frames = z.shape[-1]
    rows = args.clips * c.bins
    lines = [dict(kind="setup", clips=args.clips, samples=n, sample_rate=sr, fft_size=fft, hop=hop,
                  frames=frames, dtype="float32", **card())]
    for rate in [float(r) for r in args.rates.split(",")]:
        out_frames = sb.Effects.stretched_frames(frames, rate)
        length = sb.Effects.stretched_length(n, rate)
        voc = torch.empty(args.clips, c.bins, out_frames, dtype=torch.complex64, device="cuda")
        zt = torch.empty_like(z)
        holder = {}
        stages = {
            "transform": lambda: sb.Stft.transform(c, x, out=zt),
            "vocoder": lambda: sb.Effects.phase_vocoder(c, z, rate, out=voc),
            "invert": lambda: holder.__setitem__("y", sb.Stft.invert(c, voc, length=length)),
            "time_stretch": lambda: holder.__setitem__("y", sb.Effects.time_stretch(c, x, rate)),
        }
        for fn in stages.values():                      # warm every shape
            fn()
        torch.cuda.synchronize()
        before = sb.kernel_launch_count()
        stages["time_stretch"]()
        torch.cuda.synchronize()
        launches = sb.kernel_launch_count() - before
        ms = {k: timed(fn, args.repeat) for k, fn in stages.items()}
        vbytes = rows * 8 * (frames + out_frames)
        rate_bps = vbytes / (ms["vocoder"] * 1e-3)
        lines.append(dict(kind="rate", rate=rate, out_frames=out_frames, out_samples=length,
                          transform_ms=ms["transform"], vocoder_ms=ms["vocoder"],
                          invert_ms=ms["invert"], time_stretch_ms=ms["time_stretch"],
                          vocoder_bytes=vbytes, vocoder_tb_per_s=rate_bps / 1e12,
                          vocoder_hbm_fraction=rate_bps / HBM_BYTES_PER_S,
                          launches_per_call=launches))
        del voc, zt, holder
        torch.cuda.empty_cache()
    text = "\n".join(json.dumps(l) for l in lines)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

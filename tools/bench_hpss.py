"""Harmonic-percussive separation on one GPU: the hpss kernel against its byte floor, the
audio calls end to end, and a stock-library composition measured in the same run.

    python tools/bench_hpss.py [--clips 1024] [--seconds 10] [--repeat 5] [--out FILE]

A batch of float32 clips (22050 Hz, fft 2048 / hop 512) is transformed once; then, as
medians of --repeat passes between CUDA events after a warm-up:

* hpss on the complex64 spectrum through the C ABI into a preallocated [clips, 2, bins,
  frames] output (the kernel alone): at kernel 31 (the fused tile kernel) and at (17, 63)
  (the exact counting kernel, one pass: it is O(w^2) per output).  The fused call moves at
  least 24 bytes per element (read 8, write 2 x 8); that floor at the B200 data sheet's
  7.7 TB/s over the measured time is the kernel's share of its byte floor;
* separate / harmonic / percussive end to end (transform -> hpss -> invert in one call,
  output allocation included), with their kernel launches per call;
* the torch composition: torch.stft -> |D| -> reflect-indexed unfold + median in chunks
  of clips along each axis -> the same soft masks -> torch.istft of both parts.

``--kernel-only`` times the tile kernel alone, for A/B runs of builds with another tile
(``SOUNDML_B200_LIB`` pointing at a ``build.py -DSMB_HPSS_TILE=... --out=...`` library).

The card's name, power limit and maximum SM clock are read in the same run.  The
spectrum (3.6 GB for the default batch) and the outputs are far larger than the 126 MB
L2, so every pass reads HBM.  JSON lines go to stdout and, with --out, to FILE.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_time_stretch import HBM_BYTES_PER_S, card, timed   # noqa: E402


def torch_hpss_audio(torch, x, window, fft, hop, win, power, chunk):
    """The stock composition: torch.stft, sliding medians by unfold + median, librosa's
    soft masks, torch.istft.  Medians read reflect-indexed copies (scipy's rule)."""
    n = x.shape[-1]
    D = torch.stft(x, fft, hop, window=window, center=True, pad_mode="constant", return_complex=True)
    S = D.abs()
    bins, frames = S.shape[-2:]

    def reflect(count, w):
        q = torch.arange(count, device=x.device)[:, None] - w // 2 + torch.arange(w, device=x.device)[None, :]
        m = torch.remainder(q, 2 * count)
        return torch.where(m < count, m, 2 * count - 1 - m)

    ih, ip = reflect(frames, win), reflect(bins, win)
    harm, perc = torch.empty_like(S), torch.empty_like(S)
    for c0 in range(0, S.shape[0], chunk):
        s = S[c0:c0 + chunk]
        harm[c0:c0 + chunk] = s[:, :, ih].median(dim=-1).values
        perc[c0:c0 + chunk] = s[:, ip, :].median(dim=-2).values
    tiny = torch.finfo(S.dtype).tiny

    def softmask(a, b):
        z = torch.maximum(a, b)
        bad = z < tiny
        z = torch.where(bad, torch.ones_like(z), z)
        ma, mb = (a / z) ** power, (b / z) ** power
        return torch.where(bad, torch.full_like(z, 0.5), ma / (ma + mb))

    mh, mp = softmask(harm, perc), softmask(perc, harm)
    H, P = D * mh, D * mp
    return (torch.istft(H, fft, hop, window=window, center=True, length=n),
            torch.istft(P, fft, hop, window=window, center=True, length=n))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--chunk", type=int, default=16, help="clips per median chunk of the torch composition")
    ap.add_argument("--kernel-only", action="store_true", help="time the tile kernel at kernel 31 only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_hpss: needs a CUDA device (nothing is measured on the CPU)")
    import soundml_b200 as sb
    from soundml_b200 import _lib

    sr, fft, hop = 22050, 2048, 512
    n = int(round(args.seconds * sr))
    c = sb.Stft.Config.create(fft_size=fft, hop=hop)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(args.clips, n, device="cuda", generator=g) * 0.1
    D = sb.Stft.transform(c, x)
    bins, frames = D.shape[-2:]
    cells = args.clips * bins * frames
    lines = [dict(kind="setup", clips=args.clips, samples=n, sample_rate=sr, fft_size=fft, hop=hop,
                  bins=bins, frames=frames, dtype="float32", elements=cells, **card())]

    out = torch.empty((args.clips, 2, bins, frames), dtype=torch.complex64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def kernel(k):
        wh, wp = (k, k) if isinstance(k, int) else k
        _lib.check(_lib.lib.smb_hpss(D.data_ptr(), args.clips, bins, frames, _lib.F32, 1, wh, wp, 2.0, 1.0, 1.0,
                                     0, out.data_ptr(), _lib.MEM_DEVICE, stream))

    floor_bytes = 24 * cells
    for k, reps in ((31, args.repeat),) + (() if args.kernel_only else (((17, 63), 1),)):
        kernel(k)
        torch.cuda.synchronize()
        ms = timed(lambda: kernel(k), reps)
        floor_ms = floor_bytes / HBM_BYTES_PER_S * 1e3
        lines.append(dict(kind="hpss_kernel", kernel_size=k, path="tile" if k == 31 else "counting",
                          input="complex64", output="both", ms=ms, floor_bytes=floor_bytes,
                          byte_floor_ms=floor_ms, share_of_byte_floor=floor_ms / ms,
                          tb_per_s=floor_bytes / (ms * 1e-3) / 1e12, passes=reps,
                          library=os.environ.get("SOUNDML_B200_LIB") or "default"))
    if args.kernel_only:
        print("\n".join(json.dumps(l) for l in lines), flush=True)
        return
    del out
    torch.cuda.empty_cache()

    holder = {}
    for name, fn in (("separate", sb.Hpss.separate), ("harmonic", sb.Hpss.harmonic),
                     ("percussive", sb.Hpss.percussive)):
        call = (lambda f=fn: holder.__setitem__("y", f(c, x)))
        call()
        torch.cuda.synchronize()
        before = sb.kernel_launch_count()
        call()
        torch.cuda.synchronize()
        launches = sb.kernel_launch_count() - before
        ms = timed(call, args.repeat)
        lines.append(dict(kind="audio", call=name, kernel_size=31, ms=ms, launches_per_call=launches))
        holder.clear()
        torch.cuda.empty_cache()

    window = torch.hann_window(fft, periodic=True, device="cuda")
    comp = (lambda: holder.__setitem__("y", torch_hpss_audio(torch, x, window, fft, hop, 31, 2.0, args.chunk)))
    comp()
    torch.cuda.synchronize()
    ms = timed(comp, max(1, min(args.repeat, 3)))
    lines.append(dict(kind="torch_composition", call="separate", kernel_size=31, ms=ms, median_chunk=args.chunk,
                      torch=torch.__version__))

    text = "\n".join(json.dumps(l) for l in lines)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

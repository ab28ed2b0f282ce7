"""Spectral descriptors on one GPU: the kernel against its byte floor, features_audio end to
end, and a stock-library composition measured in the same run.

    python tools/bench_spectral.py [--clips 1024] [--seconds 10] [--repeat 5] [--out FILE]

A batch of float32 clips (22050 Hz, fft 2048 / hop 512) is turned once into its magnitude
spectrogram S [clips, 1025, frames] (Stft.power_spectrum at power 1); then, as medians of
--repeat passes between CUDA events after a warm-up:

* smb_spectral on S through the C ABI into a preallocated output (the kernel alone), with
  all four descriptors and with each alone.  The kernel must read S once: 4 bytes per
  element.  That floor at the B200 data sheet's 7.7 TB/s over the measured time is the
  kernel's share of its byte floor.  The bandwidth re-reads each frame's bins in a second
  pass; its time against the centroid's tells whether that pass reads L2 or HBM;
* Stft.power_spectrum alone and Spectral.features_audio end to end (output allocation
  included), with the launches per call;
* the torch composition: torch.stft -> abs -> the four formulas with cumsum / argmax.

``--kernel-only`` times the kernel alone, for A/B runs of builds with another CTA size or load
batch (``SOUNDML_B200_LIB`` pointing at a ``build.py -DSMB_SPECTRAL_THREADS=... --out=...`` or
``-DSMB_SPECTRAL_LOADS=...`` library; the record names the library by its file name).

The card's name, power limit and maximum SM clock are read in the same run.  S (1.8 GB for
the default batch) is far larger than the 126 MB L2, so every pass reads HBM.  JSON lines
go to stdout and, with --out, to FILE.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_time_stretch import HBM_BYTES_PER_S, card, timed   # noqa: E402

FLAGS = {"all": 15, "centroid": 1, "bandwidth": 2, "rolloff": 4, "flatness": 8}


def torch_descriptors(torch, x, window, fft, hop, sr, roll_percent=0.85, amin=1e-10, power=2.0):
    """The stock composition of librosa's four formulas over torch.stft's magnitudes."""
    S = torch.stft(x, fft, hop, window=window, center=True, pad_mode="constant", return_complex=True).abs()
    f = torch.arange(S.shape[-2], device=x.device, dtype=torch.float64)[:, None] * (sr / fft)
    f32 = f.float()
    L = S.sum(dim=-2, keepdim=True)
    L = torch.where(L < torch.finfo(S.dtype).tiny, torch.ones_like(L), L)
    centroid = (f32 * S).sum(dim=-2, keepdim=True) / L
    bandwidth = ((S / L) * (f32 - centroid) ** 2).sum(dim=-2, keepdim=True).sqrt()
    cum = S.cumsum(dim=-2)
    reached = cum >= roll_percent * cum[..., -1:, :]
    rolloff = f32[:, 0][reached.int().argmax(dim=-2, keepdim=True)]
    m = torch.clamp(S ** power, min=amin)
    flatness = m.log().mean(dim=-2, keepdim=True).exp() / m.mean(dim=-2, keepdim=True)
    return centroid, bandwidth, rolloff, flatness


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--repeat", type=int, default=5)
    ap.add_argument("--kernel-only", action="store_true", help="time the kernel with all four descriptors only")
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_spectral: needs a CUDA device (nothing is measured on the CPU)")
    import soundml_b200 as sb
    from soundml_b200 import _lib

    sr, fft, hop = 22050, 2048, 512
    n = int(round(args.seconds * sr))
    c = sb.Stft.Config.create(fft_size=fft, hop=hop)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(args.clips, n, device="cuda", generator=g) * 0.1
    S = sb.Stft.power_spectrum(c, x, power=1.0)
    bins, frames = S.shape[-2:]
    cells = args.clips * bins * frames
    lines = [dict(kind="setup", clips=args.clips, samples=n, sample_rate=sr, fft_size=fft, hop=hop,
                  bins=bins, frames=frames, dtype="float32", elements=cells, **card())]

    out = torch.empty((args.clips, 4, frames), dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def kernel(what):
        _lib.check(_lib.lib.smb_spectral(S.data_ptr(), args.clips, bins, frames, _lib.F32, _lib.DEFAULT, float(sr),
                                         what, 2.0, 1, 0.85, 1e-10, 2.0, out.data_ptr(), _lib.MEM_DEVICE, stream))

    floor_bytes = 4 * cells
    floor_ms = floor_bytes / HBM_BYTES_PER_S * 1e3
    for name in (("all",) if args.kernel_only else tuple(FLAGS)):
        what = FLAGS[name]
        kernel(what)
        torch.cuda.synchronize()
        ms = timed(lambda: kernel(what), args.repeat)
        lines.append(dict(kind="spectral_kernel", descriptors=name, input="float32 magnitude", ms=ms,
                          floor_bytes=floor_bytes, byte_floor_ms=floor_ms, share_of_byte_floor=floor_ms / ms,
                          tb_per_s=floor_bytes / (ms * 1e-3) / 1e12, passes=args.repeat,
                          library=os.path.basename(os.environ.get("SOUNDML_B200_LIB", "")) or "default"))
    if args.kernel_only:
        print("\n".join(json.dumps(l) for l in lines), flush=True)
        return
    del out, S
    torch.cuda.empty_cache()

    holder = {}
    calls = (("power_spectrum", lambda: sb.Stft.power_spectrum(c, x, power=1.0)),
             ("features_audio", lambda: sb.Spectral.features_audio(c, x, sr)))
    for name, fn in calls:
        call = (lambda f=fn: holder.__setitem__("y", f()))
        call()
        torch.cuda.synchronize()
        before = sb.kernel_launch_count()
        call()
        torch.cuda.synchronize()
        launches = sb.kernel_launch_count() - before
        ms = timed(call, args.repeat)
        lines.append(dict(kind="audio", call=name, ms=ms, launches_per_call=launches))
        holder.clear()
        torch.cuda.empty_cache()

    window = torch.hann_window(fft, periodic=True, device="cuda")
    comp = (lambda: holder.__setitem__("y", torch_descriptors(torch, x, window, fft, hop, sr)))
    comp()
    torch.cuda.synchronize()
    ms = timed(comp, args.repeat)
    lines.append(dict(kind="torch_composition", call="four descriptors", ms=ms, torch=torch.__version__))
    holder.clear()
    torch.cuda.empty_cache()

    text = "\n".join(json.dumps(l) for l in lines)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

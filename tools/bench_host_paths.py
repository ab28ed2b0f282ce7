"""Host-memory calls (pinned buffers) of the resampler (float32 and float64), the FIR, the
mel projection and the log-mel spectrogram against the copy floor of the same buffers:
cudaMemcpyAsync of input and output alone, both directions at once.  Every batch spans
several 64 MB slices.  python tools/bench_host_paths.py"""
import json
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import soundml_b200 as sb  # noqa: E402


def pinned(shape, dtype=torch.float32):
    return torch.empty(shape, dtype=dtype).pin_memory()


def timed(fn, steps=3):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / steps


def copy_floor(xh, yh):
    d_in = torch.empty_like(xh, device="cuda")
    d_out = torch.empty_like(yh, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def go():
        with torch.cuda.stream(s1):
            d_in.copy_(xh, non_blocking=True)
        with torch.cuda.stream(s2):
            yh.copy_(d_out, non_blocking=True)
    return timed(go)


def main():
    # BASELINE.json configs[3], one GPU's share: 512 clips x 30 s, 44.1 -> 16 kHz
    clips, n = 512, 30 * 44100
    cfg = sb.Resample.Config.create(sample_rate=44100, target=16000)
    xh = pinned((clips, n))
    xh.uniform_(-1, 1)
    yh = pinned((clips, cfg.output_frames(n)))
    ms = timed(lambda: sb.Resample.apply(cfg, xh.numpy(), out=yh.numpy()))
    floor = copy_floor(xh, yh)
    dev = sb.Resample.apply(cfg, xh.cuda()).cpu()
    print(json.dumps({"case": "resample 44.1->16 kHz, 512 x 30 s, pinned host buffers", "ms": round(ms, 2),
                      "copy_floor_ms": round(floor, 2), "over_floor": round(ms / floor, 3),
                      "equals_device_call": bool(torch.equal(dev, yh))}))
    del xh, yh
    lines, n = 128, 60 * 48000
    fir = sb.Fir.lowpass(k=255, cutoff=0.25)
    xh = pinned((lines, n))
    xh.uniform_(-1, 1)
    yh = pinned((lines, n))
    ms = timed(lambda: fir.apply(xh.numpy(), method="ols", out=yh.numpy()))
    floor = copy_floor(xh, yh)
    print(json.dumps({"case": "FIR 511 taps (ols), 128 lines x 60 s, pinned host buffers", "ms": round(ms, 2),
                      "copy_floor_ms": round(floor, 2), "over_floor": round(ms / floor, 3)}))
    del xh, yh
    # float64 audio: the direct kernel in double, 128 clips x 30 s (1.4 GB in)
    clips, n = 128, 30 * 44100
    xh = pinned((clips, n), torch.float64)
    xh.uniform_(-1, 1)
    yh = pinned((clips, cfg.output_frames(n)), torch.float64)
    ms = timed(lambda: sb.Resample.apply(cfg, xh.numpy(), out=yh.numpy()))
    floor = copy_floor(xh, yh)
    dev = sb.Resample.apply(cfg, xh.cuda()).cpu()
    print(json.dumps({"case": "resample float64 44.1->16 kHz, 128 x 30 s, pinned host buffers", "ms": round(ms, 2),
                      "copy_floor_ms": round(floor, 2), "over_floor": round(ms / floor, 3),
                      "equals_device_call": bool(torch.equal(dev, yh))}))
    del xh, yh
    mc = sb.Mel.Config.create(n_mels=128, sample_rate=22050, fft_size=2048)
    batch, frames = 64, 2600                                   # 680 MB of power spectrogram
    sh = pinned((batch, mc.bins, frames))
    sh.uniform_(0, 1)
    yh = pinned((batch, 128, frames))

    def mel_apply():
        sb._lib.check(sb._lib.lib.smb_mel_apply(mc._h, sh.data_ptr(), batch, frames, sb._lib.F32,
                                                yh.data_ptr(), sb._lib.MEM_HOST))
    ms = timed(mel_apply)
    floor = copy_floor(sh, yh)
    dev = sb.Mel.apply(mc, sh.cuda()).cpu()
    print(json.dumps({"case": "mel_apply fft 2048 / 128 mels, 64 x 2600 frames, pinned host buffers",
                      "ms": round(ms, 2), "copy_floor_ms": round(floor, 2), "over_floor": round(ms / floor, 3),
                      "equals_device_call": bool(torch.equal(dev, yh))}))
    del sh, yh
    sc = sb.Stft.Config.create(fft_size=2048, hop=512)
    clips, n = 512, 30 * 22050                                # 1.35 GB of audio
    xh = pinned((clips, n))
    xh.uniform_(-1, 1)
    yh = pinned((clips, 128, sb.Stft.frames(sc, n)))
    ms = timed(lambda: sb.log_mel_spectrogram(sc, mc, xh.numpy(), out=yh.numpy()))
    floor = copy_floor(xh, yh)
    dev = sb.log_mel_spectrogram(sc, mc, xh.cuda()).cpu()
    print(json.dumps({"case": "mel_spectrogram_db fft 2048 / 128 mels, 512 x 30 s, pinned host buffers",
                      "ms": round(ms, 2), "copy_floor_ms": round(floor, 2), "over_floor": round(ms / floor, 3),
                      "equals_device_call": bool(torch.equal(dev, yh))}))


if __name__ == "__main__":
    main()

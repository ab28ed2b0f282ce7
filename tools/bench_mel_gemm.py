"""The mel projection as the dense GEMM north_star names (Nx.matmul in mel.ml:231), measured:
cuBLAS through torch.matmul on a materialised power spectrogram [1024, 1025, 431] -- float32
and tf32 tensor cores -- beside the library's sparse band product (Mel.apply, standalone) and
the whole mel spectrogram in the fused frame-pair kernel.  One GPU.
python tools/bench_mel_gemm.py"""
import json
import sys

import torch

sys.path.insert(0, ".")
import soundml_b200 as sb  # noqa: E402


def timed(fn, reps=10):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    clips, bins, frames, n_mels = 1024, 1025, 431, 128
    mel = sb.Mel.Config.create(n_mels=n_mels, sample_rate=22050, fft_size=2048)
    w = torch.from_numpy(sb.Mel.filterbank(mel).astype("float32")).cuda()   # [128, 1025]
    p = torch.rand((clips, bins, frames), device="cuda")
    out = torch.empty((clips, n_mels, frames), device="cuda")
    res = {"workload": f"{clips} x [{bins}, {frames}] f32 power spectrogram -> [{n_mels}, {frames}]",
           "weights_nonzero_fraction": float((w != 0).float().mean())}
    torch.backends.cuda.matmul.allow_tf32 = False
    res["cublas_fp32_ms"] = timed(lambda: torch.matmul(w, p, out=out))
    ref = out.clone()
    torch.backends.cuda.matmul.allow_tf32 = True
    res["cublas_tf32_ms"] = timed(lambda: torch.matmul(w, p, out=out))
    res["cublas_tf32_max_err_of_peak"] = float((out - ref).abs().max() / ref.abs().max())
    res["band_product_ms"] = timed(lambda: sb.Mel.apply(mel, p))
    res["band_product_max_err_of_peak"] = float((sb.Mel.apply(mel, p) - ref).abs().max() / ref.abs().max())
    # the fused kernel: audio to mel spectrogram, the power spectrogram never materialised
    del p, out, ref
    stft = sb.Stft.Config.create(fft_size=2048, hop=512)
    x = torch.rand((clips, 220500), device="cuda") * 2 - 1
    o = torch.empty((clips, n_mels, sb.Stft.frames(stft, 220500)), device="cuda")
    res["fused_mel_spectrogram_ms"] = timed(lambda: sb.mel_spectrogram(stft, mel, x, out=o), 50)
    res["power_spectrogram_materialised_ms"] = None
    ps = torch.empty((clips, bins, sb.Stft.frames(stft, 220500)), device="cuda")
    res["power_spectrogram_materialised_ms"] = timed(lambda: sb.Stft.power_spectrum(stft, x, out=ps))
    print(json.dumps(res))


if __name__ == "__main__":
    main()

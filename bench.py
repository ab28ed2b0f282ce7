#!/usr/bin/env python
"""Headline benchmark: BASELINE.json configs[1].

    128-band mel power spectrogram of a batch of 1024 x 10 s 22.05 kHz clips,
    n_fft 2048, hop 512, Hann, centered/reflect   (per GPU)

A step is one pass of the hot path (Soundml.mel_spectrogram) over the batch.
`value` is audio-seconds per second with the clips already resident in HBM,
timed with CUDA events on the stream the kernel runs on; `e2e` is the same call
on pinned HOST buffers (H2D + kernel + D2H inside the timed region) with
`copy_floor_ms`, the same buffers through cudaMemcpyAsync alone, beside it;
`roofline` divides the algorithmic bytes of one launch by its measured duration
and carries `compute_floor_ms`, the transform skeleton alone (staging, window,
both FFT passes, transposition: smb_stft_fft_ceiling); `secondary` holds
BASELINE.json configs[2..4] (FIR 511, 44.1 -> 16 kHz, resample + STFT + mel), one
GPU's share each, with their own roofline fraction and parity; `cpu_baseline` is
the oracle (the reference's CPU arithmetic restated, see oracle/) timed on this
box's host cores on a bounded sample.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); the clips shard across ranks
with no data-path collective (weak scaling: 1024 clips per GPU), NCCL carries
only the barrier and the max-over-ranks of the timing.

--dump-outputs DIR writes, after the timed steps, what the last timed step
returned to DIR/mel_spectrogram.npy, float32: a fixed, seeded sample of rank 0's
clips (dump_sample below), or with --impl reference the oracle's output for that
arm's 64 clips (clips 0-63).  The inputs are synthesised from a fixed seed, so
two builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 22050
CLIP_SECONDS = 10
N = SR * CLIP_SECONDS            # 220 500 samples
BATCH = 1024                     # clips per GPU
FFT, HOP, N_MELS = 2048, 512, 128
FRAMES = 1 + N // HOP            # 431
METRIC = "stft_mel_audio_seconds_per_second"
UNIT = "audio-s/s"
WORKLOAD = ("mel_spectrogram 128 bands, 1024 x 10 s 22.05 kHz f32 clips per GPU, "
            "n_fft=2048 hop=512 hann centered/reflect (BASELINE.json configs[1])")
# SURVEY.md 8(d): in + out bytes per clip, intermediates stay on chip
BYTES_PER_CLIP = N * 4 + N_MELS * FRAMES * 4       # 1 102 672
ALGO_BYTES = BATCH * BYTES_PER_CLIP                # 1 129 136 128 per launch
FALLBACK_HBM_GBS = 6650.0
# --dump-outputs: 128 of the 1024 clips, 128 x [128, 431] f32 = 28 MB of the 226 MB output
DUMP_CLIPS, DUMP_SEED = 128, 0


def load_synth():
    """soundml_b200/synth.py by path: importing the package would load
    libsoundml_b200.so, which the CPU arms must not map."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "soundml_b200_synth", os.path.join(ROOT, "soundml_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def workload_config(world):
    return {"workload": WORKLOAD, "global_batch_clips": world * BATCH,
            "parallelism": f"clips sharded over {world} GPU(s), no collective",
            "l2": "inputs (903 MB per GPU) exceed L2 (126 MB); no flush needed"}


def peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}",
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc:
            self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            f = [v.strip() for v in line.split(",")]
            try:
                sm.append(float(f[0]))
                smax = max(smax, float(f[1]))
            except Exception:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_pass(x, sc, mc, workers):
    """One pass of the oracle over the clips of x on `workers` host threads: the
    clips are independent (stft.mli:216-218), so they are dealt to a thread pool
    (numpy / scipy release the GIL inside their loops); the window multiply, the
    transposed copy and |z| would otherwise run on one core."""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import mel_oracle
    parts = [p for p in np.array_split(np.arange(x.shape[0]), min(workers, x.shape[0])) if len(p)]
    if len(parts) <= 1:
        return mel_oracle.mel_spectrogram(sc, mc, x, 2.0, workers=workers)
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=1), ThreadPoolExecutor(len(parts)) as pool:   # one BLAS thread per worker
        outs = list(pool.map(lambda p: mel_oracle.mel_spectrogram(sc, mc, x[p[0]:p[-1] + 1], 2.0, workers=1), parts))
    return np.concatenate(outs, axis=0)


def time_cpu(clips, min_seconds, workers, keep=None):
    """Oracle on host cores: repeated passes over a `clips`-clip sample of the
    workload until `min_seconds` of work; returns (audio-s/s, passes, seconds).
    `keep`, a list, receives the oracle's output for the sample so the caller can
    state the GPU path's error against it next to the number."""
    os.environ["OMP_NUM_THREADS"] = str(workers)         # see run_reference
    from oracle import mel_oracle, stft_oracle
    synth = load_synth()
    from threadpoolctl import threadpool_limits
    x = synth.clips_numpy(clips, N, SR)
    sc = stft_oracle.StftConfig(FFT, HOP)
    mc = mel_oracle.MelConfig(N_MELS, SR, FFT)
    with threadpool_limits(limits=workers):
        cpu_reference_pass(x[:2], sc, mc, workers)        # warm the FFT plan cache
        t0, passes = time.perf_counter(), 0
        while True:
            y = cpu_reference_pass(x, sc, mc, workers)
            if keep is not None and not keep:
                keep.append(y)
            passes += 1
            dt = time.perf_counter() - t0
            if dt >= min_seconds:
                return clips * CLIP_SECONDS * passes / dt, passes, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port: OCaml/nx cannot
    be built here, DESIGN.md) on all host cores, rank 0 only."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    clips = 64
    steps = args.steps
    # torchrun exports OMP_NUM_THREADS=1 to every rank; scipy.fft's worker pool and
    # the BLAS behind the oracle's matmul both size themselves from it.  This arm
    # is the CPU path on all host threads at every N: undo the cap before either
    # library starts its pool (and see threadpool_limits below).
    os.environ["OMP_NUM_THREADS"] = str(cores)
    from oracle import mel_oracle, stft_oracle
    synth = load_synth()
    x = synth.clips_numpy(clips, N, SR)
    sc = stft_oracle.StftConfig(FFT, HOP)
    mc = mel_oracle.MelConfig(N_MELS, SR, FFT)
    for _ in range(max(1, min(args.warmup, 3))):
        cpu_reference_pass(x[:8], sc, mc, cores)
    # a BLAS that was loaded before the line above keeps its one thread otherwise
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=cores):
        t0 = time.perf_counter()
        for _ in range(steps):
            y = cpu_reference_pass(x, sc, mc, cores)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y)
    value = clips * CLIP_SECONDS * steps / dt
    sample = (f"{clips} of {BATCH} clips per step (same signal recipe), {steps} steps, clips dealt "
              f"to {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_sample(out):
    """The GPU arm's share of --dump-outputs: float32 [DUMP_CLIPS, N_MELS, FRAMES],
    the clips of `out` at the sorted indices
    default_rng(DUMP_SEED).choice(BATCH, DUMP_CLIPS, replace=False)."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(out.shape[0], DUMP_CLIPS, replace=False))
    return out[torch.from_numpy(idx).to(out.device)].cpu().numpy()


def dump_outputs(path, mel):
    """Write the last timed step's mel spectrograms to DIR/mel_spectrogram.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "mel_spectrogram.npy"), mel)


def timed_ms(fn, steps, warmup, barrier, dev):
    """CUDA-event time per call of fn on torch's current stream, max over ranks."""
    import torch
    from soundml_b200.parallel import max_over_ranks
    for _ in range(warmup):
        fn()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    barrier()
    return max_over_ranks(a.elapsed_time(b), device=dev) / steps


def secondary_configs(sb, dev, world, rank, barrier, peak, with_parity):
    """BASELINE.json configs[2..4], one GPU's share each (weak scaling: every rank
    runs its share, the step time is the max over ranks).  Each entry carries its
    algorithmic bytes (input + output once; taps, banks and intermediates
    excluded, SURVEY.md 8d), the roofline fraction and -- on rank 0 at N = 1 -- the
    error against the float64 oracle on a bounded sample of the same call."""
    import numpy as np
    import torch

    def peak_err(got, want):
        return float(np.abs(np.asarray(got, np.float64) - want).max() / np.abs(want).max())

    def entry(workload, ms, algo_bytes, audio_s, launches, parity):
        ach = algo_bytes / (ms * 1e-3) / 1e9
        return {"workload": workload, "ms_per_step": ms,
                "value": world * audio_s / (ms * 1e-3), "unit": UNIT,
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                             "frac": ach / peak, "algorithmic_bytes_per_launch": algo_bytes},
                "gpu_launches_per_step": launches, "parity": parity}

    out = {}
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)

    def noise(shape):
        return torch.rand(shape, device=dev, generator=gen) * 2 - 1

    def launches_of(fn):
        c0 = sb.kernel_launch_count()
        fn()
        return sb.kernel_launch_count() - c0

    # ---- configs[2]: 511-tap FIR lowpass over 256 x 60 s stereo 48 kHz clips = 512 lines
    lines, n = 512, 60 * 48000
    x = noise((lines, n))
    y = torch.empty_like(x)
    fir = sb.Fir.lowpass(k=255, cutoff=0.25)
    for method, steps in (("ols", 5), ("direct", 2)):
        ms = timed_ms(lambda: fir.apply(x, method=method, out=y), steps, 1, barrier, dev)
        parity = None
        if with_parity:
            from oracle import resample_oracle as R
            m = 200000                                   # outputs [0, m) depend on x[0, m + 255] only
            want = R.fir_apply(x[0, :m + 1024].cpu().numpy(), fir.taps)[:m]
            parity = {"max_rel_err": peak_err(y[0, :m].cpu().numpy(), want), "tolerance": 1e-5,
                      "sample": f"first {m} outputs of line 0 against the float64 oracle"}
        out[f"fir511_{method}"] = entry(
            f"511-tap FIR lowpass ({method}), {lines} lines x 60 s @48 kHz per GPU (BASELINE.json configs[2])",
            ms, 2 * lines * n * 4, lines * 60.0,
            launches_of(lambda: fir.apply(x, method=method, out=y)), parity)
    del x, y

    # ---- configs[3]: 44.1 -> 16 kHz, 4096 x 30 s clips over 8 GPUs = 512 clips per GPU
    clips, n = 512, 30 * 44100
    x = noise((clips, n))
    cfg = sb.Resample.Config.create(sample_rate=44100, target=16000)
    total = cfg.output_frames(n)
    y = torch.empty((clips, total), device=dev)
    ms = timed_ms(lambda: sb.Resample.apply(cfg, x, out=y), 5, 1, barrier, dev)
    parity = None
    if with_parity:
        from oracle import resample_oracle as R
        st = [dict(l=t["l"], m=t["m"], k=t["k"], proto=R.design_prototype(t["l"], t["k"], t["fc"], t["beta"]))
              for t in cfg.stages()]
        want = R.apply_plan(x[0].cpu().numpy(), st, cfg.l, cfg.m)
        parity = {"max_rel_err": peak_err(y[0].cpu().numpy(), want), "tolerance": 1e-5,
                  "sample": f"clip 0 at full length ({n} -> {total} samples) against the float64 oracle"}
    out["resample_44k1_16k"] = entry(
        f"{cfg.pp()}, {clips} clips x 30 s per GPU (BASELINE.json configs[3]: 4096 clips over 8 GPUs)",
        ms, clips * (n + total) * 4, clips * 30.0,
        launches_of(lambda: sb.Resample.apply(cfg, x, out=y)), parity)
    del x, y

    # ---- configs[4]: resample 44.1 -> 22.05 kHz + STFT + mel, 65536 x 10 s over 8 GPUs = 8192 per GPU
    clips, n = 8192, 10 * 44100
    x = noise((clips, n))
    cfg = sb.Resample.Config.create(sample_rate=44100, target=22050)
    mid = torch.empty((clips, cfg.output_frames(n)), device=dev)
    sc = sb.Stft.Config.create(fft_size=FFT, hop=HOP)
    mc = sb.Mel.Config.create(n_mels=N_MELS, sample_rate=SR, fft_size=FFT)
    frames = sb.Stft.frames(sc, mid.shape[1])
    y = torch.empty((clips, N_MELS, frames), device=dev)

    def step():
        sb.Resample.apply(cfg, x, out=mid)
        sb.mel_spectrogram(sc, mc, mid, out=y)
    ms = timed_ms(step, 5, 1, barrier, dev)
    parity = None
    if with_parity:
        from oracle import mel_oracle, stft_oracle
        from oracle import resample_oracle as R
        st = [dict(l=t["l"], m=t["m"], k=t["k"], proto=R.design_prototype(t["l"], t["k"], t["fc"], t["beta"]))
              for t in cfg.stages()]
        want_mid = R.apply_plan(x[:2].cpu().numpy(), st, cfg.l, cfg.m).astype(np.float32)
        want = mel_oracle.mel_spectrogram(stft_oracle.StftConfig(FFT, HOP),
                                          mel_oracle.MelConfig(N_MELS, SR, FFT), want_mid)
        got = y[:2].cpu().numpy()
        parity = {"max_rel_err": max(peak_err(got[b], want[b]) for b in range(2)), "tolerance": 1e-4,
                  "sample": "clips 0-1 at full length: oracle resampler (float64, rounded to float32 "
                            "like Resample.apply's result) -> oracle STFT + mel"}
    out["resample_stft_mel"] = entry(
        f"{cfg.pp()} -> mel_spectrogram 128 bands, {clips} clips x 10 s @44.1 kHz per GPU "
        "(BASELINE.json configs[4]: 65536 clips over 8 GPUs); the 22.05 kHz intermediate "
        f"({mid.numel() * 4 / 1e9:.1f} GB) crosses HBM once each way and is not counted",
        ms, clips * (n * 4 + N_MELS * frames * 4), clips * 10.0, launches_of(step), parity)
    del x, mid, y
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--path", default="auto", choices=["auto", "fast", "tensor", "pair"],
                    help="which fused fft-2048 kernel: auto (the library's choice: the frame-pair "
                         "kernel), the frame-pair kernel (pair), the one-frame-per-warp register FFT "
                         "(fast) or the tcgen05 one (tensor)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's mel spectrograms to "
                         f"DIR/mel_spectrogram.npy (a fixed, seeded sample of {DUMP_CLIPS} clips; "
                         "with --impl reference, that arm's 64 clips)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import soundml_b200 as sb
    from soundml_b200 import synth

    sc = sb.Stft.Config.create(fft_size=FFT, hop=HOP).set_path(args.path)
    mc = sb.Mel.Config.create(n_mels=N_MELS, sample_rate=SR, fft_size=FFT)
    # rank r owns clips [r*BATCH, (r+1)*BATCH) of the global batch: independent
    # units, no exchange (the same split tests/test_parallel_gloo.py checks)
    from soundml_b200.parallel import max_over_ranks, my_shard
    lo, hi = my_shard(world * BATCH, rank, world)
    assert hi - lo == BATCH
    x = synth.clips_torch(BATCH, N, dev, SR, first_clip=lo)
    out = torch.empty((BATCH, N_MELS, FRAMES), dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        sb.mel_spectrogram(sc, mc, x, out=out)
    barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = sb.kernel_launch_count()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    start.record()
    for _ in range(args.steps):
        sb.mel_spectrogram(sc, mc, x, out=out)
    end.record()
    barrier()
    t_wall1 = time.time()
    launches = sb.kernel_launch_count() - launches0
    ms = max_over_ranks(start.elapsed_time(end), device=dev)   # the slowest rank defines the step
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    ms_per_step = ms / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dump_sample(out))
    value = world * BATCH * CLIP_SECONDS / (ms_per_step * 1e-3)

    # ---- end to end: pinned host buffers through the same public call
    e2e = None
    if not args.no_e2e:
        xh = torch.empty((BATCH, N), dtype=torch.float32).pin_memory()
        xh.copy_(x)
        oh = torch.empty((BATCH, N_MELS, FRAMES), dtype=torch.float32).pin_memory()
        xh_np, oh_np = xh.numpy(), oh.numpy()
        e2e_steps = max(3, min(args.steps, 10))
        for _ in range(2):
            sb.mel_spectrogram(sc, mc, xh_np, out=oh_np)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            sb.mel_spectrogram(sc, mc, xh_np, out=oh_np)     # returns after D2H lands
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0, device=dev)
        e2e = {"value": world * BATCH * CLIP_SECONDS * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": BATCH * N * 4, "d2h_bytes_per_step": BATCH * N_MELS * FRAMES * 4,
               "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps}
        assert torch.equal(oh.to(dev), out), "host and device paths disagree"
        # the floor of that call: the same pinned buffers through cudaMemcpyAsync alone,
        # both directions at once on two streams (what the e2e number is bound by)
        d_in, d_out = torch.empty_like(x), torch.empty_like(out)
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            with torch.cuda.stream(s_in):
                d_in.copy_(xh, non_blocking=True)
            with torch.cuda.stream(s_out):
                oh.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize()
        e2e["copy_floor_ms"] = 1e3 * max_over_ranks(time.perf_counter() - t0, device=dev) / e2e_steps
        del d_in, d_out, xh, oh

    # ---- the compute floor of the kernel: the transform skeleton alone (tile staging,
    # window, both register-FFT passes, the transposition), same launch shape
    floor_ms = None
    if args.path in ("auto", "pair"):
        from soundml_b200 import _lib
        nbytes = _lib.lib.smb_stft_fft_ceiling_scratch_bytes(sc._h, BATCH, N)
        scratch = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
        _lib.check(_lib.lib.smb_stft_plan_set_stream(sc._h, torch.cuda.current_stream(dev).cuda_stream))
        floor_ms = timed_ms(lambda: _lib.check(_lib.lib.smb_stft_fft_ceiling(
            sc._h, x.data_ptr(), BATCH, N, scratch.data_ptr())), 20, 3, barrier, dev)
        del scratch

    peak, peak_kind = peak_hbm()
    parity_clips = 32
    got_sample = out[:parity_clips].cpu().numpy() if (rank == 0 and world == 1) else None
    del x, out
    torch.cuda.empty_cache()
    secondary = None
    if not args.no_secondary:
        secondary = secondary_configs(sb, dev, world, rank, barrier, peak, with_parity=(world == 1))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    achieved = ALGO_BYTES / (ms_per_step * 1e-3) / 1e9
    # DRAM bytes of one launch from the committed ncu capture of this kernel (not measured
    # in this run: ncu replays kernels; profiles/traffic.json names the capture)
    kernel = {"tensor": "stft2048tc_kernel<mel>", "fast": "stft2048_kernel<mel>"}.get(
        args.path, "stft2048p_kernel<mel>")
    traffic = traffic_source = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        rec = prof.get(kernel)
        if rec:
            traffic, traffic_source = rec["dram_bytes_per_launch"], rec["capture"]
    except Exception:
        pass
    cpu = parity = None
    if world == 1:                      # reported on rank 0 at N = 1 only
        cores = os.cpu_count() or 1
        clips = parity_clips
        kept = []
        v, passes, dt = time_cpu(clips, args.cpu_seconds, cores, keep=kept)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{clips} of {BATCH} clips x {passes} passes ({dt:.1f} s), oracle "
                         "(numpy/scipy float64 restatement of stft.ml + mel.ml), clips dealt to "
                         "one thread per core"}
        # the error metric that goes with the number (SURVEY.md 8d): per clip
        # max |got - ref| / max |ref| against the oracle's output for the same
        # clips, and the elementwise pass rate at the reference's float32 gate
        import numpy as np
        want = np.asarray(kept[0], dtype=np.float64)
        got = got_sample.astype(np.float64)
        per_clip = (np.abs(got - want).max(axis=(1, 2)) / np.abs(want).max(axis=(1, 2)))
        gate = np.abs(got - want) <= 1e-7 + 1e-6 * np.abs(want)
        parity = {"max_rel_err_per_clip": float(per_clip.max()), "tolerance": 1e-4,
                  "f32_gate_pass_rate": float(gate.mean()),
                  "sample": f"first {clips} clips against the oracle"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
                     "peak_source": peak_kind, "algorithmic_bytes_per_launch": ALGO_BYTES,
                     "kernel": kernel, "kernel_ms": ms_per_step, "compute_floor_ms": floor_ms,
                     "hbm_floor_ms": 1e3 * ALGO_BYTES / (peak * 1e9)},
        "cpu_baseline": cpu,
        "parity": parity,
        "e2e": e2e,
        "secondary": secondary,
        "gpu_launches": launches,
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

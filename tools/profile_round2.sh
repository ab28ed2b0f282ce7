# Round-2 evidence run (one GPU): bench lines, launch list, one full ncu capture of the
# headline kernel, the secondary benches.  Everything lands in gpurun_out/r2_*.
set -x
O=gpurun_out
timeout 300 python bench.py > $O/r2_bench_line.json 2> $O/r2_bench_err.log
timeout 200 python bench.py --impl reference --steps 5 --warmup 2 > $O/r2_bench_line_reference.json 2>> $O/r2_bench_err.log
timeout 120 python bench.py --path fast --no-e2e --no-secondary --cpu-seconds 1 --steps 100 > $O/r2_bench_line_fast.json 2>> $O/r2_bench_err.log
timeout 120 python bench.py --path tensor --no-e2e --no-secondary --cpu-seconds 1 --steps 100 > $O/r2_bench_line_tensor.json 2>> $O/r2_bench_err.log
# launch list of the bench command (cold-cache, serialised: shares only)
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:'stft2048|to_db|mfcc|resample|ols|fir' -c 60 --csv --log-file $O/r2_launches_bench.csv python bench.py --steps 10 --warmup 3 --no-e2e --no-secondary --cpu-seconds 0.3 > $O/r2_launches.log 2>&1
# full capture of the headline kernel
timeout 200 ncu --set full --clock-control none --import-source on -k regex:stft2048p -s 3 -c 1 -o $O/r2_pair python bench.py --steps 3 --warmup 3 --no-e2e --no-secondary --cpu-seconds 0.3 > $O/r2_ncu.log 2>&1
timeout 400 python bench_extra.py > $O/r2_bench_extra.jsonl 2>> $O/r2_bench_err.log
timeout 300 python tools/bench_resample_pairs.py > $O/r2_resample_pairs.jsonl 2>> $O/r2_bench_err.log
timeout 300 python tools/bench_direct.py > $O/r2_direct_kernel.jsonl 2>> $O/r2_bench_err.log
timeout 200 python tools/bench_host_paths.py > $O/r2_host_paths.jsonl 2>> $O/r2_bench_err.log
timeout 200 python tools/bench_gemm_forms.py > $O/r2_gemm_forms.jsonl 2>> $O/r2_bench_err.log
timeout 200 python tools/measure_thdn.py > $O/r2_thdn.txt 2>> $O/r2_bench_err.log
timeout 200 python tools/bench_mel_gemm.py > $O/r2_mel_gemm.json 2>> $O/r2_bench_err.log
tail -c 400 $O/r2_bench_err.log
cut -c1-300 $O/r2_bench_line.json

set -x
# headline bench line (default path) and the tensor-core path beside it
timeout 300 python bench.py > gpurun_out/bench_line.json 2> gpurun_out/bench_err.log
timeout 300 python bench.py --path tensor --no-e2e --cpu-seconds 2 > gpurun_out/bench_line_tensor.json 2> gpurun_out/bench_tensor_err.log
# launch lists (cold-cache, serialised: shares only)
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:stft2048 -c 20 --csv --log-file gpurun_out/launches.csv python bench.py --steps 10 --warmup 3 --no-e2e --cpu-seconds 0.5 > gpurun_out/launches.log 2>&1
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:stft2048 -c 20 --csv --log-file gpurun_out/launches_tensor.csv python bench.py --path tensor --steps 10 --warmup 3 --no-e2e --cpu-seconds 0.5 > gpurun_out/launches_tensor.log 2>&1
# full captures of both fused kernels
timeout 400 ncu --set full --clock-control none --import-source on -k regex:stft2048_kernel -s 3 -c 1 -o gpurun_out/r1k python bench.py --steps 3 --warmup 3 --no-e2e --cpu-seconds 0.5 > gpurun_out/r1k.log 2>&1
timeout 400 ncu --set full --clock-control none --import-source on -k regex:stft2048tc -s 3 -c 1 -o gpurun_out/tc_e python bench.py --path tensor --steps 3 --warmup 3 --no-e2e --cpu-seconds 0.5 > gpurun_out/tc_e.log 2>&1
timeout 600 python bench_extra.py > gpurun_out/bench_extra.jsonl 2> gpurun_out/bench_extra_err.log
timeout 200 python bench.py --impl reference --steps 2 --warmup 1 > gpurun_out/bench_line_reference.json 2>> gpurun_out/bench_err.log
# the bin-major outputs (Stft.transform / power_spectrum): full capture of the complex kernel
timeout 300 ncu --set full --clock-control none --import-source on -k regex:stft2048_kernel -s 6 -c 1 -o gpurun_out/cplx_c python bench_extra.py --only spectrum --steps 2 > gpurun_out/cplx_c.log 2>&1
# library yardstick (cuFFT + cuBLAS) beside the fused kernel
timeout 200 python tools/bench_library_stft.py > gpurun_out/library_stft.json 2> gpurun_out/library_stft_err.log
tail -1 gpurun_out/bench_line.json | cut -c1-200

# round 2, 1 GPU: full GPU suite, the MEASURED reference arm (full 256^3 if it fits),
# our arm, ncu launch list
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
lscpu | grep -E "^CPU\(s\)|Model name|Thread|Core|Socket" > gpurun_out/r02_lscpu.txt; free -g >> gpurun_out/r02_lscpu.txt
timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 --reps 30 2>&1 | tail -12 | tee gpurun_out/r02_probe_s3_256_v8.log
timeout -k 10 1500 python -m pytest tests -q -x -m gpu 2>&1 | tail -8 | tee gpurun_out/r02_pytest_gpu_v8.log
PS_REF_BUDGET_S=900 timeout -k 10 1500 python bench.py --impl reference 2> gpurun_out/r02_bench_ref_err_v8.log | tee gpurun_out/r02_bench_ref_n1_v8.json
tail -3 gpurun_out/r02_bench_ref_err_v8.log
timeout -k 10 900 python bench.py 2> gpurun_out/r02_bench_err_v8.log | tee gpurun_out/r02_bench_n1_v8.json
tail -3 gpurun_out/r02_bench_err_v8.log
timeout -k 10 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv --log-file gpurun_out/r02_launches_step_v8.csv python tools/probe.py --scene S3 --n 256 --steps 1 --reps 1 > gpurun_out/r02_ncu_launch_v8.log 2>&1
tail -2 gpurun_out/r02_ncu_launch_v8.log

# single-GPU round check after the PDL / one-CTA-per-region / scan changes: all GPU tests, smoke, probe, bench (both arms), ncu launch list
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv
timeout -k 10 1500 python -m pytest tests -q -m gpu --durations=10 2>&1 | tail -40 | tee gpurun_out/pytest_gpu.log
timeout -k 10 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee gpurun_out/smoke.log
timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | tail -12 | tee gpurun_out/probe_s3_256.log
timeout -k 10 900 python bench.py 2> gpurun_out/bench_err.log | tee gpurun_out/bench_n1.json
tail -3 gpurun_out/bench_err.log
timeout -k 10 600 python bench.py --impl reference --steps 1 --warmup 0 2> gpurun_out/bench_ref_err.log | tee gpurun_out/bench_ref_n1.json
timeout -k 10 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 3000 --csv --log-file gpurun_out/launches_step.csv \
    python tools/probe.py --scene S3 --n 256 --steps 1 --reps 1 > gpurun_out/ncu_launch.log 2>&1
tail -3 gpurun_out/ncu_launch.log

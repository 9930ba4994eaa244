# round 2, 2 GPUs: direct halo pushes (short push launch + wait at the consumer's head); multi handle with diagnostics
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
timeout -k 10 300 python -m pytest tests/test_gpu_distributed.py -q -x -m gpu 2>&1 | tail -15 | tee gpurun_out/r02_pytest_gpu_dist_n2_v10.log
PS_MULTI_WATCHDOG_S=45 timeout -k 10 200 python tests/multi_worker.py blob64_tile16_pad2 2 2>&1 | tail -5 | tee gpurun_out/r02_multi_worker_v10.log
timeout -k 10 400 python -m pytest tests/test_gpu_multi.py tests/test_zz_adaptor.py -q -x -m gpu 2>&1 | tail -25 | tee gpurun_out/r02_pytest_gpu_multi_n2_v10.log
timeout -k 10 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 2 --steps 10 --warmup 3 --no-cpu-baseline 2> gpurun_out/r02_bench_err_n2_v10.log | tee gpurun_out/r02_bench_n2_v10.json
tail -3 gpurun_out/r02_bench_err_n2_v10.log
PS_TRACE=100 timeout -k 10 200 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus 2 --steps 2 --warmup 1 --no-cpu-baseline 2>&1 | grep "ps trace" | tail -4 | tee gpurun_out/r02_trace_n2_v10.log

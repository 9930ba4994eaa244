# 4-GPU check: the world_size-4 distributed parity tests (both transports), bench.py at 4 ranks, per-iteration breakdown
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name,clocks.sm,clocks.max.sm --format=csv
timeout -k 10 600 python -m pytest tests/test_gpu_distributed.py -x -q -m gpu -k "tile16-4" 2>&1 | tail -6 | tee gpurun_out/pytest_gpu_dist_n4.log
PS_TRACE=60 timeout -k 10 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 4 --master-addr 127.0.0.1 --master-port 29504 \
    bench.py --gpus 4 --steps 5 --warmup 3 2> gpurun_out/bench_err_n4.log | tee gpurun_out/bench_n4.json
grep "ps trace rank 0" gpurun_out/bench_err_n4.log | tail -1
tail -3 gpurun_out/bench_err_n4.log
N=4
run() { timeout -k 10 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29530 + RANDOM % 100)) tools/dist_probe.py --tag "$1" 2>&1 | grep "dist_probe" | tee -a gpurun_out/dist_probe_n$N.log; }
run full
PS_COMM=nccl run nccl

# round 2, 2 GPUs: single-GPU probe (vectorised update), distributed parity (slab-local + replicated, peer + nccl),
# the ps_create_multi handle, bench at N = 2 (process per GPU) and through the multi handle
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv
CUDA_VISIBLE_DEVICES=0 timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | tail -12 | tee gpurun_out/r02_probe_s3_256_v5.log
timeout -k 10 1500 python -m pytest tests/test_gpu_distributed.py tests/test_gpu_multi.py -q -x -m gpu 2>&1 | tail -12 | tee gpurun_out/r02_pytest_gpu_dist_n2_v5.log
timeout -k 10 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 2 --steps 10 --warmup 3 2> gpurun_out/r02_bench_err_n2_v5.log | tee gpurun_out/r02_bench_n2_v5.json
tail -3 gpurun_out/r02_bench_err_n2_v5.log
timeout -k 10 900 python bench.py --gpus 2 --multi --steps 10 --warmup 3 2> gpurun_out/r02_bench_err_multi2_v5.log | tee gpurun_out/r02_bench_multi2_v5.json
tail -3 gpurun_out/r02_bench_err_multi2_v5.log
PS_TRACE=100 timeout -k 10 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus 2 --steps 2 --warmup 1 --no-cpu-baseline 2>&1 | grep "ps trace" | tee gpurun_out/r02_trace_n2_v5.log

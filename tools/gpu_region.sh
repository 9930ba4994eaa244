set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
for i in 1 2 3 4 5; do timeout -k 10 600 python -m pytest tests/test_gpu_parity.py -x -q -m gpu -k bicgstab 2>&1 | grep -E "^E  |passed|failed" | head -12; done | tee gpurun_out/pytest_bicg_loop.log
timeout -k 10 1500 python -m pytest tests/test_gpu_parity.py tests/test_golden.py tests/test_gpu_fullsize.py -q -m gpu --durations=5 2>&1 | tail -25 | tee gpurun_out/pytest_gpu_quick.log
echo "== chunked kernels (PS_REGION_FUSE_MAX=0)" | tee -a gpurun_out/sweep_region.log
PS_REGION_FUSE_MAX=0 timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | grep -E "^step 1|^reduced|^cg_iteration|^apply" | tee -a gpurun_out/sweep_region.log

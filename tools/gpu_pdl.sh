set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
timeout -k 10 1500 python -m pytest tests/test_gpu_parity.py tests/test_golden.py tests/test_gpu_fullsize.py -q -m gpu --durations=8 2>&1 | tail -30 | tee gpurun_out/pytest_gpu_quick.log
timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | tail -9 | tee gpurun_out/probe_s3_256.log

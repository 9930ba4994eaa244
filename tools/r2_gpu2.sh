# round 2: pass 1 with paired items + prefetching epilogue, parity subset
set -x
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
timeout -k 10 900 python -m pytest tests/test_gpu_parity.py tests/test_gpu_fullsize.py -q -x -m gpu 2>&1 | tail -5 | tee gpurun_out/r02_pytest_gpu_v2.log
timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | tail -12 | tee gpurun_out/r02_probe_s3_256_v2.log
PS_PASS1_STATIC=1 timeout -k 10 600 python tools/probe.py --scene S3 --n 256 --steps 2 2>&1 | tail -9 | tee gpurun_out/r02_probe_s3_256_v2_static.log

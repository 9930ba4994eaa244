# where does the multi-GPU CG iteration spend its time?  cg_iteration with the peer transport and with NCCL (usage: bash tools/gpu_distprobe.sh N)
N=${1:-2}
cd $GRAFT_REPO_ROOT
mkdir -p gpurun_out
run() { timeout -k 10 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29530 + RANDOM % 100)) tools/dist_probe.py --tag "$1" 2>&1 | grep "dist_probe" | tee -a gpurun_out/dist_probe_n$N.log; }
run full
PS_COMM=nccl run nccl

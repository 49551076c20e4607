#!/bin/bash
# gpurun --gpus N -- bash scripts/gpu_multi_ab.sh N [TAG] : multi-GPU parity tests, then the N-GPU bench on the production path
# (pipelined: statistics + table beside the next sweep) and, for comparison, in order (VRG_PIPELINE=0: fused tail kernel) and
# on the separate kernels (VRG_NO_FUSED_TAIL=1: cancel, halo exchange, statistics exchange and table in program order)
N=${1:-2}
TAG=${2:-r2}
set -x
mkdir -p gpurun_out
nvidia-smi -L | head -8
timeout 900 python -m pytest tests/test_gpu_multi.py -m gpu -x -q 2>&1 | tail -15 > gpurun_out/${TAG}_pytest_multi_$N.txt
cat gpurun_out/${TAG}_pytest_multi_$N.txt
run() {  # port, name, env
  env $3 timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $1 \
      bench.py --gpus $N --steps 3 --warmup 3 --quick --no-parity > gpurun_out/${TAG}_scale_${N}_$2.json 2> gpurun_out/${TAG}_scale_${N}_$2.err
  tail -c 1500 gpurun_out/${TAG}_scale_${N}_$2.json; tail -n 3 gpurun_out/${TAG}_scale_${N}_$2.err
}
run 29511 pipelined VRG_X=1
run 29512 inorder VRG_PIPELINE=0
run 29513 separate VRG_NO_FUSED_TAIL=1

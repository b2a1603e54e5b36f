#!/bin/bash
# training step (fwd + losses + CUDA backward + flat-bucket NCCL all-reduce + Adam) on N GPUs; run under `gpurun --gpus N`
N=${1:-2}
TAG=${2:-r2}
mkdir -p gpurun_out
export SNB200_GENERATOR_BACKWARD=${SNB200_GENERATOR_BACKWARD:-cuda}
timeout -k 10 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 tools/bench_configs.py --only train \
  > gpurun_out/${TAG}_train_n${N}.jsonl 2> gpurun_out/${TAG}_train_n${N}.err; echo "train n=$N rc=$?"
cat gpurun_out/${TAG}_train_n${N}.jsonl; tail -5 gpurun_out/${TAG}_train_n${N}.err
timeout -k 10 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29534 bench.py --gpus $N --steps 200 --warmup 20 \
  > gpurun_out/${TAG}_bench_n${N}.json 2> gpurun_out/${TAG}_bench_n${N}.err; echo "bench n=$N rc=$?"; cat gpurun_out/${TAG}_bench_n${N}.json

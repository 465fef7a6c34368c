#!/bin/bash
N=${1:-2}
mkdir -p gpurun_out
timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29533 tools/peer_sync_probe.py 2>&1 | grep -v -E "OMP_NUM|\*\*\*\*|NCCL version|^$" | tail -9
python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --sustained-seconds 0 2>/dev/null | cut -c1-200
for SYNC in peer; do
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus $N --steps 20 --warmup 5 --sustained-seconds 0 --sync $SYNC > gpurun_out/bench_n${N}_$SYNC.json 2> gpurun_out/bench_n${N}_$SYNC.err; echo "n$N $SYNC rc=$?"; cut -c1-200 gpurun_out/bench_n${N}_$SYNC.json
done

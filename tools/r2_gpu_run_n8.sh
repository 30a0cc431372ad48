#!/bin/bash
# Round-2 multi-GPU evidence run (8 x B200): where the host-buffer step goes at 8 ranks, the
# driver's own bench line at N = 8 (weak scaling + N-rank parity + config 5 strong scaling), the
# 2-rank GPU tests.
set -u
cd "$(dirname "$0")/.."
O=gpurun_out
N=${1:-8}
mkdir -p $O
run() { python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $((29500 + RANDOM % 400)) "$@"; }
nvidia-smi topo -m > $O/r2_topo_n$N.txt 2>&1
(lscpu | head -25; free -g) >> $O/r2_topo_n$N.txt 2>&1
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29611 tools/sharded_e2e_breakdown.py > $O/r2_e2e_breakdown_n$N.log 2>&1
echo "breakdown rc=$?"; grep -E "rank 0 rep 3|ShardedRelaxation rep 2|host link" $O/r2_e2e_breakdown_n$N.log | cut -c1-600
timeout 1200 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29612 bench.py --gpus $N --steps 10 --warmup 3 > $O/r2_bench_n$N.json 2> $O/r2_bench_n$N.err
echo "bench rc=$?"; tail -c 1500 $O/r2_bench_n$N.json
timeout 600 python -m pytest tests -m gpu -x -q -k "distributed or rank" > $O/r2_gputests_n$N.log 2>&1
echo "pytest rc=$?"; tail -3 $O/r2_gputests_n$N.log

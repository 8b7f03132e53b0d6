#!/bin/bash
# N-GPU diagnostic of the camera-block exchange: back-to-back latency (p2p vs NCCL), then the weak-scaling step with the
# peer-memory kernel and with NCCL.
N=${1:-8}
python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29640 tools/p2p_latency.py 2>&1 | tail -1
timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29600 bench.py --gpus $N --steps 100 --warmup 10 --no-lm --no-cpu --no-config5 2>/dev/null | tail -1 | python -c "
import sys,json
d=json.loads(sys.stdin.read()); print('p2p', round(d['value']), round(d['ms_per_step'],4), 'kernel', round(d['roofline']['kernel_ms'],4), d['config_detail']['exchange_check'])"
timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29603 bench.py --gpus $N --steps 100 --warmup 10 --no-lm --no-cpu --no-config5 --exchange nccl 2>/dev/null | tail -1 | python -c "
import sys,json
d=json.loads(sys.stdin.read()); print('nccl', round(d['value']), round(d['ms_per_step'],4), 'kernel', round(d['roofline']['kernel_ms'],4))"

#!/bin/bash
# 8-GPU visit: scaling variants of the data-parallel step (run with gpurun --gpus 8)
mkdir -p gpurun_out
TR="python -m torch.distributed.run --nnodes=1 --master-addr 127.0.0.1"
run() { local name=$1; shift; timeout -s KILL 300 "$@" > gpurun_out/$name.log 2>&1; echo "== $name rc=$? $(grep -o '"ms_per_step": [0-9.]*' gpurun_out/$name.log | head -1) $(grep -o '"value": [0-9.]*' gpurun_out/$name.log | head -1)" | tee -a gpurun_out/scale8_summary.txt; }
: > gpurun_out/scale8_summary.txt
B="bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-roofline"
run n1 python $B --gpus 1
run n8_default $TR --nproc-per-node 8 --master-port 29701 $B --gpus 8
run n8_ctas4 $TR --nproc-per-node 8 --master-port 29702 $B --gpus 8 --nccl-max-ctas 4
run n8_ctas8 $TR --nproc-per-node 8 --master-port 29703 $B --gpus 8 --nccl-max-ctas 8
run n8_bucket3 $TR --nproc-per-node 8 --master-port 29706 $B --gpus 8 --bucket-layers 3
python scripts/ddp_timeline.py gpurun_out/tl_n1.json > gpurun_out/tl_n1.log 2>&1
$TR --nproc-per-node 8 --master-port 29707 scripts/ddp_timeline.py gpurun_out/tl_n8.json > gpurun_out/tl_n8.log 2>&1
$TR --nproc-per-node 8 --master-port 29708 scripts/ddp_timeline.py gpurun_out/tl_n8_ctas4.json --nccl-max-ctas 4 > gpurun_out/tl_n8c4.log 2>&1
cat gpurun_out/scale8_summary.txt

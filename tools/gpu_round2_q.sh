#!/bin/bash
# GPU call Q: MMA cost with uniform issue (cta_group::1 / ::2), two-heads-per-CTA tensor-core attention: parity + A/B
set -u
mkdir -p gpurun_out
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/microbench/mma_floor2 tools/microbench/mma_floor2.cu
./tools/microbench/mma_floor2 2>&1 | tee gpurun_out/r2q_mma_floor2.log
timeout 600 python -m pytest tests/test_gpu_parity.py -q -m gpu -k "attention" --timeout 300 -p no:randomly 2>&1 | tail -5
for pm in 1000 16; do
  MEGATTS2_ATTN_PAIR_MIN=$pm BENCH_S=16,24,32,48,64 timeout 300 python tools/bench_attention.py 2>&1 | tee -a gpurun_out/r2q_attention_pair_ab.log
done
for pm in 1000 24 16; do
  echo "== PAIR_MIN=$pm"
  MEGATTS2_ATTN_PAIR_MIN=$pm timeout 600 python tools/time_stages.py --reps 2 2>&1 | grep -A13 "pass 1" | grep -E "mrte|adm|plm|full" | tee -a gpurun_out/r2q_stages_pair.log
done

#!/bin/bash
# env-steps/s of the device-resident loop versus batch size (one B200): where the fused launch, the slicing of small
# batches and the bandwidth-bound regime meet.
for n in ${SIZES:-16 64 148 149 256 512 1024 2048 4096 16384 65536}; do
  echo -n "envs=$n : "; python bench.py --envs-per-gpu $n --steps 4000 --warmup 50 --quick ${EXTRA:-} 2>/dev/null | tail -1 | cut -c1-150
done

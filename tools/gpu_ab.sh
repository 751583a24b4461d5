#!/bin/bash
# A/B of builds of the library (TRS_B200_LIB override): headline, 240x320 mask and full chain, device-resident, the builds alternating within
# each round (ROUNDS, default two).  usage: [ROUNDS=n] tools/gpu_ab.sh <libA.so> <libB.so> ...
mkdir -p gpurun_out
for rep in $(seq ${ROUNDS:-2}); do
for v in "$@"; do
  export TRS_B200_LIB=$PWD/triton-racer-sim_b200/$v
  timeout 120 python bench.py --quick --steps 20 --warmup 3 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read()); print('$v headline', round(d['value']), round(d['roofline']['frac'],4))"
  timeout 120 python bench.py --quick --workload full_house_mask_240x320 --frames 16384 --steps 10 --warmup 3 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read()); print('$v mask240', round(d['value']))"
  timeout 120 python bench.py --quick --workload full_chain_240x320 --frames 16384 --steps 10 --warmup 3 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read()); print('$v chain240', round(d['value']))"
done
done

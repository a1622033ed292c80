#!/bin/bash
# Sensitivity map of the fused GRU-layer kernel on one box: tools/ab_exp.sh <variant.so> ...
# (variants are built beforehand, in a copy of the tree with profiles/r2_k4g_sensitivity.patch applied, with
#  CF_EXTRA_DEFS=-DCF_EXP=<bits> CF_LIB_OUT=... python -m catfish_b200.build --force;
#  their results are wrong by design, only the timing is of interest)
show() { python -c "import sys,json; d=json.loads(sys.stdin.read()); k=d['kernels']; print(round(d['value']/1e6,1), round(d['ms_per_step'],2), 'k2', round(k['k2_conv_stack']['ms']/d['steps'],2), 'k4', round(k['k4_gru_recurrence']['ms']/d['steps'],2), d['clocks']['sm_mhz'], d['clocks']['power_w_max'], d['clocks']['reasons'])"; }
echo "default"; timeout 300 python bench.py --steps 5 --warmup 3 --no-cpu-baseline --legs main 2>&1 | tail -1 | show
for v in "$@"; do
  echo "variant $v"; CF_LIB_PATH=$v timeout 300 python bench.py --steps 5 --warmup 3 --no-cpu-baseline --legs main 2>&1 | tail -1 | show
done
echo "default"; timeout 300 python bench.py --steps 5 --warmup 3 --no-cpu-baseline --legs main 2>&1 | tail -1 | show

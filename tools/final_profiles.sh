#!/bin/bash
# Round-end measurements on one B200 box (run under gpurun from the repo root); everything lands in gpurun_out/.
set -u
O=gpurun_out
mkdir -p $O
timeout 600 python bench.py --steps 50 --warmup 5 --kernel-pass-json $O/kernel_pass_tf32.json > $O/r2_final_bench.json 2> $O/r2_final_bench.err
timeout 300 python bench.py --mode tf32x3 --steps 30 --warmup 5 --no-cpu-baseline > $O/r2_tf32x3_bench.json 2>/dev/null
timeout 300 python bench.py --mode bf16 --steps 30 --warmup 5 --no-cpu-baseline > $O/r2_bf16_bench.json 2>/dev/null
timeout 300 python bench.py --impl reference --steps 3 --warmup 1 > $O/r2_reference_arm.json 2>/dev/null
# launch list of the same command (cold-cache, serialised: shares)
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 800 --csv --log-file $O/r2_launches.csv \
  python bench.py --steps 2 --warmup 1 --no-cpu-baseline --no-kernel-pass --no-fp32-side > $O/r2_launches.log 2>&1
# one --set full capture of the top kernels (third launch of each: after the warm-up ones)
cap() {  # name kernel-regex args...
  local name=$1 rx=$2; shift 2
  timeout 300 ncu --set full --clock-control none --import-source on -k regex:$rx --launch-skip 2 --launch-count 1 -f -o $O/$name \
    python tools/run_conv_layer.py "$@" --reps 4 > $O/$name.log 2>&1
}
cap r2f_wgrad_L2_96x48 k_wgrad_tc --kind smc --level 2 --cin 96 --cout 48 --dir wgrad
cap r2f_wgrad_L1_64x32 k_wgrad_tc --kind smc --level 1 --cin 64 --cout 32 --dir wgrad
cap r2f_wgrad_rings_L0_32x16 k_wgrad_tc_rings --kind smc --level 0 --cin 32 --cout 16 --dir wgrad
cap r2f_conv_tc_L0_16x16 k_conv_tc --kind smc --level 0 --cin 16 --cout 16 --dir fwd
cap r2f_conv_tc_L2_96x48 k_conv_tc --kind smc --level 2 --cin 96 --cout 48 --dir fwd
ls -la $O/*.ncu-rep

#!/bin/bash
# ncu evidence (1 GPU; never a multi-rank command -- ncu replays each kernel ~40 times).  Nothing printed by a run under
# ncu is a bench value.  Outputs in gpurun_out/; summarise the .ncu-rep files HERE afterwards with tools/ncu_summary.py
# and copy the summaries into profiles/.
#   /usr/local/graft/bin/gpurun --timeout 1200 -- 'bash tools/gpu_prof.sh [steps...]'
# steps (default: launches traffic gemm decode quant layer)
set -u
mkdir -p gpurun_out
OUT=gpurun_out
STEPS=${*:-launches traffic gemm decode quant layer}
FULL="--set full --clock-control none --import-source on"
for s in $STEPS; do case $s in
  launches) # launch list of the bench command itself (shares of the step, not absolute times)
            timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv --log-file $OUT/bench_launches.csv \
                python bench.py --steps 2 --warmup 1 --no-cpu-baseline > /dev/null 2>&1; grep -c gemm_i4 $OUT/bench_launches.csv ;;
  traffic)  # DRAM bytes per launch of the GEMM at the bench shape and at prefill size -> profiles/ncu_summary.json
            for cfg in "16 0" "16 1" "64 0" "4096 2"; do set -- $cfg
              timeout 300 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -k regex:gemm_ -c 6 --csv \
                  --log-file $OUT/launch_m$1_f$2.csv python tools/prof_gemm.py $1 $2 > /dev/null 2>&1
              echo "== M=$1 flags=$2"; grep -E "gpu__time_duration|dram__bytes" $OUT/launch_m$1_f$2.csv | awk -F'","' '{print $(NF-2), $(NF-1), $NF}' | tail -6
            done ;;
  gemm)     timeout 300 ncu $FULL -k regex:gemm_ -s 3 -c 1 -f -o $OUT/prof_gemm_m16_split python tools/prof_gemm.py 16 0 > /dev/null 2>&1
            timeout 300 ncu $FULL -k regex:gemm_ -s 3 -c 1 -f -o $OUT/prof_gemm_m16_nosplit python tools/prof_gemm.py 16 1 > /dev/null 2>&1
            timeout 300 ncu $FULL -k regex:gemm_ -s 3 -c 1 -f -o $OUT/prof_gemm_m4096_tall python tools/prof_gemm.py 4096 2 > /dev/null 2>&1 ;;
  decode)   timeout 300 ncu $FULL -k regex:batch_decode -s 2 -c 1 -f -o $OUT/prof_decode python tools/layer_bench.py --copies 1 > /dev/null 2>&1 ;;
  quant)    timeout 300 ncu $FULL -k regex:rmsnorm -s 2 -c 1 -f -o $OUT/prof_rmsnorm python tools/layer_bench.py --copies 1 > /dev/null 2>&1 ;;
  layer)    # per-kernel times of one decode step of a Llama-7B layer
            timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:"gemm_i4|quant_kernel|decode_kernel|append_kv|reorder" --csv \
                --log-file $OUT/layer_launches.csv python tools/layer_bench.py --copies 2 > /dev/null 2>&1
            python - <<'PY'
import csv
rows = [r for r in csv.reader(open('gpurun_out/layer_launches.csv')) if len(r) > 10 and r[0].isdigit()]
last = rows[-9:]                                    # 9 launches per layer step (round 2: fused q/k/v, gate/up+act, add+norm)
tot = sum(float(r[-1]) for r in last)
for r in last:
    print(f"{float(r[-1]) / 1000:8.2f} us {100 * float(r[-1]) / tot:5.1f}%  {r[4].replace('atom::', '').split('(')[0][:60]}")
print("total us", tot / 1000, "launches captured", len(rows))
PY
            ;;
  *) echo "unknown step $s" ;;
esac; done
ls -la $OUT/*.ncu-rep 2>/dev/null

#!/bin/bash
# One GPU visit (1 GPU): everything a round needs, each step under its own timeout, everything into gpurun_out/.
#   /usr/local/graft/bin/gpurun --timeout 1500 -- 'bash tools/gpu_round.sh [steps...]'
# steps (default: tests smoke bench gtime trace layer harness micro; extra: sk = decode-GEMM development loop)
set -u
mkdir -p gpurun_out
OUT=gpurun_out
STEPS=${*:-tests smoke bench gtime trace layer harness micro}
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw,memory.total --format=csv > $OUT/smi.txt 2>&1
for s in $STEPS; do case $s in
  tests)   echo "== pytest -m gpu"; timeout 1500 python -m pytest tests -m gpu -q --timeout=300 -p no:cacheprovider > $OUT/pytest.txt 2>&1; echo "rc=$?"; tail -15 $OUT/pytest.txt ;;
  smoke)   echo "== smoke"; timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 ;;
  bench)   echo "== bench ours"; timeout 600 python bench.py 2> $OUT/bench.err | tee $OUT/bench_ours.json; tail -3 $OUT/bench.err
           echo "== bench reference"; timeout 600 python bench.py --impl reference 2> $OUT/bench_ref.err | tee $OUT/bench_ref.json; tail -3 $OUT/bench_ref.err ;;
  gtime)   echo "== GEMM graph timing"; timeout 600 python tools/gpu_check.py gtime 2> $OUT/gtime.err | tee $OUT/gtime.jsonl; tail -3 $OUT/gtime.err
           echo "== decode-shape table"; timeout 600 python tools/gpu_check.py gshape 2>> $OUT/gtime.err | tee $OUT/gshape.jsonl ;;
  trace)   echo "== pipeline trace"; : > $OUT/trace.jsonl
           for cfg in "16 0" "16 1" "4096 2"; do timeout 120 python tools/gpu_check.py trace $cfg 2>&1 | tail -1 | tee -a $OUT/trace.jsonl | cut -c1-2500; done ;;
  layer)   echo "== decoder-layer decode step"
           timeout 300 python tools/layer_bench.py 2>&1 | tail -1 | tee $OUT/layer_7b.json
           timeout 300 python tools/layer_bench.py --hidden 5120 --inter 13824 --heads 40 --batch 32 --kvlen 1024 --layers 40 2>&1 | tail -1 | tee $OUT/layer_13b.json ;;
  harness) echo "== continuous-batching harness (warm: one untimed batch first; cold: like the reference's script)"
           timeout 900 python tools/bench_textgen.py --model 7b --batch-size 16 --num-batches 2 --maxlen 512 2> $OUT/textgen.err | tee $OUT/textgen_7b.txt | tail -2 | cut -c1-900; tail -3 $OUT/textgen.err
           timeout 900 python tools/bench_textgen.py --model 7b --batch-size 16 --num-batches 2 --maxlen 512 --warmup-batches 0 2>> $OUT/textgen.err | tee $OUT/textgen_7b_cold.txt | tail -2 | cut -c1-900 ;;
  micro)   echo "== microbenchmarks"; for b in microbench sync_bench tma_bench tmem_bench; do timeout 120 ./tools/$b > $OUT/$b.jsonl 2>&1; echo "$b rc=$?"; done ;;
  sk)      echo "== skinny GEMM: probes, parity, timing (PDL on / off)"
           timeout 300 python tools/gpu_check.py diag 2>&1 | tee $OUT/sk_diag.jsonl | cut -c1-400
           timeout 600 python -m pytest tests/test_gpu_parity.py tests/test_gpu_vs_reference.py -m gpu -q -x --timeout=300 -p no:cacheprovider -k "gemm or fused" > $OUT/pytest_sk.txt 2>&1; echo "rc=$?"; tail -12 $OUT/pytest_sk.txt
           timeout 300 python tools/gpu_check.py gtime 16 32 64 2> $OUT/sk_gtime.err | tee $OUT/sk_gtime.jsonl; tail -3 $OUT/sk_gtime.err
           ATOM_B200_GEMM_PDL=0 timeout 300 python tools/gpu_check.py gtime 16 2>> $OUT/sk_gtime.err | tee $OUT/sk_gtime_nopdl.jsonl
           timeout 300 python tools/gpu_check.py gshape 2>> $OUT/sk_gtime.err | tee $OUT/sk_gshape.jsonl
           timeout 300 python tools/gpu_check.py gtime 128 256 1024 4096 2>> $OUT/sk_gtime.err | tee $OUT/tall_gtime.jsonl
           : > $OUT/sk_trace.jsonl
           for cfg in "16 0" "16 1" "4096 2"; do timeout 120 python tools/gpu_check.py trace $cfg 2>&1 | tail -1 | tee -a $OUT/sk_trace.jsonl | cut -c1-2500; done
           for cfg in "16 0" "16 1"; do timeout 120 python tools/gpu_check.py tracew $cfg 2>&1 | tail -1 | tee -a $OUT/sk_trace.jsonl | cut -c1-2500; done ;;
  dec)     echo "== decode attention: parity at 5e-4, timing, ncu capture"
           timeout 600 python -m pytest tests/test_gpu_parity.py tests/test_gpu_vs_reference.py -m gpu -q --timeout=300 -p no:cacheprovider -k "decode or rmsnorm" > $OUT/pytest_dec.txt 2>&1; echo "rc=$?"; tail -15 $OUT/pytest_dec.txt
           timeout 300 python tools/layer_bench.py 2>&1 | tail -1 | tee $OUT/layer_7b.json
           ;;
  ncug)    echo "== ncu --set full: prefill GEMM (128x128) at M=4096, decode GEMM at M=16 (summarised here; the .ncu-rep files are too big to travel)"
           FULL="--set full --clock-control none --import-source on"
           timeout 300 ncu $FULL -k regex:gemm_i4_tall -s 3 -c 1 -f -o $OUT/prof_gemm_m4096_tall128 python tools/prof_gemm.py 4096 2 > /dev/null 2>&1
           timeout 300 ncu $FULL -k regex:gemm_i4_skinny -s 3 -c 1 -f -o $OUT/prof_gemm_m16_skinny python tools/prof_gemm.py 16 0 > /dev/null 2>&1
           timeout 300 ncu $FULL -k regex:batch_decode -s 2 -c 1 -f -o $OUT/prof_decode python tools/layer_bench.py --copies 1 > /dev/null 2>&1
           for f in prof_gemm_m4096_tall128 prof_gemm_m16_skinny prof_decode; do
             python tools/ncu_summary.py $OUT/$f.ncu-rep $OUT/ncu_$f > /dev/null 2>&1 && echo "summarised $f" && rm -f $OUT/$f.ncu-rep
           done ;;
  *) echo "unknown step $s" ;;
esac; done

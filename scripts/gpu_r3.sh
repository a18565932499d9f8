#!/bin/bash
# Round-3 GPU iteration: selectable stages, everything logged under gpurun_out/.
#   bash scripts/gpu_r3.sh <tag> <stage> [<stage> ...]
# stages: tests | testsx (stop at first failure) | bench | bench-c0 | bench-ref | ncu-list | ncu-full | ncu-gather | smoke | gatherab | kernel
set -u
TAG=$1; shift
OUT=gpurun_out
mkdir -p $OUT
PROF_ENV="DDFA_BENCH_MIN_WARMUP=1 DDFA_BENCH_SKIP_CPU=1"
for STAGE in "$@"; do
  echo "=================== stage: $STAGE"
  case $STAGE in
    tests|testsx)
      X=""; [ $STAGE = testsx ] && X="-x"
      timeout 1800 python -m pytest tests -m gpu -q --timeout 600 -s $X > $OUT/${TAG}_pytest.log 2>&1
      echo "pytest exit: $?"; grep -E "passed|failed|error" $OUT/${TAG}_pytest.log | tail -n 5
      grep -E "^(FAILED|ERROR)|worst|max\|d|agreement|F1|adam x3|C1 variable|gradient worst" $OUT/${TAG}_pytest.log | head -n 60 ;;
    smoke)
      timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/${TAG}_smoke.log 2>&1; echo "smoke exit: $?"; tail -n 4 $OUT/${TAG}_smoke.log ;;
    bench)
      timeout 1200 python bench.py > $OUT/${TAG}_bench_c1.json 2> $OUT/${TAG}_bench_c1.err; echo "exit: $?"
      cat $OUT/${TAG}_bench_c1.json; tail -n 5 $OUT/${TAG}_bench_c1.err ;;
    bench-c0)
      timeout 900 python bench.py --graphs 256 --no-variable > $OUT/${TAG}_bench_c0.json 2> $OUT/${TAG}_bench_c0.err; echo "exit: $?"
      cat $OUT/${TAG}_bench_c0.json; tail -n 5 $OUT/${TAG}_bench_c0.err ;;
    bench-ref)
      timeout 900 python bench.py --impl reference --steps 6 --warmup 1 > $OUT/${TAG}_bench_reference.json 2> $OUT/${TAG}_bench_reference.err; echo "exit: $?"
      cat $OUT/${TAG}_bench_reference.json ;;
    ncu-list)
      env $PROF_ENV timeout 1200 ncu --metrics gpu__time_duration.sum --clock-control none -c 1200 --csv \
        --log-file $OUT/${TAG}_launches_c1.csv python bench.py --steps 2 --warmup 1 --no-secondary --no-variable > $OUT/${TAG}_ncu_list.log 2>&1
      echo "ncu launches exit: $?" ;;
    ncu-full)     # (1) --set full of the dominant kernel only (the .ncu-rep must stay well below gpurun's 64 MiB return limit);
                  # (2) a metrics-only pass over one whole step for every kernel of the path
      env $PROF_ENV timeout 900 ncu --set full --clock-control none --import-source on -k regex:"gru_fwd3_kernel" -s 12 -c 3 \
        -f -o $OUT/${TAG}_prof_fwd3_c1 python bench.py --steps 2 --warmup 1 --no-secondary --no-variable > $OUT/${TAG}_ncu_full.log 2>&1
      echo "ncu full (fwd3) exit: $?"
      env $PROF_ENV timeout 900 ncu --clock-control none --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,lts__t_bytes.sum,gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed,lts__throughput.avg.pct_of_peak_sustained_elapsed,sm__throughput.avg.pct_of_peak_sustained_elapsed,sm__warps_active.avg.pct_of_peak_sustained_active,smsp__issue_active.avg.pct_of_peak_sustained_active,sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active,launch__registers_per_thread,launch__grid_size,launch__block_size,l1tex__t_sectors_pipe_lsu_mem_global_op_st.sum \
        -k regex:"gru_fwd3_kernel|dgrad3_kernel|wgrad_kernel|gate_bwd|gather_sum|readout|embed_concat|sgemm_small" -s 80 -c 70 \
        -f -o $OUT/${TAG}_prof_step_c1 python bench.py --steps 2 --warmup 1 --no-secondary --no-variable > $OUT/${TAG}_ncu_step.log 2>&1
      echo "ncu step metrics exit: $?"; ls -la $OUT/*.ncu-rep ;;
    ncu-c0)       # --set full of the forward kernel at C0 (38 400 nodes), isolated launches (scripts/kernel_only.py), inference + training form
      timeout 600 ncu --set full --clock-control none --import-source on -k regex:"gru_fwd3_kernel" -s 2 -c 4 \
        -f -o $OUT/${TAG}_prof_fwd3_c0 python scripts/kernel_only.py fwd 256 > $OUT/${TAG}_ncu_c0.log 2>&1
      echo "ncu full (fwd3, C0) exit: $?" ;;
    ncu-gb)       # --set full + source of the gate backward kernel (two launches)
      env $PROF_ENV timeout 900 ncu --set full --clock-control none --import-source on -k regex:"gate_bwd" -s 10 -c 2 \
        -f -o $OUT/${TAG}_prof_gatebwd_c1 python bench.py --steps 2 --warmup 1 --no-secondary --no-variable > $OUT/${TAG}_ncu_gb.log 2>&1
      echo "ncu gate_bwd exit: $?" ;;
    ab-packed)    # whole-step A/B on this box: round-1 saved state (fp32 h_t + four fp32 gate planes) vs packed state
      bash scripts/gpu_ab.sh ${TAG} DDFA_PACKED_STATE 0 1 --no-secondary --no-variable 2>&1 | tee $OUT/${TAG}_ab_packed_c1.log
      bash scripts/gpu_ab.sh ${TAG}c0 DDFA_PACKED_STATE 0 1 --graphs 256 --no-variable 2>&1 | tee $OUT/${TAG}_ab_packed_c0.log ;;
    pairtest)     # the CTA-pair forward kernel alone, short timeout (first runs of a new synchronisation protocol)
      timeout 240 python -m pytest tests/test_kernels_gpu.py -m gpu -q --timeout 200 -s -x -k "cta_pair" > $OUT/${TAG}_pytest_pair.log 2>&1
      echo "pair pytest exit: $?"; tail -n 12 $OUT/${TAG}_pytest_pair.log | cut -c1-300 ;;
    ab-gbtma)     # gate backward: register-path kernel vs TMA-staged kernel, same library, same box
      bash scripts/gpu_ab.sh ${TAG} DDFA_GATE_BWD_TMA 0 1 --no-secondary --no-variable 2>&1 | tee $OUT/${TAG}_ab_gbtma_c1.log
      bash scripts/gpu_ab.sh ${TAG}c0 DDFA_GATE_BWD_TMA 0 1 --graphs 256 --no-variable 2>&1 | tee $OUT/${TAG}_ab_gbtma_c0.log ;;
    ab-csrp)      # TMA-staged gate backward: CSR scalars fetched inside the iteration (1) vs pipelined one value per lane (2)
      bash scripts/gpu_ab.sh ${TAG} DDFA_GATE_BWD_TMA 1 2 --no-secondary --no-variable 2>&1 | tee $OUT/${TAG}_ab_csrp_c1.log
      bash scripts/gpu_ab.sh ${TAG}c0 DDFA_GATE_BWD_TMA 1 2 --graphs 256 --no-variable 2>&1 | tee $OUT/${TAG}_ab_csrp_c0.log ;;
    ab-gsrc)      # image->image gather: one row group per warp (1) vs by size (0: 4 groups at C1, 2 at C0), CSR chain pipelined across groups
      bash scripts/gpu_ab.sh ${TAG} DDFA_GATHER_SRC_GROUPS 1 0 --no-secondary --no-variable 2>&1 | tee $OUT/${TAG}_ab_gsrc_c1.log
      bash scripts/gpu_ab.sh ${TAG}c0 DDFA_GATHER_SRC_GROUPS 1 0 --graphs 256 --no-variable 2>&1 | tee $OUT/${TAG}_ab_gsrc_c0.log ;;
    ab-pair)
      bash scripts/gpu_ab.sh ${TAG} DDFA_FWD_PAIR 0 1 --no-secondary --no-variable 2>&1 | tee $OUT/${TAG}_ab_pair_c1.log
      bash scripts/gpu_ab.sh ${TAG}c0 DDFA_FWD_PAIR 0 1 --graphs 256 --no-variable 2>&1 | tee $OUT/${TAG}_ab_pair_c0.log ;;
    ab-lib)       # same-box A/B of two builds: deepdfa_b200/lib/libddfa_b200_prev.so (previous commit) vs the current library
      for rep in 1 2; do
        for v in prev cur; do
          LIBP=deepdfa_b200/lib/libddfa_b200.so; [ $v = prev ] && LIBP=deepdfa_b200/lib/libddfa_b200_prev.so
          env DDFA_LIB_PATH=$PWD/$LIBP DDFA_BENCH_SKIP_CPU=1 timeout 600 python bench.py --steps 30 --warmup 5 --no-secondary --no-variable ${AB_ARGS:-} > $OUT/${TAG}_lib_${v}_r${rep}.json 2> $OUT/${TAG}_lib_${v}_r${rep}.err
          python - <<PY | tee -a $OUT/${TAG}_ab_lib.log
import json
d = json.load(open("$OUT/${TAG}_lib_${v}_r${rep}.json"))
print("lib=$v rep $rep: %.0f graphs/s  %.4f ms/step  e2e %.0f | " % (d["value"], d["ms_per_step"], d["e2e"]["value"]) +
      " ".join("%s %.1fus" % (l["kernel"][:12], l["avg_launch_us"]) for l in d["roofline_kernels"]))
PY
        done
      done ;;
    kerneltests)
      timeout 900 python -m pytest tests/test_kernels_gpu.py -m gpu -q --timeout 300 -s -x > $OUT/${TAG}_pytest_kernels.log 2>&1
      echo "pytest exit: $?"; tail -n 15 $OUT/${TAG}_pytest_kernels.log | cut -c1-300 ;;
    gatherab)
      timeout 900 python scripts/gather_bench.py > $OUT/${TAG}_gather_ab.log 2>&1; echo "gather exit: $?"; cat $OUT/${TAG}_gather_ab.log ;;
    *) echo "unknown stage $STAGE" ;;
  esac
done
ls -la $OUT | tail -n 12

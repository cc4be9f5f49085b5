#!/usr/bin/env bash
# The one GPU-side runner (everything here runs under `gpurun`; logs land in gpurun_out/ and are summarised into profiles/).
#   bash tools/gpu.sh <tag> <stage> [<stage> ...]
# stages
#   build                 compile the library (normally a no-op: the prebuilt .so travels with the snapshot)
#   pytest[:<-k expr>]    the -m gpu suite in one process (optionally filtered)
#   micro                 microbenchmarks: MUFU / polynomial exp2 mixes, TMEM load / store throughput
#   attn[:<variants>]     same-box sweep of attention variants inside the real forward (micro-batch 64); variants "kernel:polypairs ..."
#   san[:<tool,...>]      compute-sanitizer (memcheck,racecheck,synccheck) over small kernel-level cases
#   cpu0                  MEASURED CPU baseline of BASELINE config[0] (64x64, batch 4, 10+10 steps) on the box's host cores
#   bench[:<args>]        bench.py (default workload) -> bench_<tag>.json + per-op table
#   cfg                   bench.py --workload cfg
#   train[:<args>]        bench.py --workload train (SURVEY f2: one training step, batch 64/GPU);  trainlaunches[:batch]: its ncu launch list by kernel
#   ddpcheck[:fp16]       2-GPU NCCL check of the data-parallel training step (all-reduced gradient = mean of shard gradients; identical parameters);
#                         fp16: under dynamic loss scaling, plus a step that overflows on one rank only and must be skipped on every rank
#   trainprec[:<args>]    tools/bench_train_precision.py: bf16 vs fp16 training step alternated in one process (batch 64, 128x128)
#   guided                bench.py --workload guided (SURVEY f4: inversion + gradient-guided generation, batch 64)
#   train2                the same at 2 GPUs (torchrun; run under `gpurun --gpus 2`)
#   strong                strong-scaling line: total batch 256 over --gpus N ranks is not applicable at N=1; runs --batch 32 (the per-GPU share of 8)
#   launches              ncu launch list of one forward window;  dram: ncu DRAM bytes per launch
#   ncutrain:<regex>[:skip]  the same for a kernel of the training step (bench.py --workload train --batch 32)
#   ncu:<regex>[:<env>]   one ncu --set full capture of kernels matching <regex> (optionally with ENV=VAL,... set)
tag="$1"; shift
mkdir -p gpurun_out
SMIQ="index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
SHORT="python bench.py --batch 64 --no-cpu-baseline --e2e-steps 1"
for stage in "$@"; do
  name="${stage%%:*}"; arg=""; [[ "$stage" == *:* ]] && arg="${stage#*:}"
  t0=$SECONDS
  case "$name" in
    build)
      python -c "import __graft_entry__ as g; g.build()" > gpurun_out/build_${tag}.log 2>&1; echo "build exit=$?";;
    pytest)
      if [ -n "$arg" ]; then timeout 900 python -m pytest tests -q -m gpu -p no:cacheprovider --tb=short -s -k "$arg" > gpurun_out/pytest_gpu_${tag}.log 2>&1
      else timeout 900 python -m pytest tests -q -m gpu -p no:cacheprovider --tb=short -s > gpurun_out/pytest_gpu_${tag}.log 2>&1; fi
      echo "pytest exit=$?"; grep -E "^\[|passed|failed|error" gpurun_out/pytest_gpu_${tag}.log | tail -40;;
    micro)
      for m in mufu softmax_mix tmem_ld; do
        nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o gpurun_out/$m tools/microbench/$m.cu > gpurun_out/micro_build_$m.log 2>&1 \
          && timeout 120 gpurun_out/$m > gpurun_out/micro_${m}_${tag}.txt 2>&1
        echo "== $m exit=$?"; cat gpurun_out/micro_${m}_${tag}.txt; rm -f gpurun_out/$m
      done;;
    attn)
      for v in ${arg:-v3:6 tc:4 tc2:4 tc2:3 tc2p:4 v3:6}; do
        k="${v%%:*}"; pp="${v##*:}"; pipe=0; [ "$k" = "tc2p" ] && { k=tc2; pipe=1; }
        PHENDIFF_B200_ATTN_TC2_PIPE=$pipe PHENDIFF_B200_ATTN_KERNEL=$k PHENDIFF_B200_ATTN_POLYPAIRS=$pp timeout 150 $SHORT --num-inference-steps 6 --steps 2 --warmup 3 \
            --dump-ops gpurun_out/ops_${tag}_${v/:/_}.md > gpurun_out/bench_${tag}_${v/:/_}.json 2> gpurun_out/bench_${tag}_${v/:/_}.err
        python - <<PY
import json
try:
    d=json.loads(open("gpurun_out/bench_${tag}_${v/:/_}.json").read().strip().splitlines()[-1]); r=d["roofline"]
    att=[l for l in open("gpurun_out/ops_${tag}_${v/:/_}.md") if "attention S=" in l]
    print("variant $v", round(d["value"],2), "img/s (6+6 steps, batch 64)", "attn share", round(r["share_by_class"]["attention"],3), "attn ms", att[0].split("|")[4].strip() if att else None, "sm MHz", d["clocks"]["sm_mhz"])
except Exception as e:
    print("variant $v FAILED", e)
PY
      done;;
    san)
      for tool in ${arg:-memcheck racecheck synccheck}; do
        tool="${tool//,/ }"
        for t in $tool; do
          PHENDIFF_B200_SANITIZER=1 timeout 420 compute-sanitizer --tool $t --print-limit 30 python -m pytest tests/test_gpu_sanitizer_cases.py -q -m gpu -p no:cacheprovider --tb=line -x \
              > gpurun_out/sanitizer_${t}_${tag}.log 2>&1
          echo "sanitizer $t exit=$?"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed|Error" gpurun_out/sanitizer_${t}_${tag}.log | tail -6
        done
      done;;
    cpu0)
      timeout 600 python tools/cpu_baseline_config0.py > gpurun_out/cpu_config0_${tag}.json 2> gpurun_out/cpu_config0_${tag}.err; echo "cpu0 exit=$?"; cat gpurun_out/cpu_config0_${tag}.json;;
    bench)
      nvidia-smi --query-gpu=$SMIQ --format=csv -lms 500 > gpurun_out/clocks_${tag}.csv & SMI=$!
      python bench.py $arg --dump-ops gpurun_out/ops_${tag}.md > gpurun_out/bench_${tag}.json 2> gpurun_out/bench_${tag}.err; echo "bench exit=$?"
      kill $SMI; tail -c 3000 gpurun_out/bench_${tag}.json;;
    cfg)
      python bench.py --workload cfg --steps 2 --warmup 3 > gpurun_out/bench_cfg_${tag}.json 2> gpurun_out/bench_cfg_${tag}.err; echo "cfg exit=$?"; tail -c 1500 gpurun_out/bench_cfg_${tag}.json;;
    train)
      timeout 600 python bench.py --workload train --batch 64 --steps 3 --warmup 3 $arg > gpurun_out/bench_train_${tag}.json 2> gpurun_out/bench_train_${tag}.err; echo "train exit=$?"; tail -c 1800 gpurun_out/bench_train_${tag}.json; tail -3 gpurun_out/bench_train_${tag}.err;;
    trainlaunches)
      timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_train_${tag}.csv \
          python bench.py --workload train --batch ${arg:-16} --steps 1 --warmup 1 --e2e-steps 0 > gpurun_out/ncu_launches_train_${tag}.log 2>&1; echo "trainlaunches exit=$?";;   # then here: python tools/summarize_profile.py train_<tag>
    guided)
      timeout 600 python bench.py --workload guided --batch 64 --steps 1 --warmup 1 $arg > gpurun_out/bench_guided_${tag}.json 2> gpurun_out/bench_guided_${tag}.err; echo "guided exit=$?"; tail -c 1200 gpurun_out/bench_guided_${tag}.json; tail -3 gpurun_out/bench_guided_${tag}.err;;
    train2)   # needs `gpurun --gpus 2`: data-parallel training step over NCCL (one all-reduce of the flat gradient vector per step)
      timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 bench.py --gpus 2 \
          --workload train --batch 64 --steps 3 --warmup 3 $arg > gpurun_out/bench_train_n2_${tag}.json 2> gpurun_out/bench_train_n2_${tag}.err; echo "train2 exit=$?"
      tail -c 1500 gpurun_out/bench_train_n2_${tag}.json; tail -3 gpurun_out/bench_train_n2_${tag}.err;;
    trainN)    # trainN:<N> under `gpurun --gpus N`
      timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node ${arg:-8} --master-addr 127.0.0.1 --master-port 29517 bench.py --gpus ${arg:-8} \
          --workload train --batch 64 --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/bench_train_n${arg:-8}_${tag}.json 2> gpurun_out/bench_train_n${arg:-8}_${tag}.err; echo "trainN exit=$?"
      tail -c 600 gpurun_out/bench_train_n${arg:-8}_${tag}.json; tail -2 gpurun_out/bench_train_n${arg:-8}_${tag}.err;;
    ddpcheck)  # needs `gpurun --gpus 2`
      timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 tools/check_ddp_train.py ${arg:+--precision $arg} \
          > gpurun_out/ddpcheck_${tag}.log 2>&1; echo "ddpcheck exit=$?"; grep ddpcheck gpurun_out/ddpcheck_${tag}.log;;
    trainprec)   # JSON lines on stdout
      timeout 900 python tools/bench_train_precision.py $arg; echo "trainprec exit=$?";;
    strong)
      python bench.py --batch 32 --steps 3 --warmup 3 --no-cpu-baseline > gpurun_out/bench_strong32_${tag}.json 2> gpurun_out/bench_strong32_${tag}.err; echo "strong exit=$?"; tail -c 1200 gpurun_out/bench_strong32_${tag}.json;;
    launches)
      timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -s ${NCU_SKIP:-3000} -c 330 --csv \
          --log-file gpurun_out/launches_${tag}.csv $SHORT --num-inference-steps 10 --steps 1 --warmup 1 > gpurun_out/ncu_launches_${tag}.log 2>&1; echo "launches exit=$?";;
    dram)
      timeout 900 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none -s ${NCU_SKIP_DRAM:-900} -c 202 --csv \
          --log-file gpurun_out/dram_${tag}.csv $SHORT --num-inference-steps 3 --steps 1 --warmup 1 > gpurun_out/ncu_dram_${tag}.log 2>&1; echo "dram exit=$?";;
    ncu)
      rx="${arg%%:*}"; envs=""; [[ "$arg" == *:* ]] && envs="${arg#*:}"
      ( for kv in ${envs//,/ }; do export "$kv"; done
        base=function; [[ "$rx" == *"<"* ]] && base=demangled     # template arguments in the pattern: match the demangled name
        timeout 300 ncu --set full --clock-control none --import-source on --kernel-name-base $base -k "regex:$rx" -s ${NCU_KSKIP:-6} -c ${NCU_KCOUNT:-2} \
          -o gpurun_out/prof_${rx//[^a-zA-Z0-9_]/_}_${tag} -f $SHORT --num-inference-steps 1 --steps 1 --warmup 1 > gpurun_out/ncu_${rx//[^a-zA-Z0-9_]/_}_${tag}.log 2>&1 )
      echo "ncu $rx exit=$?"; tail -2 gpurun_out/ncu_${rx//[^a-zA-Z0-9_]/_}_${tag}.log;;
    ncutrain)   # ncu --set full capture of a training-step kernel: ncutrain:<regex>[:<skip>]
      rx="${arg%%:*}"; skip=4; [[ "$arg" == *:* ]] && skip="${arg#*:}"
      base=function; [[ "$rx" == *"<"* ]] && base=demangled
      timeout 600 ncu --set full --clock-control none --import-source on --kernel-name-base $base -k "regex:$rx" -s $skip -c ${NCU_KCOUNT:-2} \
          -o gpurun_out/prof_train_${rx//[^a-zA-Z0-9_]/_}_${tag} -f python bench.py --workload train --batch 32 --steps 1 --warmup 1 --e2e-steps 0 \
          > gpurun_out/ncu_train_${rx//[^a-zA-Z0-9_]/_}_${tag}.log 2>&1
      echo "ncutrain $rx exit=$?"; tail -2 gpurun_out/ncu_train_${rx//[^a-zA-Z0-9_]/_}_${tag}.log;;
    *) echo "unknown stage $stage";;
  esac
  echo "[stage $stage took $((SECONDS - t0)) s]"
done
ls gpurun_out | wc -l

#!/bin/bash
# One parameterised GPU script (replaces the round-1 gpu_*.sh collection).  Run under gpurun:
#   gpurun --timeout 900 -- 'bash tools/gpu.sh <step> [<step> ...]'
# steps: fused | unet | tests | ldmtests | time | bench | benchall | launches | ncu_conv | ncu_mem | smoke | sanitize
# Logs land in gpurun_out/ (merged back by gpurun, < 64 MiB).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv,noheader > gpurun_out/smi.txt 2>&1
run() { echo "== $1"; shift; timeout "$@"; echo "rc=$?"; }
for step in "$@"; do
case "$step" in
  linattn)  run "linattn tc tests" 600 python -m pytest tests/test_ops_gpu.py -m gpu -q -x --tb=short -k "linear_attention" > gpurun_out/t_linattn.log 2>&1; tail -15 gpurun_out/t_linattn.log ;;
  fused)    run "fused op tests" 900 python -m pytest tests/test_fused_gpu.py -m gpu -q -x --tb=short > gpurun_out/t_fused.log 2>&1; tail -15 gpurun_out/t_fused.log ;;
  unet)     run "unet tests" 1500 python -m pytest tests/test_unet_gpu.py -m gpu -q --tb=short > gpurun_out/t_unet.log 2>&1; tail -25 gpurun_out/t_unet.log ;;
  tests)    rm -f gpurun_out/parity_log.jsonl; run "pytest -m gpu" 2400 python -m pytest tests -m gpu -q -rA --tb=short > gpurun_out/pytest_gpu.log 2>&1; tail -8 gpurun_out/pytest_gpu.log ;;
  dflt)     rm -f gpurun_out/parity_log.jsonl; run "pytest -m gpu (default path)" 2400 python -m pytest tests -m gpu -q --tb=short --ignore=tests/test_ldm_gpu.py > gpurun_out/pytest_dflt.log 2>&1; tail -25 gpurun_out/pytest_dflt.log ;;
  ldmtests) run "ldm tests" 1500 python -m pytest tests/test_ldm_gpu.py -m gpu -q --tb=short > gpurun_out/t_ldm.log 2>&1; tail -5 gpurun_out/t_ldm.log ;;
  time)     rm -f gpurun_out/prof_dump.csv; NOPE_PROF_DUMP=gpurun_out/prof_dump.csv run "time_sweep" 900 python tools/time_sweep.py ${TIME_SPECS:-fp16 fp16:fuse_gn=0} --profile > gpurun_out/time_sweep.log 2>&1; cat gpurun_out/time_sweep.log ;;
  epi)      for d in ${EPI_LIST:-3 4 3 4}; do echo "NOPE_GN_EPI=$d"; NOPE_GN_EPI=$d timeout 600 python tools/time_sweep.py ${TIME_SPECS:-fp16} --steps 20 2>&1 | tail -1 | cut -c1-200; done > gpurun_out/epi_ab.log 2>&1; cat gpurun_out/epi_ab.log
            for d in 3 4; do NOPE_GN_EPI=$d NOPE_PROF_DUMP=gpurun_out/prof_dump_epi$d.csv timeout 600 python tools/time_sweep.py fp16 --profile > /dev/null 2>&1; done ;;
  dbg)      for d in ${DBG_LIST:-0 8 16 24}; do echo "NOPE_GN_DBG=$d"; NOPE_GN_DBG=$d timeout 600 python tools/time_sweep.py fp16 --profile 2>&1 | tail -1; done > gpurun_out/dbg_sweep.log 2>&1; cat gpurun_out/dbg_sweep.log ;;
  pdl)      for d in ${PDL_LIST:-0 1 3 0 1 3 0 1 3}; do echo "NOPE_PDL=$d"; NOPE_PDL=$d timeout 600 python tools/time_sweep.py fp16 --steps 20 2>&1 | tail -1 | cut -c1-120; done > gpurun_out/pdl_ab.log 2>&1; cat gpurun_out/pdl_ab.log ;;
  ts)       for k in ${TS_LAUNCHES:-2 8 20 24 30}; do NOPE_GN_TS=$k NOPE_GN_TS_FILE=gpurun_out/gn_ts_$k.csv timeout 600 python tools/time_sweep.py fp16 --steps 1 > /dev/null 2>&1; head -1 gpurun_out/gn_ts_$k.csv; done ;;
  ncu_gn)   run "ncu full: fused conv" 900 ncu --profile-from-start off --set full --clock-control none --import-source on --kernel-name-base demangled -k regex:"${NCU_KREGEX:-conv_tc2_kernel<\(int\)192, \(int\)6, \(int\)4>}" -s ${NCU_SKIP:-1} -c ${NCU_COUNT:-3} -o gpurun_out/prof_gn -f python tools/profile_step.py > gpurun_out/ncu_gn.log 2>&1
            ncu -i gpurun_out/prof_gn.ncu-rep --page raw --csv > gpurun_out/prof_gn_raw.csv 2>/dev/null ;;
  bench)    run "bench" 900 python bench.py --steps 10 --warmup 3 > gpurun_out/bench.log 2>&1; tail -1 gpurun_out/bench.log ;;
  benchall) for spec in "parity:--precision parity" "cfg2_fp16:--queries 8 --poses 2562" "cfg2_bf16:--queries 8 --poses 2562 --precision bf16" "ldm:--variant ldm" "ref:--impl reference"; do
              name=${spec%%:*}; fl=${spec#*:}; run "bench $name" 900 python bench.py --steps 10 --warmup 3 $fl > gpurun_out/bench_$name.log 2>&1; tail -1 gpurun_out/bench_$name.log | cut -c 1-900; done ;;
  smoke)    run "smoke" 900 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; tail -5 gpurun_out/smoke.log ;;
  launches2) env ${ENV_B:-NOPE_FUSE_TO_OUT=1} timeout 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches_b.csv python tools/profile_step.py > gpurun_out/ncu_list_b.log 2>&1
            python tools/summarize_launches.py gpurun_out/launches_b.csv > gpurun_out/launch_summary_b.txt 2>&1; head -12 gpurun_out/launch_summary_b.txt ;;
  pipe)     run "ncu tensor-pipe list" 900 ncu --profile-from-start off --metrics gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --csv --log-file gpurun_out/pipe.csv python tools/profile_step.py > gpurun_out/ncu_pipe.log 2>&1
            python tools/summarize_pipe.py gpurun_out/pipe.csv gpurun_out/pipe_per_launch.csv > gpurun_out/pipe_summary.txt 2>&1; cat gpurun_out/pipe_summary.txt ;;
  pipe_cfg2) NOPE_POSES=2562 NOPE_QUERIES=8 run "ncu tensor-pipe list, configs[2] size (first 420 launches)" 900 ncu --profile-from-start off -c 420 --metrics gpu__time_duration.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed,dram__bytes_read.sum,dram__bytes_write.sum --clock-control none --csv --log-file gpurun_out/pipe_cfg2.csv python tools/profile_step.py > gpurun_out/ncu_pipe_cfg2.log 2>&1
            python tools/summarize_pipe.py gpurun_out/pipe_cfg2.csv gpurun_out/pipe_cfg2_per_launch.csv > gpurun_out/pipe_cfg2_summary.txt 2>&1; cat gpurun_out/pipe_cfg2_summary.txt ;;
  launches) run "ncu launch list" 900 ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv --log-file gpurun_out/launches.csv python tools/profile_step.py > gpurun_out/ncu_list.log 2>&1
            python tools/summarize_launches.py gpurun_out/launches.csv > gpurun_out/launch_summary.txt 2>&1; head -30 gpurun_out/launch_summary.txt ;;
  ncu_conv) run "ncu full: conv" 900 ncu --profile-from-start off --set full --clock-control none --import-source on -k regex:conv_tc -c ${NCU_COUNT:-70} -o /tmp/prof_conv -f python tools/profile_step.py > gpurun_out/ncu_conv.log 2>&1
            ncu -i /tmp/prof_conv.ncu-rep --page raw --csv > gpurun_out/prof_conv_raw.csv 2>/dev/null ;;
  ncu_mem)  run "ncu full: memory-bound" 900 ncu --profile-from-start off --set full --clock-control none -k regex:'gn_|linattn|final_conv|bcast|midattn|pose_embed|topk' -c 40 -o /tmp/prof_mem -f python tools/profile_step.py > gpurun_out/ncu_mem.log 2>&1
            ncu -i /tmp/prof_mem.ncu-rep --page raw --csv > gpurun_out/prof_mem_raw.csv 2>/dev/null ;;
  dist)     N=${NGPU:-2}; run "dist_check N=$N" 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29511 tools/dist_check.py > gpurun_out/dist_check_$N.log 2>&1; tail -12 gpurun_out/dist_check_$N.log ;;
  benchN)   N=${NGPU:-2}; run "bench N=$N weak" 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29512 bench.py --gpus $N --steps 10 --warmup 3 > gpurun_out/bench_n$N.log 2>&1; tail -1 gpurun_out/bench_n$N.log | cut -c 1-600
            run "bench N=$N strong 10248" 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29513 bench.py --gpus $N --steps 10 --warmup 3 --global-poses 10248 > gpurun_out/bench_strong_n$N.log 2>&1; tail -1 gpurun_out/bench_strong_n$N.log | cut -c 1-600 ;;
  shapenet) N=${NGPU:-2}; run "test_shapeNet.py 1 GPU" 600 python test_shapeNet.py --batches 1 --batch-size 2 --grid 642 --categories bottle,mug --json-out gpurun_out/shapenet_n1.json > gpurun_out/shapenet_n1.log 2>&1
            run "test_shapeNet.py $N GPUs" 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port 29514 test_shapeNet.py --batches 1 --batch-size 2 --grid 642 --categories bottle,mug --json-out gpurun_out/shapenet_n$N.json > gpurun_out/shapenet_n$N.log 2>&1
            python -c "
import json
a=json.load(open('gpurun_out/shapenet_n1.json')); b=json.load(open('gpurun_out/shapenet_n$N.json'))
print('top-1 pose indices, 1 GPU :', a['top1_idx']); print('top-1 pose indices, $N GPUs:', b['top1_idx'])
print('scores equal:', a['scores']==b['scores'], ' top-1 equal:', a['top1_idx']==b['top1_idx'])
" | tee gpurun_out/shapenet_compare.txt ;;
  sanitize) run "memcheck smoke" 1200 compute-sanitizer --tool memcheck python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/sanitizer_memcheck.log 2>&1; tail -5 gpurun_out/sanitizer_memcheck.log ;;
  *) echo "unknown step $step" ;;
esac
done
du -sh gpurun_out

#!/bin/bash
# One parameterised GPU session script (replaces the per-session one-offs of round 1):
#   gpurun --timeout 1500 -- 'bash tools/gpu_run.sh <tag> <step> [<step> ...]'
# steps: tests | smoke | bench | bench_ab | host | micro | layers | launches | ncu_gemm | ncu_wgrad | ncu_hbm | ncu_hbm2 (light metrics, every HBM kernel of a step) | sanitize |
#        bench_cfg0 | bench_nuscenes | bench_mix3d | empty_cache
# Everything lands in gpurun_out/<tag>_*; copy what should be judged into profiles/.
tag=$1; shift
mkdir -p gpurun_out
O=gpurun_out/${tag}
# gpurun merges gpurun_out/ back only while it stays under 64 MiB: reports are exported to text on the box and removed
for step in "$@"; do
  echo "=== $step" | tee -a ${O}_steps.log
  case $step in
    tests)    timeout 1500 python -m pytest tests -m gpu -q -x 2>&1 | tail -15 | tee ${O}_gpu_tests.log ;;
    tests_all) timeout 1500 python -m pytest tests -m gpu -q --maxfail=8 2>&1 | tail -60 | tee ${O}_gpu_tests.log ;;
    tests_e2e) timeout 900 python -m pytest tests/test_gpu_fullscale.py tests/test_gpu_model.py tests/test_gpu_trainer.py -m gpu -q 2>&1 | tail -15 | tee ${O}_gpu_tests_e2e.log ;;
    smoke)    timeout 300 python __graft_entry__.py smoke 2>&1 | tail -3 | tee ${O}_smoke.log ;;
    bench)    timeout 900 python bench.py --steps 8 --warmup 3 > ${O}_bench.json 2> ${O}_bench.err; tail -2 ${O}_bench.err | cut -c1-400 ;;
    bench_ref) timeout 900 python bench.py --impl reference --steps 3 --warmup 1 > ${O}_bench_reference.json 2> ${O}_bench_reference.err; cat ${O}_bench_reference.json | cut -c1-600 ;;
    bench_default) ( time timeout 900 python bench.py ) > ${O}_bench_default.json 2> ${O}_bench_default.err; tail -5 ${O}_bench_default.err | cut -c1-300 ;;
    bench_nocpu) timeout 900 python bench.py --steps 8 --warmup 3 --no-cpu-baseline > ${O}_bench.json 2> ${O}_bench.err; tail -2 ${O}_bench.err | cut -c1-400 ;;
    bench_ab) for cfg in "LIDOG_LAYER_CALLS=0" "LIDOG_EPI_STATS=0"; do
                env $cfg timeout 600 python bench.py --steps 8 --warmup 3 --no-cpu-baseline > ${O}_bench_${cfg}.json 2> ${O}_bench_${cfg}.err
                tail -1 ${O}_bench_${cfg}.err | cut -c1-300; done ;;
    empty_cache) timeout 600 python bench.py --steps 8 --warmup 3 --no-cpu-baseline --empty-cache > ${O}_bench_empty_cache.json 2> ${O}_bench_empty_cache.err; tail -1 ${O}_bench_empty_cache.err | cut -c1-300 ;;
    bench_cfg0) timeout 900 python bench.py --steps 8 --warmup 3 --batch 1 --classes 19 > ${O}_bench_cfg0.json 2> ${O}_bench_cfg0.err; tail -1 ${O}_bench_cfg0.err | cut -c1-300 ;;
    bench_nuscenes) timeout 600 python bench.py --steps 8 --warmup 3 --shape nuscenes --batch 16 --no-cpu-baseline > ${O}_bench_nuscenes.json 2> ${O}_bench_nuscenes.err; tail -1 ${O}_bench_nuscenes.err | cut -c1-300 ;;
    bench_mix3d) timeout 600 python bench.py --steps 8 --warmup 3 --shape mix3d --batch 8 --no-cpu-baseline > ${O}_bench_mix3d.json 2> ${O}_bench_mix3d.err; tail -1 ${O}_bench_mix3d.err | cut -c1-300 ;;
    host)     timeout 300 python tools/host_profile.py > ${O}_host_profile.txt 2>&1; head -3 ${O}_host_profile.txt ;;
    micro)    timeout 900 python tools/microbench.py > ${O}_microbench.jsonl 2> ${O}_microbench.err; tail -3 ${O}_microbench.jsonl | cut -c1-300 ;;
    layers)   timeout 300 python tools/layer_table.py > ${O}_layer_table.txt 2> ${O}_layer_table.err; head -3 ${O}_layer_table.txt | cut -c1-300 ;;
    convnet)  timeout 300 python tools/conv_bench.py --cases net --sorted 1 --reps 10 > ${O}_conv_net.txt 2>&1; tail -30 ${O}_conv_net.txt | cut -c1-200 ;;
    launches) timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv \
                --log-file ${O}_launches.csv python bench.py --ncu > ${O}_ncu1.log 2>&1
              python tools/launch_summary.py ${O}_launches.csv > ${O}_launch_summary.txt 2>&1; head -45 ${O}_launch_summary.txt ;;
    envsweep) # ENVS="A=1 B=2;A=3" : one launch list per ';'-separated environment, restricted to the kernels in $KSEL
              IFS=';' read -ra VARS <<< "${ENVS:-;}"
              for E in "${VARS[@]}"; do
                echo "== env[$E]" | tee -a ${O}_envsweep.txt
                timeout 600 env $E ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv \
                  -k regex:"${KSEL:-k_wgrad2|k_reduce_partials}" --log-file ${O}_sweep.csv python bench.py --ncu > ${O}_ncu7.log 2>&1
                python tools/launch_summary.py ${O}_sweep.csv 2>&1 | head -6 | tee -a ${O}_envsweep.txt
              done; rm -f ${O}_sweep.csv ;;
    ncu_gemm) timeout 900 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:k_gemm2 -s 58 -c 2 \
                -o ${O}_ncu_gemm2 -f python bench.py --ncu > ${O}_ncu2.log 2>&1
              python tools/ncu_summary.py ${O}_ncu_gemm2.ncu-rep > ${O}_ncu_gemm2.txt; ncu -i ${O}_ncu_gemm2.ncu-rep --page source --csv > ${O}_ncu_gemm2_source.csv 2>/dev/null
              ls -la ${O}_ncu_gemm2.*; rm -f ${O}_ncu_gemm2.ncu-rep ;;
    ncu_wgrad) timeout 900 ncu --set full --clock-control none --import-source on --profile-from-start off -k regex:k_wgrad -s 0 -c 2 \
                -o ${O}_ncu_wgrad2 -f python bench.py --ncu > ${O}_ncu3.log 2>&1
              python tools/ncu_summary.py ${O}_ncu_wgrad2.ncu-rep > ${O}_ncu_wgrad2.txt; ncu -i ${O}_ncu_wgrad2.ncu-rep --page source --csv > ${O}_ncu_wgrad2_source.csv 2>/dev/null
              ls -la ${O}_ncu_wgrad2.*; rm -f ${O}_ncu_wgrad2.ncu-rep ;;
    ncu_hbm)  timeout 900 ncu --set full --clock-control none --profile-from-start off \
                -k regex:'k_bn_|k_neighbors|k_insert|k_conv_c1|k_scan' -c 70 -o ${O}_ncu_hbm -f python bench.py --ncu > ${O}_ncu4.log 2>&1
              python tools/ncu_summary.py ${O}_ncu_hbm.ncu-rep > ${O}_ncu_hbm_kernels.txt; ls -la ${O}_ncu_hbm*; rm -f ${O}_ncu_hbm.ncu-rep ;;
    ncu_hbm2) timeout 600 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,smsp__inst_executed.sum \
                --clock-control none --profile-from-start off \
                -k regex:'k_bn_|k_neighbors|k_insert|k_conv_c1|k_scan|k_bev_|k_dice|k_reduce_partials|k_head_|k_quantize|k_permute|k_sort_keys|k_relabel|k_inverse|k_up2' \
                -c 600 -o ${O}_ncu_hbm2 -f python bench.py --ncu > ${O}_ncu6.log 2>&1
              python tools/ncu_summary.py ${O}_ncu_hbm2.ncu-rep > ${O}_ncu_hbm2_kernels.txt; python tools/hbm_summary.py ${O}_ncu_hbm2_kernels.txt > ${O}_hbm_summary.txt
              ls -la ${O}_ncu_hbm2*; rm -f ${O}_ncu_hbm2.ncu-rep; head -40 ${O}_hbm_summary.txt ;;
    ncu_bev)  timeout 900 ncu --set full --clock-control none --import-source on --profile-from-start off \
                -k regex:'k_bev_' -c 4 -o ${O}_ncu_bev -f python bench.py --ncu > ${O}_ncu5.log 2>&1
              python tools/ncu_summary.py ${O}_ncu_bev.ncu-rep > ${O}_ncu_bev.txt; ncu -i ${O}_ncu_bev.ncu-rep --page source --csv > ${O}_ncu_bev_source.csv 2>/dev/null
              ls -la ${O}_ncu_bev*; rm -f ${O}_ncu_bev.ncu-rep ;;
    syncbn)   NG=${NG:-$(nvidia-smi -L | wc -l)}
              timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $NG --master-addr 127.0.0.1 --master-port 29531 \
                tools/syncbn_check.py 2>&1 | grep -E "syncbn|SYNCBN|Error|error" | tail -5 | tee ${O}_syncbn${NG}.log ;;
    bench_ddp|bench_ddp_nuscenes|bench_ddp_mix3d)
              NG=${NG:-$(nvidia-smi -L | wc -l)}
              case $step in bench_ddp) A="--shape kitti --batch 8";; bench_ddp_nuscenes) A="--shape nuscenes --batch 16";; *) A="--shape mix3d --batch 8";; esac
              timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $NG --master-addr 127.0.0.1 --master-port 29532 \
                bench.py --gpus $NG --steps 8 --warmup 3 $A > ${O}_${step}_${NG}gpu.json 2> ${O}_${step}_${NG}gpu.err
              tail -1 ${O}_${step}_${NG}gpu.err | cut -c1-200; cut -c1-400 ${O}_${step}_${NG}gpu.json ;;
    ddp_ab)   NG=${NG:-$(nvidia-smi -L | wc -l)}   # variants: "ENV=.. ENV=..|bench flags"
              for V in "|--ddp-buffers flat" "|--ddp-buffers ddp" "|--ddp-buffers off" "|--ddp-buffers flat --no-syncbn" \
                       "|--ddp-buffers flat --same-data" "|--ddp-buffers flat"; do
                E="${V%%|*}"; A="${V#*|}"
                echo "== env[$E] $A" | tee -a ${O}_ddp_ab_${NG}gpu.txt
                timeout 600 env $E python -m torch.distributed.run --nnodes=1 --nproc-per-node $NG --master-addr 127.0.0.1 --master-port 29533 \
                  bench.py --gpus $NG --steps 8 --warmup 3 $A 2>/dev/null | python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print(round(d['value'],1), 'scans/s', round(d['ms_per_step'],2), 'ms  e2e', round(d['e2e']['value'],1))" | tee -a ${O}_ddp_ab_${NG}gpu.txt
              done ;;
    tests_syncbn) timeout 900 python -m pytest tests/test_gpu_syncbn.py -m gpu -q 2>&1 | tail -5 | tee ${O}_tests_syncbn.log ;;
    sanitize) bash tools/sanitize.sh ${O} ;;
    *) echo "unknown step $step" ;;
  esac
done

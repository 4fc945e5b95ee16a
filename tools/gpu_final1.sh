#!/bin/bash
# record of the frozen kernels (1 GPU): whole GPU suite, default bench, ncu launch list + DRAM traffic, full captures, experiments
O=gpurun_out/f1; mkdir -p $O
timeout 1500 python -m pytest tests -v -m gpu -rs > $O/gpu_tests_1gpu.log 2>&1; echo "tests rc=$?"
tail -6 $O/gpu_tests_1gpu.log
timeout 900 python bench.py --dump-daily $O/hus_daily_I_E_R256.json > $O/bench_R256.json 2> $O/bench.err; echo "bench rc=$?"
timeout 600 python bench.py --impl reference --steps 1 --warmup 0 > $O/bench_reference_arm.json 2>> $O/bench.err; echo "ref rc=$?"
timeout 900 ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none --csv \
    --log-file $O/launches_traffic_R256.csv python tools/prof_run.py --replicas 256 --days 180 > $O/traffic.log 2>&1
python tools/ncu_traffic.py $O/launches_traffic_R256.csv 256 180 $O/r02_dram_traffic_R256.json "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum --clock-control none --csv python tools/prof_run.py --replicas 256 --days 180" > /dev/null 2>&1
gzip -f $O/launches_traffic_R256.csv
for k in k_sweep k_expose k_resolve k_between; do
  RB_GROUPS=1 timeout 600 ncu --set full --clock-control none --import-source on -k regex:$k -s 92 -c 1 -f \
      -o $O/day92_${k}_R256 python tools/prof_run.py --replicas 256 --days 95 > $O/full92_$k.log 2>&1
  python tools/ncu_report.py $O/day92_${k}_R256.ncu-rep 30 > $O/ncu_day92_${k}_R256.txt 2>&1
done
RB_GROUPS=1 timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_sweep -s 45 -c 1 -f \
    -o $O/day45_k_sweep_R256 python tools/prof_run.py --replicas 256 --days 47 > $O/full45.log 2>&1
python tools/ncu_report.py $O/day45_k_sweep_R256.ncu-rep 30 > $O/ncu_day45_k_sweep_R256.txt 2>&1
rm -f $O/day92_k_resolve_R256.ncu-rep $O/day92_k_between_R256.ncu-rep
for R in 256 32 1; do python tools/kern_times.py $R; done > $O/kernel_times_isolated.txt 2>&1
python tools/group_exp.py --replicas 256 --configs 1:100,2:100,4:50,4:100,8:50 --steps 3 > $O/group_experiment.txt 2>&1
python tools/group_exp.py --replicas 32 --configs 1:100,2:100,4:50,8:50 --steps 3 >> $O/group_experiment.txt 2>&1
cat $O/group_experiment.txt
ls -la $O

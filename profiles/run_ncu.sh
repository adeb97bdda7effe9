#!/bin/bash
# Profiling recipe of /opt/skills/guides/B200_PROFILING.md for the bench workload (1 GPU).
# Usage (under gpurun):  bash profiles/run_ncu.sh <tag>
#   gpurun_out/<tag>_launches.csv     every launch of one device-resident step with its device time
#   gpurun_out/<tag>_traffic.csv      DRAM bytes + time of the on-chip solver kernels of that step
#   gpurun_out/<tag>_cluster.ncu-rep  --set full capture of the dominant solver kernel (all classes of a step)
#   gpurun_out/<tag>_stream.ncu-rep   --set full capture of the streaming kernels (k_pcg_spmv / k_pcg_update,
#                                     iterations 20-22 of the streaming comparison solve, all systems active)
#   gpurun_out/<tag>_c3_traffic.csv   DRAM bytes + time of the streaming kernels on config 3 (cantilever L4)
# Every ncu pass follows a plain run of the same command that exited 0.
set -u
TAG=${1:-r02}
CMD="python bench.py --steps 1 --warmup 1 --no-cpu-baseline --skip dataset,as_sampled,c3,c1"
mkdir -p gpurun_out
# a step launches ~40 kernels (on-chip path); warm-up steps come first: skip them generously and
# keep everything until the streaming-path comparison solve starts
$CMD > gpurun_out/${TAG}_plain.log 2>&1 &&
ncu --metrics gpu__time_duration.sum --clock-control none -s 60 -c 120 --csv \
    --log-file gpurun_out/${TAG}_launches.csv $CMD > gpurun_out/${TAG}_ncu1.log 2>&1
echo "launch list rc=$?"
ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,lts__t_sectors.sum \
    --clock-control none -k regex:k_pcg_cluster -s 4 -c 4 --csv \
    --log-file gpurun_out/${TAG}_traffic.csv $CMD > gpurun_out/${TAG}_ncu2.log 2>&1
echo "traffic rc=$?"
ncu --set full --clock-control none --import-source on -k regex:k_pcg_cluster -s 4 -c 4 \
    -f -o gpurun_out/${TAG}_cluster $CMD > gpurun_out/${TAG}_ncu3.log 2>&1
echo "full capture rc=$?"
ncu --set full --clock-control none --import-source on -k "regex:k_pcg_spmv|k_pcg_update" -s 40 -c 6 \
    -f -o gpurun_out/${TAG}_stream $CMD > gpurun_out/${TAG}_ncu4.log 2>&1
echo "streaming capture rc=$?"
C3="python tools/tune_spmv_c3.py cantilever 4"
ITERS=256 $C3 > gpurun_out/${TAG}_c3_plain.log 2>&1 &&
ITERS=256 ncu --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,lts__t_sectors.sum \
    --clock-control none -k "regex:k_pcg_spmv|k_pcg_update" -s 200 -c 8 --csv \
    --log-file gpurun_out/${TAG}_c3_traffic.csv $C3 > gpurun_out/${TAG}_ncu5.log 2>&1
echo "c3 traffic rc=$?"
for f in cluster stream; do
  ncu -i gpurun_out/${TAG}_$f.ncu-rep --page raw --csv > gpurun_out/${TAG}_${f}_raw_full.csv 2>/dev/null
done
tail -2 gpurun_out/${TAG}_plain.log | cut -c1-400

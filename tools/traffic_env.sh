#!/bin/bash
# DRAM traffic of one kernel at the full default workload under environment settings (run on the GPU machine): tools/traffic_env.sh al_kernel "" "IDL_DP_CTAS_PER_SM=3"
K=$1; shift
mkdir -p gpurun_out
M=dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,smsp__thread_inst_executed.sum,lts__t_sectors_srcunit_tex_op_read.sum,lts__t_sectors_srcunit_tex_op_write.sum
for V in "$@"; do
  env $V ncu --metrics $M --clock-control none -k regex:$K -s 1 -c 1 --csv --log-file gpurun_out/tv.csv python bench.py --steps 1 --warmup 1 --cpu-sample 100 > gpurun_out/tv.log 2>&1
  python - "$V" <<'PY'
import csv, sys
rows = [r for r in csv.reader(open("gpurun_out/tv.csv")) if len(r) > 10]
hdr = rows[0]
print("env [%s]" % sys.argv[1])
for r in rows[1:]:
    d = dict(zip(hdr, r)); print("   %-22s %-50s %s %s" % (d["Kernel Name"][:22], d["Metric Name"], d["Metric Value"], d["Metric Unit"]))
PY
done

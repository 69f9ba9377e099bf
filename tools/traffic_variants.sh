#!/bin/bash
# DRAM traffic / instruction counts of one kernel of the chain at the full default workload, for compile-time variants (run under gpurun):
#   tools/traffic_variants.sh al_kernel "" "-DKSW_UNB_WARPS=8 -DKSW_UNB_CTAS=2" ...
K=$1; shift
mkdir -p gpurun_out
M=dram__bytes_read.sum,dram__bytes_write.sum,gpu__time_duration.sum,smsp__thread_inst_executed.sum,lts__t_sectors_srcunit_tex_op_read.sum,lts__t_sectors_srcunit_tex_op_write.sum,lts__t_sectors_srcunit_tex_op_read_lookup_miss.sum,lts__t_sectors_srcunit_tex_op_write_lookup_miss.sum
for V in "$@"; do
  IDL_NVCC_EXTRA="$V" python -c "from indelope_b200 import build as b; b.build_cuda(force=True)" > /dev/null 2>&1 || { echo "$V: build failed"; continue; }
  ncu --metrics $M --clock-control none -k regex:$K -s 1 -c 1 --csv --log-file gpurun_out/tv.csv python bench.py --steps 1 --warmup 1 --cpu-sample 100 > gpurun_out/tv.log 2>&1
  python - "$V" <<'PY'
import csv, sys
rows = [r for r in csv.reader(open("gpurun_out/tv.csv")) if len(r) > 10]
hdr = rows[0]; out = {}
for r in rows[1:]:
    d = dict(zip(hdr, r)); out[d["Metric Name"]] = (d["Metric Value"], d["Metric Unit"])
print("variant [%s]" % sys.argv[1])
for k, v in out.items():
    print("   %-60s %s %s" % (k, v[0], v[1]))
PY
done
python -c "from indelope_b200 import build as b; b.build_cuda(force=True)" > /dev/null 2>&1

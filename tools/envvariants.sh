#!/bin/bash
# time the bench under different environment settings (run under gpurun):  tools/envvariants.sh "IDL_ASM_CTAS_PER_SM=3" ...
mkdir -p gpurun_out
for V in "$@"; do
  env $V timeout 300 python bench.py --steps 3 --warmup 2 --cpu-sample 100 --e2e-batches 2 > gpurun_out/var.json 2> gpurun_out/var.err
  python - "$V" <<'PY'
import json, sys
try:
    d = json.load(open("gpurun_out/var.json")); k = d["kernel_ms"]
    print("%-60s step %.2f ms  asm %.2f  align %.2f  al %.2f  kmer %.3f" % (sys.argv[1], d["ms_per_step"], k["assemble_kernel"], k["align4_kernel"], k["al_kernel"], k["kmer_kernel"]))
except Exception as e:
    print(sys.argv[1], "bench failed", e)
PY
done

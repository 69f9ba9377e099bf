#!/bin/bash
# build-and-time loop for compile-time variants of the kernels (run under gpurun; nvcc is on the box):
#   tools/variants.sh "-DASM_BLOCKS=0" "-DASM_BLOCKS=1 -DASM_EVAL_NOINLINE=0" ...
mkdir -p gpurun_out
for V in "$@"; do
  IDL_NVCC_EXTRA="$V" python -c "from indelope_b200 import build as b; b.build_cuda(force=True)" > /dev/null 2>&1 || { echo "$V: build failed"; continue; }
  timeout 300 python bench.py --steps 3 --warmup 2 --cpu-sample 100 --e2e-batches 2 > gpurun_out/var.json 2> gpurun_out/var.err
  python - "$V" <<'PY'
import json, sys
try:
    d = json.load(open("gpurun_out/var.json")); k = d["kernel_ms"]
    print("%-60s step %.2f ms  asm %.2f  align %.2f  al %.2f  kmer %.3f" % (sys.argv[1], d["ms_per_step"], k["assemble_kernel"], k["align4_kernel"], k["al_kernel"], k["kmer_kernel"]))
except Exception as e:
    print(sys.argv[1], "bench failed", e)
PY
done
python -c "from indelope_b200 import build as b; b.build_cuda(force=True)" > /dev/null 2>&1

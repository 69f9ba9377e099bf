#!/bin/bash
# compute-sanitizer over the kernels that changed in round 2 (run under gpurun): the 4-thread ring variant and the cp.async tile fetch through
# idl_ksw2_batch and the pipeline, idl_sweep; then a soak of kernel 2 against the compiled reference
OUT=gpurun_out; mkdir -p $OUT
SEL="known_answers or edge_shapes or production or four_threads or row_owned_variant or golden or directed_boundaries or evidence_array or status_bits"
{
echo "compute-sanitizer (B200, round 2) on pytest tests/test_gpu_ksw2.py tests/test_gpu_pipeline.py tests/test_gpu_sweep.py -m gpu -k \"$SEL\""
for T in memcheck synccheck; do
  echo "== $T"
  timeout 1500 compute-sanitizer --tool $T --error-exitcode 0 python -m pytest tests/test_gpu_ksw2.py tests/test_gpu_pipeline.py tests/test_gpu_sweep.py -m gpu -q -k "$SEL" 2>&1 | grep -E "passed|failed|ERROR SUMMARY|Invalid|hazard|error" | tail -8
done
echo "== racecheck (kernel 2 unit tests + sweep)"
timeout 1500 compute-sanitizer --tool racecheck --error-exitcode 0 python -m pytest tests/test_gpu_ksw2.py tests/test_gpu_sweep.py -m gpu -q -k "known_answers or edge_shapes or directed_boundaries or evidence_array" 2>&1 | grep -E "passed|failed|RACECHECK SUMMARY|hazard|error" | tail -8
echo "== soak"
timeout 900 python tools/ksw_soak.py 30000 777
IDL_KSW2_COLUMNS=1 timeout 900 python tools/ksw_soak.py 8000 779
} > $OUT/r02_sanitizer.txt 2>&1
cat $OUT/r02_sanitizer.txt

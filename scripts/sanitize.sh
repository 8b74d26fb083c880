#!/bin/bash
# Run on a machine with the GPU: compute-sanitizer memcheck + racecheck over smoke-size runs of both variants and of a
# batch of tiny utterances.  Uses the sanitizer build of the library (make -C nhans_b200/csrc sanitizer: barrier time-outs
# raised from 2 s to 15 min, everything else identical).  Logs -> gpurun_out/san_*.txt (summaries go to profiles/).
set -u
mkdir -p gpurun_out
export NHANS_B200_LIB=$PWD/nhans_b200/libnhans_b200_san.so
for tool in memcheck racecheck; do
  for mode in sn ss tiny; do
    timeout ${SAN_TIMEOUT:-900} compute-sanitizer --tool $tool --error-exitcode 9 --log-file gpurun_out/san_${tool}_${mode}.txt \
        python scripts/sanitize_run.py $mode > gpurun_out/san_${tool}_${mode}.out 2>&1
    echo "$tool $mode rc=$? : $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' gpurun_out/san_${tool}_${mode}.txt | tail -1) $(tail -1 gpurun_out/san_${tool}_${mode}.out | cut -c1-100)"
  done
done

#!/bin/bash
# The parity suites (device decode and model-input rows included) and the randomised sweep under the bounds-checked build (make variant NAME=bounds
# DEFS=-DWP_DEBUG_BOUNDS): every scratch / list / output index asserted on the device.  usage: bash tools/gpu_bounds.sh <tag>
TAG=${1:-s}; OUT=gpurun_out; mkdir -p $OUT
export WORDPIECE_B200_LIB=$PWD/wordpiece_b200/lib/variants/libwordpiece_b200_bounds.so
PYT="python -m pytest -m gpu -q -p no:cacheprovider --timeout 600 --timeout-method thread"
timeout -k 10 1200 $PYT -x tests/test_gpu_parity.py tests/test_gpu_batch.py tests/test_gpu_decode_device.py tests/test_gpu_rows_device.py > $OUT/t_bounds_$TAG.log 2>&1; echo "bounds parity+batch rc=$?"; tail -n 4 $OUT/t_bounds_$TAG.log
timeout -k 10 900 $PYT tests/test_gpu_configs.py -k "dirty or stress or sharded or zh or adv" > $OUT/t_bounds_configs_$TAG.log 2>&1; echo "bounds configs rc=$?"; tail -n 4 $OUT/t_bounds_configs_$TAG.log
timeout -k 10 600 python tools/fuzz_gpu.py > $OUT/fuzz_bounds_$TAG.log 2>&1; echo "bounds fuzz rc=$?"; tail -n 3 $OUT/fuzz_bounds_$TAG.log
grep -h "WP_CHECK failed" $OUT/t_bounds_$TAG.log $OUT/t_bounds_configs_$TAG.log $OUT/fuzz_bounds_$TAG.log | sort | uniq -c | head

#!/bin/bash
# The pool's compute-sanitizer is closed (profiles/r2_sanitizer_closed.log), so the memory check is our own: build the
# library with -DOK_CHECKED=1 (every table row / chunk / segment / ray / agent index is range-checked and violations are
# COUNTED instead of used) and run the parity suites on it; tests/test_gpu_checked.py then requires the count to be zero.
# usage (on the GPU box, after `make -C openkitchen_b200/csrc variant NAME=checked DEFS=-DOK_CHECKED=1` here): tools/checked_build.sh
cd "$(dirname "$0")/.."
lib=$PWD/openkitchen_b200/lib/variants/lib_checked.so
[ -f "$lib" ] || { echo "build it first: make -C openkitchen_b200/csrc variant NAME=checked DEFS=-DOK_CHECKED=1"; exit 2; }
mkdir -p gpurun_out
OK_B200_LIB=$lib timeout 900 python -m pytest tests/test_gpu_checked.py tests/test_gpu_lidar_query.py tests/test_gpu_bev.py tests/test_gpu_parity.py tests/test_gpu_parity_gaps.py tests/test_gpu_kernel_shapes.py tests/test_gpu_races.py tests/test_gpu_beam_geometry.py -q -x -k "not reference_cuda_kernel" \
  > gpurun_out/checked_build.log 2>&1
echo "checked build: exit $? -- $(tail -1 gpurun_out/checked_build.log)"

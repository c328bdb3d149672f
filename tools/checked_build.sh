#!/bin/bash
# The memory-safety run of this repo (compute-sanitizer is closed on the GPU pool): the library compiled with device-side
# bounds / invariant checks (-DDAISY_BOUNDS_CHECK -> DZ_ASSERT traps) driven through the small parity cases, every result
# compared with the CPU oracle.  Build here (`make -C daisyriot_b200/csrc TAG=check EXTRA=-DDAISY_BOUNDS_CHECK`), run on the GPU box.
cd ${GRAFT_REPO_ROOT:-.}
export DAISY_B200_LIB=$PWD/daisyriot_b200/libdaisy_b200_check.so
for t in ff gather9 gather32; do
  timeout 600 python tools/sanitize_target.py $t 2>&1 | tail -2
done
timeout 1800 python -m pytest tests/test_gpu_parity.py tests/test_gpu_gather_shapes.py -x -q -m gpu -k "(radmat or fixture_scene_rows or sample_counts or edge_heavy or irregular or empty_and_single or gather or closest or trace_screen or face_grids or perforated or chained) and not fused_exchange" 2>&1 | tail -4
timeout 1800 python -m pytest tests/test_gpu_far_geometry.py -x -q -m gpu 2>&1 | tail -4
timeout 1800 python -m pytest tests/test_gpu_converge_device.py -x -q -m gpu -k "not group and not two_process and not shim" 2>&1 | tail -4

#!/bin/bash
# compute-sanitizer over the GPU parity tests: memcheck on everything, racecheck on the kernels with shared-memory pipelines
# (fused forward / backward, gradient rows, voxelizer finalize + claim)
mkdir -p gpurun_out
timeout 900 compute-sanitizer --tool memcheck --error-exitcode 3 python -m pytest tests -m gpu -x -q --timeout 800 > gpurun_out/memcheck_all.log 2>&1; echo memcheck rc=$?
timeout 500 compute-sanitizer --tool racecheck --error-exitcode 3 python -m pytest tests/test_gpu_run_plan.py tests/test_gpu_voxel_pool.py tests/test_gpu_nchw_rig.py -x -q -k "run_plan_and_forward or camera_rig or fused_forward_backward_random or nchw_tensor_map or gradient_rows" --timeout 450 > gpurun_out/racecheck_fused.log 2>&1; echo racecheck fused rc=$?
timeout 300 compute-sanitizer --tool racecheck --error-exitcode 3 python -m pytest tests/test_gpu_pool_mixed.py -x -q -k "mixed_equals_upcast or cold_call_from_geom" --timeout 250 2>&1 | tail -n 4; echo racecheck mixed rc=${PIPESTATUS[0]}
timeout 400 compute-sanitizer --tool racecheck --error-exitcode 3 python -m pytest tests/test_gpu_voxelize.py -x -q -k "random_small_grids or adversarial or batched_ragged or contention or canvas_without" --timeout 350 > gpurun_out/racecheck_vox.log 2>&1; echo racecheck voxelizer rc=$?
for f in gpurun_out/memcheck_all.log gpurun_out/racecheck_fused.log gpurun_out/racecheck_vox.log; do tail -n 4 $f; done # gpurun_out/racecheck_fused.log gpurun_out/racecheck_vox.log

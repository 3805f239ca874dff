# the opt-in code paths must give the same answers as the defaults
for v in "SMPLGPU_V32_EDGE_BATCH=1" "SMPLGPU_WARP_RESOLVE=0" "SMPLGPU_V32_PERSISTENT=1" "SMPLGPU_BFS_MODE=1" "SMPLGPU_BFS_MODE=1 SMPLGPU_BANK_STEPWISE=1" "SMPLGPU_BANK_COOPERATIVE=1" "SMPLGPU_BFS_TILE_RPT=4" "SMPLGPU_LATTICE_FUSED=1" "SMPLGPU_V32_FOLD=0" "SMPLGPU_BANK_TILE_CHUNK=1" "SMPLGPU_BANK_TILE_CHUNK=5"; do
  echo "== $v"
  env $v timeout 900 python -m pytest tests/test_gpu_validity.py tests/test_gpu_planner.py tests/test_gpu_reference_golden.py tests/test_gpu_bfs.py tests/test_gpu_goal_types.py tests/test_gpu_ik_snap.py tests/test_gpu_goal_sets.py tests/test_gpu_planner_limits.py tests/test_gpu_snap_kinds.py -x -q 2>&1 | tail -1
done

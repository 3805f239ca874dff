"""Plan queries/s of BASELINE configuration 5: the PR2 torso and both arms (15-DOF) on the dense shelf scene at 1 cm
(smpl_b200.scenes.pr2_dual_arm_planning_scene, DualArmPlanParams), on 1, 2, 4 and 8 GPUs in one process.

The distance field is built once on GPU 0 and copied to the other GPUs with api.clone_context(..., device=d); each GPU
runs --threads-per-gpu planner threads (one context each) and plan_batch shares the queries over the whole context
list.  The queries are 16 384 reachable XYZ_RPY goals (0.015 m, 0.05 rad) at the target-offset poses of lattice states
--walk random primitive steps from scenes.DUAL_ARM_START (edges checked on the device), the SNAP_TO_XYZ_RPY action at
0.2 m.  Each GPU count gets a warm-up call of the same shape on its first queries, then one timed call.  Prints one JSON
line per GPU count with queries/s, expansions/s, the solved fraction, the share of planner time in BFS bank runs
(setup_seconds / total_seconds) and the scaling against one GPU; every line carries the name and power limit of each
GPU used, read in the same run.

    python tools/dual_arm_plan_time.py [--queries 16384] [--gpus 1 2 4 8] [--threads-per-gpu 4] [--concurrent 96]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from smpl_b200 import api, scenes  # noqa: E402


def gpu_info(n):
    out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30, check=True).stdout.strip().splitlines()
    return out[:n]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--queries", type=int, default=16384)
    ap.add_argument("--max-expansions", type=int, default=2000)
    ap.add_argument("--walk", type=int, default=16, help="primitive steps from the start to each goal state")
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--threads-per-gpu", type=int, default=4)
    ap.add_argument("--concurrent", type=int, default=96, help="queries in flight per planner thread")
    args = ap.parse_args()

    import torch   # the device count only
    n_dev = torch.cuda.device_count()
    gpus = [g for g in args.gpus if g <= n_dev]
    if not gpus:
        raise SystemExit("no GPU")

    t0 = time.perf_counter()
    scene = scenes.pr2_dual_arm_planning_scene(0.01)
    ctx, tables = api.setup_context(scene, device=0)
    field_seconds = time.perf_counter() - t0
    params = scenes.DualArmPlanParams()
    params.max_expansions = args.max_expansions
    nq = args.queries
    starts = np.ascontiguousarray(np.tile(np.array(scenes.DUAL_ARM_START, np.float64), (nq, 1)))
    valid = lambda q0, q1: ctx.check_joint_limits(q1).astype(bool) & ctx.is_edges_valid(q0, q1)[0].astype(bool)
    goals_q = scenes.lattice_walks(starts, params, args.walk, seed=101, valid=valid)
    goals = api.pose_goals(ctx.planning_frame_fk(goals_q), params.xyz_tolerance, rpy_tolerance=0.05)
    snap = api.SnapParams(dist_thresh=0.2)

    per_dev = {0: [ctx] + [api.clone_context(ctx, scene, tables, device=0) for _ in range(args.threads_per_gpu - 1)]}
    for d in range(1, max(gpus)):
        per_dev[d] = [api.clone_context(ctx, scene, tables, device=d) for _ in range(args.threads_per_gpu)]
    base = None
    for g in gpus:
        ctxs = [c for d in range(g) for c in per_dev[d]]
        m = min(nq, len(ctxs) * 8)
        api.plan_batch(ctxs, scene, tables, params, starts[:m], goals[:m], max_concurrent=args.concurrent, snap=snap)
        t1 = time.perf_counter()
        res, st = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=args.concurrent, snap=snap)
        dt = time.perf_counter() - t1
        qps = nq / dt
        base = base or qps
        print(json.dumps(dict(gpus=g, planner_threads=len(ctxs), queries=nq, max_expansions=args.max_expansions,
                              walk=args.walk, seconds=round(dt, 3), queries_per_s=round(qps, 1),
                              expansions_per_s=round(sum(r["expansions"] for r in res) / dt, 1),
                              solved_fraction=round(sum(r["success"] for r in res) / nq, 4),
                              setup_seconds_share=round(st["setup_seconds"] / max(st["total_seconds"], 1e-12), 4),
                              bfs_runs=st["bfs_runs"], scaling_vs_1_gpu=round(qps / base, 3),
                              field_build_seconds=round(field_seconds, 3), gpu_info=gpu_info(g))), flush=True)
    for d, cs in per_dev.items():
        for c in cs:
            c.close()


if __name__ == "__main__":
    main()

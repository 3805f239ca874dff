"""Plan rate of the batched planner per goal type (smplhost_plan_batch_goals) on one GPU.

The PR2 tabletop queries of bench.py's plan leg (2048 queries, at most 2000 expansions, first solution at eps 100,
planner threads as bench.py picks them) are planned four ways:
  xyz         the (nq, 3) goal positions through smplhost_plan_batch_multi (what bench.py times)
  rpy 0.05    the same positions with the demo's orientation, roll = pitch = yaw = 0 (call_planner.cpp:93-96), as
  rpy 0.2     XYZ_RPY goals within 0.05 and 0.2 rad
  joint       joint goals at half a lattice resolution: the configurations reached from the start by 20 random valid
              motion primitive steps
Each variant is warmed up with the same call on the first batch of its queries (same shape: the lattices and the BFS
bank are sized by concurrency and expansion bound, DESIGN.md section 7) and then timed once.  Prints one JSON line per
variant with queries/s, expansions/s, success rate, rounds and device seconds, plus the GPU name and power limit.

    python tools/goal_types_time.py [--queries 2048] [--max-expansions 2000] [--threads 0]
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


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # noqa: BLE001
        out = "unknown (%s)" % e
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--queries", type=int, default=2048)
    ap.add_argument("--max-expansions", type=int, default=2000)
    ap.add_argument("--threads", type=int, default=0, help="planner threads (= contexts); 0 = bench.py's choice")
    args = ap.parse_args()

    scene = scenes.pr2_tabletop_scene()
    ctx, tables = api.setup_context(scene)
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = args.max_expansions
    nq = args.queries
    starts, xyz = scenes.tabletop_queries(nq, seed=13)
    cores = os.cpu_count() or 1
    n_thr = args.threads if args.threads > 0 else max(1, min(6, int(0.75 * cores)))
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(n_thr - 1)]
    per_ctx = (nq + n_thr - 1) // n_thr

    valid = lambda q0, q1: ctx.check_joint_limits(q1).astype(bool) & ctx.is_edges_valid(q0, q1)[0].astype(bool)
    targets = scenes.lattice_walks(starts, params, 20, seed=17, valid=valid)
    poses = np.concatenate([xyz, np.zeros((nq, 3))], axis=1)
    variants = [
        ("xyz", xyz),
        ("xyz_rpy 0.05 rad", api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)),
        ("xyz_rpy 0.2 rad", api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.2)),
        ("joint", api.joint_goals(targets, 0.5 * np.asarray(params.resolutions))),
    ]
    gpu = gpu_info()
    for name, goals in variants:
        wq = min(nq, per_ctx * n_thr)
        api.plan_batch(ctxs, scene, tables, params, starts[:wq], goals[:wq], max_concurrent=per_ctx)
        t0 = time.perf_counter()
        res, st = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=per_ctx)
        dt = time.perf_counter() - t0
        exp = sum(r["expansions"] for r in res)
        print(json.dumps({"goal": name, "queries": nq, "planner_threads": n_thr, "max_expansions": args.max_expansions,
                          "seconds": round(dt, 4), "queries_per_s": round(nq / dt, 1), "expansions_per_s": round(exp / dt, 1),
                          "expansions": exp, "solved": sum(r["success"] for r in res),
                          "success_rate": round(sum(r["success"] for r in res) / nq, 4), "rounds": st["rounds"],
                          "device_seconds_max_thread": round(st["device_seconds"], 4), "gpu": gpu}), flush=True)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()

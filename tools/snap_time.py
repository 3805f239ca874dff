"""Plan rate of the batched planner with and without the snap-to-goal action (smplhost_plan_batch_snap) on one GPU,
and the time of the standalone planning-link IK (smplgpu_planning_link_ik).

The setup of tools/goal_types_time.py: the PR2 tabletop queries of bench.py's plan leg (2048 queries, at most 2000
expansions, first solution at eps 100, 6 planner threads), each variant warmed up with the same call on the first
batch of its queries and then timed once.  Workloads, each with snaps off and with snaps at thresholds 0.0 (the
reference demo's) and 0.2 m:
  pose 0.05     DESIGN.md section 5's pose workload: the goal positions with roll = pitch = yaw = 0, within 0.05 rad
  reachable     XYZ_RPY goals (0.05 rad) at the target-offset poses of random valid states
  joint         joint goals at half a lattice resolution, 20 random valid primitive steps from the start
Prints one JSON line per (workload, snap) with queries/s, expansions/s, solved, rounds, IK solves, convergence rate
and the mean IK iterations of the standalone IK on the same kind of targets, then the standalone IK's time per call at
n = 1, 64 and 4096; every line carries the GPU name and power limit, read in the same run.

    python tools/snap_time.py [--queries 2048] [--max-expansions 2000] [--threads 6]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from smpl_b200 import api, scenes  # noqa: E402
from goal_types_time import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--queries", type=int, default=2048)
    ap.add_argument("--max-expansions", type=int, default=2000)
    ap.add_argument("--threads", type=int, default=6, help="planner threads (= contexts)")
    args = ap.parse_args()

    scene = scenes.pr2_tabletop_scene()
    ctx, tables = api.setup_context(scene)
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = args.max_expansions
    nq = args.queries
    starts, xyz = scenes.tabletop_queries(nq, seed=13)
    n_thr = args.threads
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(n_thr - 1)]
    per_ctx = (nq + n_thr - 1) // n_thr
    gpu = gpu_info()

    valid = lambda q0, q1: ctx.check_joint_limits(q1).astype(bool) & ctx.is_edges_valid(q0, q1)[0].astype(bool)
    targets = scenes.lattice_walks(starts, params, 20, seed=17, valid=valid)
    lo, hi, cont = tables.limits()
    lo = np.where(cont, -np.pi, lo)
    hi = np.where(cont, np.pi, hi)
    rng = np.random.default_rng(31)
    q = rng.uniform(lo, hi, (8 * nq, scene.dof))
    q = q[ctx.is_states_valid(q).astype(bool)][:nq]
    reach = ctx.planning_frame_fk(q)
    poses = np.concatenate([xyz, np.zeros((nq, 3))], axis=1)
    workloads = [
        ("pose 0.05", api.pose_goals(poses, params.xyz_tolerance, rpy_tolerance=0.05)),
        ("reachable pose 0.05", api.pose_goals(reach, params.xyz_tolerance, rpy_tolerance=0.05)),
        ("joint", api.joint_goals(targets, 0.5 * np.asarray(params.resolutions))),
    ]
    snaps = [("off", None), ("0.0", api.SnapParams(dist_thresh=0.0)), ("0.2", api.SnapParams(dist_thresh=0.2))]
    for name, goals in workloads:
        for sname, snap in snaps:
            wq = min(nq, per_ctx * n_thr)
            api.plan_batch(ctxs, scene, tables, params, starts[:wq], goals[:wq], max_concurrent=per_ctx, snap=snap)
            t0 = time.perf_counter()
            res, st = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=per_ctx, snap=snap)
            dt = time.perf_counter() - t0
            exp = sum(r["expansions"] for r in res)
            att, conv = st.get("ik_attempted", 0), st.get("ik_converged", 0)
            print(json.dumps({"goal": name, "snap": sname, "queries": nq, "planner_threads": n_thr,
                              "max_expansions": args.max_expansions, "seconds": round(dt, 4),
                              "queries_per_s": round(nq / dt, 1), "expansions_per_s": round(exp / dt, 1),
                              "solved": sum(r["success"] for r in res), "rounds": st["rounds"], "ik_solves": att,
                              "ik_converged_rate": round(conv / att, 4) if att else None, "gpu": gpu}), flush=True)

    # standalone IK: targets = FK poses of valid states, seeds 0.1 rad away
    seeds = q + rng.uniform(-0.1, 0.1, q.shape)
    for n in (1, 64, 4096):
        k = min(n, len(q))
        P, S = reach[np.arange(n) % len(q)], seeds[np.arange(n) % len(q)]
        for _ in range(3):
            ctx.planning_link_ik(P, S)
        reps = 200 if n < 4096 else 50
        t0 = time.perf_counter()
        for _ in range(reps):
            _, ok, it = ctx.planning_link_ik(P, S)
        dt = (time.perf_counter() - t0) / reps
        print(json.dumps({"ik_n": n, "us_per_call": round(dt * 1e6, 1), "converged_rate": round(float(ok.mean()), 4),
                          "mean_iterations": round(float(it[ok].mean()), 2) if ok.any() else None,
                          "distinct_problems": k, "gpu": gpu}), flush=True)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()

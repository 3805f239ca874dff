"""Plan rate of the batched planner with the snap kinds SNAP_TO_XYZ, SNAP_TO_RPY and SNAP_TO_XYZ_RPY
(smplhost_plan_batch_snaps) on one GPU, and the time of the standalone position-only IK
(smplgpu_planning_link_ik_position).

The setup of tools/snap_time.py: the PR2 tabletop queries of bench.py's plan leg (2048 queries, at most 2000
expansions, first solution at eps 100, 6 planner threads), each variant warmed up with the same call on the first
batch of its queries and then timed once.  Workloads:
  xyz            the bench's XYZ goals: snaps off, SNAP_TO_XYZ at 0.0 and at 0.2 m
  reachable      XYZ_RPY goals (0.05 rad) at the target-offset poses of random valid states: SNAP_TO_XYZ_RPY alone at
                 0.0, SNAP_TO_RPY alone at 0.2, and RPY 0.2 + XYZ 0.2 + XYZ_RPY 0.0
Prints one JSON line per (workload, snaps) with queries/s, expansions/s, solved, rounds, and the IK solves and
converged share of every kind; then the position-only IK's time per call at n = 1, 64 and 4096 (targets: FK positions
of valid states, seeds 0.1 rad away).  Every line carries the GPU name, power limit and max SM clock, read in the same
run.

    python tools/snap_kinds_time.py [--queries 2048] [--max-expansions 2000] [--threads 6]
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

    lo, hi, cont = tables.limits()
    lo = np.where(cont, -np.pi, lo)
    hi = np.where(cont, np.pi, hi)
    rng = np.random.default_rng(31)
    q = rng.uniform(lo, hi, (8 * nq, scene.dof))
    q = q[ctx.is_states_valid(q).astype(bool)][:nq]
    reach = ctx.planning_frame_fk(q)
    S = api.SnapParams
    runs = [
        ("xyz", api.pose_goals(xyz, params.xyz_tolerance), [
            ("off", None),
            ("XYZ 0.0", S(enabled=False, xyz_dist_thresh=0.0)),
            ("XYZ 0.2", S(enabled=False, xyz_dist_thresh=0.2))]),
        ("reachable pose 0.05", api.pose_goals(reach, params.xyz_tolerance, rpy_tolerance=0.05), [
            ("XYZ_RPY 0.0", S(dist_thresh=0.0)),
            ("RPY 0.2", S(enabled=False, rpy_dist_thresh=0.2)),
            ("RPY 0.2 + XYZ 0.2 + XYZ_RPY 0.0", S(dist_thresh=0.0, xyz_dist_thresh=0.2, rpy_dist_thresh=0.2))]),
    ]
    for name, goals, snaps in runs:
        for sname, snap in snaps:
            wq = min(nq, per_ctx * n_thr)
            api.plan_batch(ctxs, scene, tables, params, starts[:wq], goals[:wq], max_concurrent=per_ctx, snap=snap)
            t0 = time.perf_counter()
            res, st = api.plan_batch(ctxs, scene, tables, params, starts, goals, max_concurrent=per_ctx, snap=snap)
            dt = time.perf_counter() - t0
            exp = sum(r["expansions"] for r in res)
            ik = {}
            for kind in api.SNAP_KIND_NAMES:
                att, conv = st.get("ik_attempted_" + kind, 0), st.get("ik_converged_" + kind, 0)
                ik[kind] = {"ik_solves": att, "converged_rate": round(conv / att, 4) if att else None}
            print(json.dumps({"goal": name, "snaps": sname, "queries": nq, "planner_threads": n_thr,
                              "max_expansions": args.max_expansions, "seconds": round(dt, 4),
                              "queries_per_s": round(nq / dt, 1), "expansions_per_s": round(exp / dt, 1),
                              "solved": sum(r["success"] for r in res), "rounds": st["rounds"], "ik": ik, "gpu": gpu}),
                  flush=True)

    seeds = q + rng.uniform(-0.1, 0.1, q.shape)
    for n in (1, 64, 4096):
        idx = np.arange(n) % len(q)
        P, Sd = reach[idx, :3], seeds[idx]
        for _ in range(3):
            ctx.planning_link_ik(P, Sd)
        reps = 200 if n < 4096 else 50
        t0 = time.perf_counter()
        for _ in range(reps):
            _, ok, it = ctx.planning_link_ik(P, Sd)
        dt = (time.perf_counter() - t0) / reps
        print(json.dumps({"position_ik_n": n, "us_per_call": round(dt * 1e6, 1),
                          "converged_rate": round(float(ok.mean()), 4),
                          "mean_iterations": round(float(it[ok].mean()), 2) if ok.any() else None, "gpu": gpu}),
              flush=True)
    for c in ctxs:
        c.close()


if __name__ == "__main__":
    main()

"""Goal sets against separate queries in the batched planner (smplhost_plan_batch_goal_sets) on one GPU.

The setup of tools/snap_time.py: the PR2 tabletop queries of bench.py's plan leg (2048 queries, at most 2000 expansions,
first solution at eps 100, 6 planner threads), each call warmed up with the same call (same shape) on the first batch
of its queries and then timed once.  Each query gets K candidate goals, XYZ_RPY records (0.015 m, 0.05 rad) at the
target-offset poses of random valid states, for K = 1, 4 and 16, with snaps off and at 0.0 m.  Two ways to plan them:
  set        one query per original query, its K candidates as one goal set
  separate   K x 2048 single-goal queries, keeping per original query the cheapest success
Prints one JSON line per (K, snap, mode) with original queries/s, expansions/s, original queries solved, IK solves and
converged, and (set mode) the histogram of reached_goal; every line carries the GPU name and power limit, read in the
same run.

    python tools/goal_set_time.py [--queries 2048] [--max-expansions 2000] [--threads 6] [--k 1 4 16]
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
    ap.add_argument("--k", type=int, nargs="+", default=[1, 4, 16])
    args = ap.parse_args()

    scene = scenes.pr2_tabletop_scene()
    ctx, tables = api.setup_context(scene)
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = args.max_expansions
    nq = args.queries
    starts, _ = scenes.tabletop_queries(nq, seed=13)
    n_thr = args.threads
    ctxs = [ctx] + [api.clone_context(ctx, scene, tables) for _ in range(n_thr - 1)]
    per_ctx = (nq + n_thr - 1) // n_thr
    gpu = gpu_info()

    kmax = max(args.k)
    lo, hi, cont = tables.limits()
    lo = np.where(cont, -np.pi, lo)
    hi = np.where(cont, np.pi, hi)
    rng = np.random.default_rng(31)
    q = rng.uniform(lo, hi, (8 * nq * kmax, scene.dof))
    q = q[ctx.is_states_valid(q).astype(bool)][:nq * kmax]
    assert len(q) == nq * kmax, "not enough valid states"
    cands = api.pose_goals(ctx.planning_frame_fk(q), params.xyz_tolerance, rpy_tolerance=0.05).reshape(nq, kmax)

    def run(starts_, goals_, snap, m):
        """one warm-up call of the same shape on the first m queries, then the timed call"""
        api.plan_batch(ctxs, scene, tables, params, starts_[:m], _head(goals_, m), max_concurrent=per_ctx, snap=snap)
        t0 = time.perf_counter()
        res, st = api.plan_batch(ctxs, scene, tables, params, starts_, goals_, max_concurrent=per_ctx, snap=snap)
        return res, st, time.perf_counter() - t0

    for k in args.k:
        sets = api.goal_sets([cands[i, :k] for i in range(nq)])
        sep_starts = np.repeat(starts, k, axis=0)
        sep_goals = np.ascontiguousarray(cands[:, :k].reshape(-1))
        for sname, snap in (("off", None), ("0.0", api.SnapParams(dist_thresh=0.0))):
            res, st, dt = run(starts, sets, snap, min(nq, per_ctx * n_thr))
            hist = np.bincount([r["reached_goal"] for r in res if r["success"]], minlength=k).tolist()
            print(json.dumps(dict(k=k, snap=sname, mode="set", queries=nq, planner_threads=n_thr,
                                  max_expansions=args.max_expansions, seconds=round(dt, 4),
                                  queries_per_s=round(nq / dt, 1),
                                  expansions_per_s=round(sum(r["expansions"] for r in res) / dt, 1),
                                  solved=sum(r["success"] for r in res), ik_solves=st.get("ik_attempted", 0),
                                  ik_converged=st.get("ik_converged", 0), reached_goal_histogram=hist, gpu=gpu)),
                  flush=True)
            res, st, dt = run(sep_starts, sep_goals, snap, min(nq * k, per_ctx * n_thr))
            best = {}
            for j, r in enumerate(res):
                if r["success"]:
                    i = j // k
                    best[i] = min(best.get(i, r["cost"]), r["cost"])
            print(json.dumps(dict(k=k, snap=sname, mode="separate", queries=nq, submitted=nq * k,
                                  planner_threads=n_thr, max_expansions=args.max_expansions, seconds=round(dt, 4),
                                  queries_per_s=round(nq / dt, 1),
                                  expansions_per_s=round(sum(r["expansions"] for r in res) / dt, 1),
                                  solved=len(best), ik_solves=st.get("ik_attempted", 0),
                                  ik_converged=st.get("ik_converged", 0), gpu=gpu)), flush=True)
    for c in ctxs:
        c.close()


def _head(goals, m):
    """the goals of the first m queries (records, or a (records, offsets) goal-set pair)"""
    if isinstance(goals, tuple):
        recs, off = goals
        return recs[:off[m]], off[:m + 1]
    return goals[:m]


if __name__ == "__main__":
    main()

"""Time of the EUCLID_SPACE path shortcut (smplhost_shortcut_paths_euclid) on one GPU, against the sequential oracle
(oracle/euclid_shortcut) on a subset.

Inputs: planned PR2 tabletop paths (bench.py's plan-leg queries, at most 2000 expansions, first solution at eps 100)
for 64, 256 and 1024 queries; the successful paths are shortcut with the default EuclidParams.  Each size is warmed up
with one call and then timed once.  Prints one JSON line per size with the paths, points, motions decided, IK solves
and converged, waypoint edges checked, device calls, device seconds, host seconds and wall seconds, and the oracle's
CPU seconds on the first --oracle-paths paths with the device's wall seconds on the same paths.  Every line carries
the GPU name, power limit and max SM clock, read in the same run.

    python tools/euclid_shortcut_time.py [--sizes 64,256,1024] [--oracle-paths 16]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from smpl_b200 import api, scenes  # noqa: E402
from goal_types_time import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--sizes", default="64,256,1024")
    ap.add_argument("--max-expansions", type=int, default=2000)
    ap.add_argument("--oracle-paths", type=int, default=16)
    args = ap.parse_args()

    import euclid_shortcut_oracle as eo
    from helpers import make_oracle

    scene = scenes.pr2_tabletop_scene()
    ctx, tables = api.setup_context(scene)
    o = make_oracle(scene)
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = args.max_expansions
    prm = api.EuclidParams()
    gpu = gpu_info()
    for nq in [int(s) for s in args.sizes.split(",")]:
        starts, goals = scenes.tabletop_queries(nq, seed=13)
        got, _ = api.plan_batch(ctx, scene, tables, params, starts, goals, max_concurrent=min(nq, 256), want_states=True)
        paths = [r["path_states"] for r in got if r["success"]]
        api.shortcut_paths_euclid(ctx, tables, paths, prm)   # warm-up
        t0 = time.perf_counter()
        out, src, st = api.shortcut_paths_euclid(ctx, tables, paths, prm)
        wall = time.perf_counter() - t0
        sub = paths[:args.oracle_paths]
        t0 = time.perf_counter()
        api.shortcut_paths_euclid(ctx, tables, sub, prm)
        dev_sub = time.perf_counter() - t0
        t0 = time.perf_counter()
        for p in sub:
            eo.shortcut_path_euclid(o, scene.T_kin_to_planning, p, prm)
        cpu_sub = time.perf_counter() - t0
        line = dict(queries=nq, paths=len(paths), points_in=int(sum(len(p) for p in paths)),
                    points_out=int(sum(len(p) for p in out)), ik_states_out=int(sum((s < 0).sum() for s in src)),
                    motions=st["motions"], ik_solves=st["ik_solves"], ik_converged=st["ik_converged"],
                    edges_checked=st["edges_checked"], device_calls=st["device_calls"],
                    device_s=round(st["device_seconds"], 4), host_s=round(st["host_seconds"], 4), wall_s=round(wall, 4),
                    motions_per_s=round(st["motions"] / wall, 1), oracle_paths=len(sub),
                    oracle_cpu_s=round(cpu_sub, 4), device_wall_s_same_paths=round(dev_sub, 4), gpu=gpu)
        print(json.dumps(line), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()

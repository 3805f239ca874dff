#!/usr/bin/env python3
"""Benchmark of the validity + BFS hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W          our CUDA path
    python bench.py --impl reference ...                    the reference's CPU algorithm on the host cores
    python bench.py ... --dump-outputs DIR                  also the last timed step's outputs, DIR/<name>.npy

A step = one pass of the hot path over one batch of synthetic input of the shape
BASELINE.json configs[1] names: `--states` random PR2 right-arm states plus as many
motion-primitive edges, against the 2 m^3 / 2 cm clutter scene.  The states are uniformly
random LATTICE states (1 degree, ManipLattice::coordToState): what the path's real caller
holds.  Every rank (GPU) processes its own full batch (weak scaling: independent queries, no
collective on the data path; the distance field is built on rank 0 and broadcast once over
NCCL, device to device).  The unit is a validated state: one per state plus `waypoint_count`
per edge, the states CollisionSpace::isStateToStateValid accounts for (collision_space.cpp:538-581).

The driver's record keeps scalars of the dicts the contract names and drops everything else, so
every BASELINE metric is ALSO written as a scalar: device-side fractions under `roofline`, the
other legs' throughputs (plan, drop-in, BFS, config[3] UBR1, config[4] 15-DOF) under `e2e`, their
CPU counterparts under `cpu_baseline`.  `config` is identical in both arms.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True     # no __pycache__: a benchmark run leaves the source tree as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "states validated/s"
UNIT = "states/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_oracle(scene, prime_q, attach=None):
    from oracle_api import OracleScene
    o = OracleScene(scene.robot_path, scene.group, scene.planning_joints, scene.origin, scene.size, scene.res,
                    scene.max_dist)
    for k, v in scene.fixed_joints.items():
        o.set_joint(k, v)
    if scene.use_desc_acm:
        o.use_desc_acm()
    for a, b, allowed in scene.acm_extra:
        o.acm_set(a, b, allowed)
    if attach is not None:
        o.attach_box(*attach)
    if len(scene.cells):
        o.add_cells(scene.cells)
    if len(getattr(scene, "boxes", [])):
        o.insert_boxes(scene.boxes)
    o.prime(prime_q)
    return o


def make_reference_checker(scene, prime_q, attach=None):
    """The reference's OWN collision checker (sbpl_collision_checking compiled from its sources into
    oracle/_ref/libref_collision.so, see oracle/ref_collision_shim.cpp) set up for `scene`, or None when that library
    was not built (then the CPU legs time the oracle port)."""
    from oracle_api import RefCollisionScene, ref_collision_lib
    if ref_collision_lib() is None or os.environ.get("SMPL_BENCH_CPU_PORT"):
        return None
    r = RefCollisionScene(scene.robot_path, scene.group, scene.planning_joints, scene.origin, scene.size, scene.res,
                          scene.max_dist)
    for k, v in scene.fixed_joints.items():
        r.set_joint(k, v)
    if scene.use_desc_acm:
        r.use_desc_acm()
    for a, b, allowed in scene.acm_extra:
        r.acm_set(a, b, allowed)
    if attach is not None:
        r.attach_box(*attach)     # CollisionSpace::attachObject: the reference generates the body's spheres itself
    if len(scene.cells):
        r.add_cells(scene.cells)
    if len(getattr(scene, "boxes", [])):
        r.insert_boxes(scene.boxes)
    r.prime(prime_q)
    return r


def make_cpu_checker(scene, prime_q):
    """-> (checker, kind, description): the compiled reference when available ("reference"), else the port."""
    r = make_reference_checker(scene, prime_q)
    if r is not None:
        return r, "reference", "the reference's own sbpl_collision_checking CollisionSpace (oracle/_ref/libref_collision.so)"
    return make_oracle(scene, prime_q), "port", "oracle (CPU port of sbpl_collision_checking)"


def cpu_validity_rate(scene, q, q0, q1, threads, checkers=None):
    """The CPU checker (one instance per thread: CollisionSpace is not reentrant) on `threads` host threads;
    returns (units/s, units, seconds)."""
    n = len(q)
    parts = np.array_split(np.arange(n), threads)
    oracles = checkers if checkers is not None else [make_cpu_checker(scene, q[0])[0] for _ in range(threads)]
    units = [0] * threads

    def work(i):
        idx = parts[i]
        if len(idx) == 0:
            return
        oracles[i].time_states_valid(q[idx])
        _, _, c = oracles[i].time_edges_valid(q0[idx], q1[idx])
        units[i] = len(idx) + int(c.sum())

    t0 = time.perf_counter()
    if threads == 1:
        work(0)
    else:
        ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
    dt = time.perf_counter() - t0
    return sum(units) / dt, sum(units), dt


def cpu_bfs_rate(n):
    """The reference's own BFS_3D (oracle/_ref) when present, else the port; Mvoxel/s on one core (+1 search thread)."""
    from oracle_api import OracleBfs, RefBfs, ref_lib
    from smpl_b200 import scenes
    walls = scenes.bfs_clutter_walls(n, seed=11)
    seed = scenes.first_free_cell(walls, (n // 2, n // 2, n // 2))
    kind = "reference" if ref_lib() is not None else "port"
    b = RefBfs(n, n, n) if kind == "reference" else OracleBfs(n, n, n)
    b.set_walls(walls)
    dt = b.time_run(*seed)
    b.close()
    return n ** 3 / dt / 1e6, kind, dt


class StdoutToStderr:
    """stdout carries exactly one JSON line: anything a library prints while this is active (NCCL's version
    banner at the first collective, at file-descriptor level) goes to stderr instead."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def setup_shared_scene(scene, local_rank, rank, world, dev, timing=None):
    """Context for `scene` on this rank's GPU: rank 0 builds the distance field on its GPU, every other rank
    receives it in ONE broadcast (NCCL over NVLink) -- the only collective of the data path -- straight from rank 0's
    resident field (smplgpu_distance_field_dev_ptr) into its own reserved buffer (smplgpu_reserve_distance_field):
    device to device, no host hop, no staging tensor.  timing (dict, optional) receives build_ms / broadcast_ms."""
    import torch
    from smpl_b200 import api, sharding
    ctx = api.GpuContext(local_rank)
    tables = api.build_tables(scene)
    ctx.set_robot(tables)
    t0 = time.perf_counter()
    if rank == 0:
        ctx.build_distance_field(api.scene_cells(scene, tables), scene.dims, scene.origin, scene.res, scene.max_dist,
                                 scene.padding)
        ctx.synchronize()
    t1 = time.perf_counter()
    if world > 1:
        ptr, nbytes = ctx.distance_field_dev_ptr() if rank == 0 else ctx.reserve_distance_field(scene.dims)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sharding.broadcast_field_in_place(ptr, nbytes, src=0, device=dev)
        e1.record()
        torch.cuda.synchronize()
        if rank != 0:
            dmax = int(np.ceil(scene.max_dist * (1.0 / scene.res)))
            ctx.set_distance_field_dev(ptr, scene.dims, scene.origin, scene.res, dmax * dmax, scene.padding)   # adopts in place
        if timing is not None:
            timing["broadcast_ms"] = e0.elapsed_time(e1)
            timing["broadcast_bytes"] = nbytes
    if timing is not None:
        timing["build_ms"] = (t1 - t0) * 1e3
    return ctx, tables


WORKLOAD = "config[1] validity sweep: PR2 right arm (7-DOF) lattice states + mprim edges vs 2 m^3 clutter scene @ 2 cm"


def sweep_inputs(lo, hi, cont, n, rank):
    """The step's inputs, identical for both arms: n uniformly random lattice states (1 degree discretisation,
    ManipLattice::coordToState joint values) and n edges, edge i = state i + motion primitive i mod 22."""
    from smpl_b200 import scenes
    res = scenes.PlanParams(len(lo)).resolutions
    coords, q = scenes.random_lattice_coords(n, lo, hi, cont, res, seed=20260101 + rank)
    deltas = np.ascontiguousarray(scenes.pr2_mprim_deltas())
    pid = (np.arange(n) % len(deltas)).astype(np.uint8)
    q1 = np.ascontiguousarray(q + deltas[pid])
    return res, coords, q, pid, deltas, q1


def sweep_config(n, units_per_step):
    return {"workload": WORKLOAD, "states_per_step_per_gpu": int(n), "edges_per_step_per_gpu": int(n),
            "validated_states_per_step_per_gpu": int(units_per_step),
            "input": "uniformly random lattice states (1 deg, coordToState); edge i = state i + primitive i mod 22",
            "l2_policy": "inputs (%.0f MB/step as doubles) exceed the 126 MB L2; the 2 MB distance field is L2-resident by design"
                         % ((3 * n * 7 * 8) / 1e6)}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU collision checker (oracle/_ref/libref_collision.so; the oracle port
    when that was not built) on all host threads, one CollisionSpace per thread."""
    if rank != 0:
        return
    from smpl_b200 import scenes
    scene = scenes.pr2_clutter_scene()
    o = make_oracle(scene, np.zeros(scene.dof))
    o.init_kdl(scene.chain_root, scene.chain_tip, scene.planning_link, scene.T_kin_to_planning)
    lo, hi, cont = o.joint_limits()
    n = args.ref_sample if args.ref_sample > 0 else args.states     # default: the GPU arm's step (same config)
    threads = os.cpu_count() or 1
    _, _, q, _, _, q1 = sweep_inputs(lo, hi, cont, n, 0)
    q0 = q
    made = [make_cpu_checker(scene, q[0]) for _ in range(threads)]
    checkers, kind, what = [m[0] for m in made], made[0][1], made[0][2]
    for _ in range(args.warmup):
        cpu_validity_rate(scene, q[: n // 8], q0[: n // 8], q1[: n // 8], threads, checkers)
    total_units, total_t = 0, 0.0
    steps_run = args.steps
    for _ in range(steps_run):
        _, u, dt = cpu_validity_rate(scene, q, q0, q1, threads, checkers)
        total_units += u
        total_t += dt
    value = total_units / total_t
    units_per_step = total_units // steps_run
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / steps_run,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": sweep_config(n, units_per_step),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "steps_timed": steps_run,
                         "sample": "%d states + %d edges per step on %d threads, %s; Eigen arithmetic is the stand-in "
                                   "oracle/ref_stubs/eigen_arith (real Eigen is absent here)" % (n, n, threads, what)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def wandering_paths(anchors, n_paths, dof, seed):
    """Joint-space paths for the shortcut leg: random walks of small steps, jittered straight lines and detours
    between valid states (20 to 60 points), the shapes tests/test_gpu_postprocessing.py checks against the oracle."""
    rng = np.random.default_rng(seed)
    paths = []
    for p in range(n_paths):
        m = int(rng.integers(20, 61))
        a, b = anchors[rng.integers(0, len(anchors), 2)]
        if p % 3 == 0:
            pts = a + np.cumsum(rng.normal(0.0, 0.06, (m, dof)), axis=0)
        elif p % 3 == 1:
            pts = a + np.linspace(0.0, 1.0, m)[:, None] * (b - a) * 0.5 + rng.normal(0.0, 0.02, (m, dof))
        else:
            t = np.concatenate([np.linspace(0, 1, m // 2 + 1), np.linspace(1, 0.2, m - m // 2 - 1)])[:, None]
            pts = a + t * (b - a) * 0.4
        paths.append(np.ascontiguousarray(pts[:m]))
    return paths


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each equal-length device array as out_dir/<name>.npy in float32 (verdicts and waypoint counts are
    exact in it).  Above DUMP_BYTES in all, every array keeps the same elements: a sorted sample drawn with seed 0,
    so that two builds run with the same arguments still compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.cpu().numpy() for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    room = (DUMP_BYTES - 128 * len(host)) // (4 * len(host))     # elements per array, 128-byte .npy headers included
    if n > room:
        idx = np.sort(np.random.default_rng(0).choice(n, room, replace=False))
        host = {k: v[idx] for k, v in host.items()}
    for k, v in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.astype(np.float32))


def timed_events(torch, fn, reps):
    """mean milliseconds of fn() over reps calls, CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def plan_leg(api, scenes, sharding, dist, torch, dev, scene, starts_all, goals_all, params, args, rank, world, local_rank,
             barrier, label, attach=None):
    """Planning queries sharded round-robin over the ranks (no collective); -> (dict, results of this rank, contexts'
    scene objects for the CPU comparison)."""
    pctx, ptables = setup_shared_scene(scene, local_rank, rank, world, dev)
    if attach is not None:
        # AttachedBodiesCollisionModel::generateSpheresModel on the device voxeliser (smplhost_tables_attach_box)
        ptables.attach_box(pctx, *attach)
        ptables.apply(pctx)
    nq_total = len(starts_all)
    mine = sharding.round_robin_shard(nq_total, rank, world)
    cores = os.cpu_count() or 1
    # planner threads (= contexts) per GPU: host work per query is light since the lattices moved to the device, and
    # more contexts mean more and smaller rounds (measured on one B200, 2048 queries: 4 threads 1810-1930 q/s, 6: 1940-2000,
    # 8: 1610, 12: 1470); the 8-GPU box has 4 cores per GPU
    n_thr = args.plan_threads if args.plan_threads > 0 else max(1, min(6, int(0.75 * cores / max(1, world))))
    n_thr = max(n_thr, (args.plan_concurrent + 511) // 512)
    pctxs = [pctx] + [api.clone_context(pctx, scene, ptables, device=local_rank) for _ in range(n_thr - 1)]
    per_ctx = max(1, (min(args.plan_concurrent, max(1, len(mine))) + n_thr - 1) // n_thr)
    # warm-up = the same call on the first batch of queries, with the SAME expansion bound: the lattices and the BFS bank
    # are scene-level allocations sized by (concurrent queries, expansion bound) and kept across calls; a warm-up with a
    # smaller bound made the timed call re-allocate ~5 GB per context (0.1 to 1.2 s of its "setup", run to run)
    wq = min(len(mine), per_ctx * n_thr)
    api.plan_batch(pctxs, scene, ptables, params, starts_all[mine][:wq], goals_all[mine][:wq], max_concurrent=per_ctx)
    barrier()
    psampler = ClockSampler(local_rank)
    if rank == 0:
        psampler.start()
    t0 = time.perf_counter()
    pres, pstats = api.plan_batch(pctxs, scene, ptables, params, starts_all[mine], goals_all[mine], max_concurrent=per_ctx)
    dt = time.perf_counter() - t0
    pclocks = psampler.stop() if rank == 0 else None
    pstats["planner_threads"] = n_thr
    t_plan = torch.tensor([dt], device=dev, dtype=torch.float64)
    n_exp = torch.tensor([float(sum(r["expansions"] for r in pres)), float(sum(r["success"] for r in pres))],
                         device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_plan, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_exp, op=dist.ReduceOp.SUM)
    secs = float(t_plan.item())
    plan = {"scene": label, "queries": nq_total, "solved": int(n_exp[1].item()), "expansions": int(n_exp[0].item()),
            "seconds": secs, "queries_per_s": nq_total / secs, "expansions_per_s": float(n_exp[0].item()) / secs,
            "concurrent_per_gpu": args.plan_concurrent, "planner_threads_per_gpu": n_thr, "rank0": pstats, "clocks": pclocks}
    for c in pctxs:
        c.close()
    return plan, pres


def plan_cpu_compare(plan, scene, starts_all, goals_all, params, pres, k, world, attach=None):
    """The reference's own ManipLattice + BfsHeuristic + ARAStar + CollisionSpace (oracle/ref_planner_shim.cpp) on the
    first k queries, 1 thread, with the parity count of this rank's results."""
    po = make_oracle(scene, np.zeros(scene.dof), attach)
    po.init_kdl(scene.chain_root, scene.chain_tip, scene.planning_link, scene.T_kin_to_planning, scene.xyz_offset)
    pref = make_reference_checker(scene, np.zeros(scene.dof), attach)
    k = min(k, len(starts_all))
    secs, cexp, same = 0.0, 0, 0
    for qi, (s_, g_) in enumerate(zip(starts_all[:k], goals_all[:k])):
        po.heur_init(scene.inflation_radius, scene.cost_per_cell)
        t0 = time.perf_counter()
        pr = pref.plan(scene, s_, g_, params) if pref is not None else po.plan(s_, g_, params)
        secs += time.perf_counter() - t0      # includes the per-query BFS, as the GPU figure does
        cexp += pr["expansions"]
        if world == 1 or qi % world == 0:     # rank 0 planned queries 0, world, 2 world, ...
            gr = pres[qi // world]
            same += int((gr["success"], gr["expansions"], gr["cost"]) == (pr["success"], pr["expansions"], pr["cost"])
                        and np.array_equal(gr["path_ids"], pr["path_ids"]))
        else:
            same += 1
    plan["parity_checked_queries"] = k
    plan["parity_identical"] = same
    plan["cpu_queries_per_s"] = k / secs
    plan["cpu_expansions_per_s"] = cexp / secs
    plan["cpu_kind"] = "reference" if pref is not None else "port"
    plan["cpu_sample"] = "first %d queries, %s, 1 thread" % (
        k, "the reference's own ManipLattice + BfsHeuristic + ARAStar + CollisionSpace (oracle/_ref/libref_collision.so; "
           "RobotModel and action-space plug-ins from the oracle)" if pref is not None else "oracle ManipLattice + ARA*")


def dropin_leg(api, scenes, local_rank):
    """north_star's acceptance test: the REFERENCE's own ManipLattice + ARAStar (compiled from /root/reference into
    oracle/_ref/libref_dropin.so, the caller -- not the thing measured) plan over the product's plug-ins, unchanged,
    one virtual call per question; the adapters answer from one smplgpu_expand_state launch per expansion.  Beside it
    the all-reference run (its own CollisionSpace + BfsHeuristic + BFS_3D on one host thread) on the same queries."""
    import ctypes as C
    lib_path = os.path.join(ROOT, "oracle", "_ref", "libref_dropin.so")
    if not os.path.exists(lib_path):
        return None
    from test_gpu_dropin import dropin_plan
    lib = C.CDLL(lib_path)
    scene = scenes.pr2_tabletop_scene()
    params = scenes.PlanParams(scene.dof)
    params.max_expansions = 2000
    starts, goals = scenes.tabletop_queries(8, seed=3)
    ctx, tables = api.setup_context(scene, device=local_rank)
    try:
        dropin_plan(lib, ctx, scene, starts[0], goals[0], params, batched=2)      # warm-up
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        got, cache_launches = [], 0
        for s_, g_ in zip(starts, goals):
            got.append(dropin_plan(lib, ctx, scene, s_, g_, params, batched=2))
            cache_launches += dropin_plan.last_batched[0]
        secs = time.perf_counter() - t0
        launches = ctx.launch_count() - l0
        # the same queries through the reference's LAZY successors (GetLazySuccs / GetTrueCost under its LazyARAStar)
        lazy = None
        if hasattr(lib, "refdrop_plan_lazy"):
            dropin_plan(lib, ctx, scene, starts[1], goals[1], params, batched=2, lazy=True)
            l1 = ctx.launch_count()
            t1 = time.perf_counter()
            lgot, evals = [], 0
            for s_, g_ in zip(starts, goals):
                lgot.append(dropin_plan(lib, ctx, scene, s_, g_, params, batched=2, lazy=True))
                evals += dropin_plan.last_evaluations
            lazy = {"seconds": time.perf_counter() - t1, "launches": int(ctx.launch_count() - l1),
                    "expansions": sum(g[1] for g in lgot), "evaluations": int(evals), "_got": lgot}
    finally:
        ctx.close()
    expansions = sum(g[1] for g in got)
    out = {"queries": len(got), "expansions": expansions, "seconds": secs, "expansions_per_s": expansions / secs,
           "queries_per_s": len(got) / secs, "launches": int(launches), "launches_per_expansion": launches / max(1, expansions),
           "caller": "the reference's ManipLattice::GetSuccs + ARAStar, unchanged (oracle/_ref/libref_dropin.so)",
           "_got": got, "_scene": scene, "_params": params, "_starts": starts, "_goals": goals}
    if lazy is not None:
        out["lazy"] = lazy
    return out


def dropin_cpu_compare(drop):
    scene, params = drop.pop("_scene"), drop.pop("_params")
    starts, goals, got = drop.pop("_starts"), drop.pop("_goals"), drop.pop("_got")
    pref = make_reference_checker(scene, np.zeros(scene.dof))
    if pref is None:
        return
    t0 = time.perf_counter()
    same, cexp = 0, 0
    for s_, g_, g in zip(starts, goals, got):
        pr = pref.plan(scene, s_, g_, params)
        cexp += pr["expansions"]
        same += int([int(pr["success"]), int(pr["expansions"]), int(pr["cost"]), int(pr["num_states"]),
                     [int(i) for i in pr["path_ids"]]] == g)
    secs = time.perf_counter() - t0
    drop["cpu_seconds"] = secs
    drop["cpu_expansions_per_s"] = cexp / secs
    drop["identical_plans"] = same
    drop["cpu_sample"] = "the same %d queries through the reference's own CollisionSpace + BfsHeuristic + BFS_3D, 1 thread" % len(got)
    lazy = drop.get("lazy")
    if lazy is not None:
        lgot = lazy.pop("_got")
        t0 = time.perf_counter()
        same = 0
        for s_, g_, g in zip(starts, goals, lgot):
            pr = pref.plan(scene, s_, g_, params, lazy=True)
            same += int([int(pr["success"]), int(pr["expansions"]), int(pr["cost"]), int(pr["num_states"]),
                         [int(i) for i in pr["path_ids"]]] == g)
        lazy["cpu_seconds"] = time.perf_counter() - t0
        lazy["identical_plans"] = same


def dual_arm_leg(api, scenes, sharding, dist, torch, dev, args, rank, world, local_rank, barrier, stream):
    """BASELINE config[4] at the validity level (the reference's only RobotModel on this path refuses two chains,
    kdl_robot_model.cpp:96-108, so there is no reference lattice to plan on): PR2 torso + both arms (15-DOF), 3 x 3 x 2 m
    dense shelf at 1 cm = 300 x 300 x 200 cells; the 36 MB field is built on rank 0 and broadcast device to device."""
    scene = scenes.pr2_dual_arm_scene()
    timing = {}
    ctx, tables = setup_shared_scene(scene, local_rank, rank, world, dev, timing)
    ctx.set_stream(stream.cuda_stream)
    lo, hi, cont = tables.limits()
    n = args.dual_states
    q = scenes.random_states(n, lo, hi, cont, seed=4040 + rank)
    prm = scenes.PlanParams(scene.dof)
    deltas = np.concatenate([prm.mprims, -prm.mprims])
    q0, q1 = scenes.mprim_edges(q, deltas)
    d_q0, d_q1 = torch.from_numpy(q0).to(dev), torch.from_numpy(q1).to(dev)
    d_v = torch.empty(n, dtype=torch.uint8, device=dev)
    d_ev = torch.empty(n, dtype=torch.uint8, device=dev)
    d_cnt = torch.empty(n, dtype=torch.int32, device=dev)

    def step():
        ctx.is_states_valid_dev(d_q0.data_ptr(), n, d_v.data_ptr())
        ctx.is_edges_valid_dev(d_q0.data_ptr(), d_q1.data_ptr(), n, d_ev.data_ptr(), d_cnt.data_ptr())

    for _ in range(3):
        step()
    barrier()
    ms_plain = timed_events(torch, step, 5)
    stats = ctx.last_validity_stats()
    resolved = ctx.last_f64_resolved()
    units = n + int(d_cnt.sum().item())
    ms_l2, set_aside = None, 0.0
    try:
        set_aside = ctx.set_distance_field_l2_persistence(True)
        for _ in range(2):
            step()
        ms_l2 = timed_events(torch, step, 5)
        ctx.set_distance_field_l2_persistence(False)
    except api.SmplGpuError as e:
        sys.stderr.write("[bench] L2 persistence window unavailable: %s\n" % e)
    best = min(ms_plain, ms_l2) if ms_l2 else ms_plain
    t = torch.tensor([best], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cert_in_use, e_pos, eps_cells = ctx.certified_bounds()
    out = {"scene": "PR2 torso + both arms (15-DOF), 300x300x200 field @ 1 cm (36 MB), dense shelf", "states_per_gpu": n,
           "edges_per_gpu": n, "validated_states_per_gpu": units, "ms_per_step": float(t.item()),
           "states_per_s": world * units / (float(t.item()) * 1e-3), "ms_default_l2": ms_plain, "ms_l2_window": ms_l2,
           "l2_set_aside_mb": set_aside, "field_build_ms": timing.get("build_ms"), "broadcast_ms": timing.get("broadcast_ms"),
           "broadcast_bytes": timing.get("broadcast_bytes"),
           "broadcast_gbs": (timing["broadcast_bytes"] / (timing["broadcast_ms"] * 1e-3) / 1e9) if timing.get("broadcast_ms") else None,
           "lookups_per_checked_state": stats["df_lookups"] / max(1, stats["waypoints"]),
           "pair_tests_per_checked_state": stats["pair_tests"] / max(1, stats["waypoints"]),
           "f64_resolved_edge_fraction": resolved / n, "certified_f32": bool(cert_in_use), "valid_fraction_states": float(d_v.float().mean().item()),
           "_scene": scene, "_q0": q0, "_q1": q1, "_v": d_v.cpu().numpy(), "_ev": d_ev.cpu().numpy(), "_cnt": d_cnt.cpu().numpy()}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the validity sweep (the value); the e2e legs time max(3, steps // 2) steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="smpl_b200", choices=["smpl_b200", "reference"])
    ap.add_argument("--states", type=int, default=1 << 20, help="states (and edges) per step per GPU")
    ap.add_argument("--bfs-n", type=int, default=400)
    ap.add_argument("--cpu-sample", type=int, default=1 << 19, help="states (and edges) timed on the CPU oracle")
    ap.add_argument("--ref-sample", type=int, default=0, help="--impl reference: states (and edges) per step; 0 = --states")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--plan-queries", type=int, default=2048, help="planning queries per GPU (0 = skip)")
    ap.add_argument("--plan-concurrent", type=int, default=2048, help="queries in flight per GPU (one BFS grid each)")
    ap.add_argument("--plan-max-expansions", type=int, default=2000)
    ap.add_argument("--plan-cpu-queries", type=int, default=12)
    ap.add_argument("--ubr1-queries", type=int, default=4096, help="config[3]: UBR1 + attached object queries in TOTAL, sharded over the ranks (0 = skip)")
    ap.add_argument("--ubr1-max-expansions", type=int, default=1000)
    ap.add_argument("--dual-states", type=int, default=1 << 18, help="config[4]: 15-DOF states (and edges) per GPU (0 = skip)")
    ap.add_argument("--no-dropin", dest="dropin", action="store_false", help="skip the unchanged-caller leg")
    ap.add_argument("--post-paths", type=int, default=1024, help="joint-space paths shortcut in one call (0 = skip)")
    ap.add_argument("--post-cpu-paths", type=int, default=48)
    ap.add_argument("--no-ingest", dest="ingest", action="store_false", help="skip the scene-ingest leg")
    ap.add_argument("--e2e-threads", type=int, default=0, help="host threads (= contexts) of the end-to-end leg; 0 = min(8, cores per rank)")
    ap.add_argument("--plan-threads", type=int, default=0, help="planner threads (= contexts) per GPU; 0 = 75 %% of the rank's cores, at most 6")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the verdicts and waypoint counts of the last timed step to DIR/<name>.npy (float32); with "
                         "several ranks, rank 0's (each rank sweeps its own seeded batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "smpl_b200":
        ap.error("--dump-outputs writes the outputs of --impl smpl_b200")
    args.warmup = max(args.warmup, 3) if args.impl == "smpl_b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes as C

    import torch
    import torch.distributed as dist
    from smpl_b200 import api, scenes, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # ---- scene: rank 0 builds the distance field on its GPU, then ONE broadcast over NCCL ----
    scene = scenes.pr2_clutter_scene()
    with StdoutToStderr():
        if world > 1:
            dist.init_process_group("nccl", device_id=dev)
        ctx, tables = setup_shared_scene(scene, local_rank, rank, world, dev)
        if world > 1:
            dist.barrier()
    # time on ONE explicit stream shared by torch (events) and the library (kernels, copies)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    lo, hi, cont = tables.limits()

    n = args.states
    dof = scene.dof
    res, coords, q, pid8, deltas, q1 = sweep_inputs(lo, hi, cont, n, rank)
    q0 = q
    ctx.set_lattice(res)

    # ---- resident inputs (value) ----
    d_q = torch.from_numpy(q).to(dev)
    d_q1 = torch.from_numpy(q1).to(dev)
    d_v = torch.empty(n, dtype=torch.uint8, device=dev)
    d_ev = torch.empty(n, dtype=torch.uint8, device=dev)
    d_cnt = torch.empty(n, dtype=torch.int32, device=dev)

    def step_resident():
        ctx.is_states_valid_dev(d_q.data_ptr(), n, d_v.data_ptr())
        ctx.is_edges_valid_dev(d_q.data_ptr(), d_q1.data_ptr(), n, d_ev.data_ptr(), d_cnt.data_ptr())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident()
    barrier()
    units_per_step = n + int(d_cnt.sum().item())
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    barrier()
    ev[0].record()
    for s in range(args.steps):
        ctx.is_states_valid_dev(d_q.data_ptr(), n, d_v.data_ptr())
        ev[2 * s + 1].record()
        ctx.is_edges_valid_dev(d_q.data_ptr(), d_q1.data_ptr(), n, d_ev.data_ptr(), d_cnt.data_ptr())
        ev[2 * s + 2].record()
    barrier()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"states_valid": d_v, "edges_valid": d_ev, "edges_waypoint_count": d_cnt})
    gpu_launches = ctx.launch_count() - launches0
    total_ms = ev[0].elapsed_time(ev[-1])
    states_ms = np.mean([ev[2 * s].elapsed_time(ev[2 * s + 1]) for s in range(args.steps)])
    edges_ms = np.mean([ev[2 * s + 1].elapsed_time(ev[2 * s + 2]) for s in range(args.steps)])
    t_ms = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    total_ms_max = float(t_ms.item())
    gpu_stats = ctx.last_validity_stats()       # of the last launch (the edges)
    gpu_stats["f64_resolved_edges_last_launch"] = ctx.last_f64_resolved()
    cert_in_use, e_pos, eps_cells = ctx.certified_bounds()
    gpu_stats["certified_f32"] = {"in_use": cert_in_use, "e_pos_m": e_pos, "eps_cells": eps_cells}
    df_lookup_peak = ctx.probe_df_lookup_rate() if rank == 0 else None   # independent random lookups/s on this field

    # ---- end to end through the C ABI with HOST buffers (pinned), copies inside the timed region ----
    # lattice states on the wire as the real caller holds them: 16-bit RobotCoord + one primitive byte per edge
    hc = torch.from_numpy(coords).pin_memory()
    hp = torch.from_numpy(pid8).pin_memory()
    hv = torch.empty(n, dtype=torch.uint8).pin_memory()
    hev = torch.empty(n, dtype=torch.uint8).pin_memory()
    L = ctx.L
    c_i16_p = C.POINTER(C.c_int16)
    deltas_p = deltas.ctypes.data_as(api.c_double_p)

    def step_e2e():
        r = L.smplgpu_is_lattice_states_valid(ctx.h, C.cast(hc.data_ptr(), c_i16_p), n, C.cast(hv.data_ptr(), api.c_uint8_p))
        r |= L.smplgpu_is_lattice_edges_valid(ctx.h, C.cast(hc.data_ptr(), c_i16_p), C.cast(hp.data_ptr(), api.c_uint8_p), n,
                                              deltas_p, len(deltas), C.cast(hev.data_ptr(), api.c_uint8_p), None)
        if r != 0:
            raise RuntimeError(L.smplgpu_last_error(ctx.h).decode())

    # the same step with the states as doubles (arbitrary, off-lattice states take this path)
    hq = torch.from_numpy(q).pin_memory()
    hpid = torch.from_numpy(pid8.astype(np.int32)).pin_memory()
    hv2 = torch.empty(n, dtype=torch.uint8).pin_memory()
    hev2 = torch.empty(n, dtype=torch.uint8).pin_memory()

    def step_e2e_f64():
        r = L.smplgpu_is_states_valid(ctx.h, C.cast(hq.data_ptr(), api.c_double_p), n, C.cast(hv2.data_ptr(), api.c_uint8_p))
        r |= L.smplgpu_is_mprim_edges_valid(ctx.h, C.cast(hq.data_ptr(), api.c_double_p), C.cast(hpid.data_ptr(), api.c_int32_p),
                                            n, deltas_p, len(deltas), C.cast(hev2.data_ptr(), api.c_uint8_p), None)
        if r != 0:
            raise RuntimeError(L.smplgpu_last_error(ctx.h).decode())

    def time_e2e(fn, steps):
        for _ in range(2):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * units_per_step * steps / (float(t.item()) * 1e-3)

    e2e_steps = max(3, args.steps // 2)
    e2e_single = time_e2e(step_e2e, e2e_steps)
    e2e_f64_value = time_e2e(step_e2e_f64, max(3, e2e_steps // 2))
    assert torch.equal(hv.to(dev), d_v) and torch.equal(hev.to(dev), d_ev), "host-buffer (lattice) path disagrees with resident path"
    assert torch.equal(hv2.to(dev), d_v) and torch.equal(hev2.to(dev), d_ev), "host-buffer (double) path disagrees with resident path"

    # The headline e2e: the same step issued the way the reference is used at scale -- K host threads, one context each
    # (its CollisionSpace is one-per-thread too; `--impl reference` runs one per host thread), thread k validating the
    # k-th share of the step's states and edges from the same pinned buffers.  The callers' copies and kernels overlap.
    # Timed by the host clock between a barrier in front of the K synchronous callers and the join behind them.
    e2e_threads = args.e2e_threads if args.e2e_threads > 0 else max(1, min(8, (os.cpu_count() or 1) // max(1, world)))
    hv.zero_()
    hev.zero_()
    ectxs = [ctx] + [api.clone_context(ctx, scene, tables, device=local_rank) for _ in range(e2e_threads - 1)]
    for c in ectxs[1:]:
        c.set_lattice(res)
    bounds = np.linspace(0, n, e2e_threads + 1).astype(np.int64)
    gate = threading.Barrier(e2e_threads + 1)
    e2e_errors = []

    def e2e_worker(k):
        try:
            c = ectxs[k]
            L.smplgpu_bind_thread(c.h)
            b, e = int(bounds[k]), int(bounds[k + 1])
            pc = C.cast(hc.data_ptr() + b * dof * 2, c_i16_p)
            pp = C.cast(hp.data_ptr() + b, api.c_uint8_p)
            pv = C.cast(hv.data_ptr() + b, api.c_uint8_p)
            pe = C.cast(hev.data_ptr() + b, api.c_uint8_p)
            for it in range(e2e_steps + 2):
                if it == 2:
                    gate.wait(timeout=300)
                r = L.smplgpu_is_lattice_states_valid(c.h, pc, e - b, pv)
                r |= L.smplgpu_is_lattice_edges_valid(c.h, pc, pp, e - b, deltas_p, len(deltas), pe, None)
                if r != 0:
                    raise RuntimeError(L.smplgpu_last_error(c.h).decode())
        except Exception as ex:   # a failing caller must not leave the others (or the main thread) at the barrier
            e2e_errors.append(repr(ex))
            gate.abort()

    workers = [threading.Thread(target=e2e_worker, args=(k,)) for k in range(e2e_threads)]
    for w in workers:
        w.start()
    barrier()
    try:
        gate.wait(timeout=300)
    except threading.BrokenBarrierError:
        pass
    t0 = time.perf_counter()
    for w in workers:
        w.join()
    e2e_wall = time.perf_counter() - t0
    if e2e_errors:
        raise RuntimeError(e2e_errors[0])
    t_e2e = torch.tensor([e2e_wall], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = world * units_per_step * e2e_steps / float(t_e2e.item())
    for c in ectxs[1:]:
        c.close()
    L.smplgpu_bind_thread(ctx.h)
    assert torch.equal(hv.to(dev), d_v) and torch.equal(hev.to(dev), d_ev), "multi-context host-buffer path disagrees with resident path"
    verdict_s, verdict_e, counts_e = hv.numpy().copy(), hev.numpy().copy(), d_cnt.cpu().numpy()

    # ---- BFS (config[2]): 400^3 cluttered occupancy (+ the planner's 150^3 size), rank 0 only ----
    bfs = None
    if rank == 0 and args.bfs_n > 0:
        def bfs_time(nb):
            walls = scenes.bfs_clutter_walls(nb, seed=11)
            seed = scenes.first_free_cell(walls, (nb // 2, nb // 2, nb // 2))
            ctx.bfs_set_walls(walls)
            for _ in range(2):
                ctx.bfs_run([seed])
            return timed_events(torch, lambda: ctx.bfs_run([seed]), 5), ctx.bfs_last_levels()
        nb = args.bfs_n
        ms150, lv150 = bfs_time(150) if nb != 150 else (None, None)
        bfs_ms, levels = bfs_time(nb)
        alg_bytes = (nb + 2) ** 3 * (1.0 / 8 + 4)
        bfs = {"grid": "%d^3" % nb, "levels": levels, "ms": bfs_ms,
               "mvoxel_s": nb ** 3 / (bfs_ms * 1e-3) / 1e6,
               "algorithmic_bytes": alg_bytes, "achieved_gbs": alg_bytes / (bfs_ms * 1e-3) / 1e9,
               "ms_150": ms150, "levels_150": lv150}

    # ---- path post-processing (SURVEY 8f row 4): shortcut many paths with ONE batch of candidate motions ----
    post = None
    post_paths = None
    if rank == 0 and args.post_paths > 0:
        post_paths = wandering_paths(q[d_v.cpu().numpy().astype(bool)], args.post_paths, dof, seed=5)
        api.shortcut_paths(ctx, tables, post_paths, kind=0)     # warm-up at full size (buffers, lazily loaded kernels)
        t0 = time.perf_counter()
        short, pst = api.shortcut_paths(ctx, tables, post_paths, kind=0)
        dt = time.perf_counter() - t0
        post = {"paths": len(post_paths), "points": int(sum(len(p) for p in post_paths)),
                "points_after": int(sum(len(g) for g in short)), "candidate_motions": pst["edges_checked"],
                "seconds": dt, "device_seconds": pst["device_seconds"], "paths_per_s": len(post_paths) / dt,
                "call": "smplhost_shortcut_paths (ShortcutPath JOINT_SPACE): all point pairs of every path in one "
                        "smplgpu_is_indexed_edges_valid call", "_short": short}

    # ---- scene ingest (SURVEY 8f row 3): box objects -> surface voxels -> distance field, all on the device ----
    ingest = None
    if rank == 0 and args.ingest:
        iscene = scenes.pr2_shelf_objects_scene()
        ictx = api.GpuContext(local_rank)
        itables = api.build_tables(iscene)
        ictx.set_robot(itables)
        icells = api.scene_cells(iscene, itables)
        iv, it = api.box_meshes(iscene.boxes)
        for _ in range(2):
            ictx.build_distance_field_from_meshes(iv, it, icells, iscene.dims, iscene.origin, iscene.res, iscene.max_dist)
        t0 = time.perf_counter()
        reps = 10
        for _ in range(reps):
            ictx.build_distance_field_from_meshes(iv, it, icells, iscene.dims, iscene.origin, iscene.res, iscene.max_dist)
        dt = (time.perf_counter() - t0) / reps
        d2 = ictx.download_distance_field()
        ingest = {"scene": "34 box objects (12 triangles each, arbitrary poses) in 2 m^3 @ 2 cm", "triangles": int(len(it)),
                  "grid_cells": int(d2.size), "occupied_cells": int((d2 == 0).sum()), "ms": dt * 1e3,
                  "call": "smplgpu_build_distance_field_from_meshes: voxelise + addPointsToField + distance field, host call to field ready",
                  "_d2": d2, "_scene": iscene}
        ictx.close()

    # ---- the unchanged caller (north_star's acceptance test), rank 0 ----
    drop = None
    if rank == 0 and args.dropin:
        with StdoutToStderr():
            drop = dropin_leg(api, scenes, local_rank)

    clocks = sampler.stop() if rank == 0 else None   # sampled across the validity, end-to-end, BFS, shortcut, ingest, drop-in regions

    # ---- config[4]: 15-DOF validity at 1 cm, field broadcast device to device (all ranks) ----
    dual = None
    if args.dual_states > 0:
        with StdoutToStderr():
            dual = dual_arm_leg(api, scenes, sharding, dist, torch, dev, args, rank, world, local_rank, barrier, stream)

    # ---- plan queries/s (config[0] shape): PR2 right arm on the tabletop scene, queries sharded over ranks ----
    plan, pres = None, None
    if args.plan_queries > 0:
        pscene = scenes.pr2_tabletop_scene()
        pparams = scenes.PlanParams(pscene.dof)
        pparams.max_expansions = args.plan_max_expansions
        starts_all, goals_all = scenes.tabletop_queries(args.plan_queries * world, seed=13)
        with StdoutToStderr():
            plan, pres = plan_leg(api, scenes, sharding, dist, torch, dev, pscene, starts_all, goals_all, pparams, args, rank,
                                  world, local_rank, barrier,
                                  "PR2 right arm, tabletop env, 150^3 field @ 2 cm, ARA* eps 100, first solution, <= %d expansions; "
                                  "%d queries per GPU" % (args.plan_max_expansions, args.plan_queries))

    # ---- config[3]: UBR1 arm + attached object + ACM, 4096 queries in total sharded over the ranks ----
    ubr1, ures = None, None
    if args.ubr1_queries > 0:
        uscene = scenes.ubr1_tabletop_scene()
        # the grasped object goes through attachObject on both sides (device voxeliser here, the reference's own there)
        uscene.attached = None
        uattach = ("object", "wrist_roll_link", (0.05, 0.05, 0.20),
                   np.array([[1.0, 0.0, 0.0, 0.26], [0.0, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.0]]))
        uparams = scenes.PlanParams(uscene.dof)
        uparams.max_expansions = args.ubr1_max_expansions
        ustarts, ugoals = scenes.ubr1_tabletop_queries(args.ubr1_queries, seed=13)
        with StdoutToStderr():
            ubr1, ures = plan_leg(api, scenes, sharding, dist, torch, dev, uscene, ustarts, ugoals, uparams, args, rank, world,
                                  local_rank, barrier,
                                  "config[3]: UBR1 arm + attached 5x5x20 cm object + self-collision ACM, tabletop_ubr1 env, 100^3 field @ "
                                  "2 cm, <= %d expansions; %d queries in TOTAL over the ranks" % (args.ubr1_max_expansions, args.ubr1_queries),
                                  attach=uattach)
            ubr1["scaling"] = "strong (fixed total)"

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU legs + roofline of the dominant kernel (rank 0) ----
    peak, peak_src = load_peaks()
    cpu = None
    Lbar_state, Lbar_edge = None, None
    if not args.no_cpu:
        m = min(args.cpu_sample, n)
        o = make_oracle(scene, q[0])
        checker, cpu_kind, cpu_what = make_cpu_checker(scene, q[0])
        t_s, v_s = checker.time_states_valid(q[:m])
        t_e, v_e, c = checker.time_edges_valid(q0[:m], q1[:m])
        cpu_units = m + int(c.sum())
        cpu_rate = cpu_units / (t_s + t_e)
        cpu_agree = {"states_differing": int((v_s != verdict_s[:m]).sum()), "edges_differing": int((v_e != verdict_e[:m]).sum()),
                     "waypoint_counts_differing": int((c != counts_e[:m]).sum()), "of": m}
        # L-bar: DF lookups the reference semantics requires (no early-out), from the oracle on a sub-sample
        ms = min(m, 1 << 15)
        _, Ls, _, _ = o.report_states(q[:ms])
        _, _, Le = o.report_edges(q0[:ms], q1[:ms])
        Lbar_state, Lbar_edge = float(Ls.mean()), float(Le.mean())
        cpu = {"value": cpu_rate, "unit": UNIT, "cores": 1, "kind": cpu_kind,
               "sample": "%d states + %d edges of the same workload, 1 thread, %s (stand-in Eigen arithmetic); "
                         "states %.0f/s, edge waypoints %.0f/s" % (m, m, cpu_what, m / t_s, int(c.sum()) / t_e),
               "device_verdicts_differing": cpu_agree["states_differing"] + cpu_agree["edges_differing"] + cpu_agree["waypoint_counts_differing"],
               "device_verdicts_checked": 2 * m,
               "device_verdicts_vs_this_run": cpu_agree}
        if plan is not None and args.plan_cpu_queries > 0:
            plan_cpu_compare(plan, pscene, starts_all, goals_all, pparams, pres, args.plan_cpu_queries, world)
        if ubr1 is not None and args.plan_cpu_queries > 0:
            plan_cpu_compare(ubr1, uscene, ustarts, ugoals, uparams, ures, max(4, args.plan_cpu_queries // 2), world, uattach)
        if drop is not None:
            dropin_cpu_compare(drop)
        if dual is not None:
            dsc = dual["_scene"]
            # the oracle port: the reference's 48-byte cells make this 18 M-cell grid a gigabyte
            dchk, dkind = make_oracle(dsc, dual["_q0"][0]), "port"
            k = min(32768, len(dual["_q0"]))
            t_s, v_s = dchk.time_states_valid(dual["_q0"][:k])
            t_e, v_e, c = dchk.time_edges_valid(dual["_q0"][:k], dual["_q1"][:k])
            dual["cpu_states_per_s"] = (k + int(c.sum())) / (t_s + t_e)
            dual["cpu_kind"] = dkind
            dual["cpu_sample"] = "first %d states + edges, 1 thread" % k
            dual["device_verdicts_differing"] = int((v_s != dual["_v"][:k]).sum() + (v_e != dual["_ev"][:k]).sum() + (c != dual["_cnt"][:k]).sum())
        if post is not None:
            k = min(args.post_cpu_paths, len(post_paths))
            t0 = time.perf_counter()
            same = 0
            # the reference's own ShortcutPath (post_processing.cpp over its CollisionSpace) when its build is there
            if cpu_kind == "reference":
                for p_, g_ in zip(post_paths[:k], post["_short"][:k]):
                    same += int(np.array_equal(checker.post_process(scene, p_, 0), p_[g_]))
            else:
                for p_, g_ in zip(post_paths[:k], post["_short"][:k]):
                    ref_idx, _ = o.shortcut_path(p_, cont, kind=0)
                    same += int(np.array_equal(ref_idx, g_))
            dt = time.perf_counter() - t0
            post["cpu_paths_per_s"] = k / dt
            post["cpu_kind"] = cpu_kind
            post["cpu_sample"] = "first %d paths, %s ShortcutPath JOINT_SPACE (one isStateToStateValid per request), 1 thread" % (
                k, "the reference's own" if cpu_kind == "reference" else "oracle")
            post["parity_identical"] = "%d / %d" % (same, k)
        if ingest is not None:
            t0 = time.perf_counter()
            io = make_reference_checker(ingest["_scene"], np.zeros(dof))   # WorldCollisionModel::insertObject per box
            ingest_kind = "reference"
            if io is None:
                io = make_oracle(ingest["_scene"], np.zeros(dof))  # VoxelizeBox per object + addPointsToField + propagation
                ingest_kind = "port"
            dt = time.perf_counter() - t0
            ref_d2 = io.df_d2()
            ingest["cpu_ms"] = dt * 1e3
            ingest["cpu_kind"] = ingest_kind
            ingest["cpu_sample"] = "%s: scene construction incl. insertObject (VoxelizeBox + addPointsToField) + DistanceMap propagation, 1 thread" % (
                "the reference's own CollisionSpace + OccupancyGrid" if ingest_kind == "reference" else "oracle")
            ingest["occupied_cells_identical"] = bool(np.array_equal(ref_d2 == 0, ingest["_d2"] == 0))
            ingest["cells_where_reference_propagation_is_inexact"] = int((ref_d2 != ingest["_d2"]).sum())
        if bfs is not None:
            mv, kind, dt = cpu_bfs_rate(args.bfs_n)
            bfs["cpu_mvoxel_s"] = mv
            bfs["cpu_kind"] = kind
            bfs["cpu_seconds"] = dt
    if Lbar_state is None:
        Lbar_state = gpu_stats["df_lookups"] / max(1, gpu_stats["waypoints"])
        Lbar_edge = Lbar_state * (units_per_step - n) / n
    state_bytes = n * (8 * dof + 1 + 32 * Lbar_state)
    edge_bytes = n * (16 * dof + 1 + 32 * Lbar_edge)
    k_states = {"kernel": "states_valid32_kernel (+ f64 resolve pass)", "ms": float(states_ms), "algorithmic_bytes": state_bytes,
                "achieved": state_bytes / (states_ms * 1e-3) / 1e9}
    k_edges = {"kernel": "edges_valid32_kernel (+ f64 resolve pass)", "ms": float(edges_ms), "algorithmic_bytes": edge_bytes,
               "achieved": edge_bytes / (edges_ms * 1e-3) / 1e9}
    dom, other = (k_edges, k_states) if edges_ms >= states_ms else (k_states, k_edges)
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (profiles/), scaled to this
    # launch's item count (the traffic is the streamed inputs; the distance field stays in L2)
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "edges_valid32_kernel" if dom is k_edges else "states_valid32_kernel"
        traffic = tr[key]["dram_bytes"] * n / tr[key]["items"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s",
                "frac": dom["achieved"] / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom["algorithmic_bytes"], "launch_ms": dom["ms"],
                "Lbar_state": Lbar_state, "Lbar_edge": Lbar_edge,
                "note": "issue/latency bound (FK arithmetic + dependent L2 lookups), not HBM bound; L-bar counts lookups "
                        "WITHOUT early-out, see l2_frac / lookups_performed_frac and DESIGN.md",
                "states_ms": float(states_ms), "edges_ms": float(edges_ms),
                "states_frac": k_states["achieved"] / peak, "edges_frac": k_edges["achieved"] / peak,
                "other_kernel": other}
    # SURVEY 8d's two fractions for the dominant kernel: HBM = streamed bytes only; L2 = the lookups the reference
    # semantics requires (one 32-byte sector each) against the measured rate of INDEPENDENT random lookups on the
    # same field (smplgpu_probe_df_lookup_rate): the kernels' lookups are dependent, so this ceiling is not reachable
    if df_lookup_peak:
        Lb, per_item = (Lbar_edge, 16 * dof + 1) if dom is k_edges else (Lbar_state, 8 * dof + 1)
        roofline["hbm_frac_streamed_bytes"] = n * per_item / (dom["ms"] * 1e-3) / 1e9 / peak
        roofline["l2_frac"] = n * Lb / (dom["ms"] * 1e-3) / df_lookup_peak
        roofline["l2_peak_glookups_s"] = df_lookup_peak / 1e9
        roofline["l2_achieved_glookups_s"] = n * Lb / (dom["ms"] * 1e-3) / 1e9
        if dom is k_edges:   # gpu_stats is the last launch = the edges
            roofline["lookups_performed_frac"] = gpu_stats["df_lookups"] / (dom["ms"] * 1e-3) / df_lookup_peak
        roofline["l2"] = {"required_lookups_per_launch": n * Lb, "achieved_glookups_s": n * Lb / (dom["ms"] * 1e-3) / 1e9,
                          "peak_glookups_s": df_lookup_peak / 1e9, "frac": n * Lb / (dom["ms"] * 1e-3) / df_lookup_peak,
                          "achieved_gbs": 32 * n * Lb / (dom["ms"] * 1e-3) / 1e9, "peak_gbs": 32 * df_lookup_peak / 1e9,
                          "peak_source": "measured live: independent random lookups on the loaded field, 8 in flight per thread"}
    if bfs is not None:
        roofline["bfs_frac"] = bfs["achieved_gbs"] / peak
        roofline["bfs_achieved_gbs"] = bfs["achieved_gbs"]
        roofline["bfs_ms"] = bfs["ms"]
        roofline["bfs"] = {"bound": "hbm", "achieved": bfs["achieved_gbs"], "peak": peak, "unit": "GB/s",
                           "frac": bfs["achieved_gbs"] / peak}

    value = world * units_per_step * args.steps / (total_ms_max * 1e-3)
    # the early-out means fewer states are actually evaluated than the unit credits: both rates are printed
    checked_per_step = n + gpu_stats["waypoints"] if dom is k_edges else None
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * (2 * dof * n) + n, "d2h_bytes_per_step": 2 * n,
           "calls": "smplgpu_is_lattice_states_valid + smplgpu_is_lattice_edges_valid: 16-bit RobotCoord (+ 1 primitive byte per edge) in pinned host buffers, verdicts out",
           "host_threads": e2e_threads, "timing": "host clock around K synchronous callers (one context per thread), max over ranks",
           "single_context_value": e2e_single,
           "f64_value": e2e_f64_value, "f64_h2d_bytes_per_step": 2 * n * dof * 8 + 4 * n,
           "f64_calls": "smplgpu_is_states_valid + smplgpu_is_mprim_edges_valid (joint values as doubles)"}
    if checked_per_step:
        e2e["checked_states_per_s"] = world * checked_per_step * args.steps / (total_ms_max * 1e-3)
    if plan is not None:
        e2e.update({"plan_queries_per_s": plan["queries_per_s"], "plan_expansions_per_s": plan["expansions_per_s"],
                    "plan_queries": plan["queries"], "plan_solved": plan["solved"], "plan_seconds": plan["seconds"],
                    "plan_threads_per_gpu": plan["planner_threads_per_gpu"],
                    "plan_parity_identical": plan.get("parity_identical"), "plan_parity_checked": plan.get("parity_checked_queries")})
    if ubr1 is not None:
        e2e.update({"ubr1_queries_per_s": ubr1["queries_per_s"], "ubr1_expansions_per_s": ubr1["expansions_per_s"],
                    "ubr1_queries": ubr1["queries"], "ubr1_solved": ubr1["solved"], "ubr1_seconds": ubr1["seconds"],
                    "ubr1_parity_identical": ubr1.get("parity_identical"), "ubr1_parity_checked": ubr1.get("parity_checked_queries")})
    if drop is not None:
        e2e.update({"dropin_expansions_per_s": drop["expansions_per_s"], "dropin_seconds": drop["seconds"],
                    "dropin_queries": drop["queries"], "dropin_launches_per_expansion": drop["launches_per_expansion"],
                    "dropin_identical_plans": drop.get("identical_plans")})
        if drop.get("lazy"):
            e2e.update({"dropin_lazy_seconds": drop["lazy"]["seconds"], "dropin_lazy_launches": drop["lazy"]["launches"],
                        "dropin_lazy_expansions": drop["lazy"]["expansions"], "dropin_lazy_evaluations": drop["lazy"]["evaluations"],
                        "dropin_lazy_identical_plans": drop["lazy"].get("identical_plans")})
    if dual is not None:
        e2e.update({"dual_arm_states_per_s": dual["states_per_s"], "dual_arm_broadcast_ms": dual["broadcast_ms"],
                    "dual_arm_broadcast_gbs": dual["broadcast_gbs"], "dual_arm_field_build_ms": dual["field_build_ms"],
                    "dual_arm_ms_default_l2": dual["ms_default_l2"], "dual_arm_ms_l2_window": dual["ms_l2_window"],
                    "dual_arm_lookups_per_checked_state": dual["lookups_per_checked_state"],
                    "dual_arm_f64_resolved_edge_fraction": dual["f64_resolved_edge_fraction"],
                    "dual_arm_device_verdicts_differing": dual.get("device_verdicts_differing")})
    if bfs is not None:
        e2e.update({"bfs_mvoxel_s": bfs["mvoxel_s"], "bfs_ms": bfs["ms"], "bfs_levels": bfs["levels"], "bfs_ms_150": bfs["ms_150"]})
    if post is not None:
        e2e["post_paths_per_s"] = post["paths_per_s"]
    if ingest is not None:
        e2e["ingest_ms"] = ingest["ms"]
    if cpu is not None:
        if plan is not None and "cpu_queries_per_s" in plan:
            cpu.update({"plan_queries_per_s": plan["cpu_queries_per_s"], "plan_expansions_per_s": plan["cpu_expansions_per_s"]})
        if ubr1 is not None and "cpu_queries_per_s" in ubr1:
            cpu.update({"ubr1_queries_per_s": ubr1["cpu_queries_per_s"], "ubr1_expansions_per_s": ubr1["cpu_expansions_per_s"]})
        if drop is not None and "cpu_expansions_per_s" in drop:
            cpu.update({"dropin_expansions_per_s": drop["cpu_expansions_per_s"], "dropin_seconds": drop["cpu_seconds"]})
            if drop.get("lazy") and "cpu_seconds" in drop["lazy"]:
                cpu["dropin_lazy_seconds"] = drop["lazy"]["cpu_seconds"]
        if dual is not None and "cpu_states_per_s" in dual:
            cpu["dual_arm_states_per_s"] = dual["cpu_states_per_s"]
        if bfs is not None and "cpu_mvoxel_s" in bfs:
            cpu["bfs_mvoxel_s"] = bfs["cpu_mvoxel_s"]
        if post is not None and "cpu_paths_per_s" in post:
            cpu["post_paths_per_s"] = post["cpu_paths_per_s"]
        if ingest is not None and "cpu_ms" in ingest:
            cpu["ingest_ms"] = ingest["cpu_ms"]
    gpu_stats["valid_fraction_states"] = float(d_v.float().mean().item())
    gpu_stats["valid_fraction_edges"] = float(d_ev.float().mean().item())
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 certified, f64 resolves the undecidable items (verdicts = all-f64)", "data": "synthetic",
        "config": sweep_config(n, units_per_step),
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": int(gpu_launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "bfs": bfs,
        "plan": plan,
        "ubr1_plan": ubr1,
        "dual_arm": dual,
        "dropin": drop,
        "post_processing": post,
        "scene_ingest": ingest,
        "host_cores": os.cpu_count(),
        "gpu_stats_last_launch": gpu_stats,
    }
    if post is not None:
        post.pop("_short", None)
    if ingest is not None:
        ingest.pop("_d2", None)
        ingest.pop("_scene", None)
    if dual is not None:
        for k in ("_scene", "_q0", "_q1", "_v", "_ev", "_cnt"):
            dual.pop(k, None)
    if drop is not None:
        for k in ("_got", "_scene", "_params", "_starts", "_goals"):
            drop.pop(k, None)
        if drop.get("lazy"):
            drop["lazy"].pop("_got", None)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

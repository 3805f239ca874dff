"""Per-kernel time of the certified single-precision validity kernels at bench.py's config[1] sweep.

The inputs of bench.py's value leg (PR2 right arm, clutter scene, 2^20 lattice states and 2^20 primitive edges,
device-resident), on one explicit stream shared with the library:
  * CUDA events around each is_states_valid_dev / is_edges_valid_dev call (the single-precision kernel plus the
    double-precision resolve pass of its undecided items), averaged over --iters calls after --warmup calls;
  * the items each call left to the double-precision pass (smplgpu_last_f64_resolved) and the certified bounds;
  * in a separate run under torch.profiler, the device time per launch of every kernel of those calls.
Prints one JSON line, with the GPU name, power limit and maximum SM clock read in the same run.

    python tools/validity32_time.py [--states 1048576] [--iters 20] [--warmup 3]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import sweep_inputs  # noqa: E402
from goal_types_time import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--states", type=int, default=1 << 20, help="states (and edges) per call")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from smpl_b200 import api, scenes

    if not torch.cuda.is_available():
        raise SystemExit("validity32_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    scene = scenes.pr2_clutter_scene()
    ctx, tables = api.setup_context(scene, device=0)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    lo, hi, cont = tables.limits()
    n = args.states
    _, _, q, _, _, q1 = sweep_inputs(lo, hi, cont, n, 0)
    d_q = torch.from_numpy(q).to(dev)
    d_q1 = torch.from_numpy(q1).to(dev)
    d_v = torch.empty(n, dtype=torch.uint8, device=dev)
    d_ev = torch.empty(n, dtype=torch.uint8, device=dev)
    d_cnt = torch.empty(n, dtype=torch.int32, device=dev)

    def states():
        ctx.is_states_valid_dev(d_q.data_ptr(), n, d_v.data_ptr())

    def edges():
        ctx.is_edges_valid_dev(d_q.data_ptr(), d_q1.data_ptr(), n, d_ev.data_ptr(), d_cnt.data_ptr())

    def time_call(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
        return {"mean_ms": float(np.mean(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}

    out = {"gpu": gpu_info(), "items": n}
    out["states_call"] = time_call(states)
    out["states_f64_resolved"] = int(ctx.last_f64_resolved())
    out["edges_call"] = time_call(edges)
    out["edges_f64_resolved"] = int(ctx.last_f64_resolved())
    in_use, e_pos, eps_cells = ctx.certified_bounds()
    out["certified_f32"] = {"in_use": bool(in_use), "e_pos_m": e_pos, "eps_cells": eps_cells}

    steps = 5
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            states()
            edges()
        torch.cuda.synchronize()
    kernels = {}
    for evt in prof.key_averages():
        t = getattr(evt, "device_time_total", None)
        if t is None:
            t = evt.cuda_time_total
        if t <= 0 or "Memcpy" in evt.key or "Memset" in evt.key:
            continue
        name = evt.key.split("(")[0].replace("smplgpu::", "").replace("void ", "")
        kernels[name] = {"launches": int(evt.count), "us_per_launch": float(t) / evt.count}
    out["kernels_profiled"] = dict(sorted(kernels.items(), key=lambda kv: -kv[1]["us_per_launch"] * kv[1]["launches"]))
    print(json.dumps(out))
    ctx.close()


if __name__ == "__main__":
    main()

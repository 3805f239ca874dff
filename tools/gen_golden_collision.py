#!/usr/bin/env python
"""Writes tests/golden/collision_reference.npz: outputs of the REFERENCE's own collision checker and what regenerates
its inputs (oracle/_ref/libref_collision.so, built by `make -C oracle ref REF=<checkout of the reference sources>`;
see oracle/ref_collision_shim.cpp) for the cases of tests/test_oracle_collision.py.  Needs that build."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import test_oracle_collision as T  # noqa: E402


def main():
    out = {}
    for name in T.CASES:
        scene, attach = T.case_scene(name)
        r = T.make_reference(scene, attach)
        lo, hi, cont = r.limits()
        q, q0, q1 = T.case_inputs(scene, (lo, hi, cont), 1500, 600, seed=211)
        nt = r.node_table()
        e, n = r.is_edges_valid(q0, q1)
        # the inputs are regenerated from the seed (T.golden_inputs); every 50th row is kept to check that
        out[name + "/limits_lo"] = lo
        out[name + "/limits_hi"] = hi
        out[name + "/limits_continuous"] = cont
        out[name + "/q_rows"] = q[::50]
        out[name + "/q1_rows"] = q1[::50]
        out[name + "/node_table"] = nt
        out[name + "/centers"] = r.sphere_centers(q[:64], len(nt))
        out[name + "/states_valid"] = r.is_states_valid(q)
        out[name + "/edges_valid"] = e
        out[name + "/waypoint_counts"] = n
        out[name + "/df_d2_sum"] = np.int64(r.df_d2().astype(np.int64).sum())
        print("%-22s nodes %3d  valid states %.3f  valid edges %.3f  max waypoints %d" %
              (name, len(nt), out[name + "/states_valid"].mean(), e.mean(), n.max()))
    path = os.path.join(ROOT, "tests", "golden", "collision_reference.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

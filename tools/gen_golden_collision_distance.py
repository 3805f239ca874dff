#!/usr/bin/env python3
"""Golden outputs of the REFERENCE's own CollisionSpace::collisionDistance (collision_space.cpp:496-500 ->
self_collision_model.cpp:503-531, 1386-1468), run here from oracle/_ref/libref_collision.so (the reference's sources
compiled where they lie, see oracle/Makefile `ref`).  /root/reference does not travel to the GPU box, these vectors do.

    python tools/gen_golden_collision_distance.py   ->  tests/golden/collision_distance_reference.npz
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_oracle_collision import case_inputs, case_scene, make_reference  # noqa: E402

CASES = ["pr2_tabletop", "pr2_clutter", "pr2_clutter_padded", "ubr1_attached_box", "pr2_dual_arm_15dof"]


def main():
    out = {}
    for name in CASES:
        scene, attach = case_scene(name)
        r = make_reference(scene, attach)
        q, _, _ = case_inputs(scene, r.limits(), 1500, 10, seed=77)
        out[name + "/q"] = q
        out[name + "/distance"] = r.collision_distance(q)
        print(name, "min %.4f max %.4f zero %.2f" % (out[name + "/distance"].min(), out[name + "/distance"].max(),
                                                     (out[name + "/distance"] == 0).mean()))
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "collision_distance_reference.npz"), **out)


if __name__ == "__main__":
    main()

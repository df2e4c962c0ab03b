#!/usr/bin/env python
"""Derive the robot descriptions used by tests and bench.py from the reference's URDF fixtures.

    python tools/make_fixtures.py <RigidBodyDynamics.jl checkout>

Reads the reference's test URDFs (test/urdf/*.urdf of the checkout) with ``read_urdf`` (only the fields the reference's parser
reads: link inertials, joint type / parent / child / origin / axis, in document order) and writes

  * the JSON robot descriptions of Atlas and Valkyrie to ``rigidbodydynamics/jl_b200/models/``;
  * ``tests/golden/reference_urdf.npz``: the flattened mechanisms ``parse_urdf`` builds from the original atlas.urdf and
    valkyrie.urdf (fixed and floating base), which ``tests/test_urdf.py`` compares the JSON descriptions against;
  * copies of the two small URDFs ``tests/test_urdf.py`` parses (Acrobot, planar slider) to ``tests/golden/urdf/``.
"""
import json
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rigidbodydynamics.jl_b200.urdf import parse_urdf, read_urdf  # noqa: E402

DST = os.path.join(ROOT, "rigidbodydynamics", "jl_b200", "models")
GOLD = os.path.join(ROOT, "tests", "golden")
FLAT_FIELDS = ("parent", "jtype", "X_tree", "jparam", "inertia")

if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    src = os.path.join(sys.argv[1], "test", "urdf")
    os.makedirs(DST, exist_ok=True)
    flat = {}
    for name in ("atlas", "valkyrie"):
        d = read_urdf(os.path.join(src, name + ".urdf"))
        d["source"] = f"derived from RigidBodyDynamics.jl test/urdf/{name}.urdf by tools/make_fixtures.py"
        with open(os.path.join(DST, name + ".json"), "w") as f:
            json.dump(d, f, separators=(",", ":"))
        print(name, len(d["links"]), "links", len(d["joints"]), "joints")
        for floating in (False, True):
            m = parse_urdf(os.path.join(src, name + ".urdf"), floating=floating).flatten()
            key = f"{name}_{'floating' if floating else 'fixed'}"
            flat[key + "_joint_names"] = np.array(m.joint_names)
            for fld in FLAT_FIELDS:
                flat[f"{key}_{fld}"] = getattr(m, fld)
    np.savez_compressed(os.path.join(GOLD, "reference_urdf.npz"), **flat)
    os.makedirs(os.path.join(GOLD, "urdf"), exist_ok=True)
    for name in ("Acrobot", "planar_slider"):
        shutil.copyfile(os.path.join(src, name + ".urdf"), os.path.join(GOLD, "urdf", name + ".urdf"))
    print("wrote", os.path.join(GOLD, "reference_urdf.npz"), "and", os.path.join(GOLD, "urdf"))

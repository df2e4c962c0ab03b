"""Host model loading: URDF rules of the reference (src/urdf/parse.jl) and fixed-joint removal."""
import os

import numpy as np
import pytest

import rigidbodydynamics.jl_b200 as rbd
from oracle import Oracle
from tests.util import GOLD, rand_inputs

ATLAS_ORDER = ["pelvis_to_world", "back_bkz", "l_leg_hpz", "r_leg_hpz", "back_bky", "l_leg_hpx", "r_leg_hpx", "back_bkx",
               "l_leg_hpy", "r_leg_hpy", "l_arm_shz", "neck_ay", "r_arm_shz", "l_leg_kny", "r_leg_kny", "l_arm_shx",
               "r_arm_shx", "l_leg_aky", "r_leg_aky", "l_arm_ely", "r_arm_ely", "l_leg_akx", "r_leg_akx", "l_arm_elx",
               "r_arm_elx", "l_arm_uwy", "r_arm_uwy", "l_arm_mwx", "r_arm_mwx", "l_arm_lwy", "r_arm_lwy"]


def test_rpy_goldens():
    """test/test_urdf.jl:79-102 (from ROS tf): rpy -> Rz(y) Ry(p) Rx(r)."""
    assert np.allclose(rbd.rot_rpy(1, 2, 3), [[0.41198225, -0.83373765, -0.36763046],
                                              [-0.05872664, -0.42691762, 0.90238159],
                                              [-0.90929743, -0.35017549, -0.2248451]], atol=1e-7)
    assert np.allclose(rbd.rot_rpy(0.5, 0.1, 0.2), [[0.97517033, -0.12744012, 0.18111281],
                                                    [0.19767681, 0.86959819, -0.45246312],
                                                    [-0.09983342, 0.47703041, 0.8731983]], atol=1e-7)
    assert np.allclose(rbd.rot_rpy(0, 0, 0.1), rbd.rot_z(0.1))


def test_atlas_joint_order_and_sizes():
    """SURVEY 8(b) 'Joint / index order': BFS + fixed-joint removal gives this exact order; nq 37 / nv 36; 175.118 kg."""
    m = rbd.load_model("atlas", floating=True)
    d = m.flatten()
    assert d.joint_names == ATLAS_ORDER
    assert (d.nq, d.nv, d.nb) == (37, 36, 31)
    assert abs(m.mass() - 175.117964) < 1e-9
    fixed = rbd.load_model("atlas").flatten()
    assert (fixed.nq, fixed.nv, fixed.nb) == (30, 30, 30)
    assert fixed.joint_names == ATLAS_ORDER[1:]


@pytest.mark.parametrize("name", ["atlas", "valkyrie"])
def test_json_description_equals_reference_urdf(name):
    """The JSON description gives the mechanism parse_urdf built from the reference's test/urdf/<name>.urdf (stored flattened in
    tests/golden/reference_urdf.npz by tools/make_fixtures.py)."""
    ref = np.load(os.path.join(GOLD, "reference_urdf.npz"))
    for floating in (False, True):
        a = rbd.load_model(name, floating=floating).flatten()
        key = f"{name}_{'floating' if floating else 'fixed'}"
        assert a.joint_names == ref[key + "_joint_names"].tolist()
        for f in ("parent", "jtype", "X_tree", "jparam", "inertia"):
            assert np.array_equal(getattr(a, f), ref[f"{key}_{f}"]), f


def test_reference_small_urdfs_parse():
    acro = rbd.parse_urdf(os.path.join(GOLD, "urdf", "Acrobot.urdf"))
    assert (acro.num_positions(), acro.num_velocities()) == (2, 2)
    slider = rbd.parse_urdf(os.path.join(GOLD, "urdf", "planar_slider.urdf"))
    assert all(isinstance(j.joint_type, rbd.Planar) for j in slider.joints)


@pytest.mark.parametrize("name", ["atlas", "valkyrie"])
def test_remove_fixed_joints_preserves_mass_matrix(name):
    """'remove fixed joints' testset of test/test_mechanism_modification.jl: M unchanged (1e-12), and inverse dynamics
    match (test/test_urdf.jl:106-119)."""
    kept = rbd.load_model(name, floating=True, remove_fixed_tree_joints=False)
    merged = rbd.load_model(name, floating=True)
    assert kept.num_velocities() == merged.num_velocities()
    ok, om = Oracle(kept.flatten()), Oracle(merged.flatten())
    q, v, tau, vd, _ = rand_inputs(merged, 3, 11)
    # fixed joints carry no coordinates, but the joint ORDER differs (fixed ones interleaved): map by joint name
    names_k = [j.name for j in kept.joints if j.nv > 0]
    names_m = [j.name for j in merged.joints]
    assert names_k == names_m
    assert np.abs(ok.mass_matrix(q) - om.mass_matrix(q)).max() < 1e-11
    assert np.abs(ok.inverse_dynamics(q, v, vd) - om.inverse_dynamics(q, v, vd)).max() < 1e-9


def test_modcount_and_loops():
    m = rbd.load_model("iiwa14")
    mc = m.modcount
    body = rbd.RigidBody("tool", rbd.SpatialInertia.rand(np.random.default_rng(0)))
    m.attach(m.bodies[-1], body, rbd.Joint("tool_joint", rbd.Fixed()))
    assert m.modcount == mc + 1
    m.attach(m.bodies[1], body, rbd.Joint("loop", rbd.Fixed()))      # successor already present -> non-tree joint
    assert m.has_loops()

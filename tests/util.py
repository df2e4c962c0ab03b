"""Shared helpers for the test-suite: models, seeded inputs, error metrics."""
import os

import numpy as np

import rigidbodydynamics.jl_b200 as rbd

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ALL_JOINT_TYPES = ([rbd.QuaternionFloating] + [rbd.Revolute] * 5 + [rbd.Fixed] * 5 + [rbd.Prismatic] * 5
                   + [rbd.Planar] * 5 + [rbd.SPQuatFloating] * 2 + [rbd.SinCosRevolute] * 2
                   + [rbd.QuaternionSpherical] * 2)


def randmech(seed, shuffle=False):
    """The reference's `randmech()` fixture (test/test_mechanism_algorithms.jl:1-11) plus QuaternionSpherical joints."""
    rng = np.random.default_rng(seed)
    jts = list(ALL_JOINT_TYPES)
    if shuffle:
        jts = [jts[i] for i in rng.permutation(len(jts))]
    return rbd.rand_tree_mechanism(rng, jts)


def double_pendulum(I1=0.333, I2=0.333, lc1=-0.5, lc2=-0.5, l1=-1.0, m1=1.0, m2=1.0, g=-9.81):
    """The reference's double pendulum built through the API (test/test_double_pendulum.jl:2-32, examples/1)."""
    axis = np.array([0.0, 1.0, 0.0])
    mech = rbd.Mechanism(rbd.RigidBody("world"), gravity=(0, 0, g))
    b1 = rbd.RigidBody("upper_link", rbd.SpatialInertia(I1 * np.outer(axis, axis), None, m1, com=[0, 0, lc1]))
    mech.attach(mech.root_body, b1, rbd.Joint("shoulder", rbd.Revolute(axis)))
    b2 = rbd.RigidBody("lower_link", rbd.SpatialInertia(I2 * np.outer(axis, axis), None, m2, com=[0, 0, lc2]))
    mech.attach(b1, b2, rbd.Joint("elbow", rbd.Revolute(axis)), joint_pose=rbd.Transform3D(None, [0, 0, l1]))
    return mech


def rand_inputs(mech, B, seed, wext=False):
    rng = np.random.default_rng(seed)
    nq, nv, nb = mech.num_positions(), mech.num_velocities(), len(mech.joints)
    q = np.stack([mech.rand_configuration(rng) for _ in range(B)], 1) if nq else np.zeros((0, B))
    v = rng.random((nv, B))
    tau = rng.random((nv, B))
    vd = rng.random((nv, B))
    w = rng.random((6 * nb, B)) if wext else None
    return q, v, tau, vd, w


def rel_err(got, ref):
    """max over the batch of |got - ref|_inf / max(1, |ref|_inf)   (SURVEY 8(d) 'Accuracy')."""
    got, ref = np.asarray(got, float), np.asarray(ref, float)
    return float((np.abs(got - ref).max(0) / np.maximum(1.0, np.abs(ref).max(0))).max())


def make_duals(mech, q, v, tau, seed):
    """Dual{Float64,6} versions [rows, B, 7] of (q, v, tau): value + 6 random partials.  Partials of unit-quaternion
    coordinates are projected onto the tangent space of the unit sphere: off-manifold derivatives depend on how an algorithm
    happens to extend R(q) to non-unit quaternions and are not comparable between formulations (SURVEY 8(c): parity unpinned)."""
    rng = np.random.default_rng(seed)

    def dual(x):
        a = np.zeros(x.shape + (7,))
        a[..., 0] = x
        a[..., 1:] = rng.standard_normal(x.shape + (6,))
        return a
    Q, V, T = dual(q), dual(v), dual(tau)
    qs = 0
    for j in mech.joints:
        if isinstance(j.joint_type, (rbd.QuaternionFloating, rbd.QuaternionSpherical)):
            qq = Q[qs:qs + 4, :, 0]
            for k in range(6):
                dq = Q[qs:qs + 4, :, 1 + k]
                dq -= qq * (qq * dq).sum(0)
        elif isinstance(j.joint_type, rbd.SinCosRevolute):
            qq = Q[qs:qs + 2, :, 0]
            for k in range(6):
                dq = Q[qs:qs + 2, :, 1 + k]
                dq -= qq * (qq * dq).sum(0)
        qs += j.nq
    return Q, V, T


def config_distance(mech, qa, qb):
    """max over joints / samples of the distance between two configurations, insensitive to the sign of unit quaternions
    (q and -q are the same rotation; the reference's matrix -> quaternion conversion fixes a sign this code does not need)."""
    qa, qb = np.asarray(qa, float), np.asarray(qb, float)
    d, qs = 0.0, 0
    for j in mech.joints:
        a, b = qa[qs:qs + j.nq], qb[qs:qs + j.nq]
        if isinstance(j.joint_type, (rbd.QuaternionFloating, rbd.QuaternionSpherical)):
            sgn = np.sign((a[:4] * b[:4]).sum(0))
            d = max(d, np.abs(a[:4] - sgn * b[:4]).max(initial=0.0), np.abs(a[4:] - b[4:]).max(initial=0.0))
        elif j.nq:
            d = max(d, np.abs(a - b).max())
        qs += j.nq
    return d


def axis_aligned_tree(seed, n=24):
    """Random tree whose joint axes are coordinate axes and whose tree rotations are multiples of 90 degrees (like real robots),
    with every joint type present, some zero tree offsets, and a floating base: exercises the fast joint classes of
    csrc/rbd_model.cpp (parallel / perpendicular axes, zero origin shift) next to the general path."""
    rng = np.random.default_rng(seed)
    eye = np.eye(3)

    def rot90():
        perm = rng.permutation(3)
        R = eye[:, perm] * rng.choice([-1.0, 1.0], 3)
        if np.linalg.det(R) < 0:
            R[:, 0] = -R[:, 0]
        return R

    def axis():
        return eye[int(rng.integers(3))] * rng.choice([-1.0, 1.0])

    mech = rbd.Mechanism(rbd.RigidBody("world"))
    base = rbd.RigidBody("base", rbd.SpatialInertia.rand(rng))
    mech.attach(mech.root_body, base, rbd.Joint("floating", rbd.QuaternionFloating()))
    kinds = [rbd.Revolute] * (n - 6) + [rbd.Prismatic, rbd.Fixed, rbd.SinCosRevolute, rbd.Revolute, rbd.Prismatic, rbd.Revolute]
    for i, K in enumerate(kinds):
        parent = mech.bodies[int(rng.integers(1, len(mech.bodies)))]
        jt = K() if K is rbd.Fixed else K(axis())
        trans = np.zeros(3) if rng.random() < 0.3 else rng.standard_normal(3) * (rng.random(3) < 0.6)
        general = rng.random() < 0.15            # a few arbitrary rotations: general path
        R = rbd.Transform3D.rand(rng).rot if general else rot90()
        mech.attach(parent, rbd.RigidBody(f"b{i}", rbd.SpatialInertia.rand(rng)), rbd.Joint(f"j{i}", jt),
                    joint_pose=rbd.Transform3D(R, trans))
    return mech


def oracle_dynamics_derivatives(oracle, mech, q, v, tau):
    """Tangent-space Jacobians of forward dynamics from the ORACLE's dual-number run of the reference's own algorithm, the way a
    ForwardDiff user gets them (examples/5, test_mechanism_algorithms.jl:600-675): partial k of q is seeded with
    q̇ = velocity_to_configuration_derivative(e_k) (mechanism_state.jl:905-910), partial k of v with e_k; six partials per sweep.
    Returns (dvd_dq, dvd_dv), each [nv*nv, B] with entry (i, j) at row i + j*nv."""
    q, v, tau = np.asarray(q, float), np.asarray(v, float), np.asarray(tau, float)
    nq, B = q.shape
    nv = v.shape[0]
    N = np.zeros((nq, nv, B))                       # velocity_to_configuration_derivative_jacobian, column by column
    for k in range(nv):
        e = np.zeros((nv, B)); e[k] = 1.0
        N[:, k] = oracle.dynamics(q, e, tau, want_qd=True)[1]
    out = []
    for which in range(2):
        J = np.zeros((nv, nv, B))
        for k0 in range(0, nv, 6):
            Q = np.zeros((nq, B, 7)); V = np.zeros((nv, B, 7)); T = np.zeros((nv, B, 7))
            Q[..., 0], V[..., 0], T[..., 0] = q, v, tau
            ks = range(k0, min(k0 + 6, nv))
            for s, k in enumerate(ks):
                if which == 0:
                    Q[:, :, 1 + s] = N[:, k]
                else:
                    V[k, :, 1 + s] = 1.0
            r = oracle.dynamics_dual6(Q, V, T)
            for s, k in enumerate(ks):
                J[:, k] = r[:, :, 1 + s]
        out.append(J.transpose(1, 0, 2).reshape(nv * nv, B))   # row i + j*nv  <->  [j, i]
    return out[0], out[1]

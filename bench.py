#!/usr/bin/env python
"""bench.py -- headline benchmark: Atlas (floating base, nv = 36) forward-dynamics evaluations per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dtype f32|f64] [--dump-outputs DIR]

Workload (BASELINE.json metric, SURVEY 8(d) "Headline"): Atlas v5 with a QuaternionFloating root (nq 37, nv 36, 31 bodies),
`dynamics!` with joint torques, fp32, batch 2^20 per GPU.  A "step" is one pass of the forward-dynamics kernel over the whole
batch.  Inputs follow `rand!(state)` and perf/runbenchmarks.jl:59-67 (q: N(0,1) angles, uniform random unit quaternion,
base position U(-0.5,0.5)^3; v, tau ~ U[0,1)), generated with numpy PCG64 seed 1 on the host in fp64 and cast.

One JSON line on stdout (rank 0).  `value` = evaluations/s with inputs resident in HBM (CUDA events around K launches);
`e2e` = the same through the host-pointer C-ABI call (pinned host buffers, H2D and D2H inside the timed region);
`roofline` = algorithmic bytes (580 B/eval fp32, BASELINE.md section 4) x evals/s against the measured HBM peak;
`cpu_baseline` = the CPU oracle (port of the reference's CRBA + RNEA + Cholesky path) on a bounded sample.

`--impl reference` times that CPU path alone (the reference itself is Julia and cannot run here; see DESIGN.md).

`--dump-outputs DIR` writes what the last timed step computed, v̇ of rank 0, as DIR/vd.npy ([36, n], the run's dtype): the whole
batch when it fits in 48 MB, else the same seeded sample of n columns in every run with the same arguments.  The inputs depend on
the arguments alone, so two builds can be compared output for output.

Nothing is written into the source tree: cubins compiled at run time go to a temporary copy of the build's cubin cache.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

BYTES_PER_EVAL = {"f32": 580, "f64": 1160}      # (37 + 36 + 36 in, 36 out) scalars, BASELINE.md section 4
DUMP_BYTES = 48 << 20
METRIC = "ABA evals/sec for Atlas 30-DoF at batch 2^20; achieved HBM GB/s vs peak"


def make_inputs(mech, B, seed):
    """rand!(state) + random torques, host fp64, [rows, B]."""
    rng = np.random.Generator(np.random.PCG64(seed))
    nq, nv = mech.num_positions(), mech.num_velocities()
    q = np.empty((nq, B))
    x = rng.standard_normal((4, B))
    q[0:4] = x / np.linalg.norm(x, axis=0)                 # uniform random rotation, unit norm, [w x y z]
    q[4:7] = rng.random((3, B)) - 0.5
    q[7:] = rng.standard_normal((nq - 7, B))
    v = rng.random((nv, B))
    tau = rng.random((nv, B))
    return q, v, tau


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the GPU is under load (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [s for (t, s) in self.samples if (t0 is None or t >= t0) and (t1 is None or t <= t1 + 0.15)]
        if not rows:
            rows = [s for (_, s) in self.samples]
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            p = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(p[0])); smax.append(float(p[1]))
            except (ValueError, IndexError):
                continue
            for n, val in zip(names, p[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def effective_cores():
    """CPU cores this process may actually use: the cgroup CPU quota when there is one (the GPU boxes expose 128 logical CPUs
    but cap the container at 16 -- running 128 threads there is 2x SLOWER than 16), else the affinity mask."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                quota, period = int(f.read()), int(g.read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except (OSError, ValueError):
            pass
    return n


def cpu_baseline(mech, q, v, tau, dtype, seconds_target=12.0):
    """Oracle (CPU port of the reference's dynamics!: RNEA bias + CRBA + Cholesky) on a bounded sample, all host cores."""
    from oracle import Oracle
    o = Oracle(mech.flatten())
    cores = effective_cores()
    dt = np.float32 if dtype == "f32" else np.float64
    n = min(q.shape[1], 8192 * cores)
    qs, vs, ts = (np.ascontiguousarray(a[:, :n], dt) for a in (q, v, tau))
    o.dynamics(qs[:, :256], vs[:, :256], ts[:, :256], nthreads=cores)     # warm
    t0 = time.perf_counter()
    reps = 0
    while True:
        o.dynamics(qs, vs, ts, nthreads=cores)
        reps += 1
        el = time.perf_counter() - t0
        if el > seconds_target or reps >= 64:
            break
    return {"value": reps * n / el, "unit": "evals/s", "cores": cores, "kind": "port",
            "sample": f"{n} Atlas states x {reps} repeats, CRBA+RNEA+Cholesky (the reference's dynamics! algorithm), "
                      f"{np.dtype(dt).name}, {cores} threads"}


def time_fn(fn, steps, warmup=3):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def other_configs(steps):
    """The remaining BASELINE.json configs as secondary measurements (kernel time, CUDA events, inputs resident in HBM):
    config 2 (Atlas fp64 dynamics, batch 65536), config 3 (7-DoF arm fp32 inverse_dynamics / mass_matrix, batch 2^20), and the
    reference's own benchmark variant with an external wrench on every body (perf/runbenchmarks.jl:59-67)."""
    import torch
    import rigidbodydynamics.jl_b200 as rbd
    out = {}
    rng = np.random.default_rng(1)
    atlas = rbd.load_model("atlas", floating=True)
    st = rbd.MechanismState(atlas, 1 << 16, torch.float64)
    rbd.rand_(st, rng)
    tau = torch.rand((36, 1 << 16), dtype=torch.float64, device="cuda")
    res = rbd.DynamicsResult(atlas, 1 << 16, torch.float64)
    ms = time_fn(lambda: rbd.dynamics_(res, st, tau, want_qd=False), steps)
    out["atlas_f64_dynamics_b65536"] = {"evals_per_s": (1 << 16) / (ms * 1e-3), "ms": ms, "algorithmic_GBps": (1 << 16) * 1160 / (ms * 1e-3) / 1e9}
    B = 1 << 20
    st = rbd.MechanismState(atlas, B, torch.float32)
    rbd.rand_(st, rng)
    tau = torch.rand((36, B), dtype=torch.float32, device="cuda")
    wext = torch.rand((6 * 31, B), dtype=torch.float32, device="cuda")
    res = rbd.DynamicsResult(atlas, B, torch.float32)
    ms = time_fn(lambda: rbd.dynamics_(res, st, tau, wext, want_qd=False), steps)
    out["atlas_f32_dynamics_extwrench_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * (580 + 744) / (ms * 1e-3) / 1e9}
    ms = time_fn(lambda: rbd.dynamics_(res, st, tau, want_qd=True), steps)
    out["atlas_f32_dynamics_with_qdot_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 728 / (ms * 1e-3) / 1e9}
    vd = torch.rand((36, B), dtype=torch.float32, device="cuda")
    tout = torch.empty_like(vd)
    ms = time_fn(lambda: rbd.inverse_dynamics_(tout, st, vd), steps)
    out["atlas_f32_inverse_dynamics_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 580 / (ms * 1e-3) / 1e9}
    ms = time_fn(lambda: rbd.simulate_(st, 1e-4, tau, dt=1e-4), max(3, steps // 4))      # one Munthe-Kaas RK4 step (4 dynamics)
    out["atlas_f32_rk4_step_b1048576"] = {"sample_steps_per_s": B / (ms * 1e-3), "ms": ms, "kernel_launches_per_step": rbd.launch_info().kernels_launched}
    # kinematics by-products (perf/runbenchmarks.jl:69-110): algorithmic bytes = q (+ v) in, the requested outputs out
    A = torch.empty((6 * 36, B), dtype=torch.float32, device="cuda")
    ms = time_fn(lambda: rbd.momentum_matrix_(A, st), steps)
    out["atlas_f32_momentum_matrix_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * (37 + 216) * 4 / (ms * 1e-3) / 1e9}
    pth = rbd.path(atlas, atlas.findbody("r_foot"), atlas.findbody("l_hand"))    # perf/runbenchmarks.jl:29-31
    ms = time_fn(lambda: rbd.geometric_jacobian_(A, st, pth), steps)
    out["atlas_f32_geometric_jacobian_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * (37 + 216) * 4 / (ms * 1e-3) / 1e9}
    trs = torch.empty((12 * 31, B), dtype=torch.float32, device="cuda")
    ms = time_fn(lambda: rbd.transforms_to_root_(trs, st), steps)
    out["atlas_f32_transforms_to_root_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * (37 + 372) * 4 / (ms * 1e-3) / 1e9}
    del trs
    small = {k: torch.empty((r, B), dtype=torch.float32, device="cuda") for k, r in
             (("center_of_mass", 3), ("kinetic_energy", 1), ("gravitational_potential_energy", 1), ("momentum", 6),
              ("momentum_rate_bias", 6))}
    ms = time_fn(lambda: rbd.kinematics_(st, None, **small), steps)
    out["atlas_f32_com_energies_momentum_fused_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * (37 + 36 + 17) * 4 / (ms * 1e-3) / 1e9}
    Mfull = torch.empty((36 * 36, 1 << 18), dtype=torch.float32, device="cuda")          # 5.2 KB/sample out: batch 2^18
    st18 = rbd.MechanismState(atlas, 1 << 18, torch.float32)
    rbd.rand_(st18, rng)
    ms = time_fn(lambda: rbd.mass_matrix_(Mfull, st18), steps)
    out["atlas_f32_mass_matrix_b262144"] = {"evals_per_s": (1 << 18) / (ms * 1e-3), "ms": ms, "algorithmic_GBps": (1 << 18) * (37 + 1296) * 4 / (ms * 1e-3) / 1e9}
    ms = time_fn(lambda: rbd.mass_matrix_(Mfull, st18, uplo="L"), steps)          # the triangle the reference's mass_matrix! fills
    out["atlas_f32_mass_matrix_lower_b262144"] = {"evals_per_s": (1 << 18) / (ms * 1e-3), "ms": ms, "algorithmic_GBps": (1 << 18) * (37 + 666) * 4 / (ms * 1e-3) / 1e9}
    st17 = rbd.MechanismState(atlas, 1 << 17, torch.float64)
    rbd.rand_(st17, rng)
    M64 = torch.empty((36 * 36, 1 << 17), dtype=torch.float64, device="cuda")
    ms = time_fn(lambda: rbd.mass_matrix_(M64, st17), steps)
    out["atlas_f64_mass_matrix_b131072"] = {"evals_per_s": (1 << 17) / (ms * 1e-3), "ms": ms, "algorithmic_GBps": (1 << 17) * (37 + 1296) * 8 / (ms * 1e-3) / 1e9}
    del M64, st17
    # SURVEY 8(f) rank 4: contact_dynamics! -- one contact point per foot corner against the ground half-space (8 points), fp32
    catlas = rbd.load_model("atlas", floating=True)
    cmodel = rbd.SoftContactModel(rbd.hunt_crossley_hertz(), rbd.ViscoelasticCoulombModel(0.8, 20e3, 100.0))
    for foot in ("l_foot", "r_foot"):
        for x in (-0.08, 0.17):
            for y in (-0.06, 0.06):
                rbd.add_contact_point(catlas.findbody(foot), rbd.ContactPoint([x, y, -0.08], cmodel))
    rbd.add_environment_primitive(catlas, rbd.HalfSpace3D([0.0, 0.0, 0.0], [0.0, 0.0, 1.0]))
    cst = rbd.MechanismState(catlas, B, torch.float32)
    cst.q.copy_(st.q); cst.v.copy_(st.v)
    cw = torch.empty((6 * 31, B), dtype=torch.float32, device="cuda")
    ns = rbd.num_contact_states(catlas)
    cs = torch.zeros((ns, B), dtype=torch.float32, device="cuda")
    csd = torch.empty_like(cs)
    ms = time_fn(lambda: rbd.contact_dynamics_(cst, cw, cs, csd), steps)
    out["atlas_f32_contact_dynamics_8points_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms,
                                                          "algorithmic_GBps": B * (37 + 36 + 2 * ns + 6 * 31) * 4 / (ms * 1e-3) / 1e9}
    del cst, cw, cs, csd
    del res, wext, tau, vd, tout, st, A, small, Mfull, st18
    # config 4: dynamics! on ForwardDiff.Dual{Tag,Float64,6} (value + 6 partials per scalar), batch 8192
    Bd = 8192
    std = rbd.MechanismState(atlas, 1, torch.float64)
    qd_ = torch.zeros((37, Bd, 7), dtype=torch.float64, device="cuda")
    stq = rbd.MechanismState(atlas, Bd, torch.float64)
    rbd.rand_(stq, rng)
    qd_[..., 0] = stq.q
    qd_[4:, :, 1:] = torch.rand((33, Bd, 6), dtype=torch.float64, device="cuda")          # partials of the non-quaternion coordinates
    vdual = torch.rand((36, Bd, 7), dtype=torch.float64, device="cuda")
    tdual = torch.rand((36, Bd, 7), dtype=torch.float64, device="cuda")
    odual = torch.empty((36, Bd, 7), dtype=torch.float64, device="cuda")
    ms = time_fn(lambda: rbd.dynamics_dual_(odual, std, qd_, vdual, tdual), max(3, steps // 2))
    out["atlas_dual64x6_dynamics_b8192"] = {"evals_per_s": Bd / (ms * 1e-3), "ms": ms, "algorithmic_GBps": Bd * 8120 / (ms * 1e-3) / 1e9}
    dual_sweeps_per_s = Bd / (ms * 1e-3)
    del std, stq, qd_, vdual, tdual, odual
    # SURVEY 8(f) rank 3: the full Jacobians dv̇/dq, dv̇/dv analytically (rbd_dynamics_derivatives) -- what 2 nv / 6 = 12 of the Dual
    # sweeps above produce for one Atlas sample.  Algorithmic bytes: q, v, tau in; v̇ and two nv x nv matrices out.
    for tdt, key, Bj in ((torch.float64, "f64", 1 << 15), (torch.float32, "f32", 1 << 16)):
        stj = rbd.MechanismState(atlas, Bj, tdt)
        rbd.rand_(stj, rng)
        tauj = torch.rand((36, Bj), dtype=tdt, device="cuda")
        resj = rbd.DynamicsResult(atlas, Bj, tdt)
        dq = torch.empty((36 * 36, Bj), dtype=tdt, device="cuda")
        dv = torch.empty_like(dq)
        ms = time_fn(lambda: rbd.dynamics_derivatives_(dq, dv, resj, stj, tauj), max(3, steps // 2))
        es = dq.element_size()
        out[f"atlas_{key}_dynamics_derivatives_b{Bj}"] = {
            "jacobian_pairs_per_s": Bj / (ms * 1e-3), "ms": ms, "dual_sweep_equivalents_per_s": Bj / (ms * 1e-3) * 12,
            "vs_own_dual_sweeps": Bj / (ms * 1e-3) * 12 / dual_sweeps_per_s,
            "algorithmic_GBps": Bj * (37 + 36 + 36 + 36 + 2 * 1296) * es / (ms * 1e-3) / 1e9,
            "kernel_launches": rbd.launch_info().kernels_launched}
        del stj, tauj, resj, dq, dv
    iiwa = rbd.load_model("iiwa14")
    st = rbd.MechanismState(iiwa, B, torch.float32)
    rbd.rand_(st, rng)
    vd = torch.rand((7, B), dtype=torch.float32, device="cuda")
    tout = torch.empty_like(vd)
    ms = time_fn(lambda: rbd.inverse_dynamics_(tout, st, vd), steps)
    out["iiwa14_f32_inverse_dynamics_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 112 / (ms * 1e-3) / 1e9}
    Mout = torch.empty((49, B), dtype=torch.float32, device="cuda")
    ms = time_fn(lambda: rbd.mass_matrix_(Mout, st), steps)
    out["iiwa14_f32_mass_matrix_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 224 / (ms * 1e-3) / 1e9}
    res = rbd.DynamicsResult(iiwa, B, torch.float32)
    tau = torch.rand((7, B), dtype=torch.float32, device="cuda")
    ms = time_fn(lambda: rbd.dynamics_(res, st, tau, want_qd=False), steps)
    out["iiwa14_f32_dynamics_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 112 / (ms * 1e-3) / 1e9}
    Mlow = torch.empty((49, B), dtype=torch.float32, device="cuda")
    ms = time_fn(lambda: rbd.mass_matrix_(Mlow, st, uplo="L"), steps)
    out["iiwa14_f32_mass_matrix_lower_b1048576"] = {"evals_per_s": B / (ms * 1e-3), "ms": ms, "algorithmic_GBps": B * 140 / (ms * 1e-3) / 1e9}
    del st, res, tau, vd, tout, Mout, Mlow
    # throughput against batch size (VERDICT r1 item 7): Atlas forward dynamics, kernel time per call, fp32 and fp64
    curve = {}
    for tdt, key in ((torch.float32, "f32"), (torch.float64, "f64")):
        pts = []
        stc = rbd.MechanismState(atlas, 1 << 20, tdt)
        rbd.rand_(stc, rng)
        tauc = torch.rand((36, 1 << 20), dtype=tdt, device="cuda")
        for lg in range(10, 21, 2 if key == "f64" else 1):
            n = 1 << lg
            sub = rbd.MechanismState(atlas, n, tdt)
            sub.q.copy_(stc.q[:, :n]); sub.v.copy_(stc.v[:, :n])
            tn = tauc[:, :n].contiguous()
            rn = rbd.DynamicsResult(atlas, n, tdt)
            ms = time_fn(lambda: rbd.dynamics_(rn, sub, tn, want_qd=False), max(steps, 10))
            pts.append({"batch": n, "us_per_call": round(ms * 1e3, 2), "evals_per_s": n / (ms * 1e-3),
                        "specialised": bool(rbd.launch_info().specialised)})
        curve[key] = pts
        del stc, tauc
    out["atlas_dynamics_batch_curve"] = curve
    return out


def private_jit_cache():
    """Point the cubin cache at a temporary copy of the one build() filled (csrc/jit_cache), so that kernels compiled during the run
    never land in the source tree, which may be read-only.  Returns the TemporaryDirectory (removed when it is closed)."""
    import shutil
    import tempfile
    if os.environ.get("RBD_JIT_CACHE"):
        return None
    tmp = tempfile.TemporaryDirectory(prefix="rbd_jit_cache_")
    src = os.path.join(ROOT, "rigidbodydynamics", "jl_b200", "csrc", "jit_cache")
    if os.path.isdir(src):
        for f in os.listdir(src):
            if f.endswith(".cubin"):
                shutil.copyfile(os.path.join(src, f), os.path.join(tmp.name, f))
    os.environ["RBD_JIT_CACHE"] = tmp.name
    return tmp


def output_sample(vd):
    """Device copy of what --dump-outputs writes: v̇ [rows, B], or above DUMP_BYTES a fixed seeded sample of its columns."""
    import torch
    rows, B = vd.shape
    n = min(B, DUMP_BYTES // (rows * vd.element_size()))
    if n == B:
        return vd.clone()
    idx = np.sort(np.random.Generator(np.random.PCG64(0)).choice(B, n, replace=False))
    return vd[:, torch.from_numpy(idx).to(vd.device)]


def add_rooflines(cfgs, peak):
    """Per-config roofline objects (HBM, algorithmic bytes) next to the raw rates; ncu summaries of the kernels behind them are under
    profiles/r2_*_summary.txt (dram__bytes_read/write, issue-active, stall reasons)."""
    for k, c in cfgs.items():
        if isinstance(c, dict) and "algorithmic_GBps" in c:
            c["roofline"] = {"bound": "hbm", "achieved": c["algorithmic_GBps"], "peak": peak, "unit": "GB/s",
                             "frac": c["algorithmic_GBps"] / peak}
    return cfgs


def run_config5(rbd, mech, dist, world, rank, args, tdt):
    """BASELINE config 5: 2^22 Atlas states in total, sharded over the ranks; returns the dicts rank 0 prints."""
    import torch
    from rigidbodydynamics.jl_b200.sharding import GatheredResult, dynamics_gather_
    total = 1 << 22
    Bl = total // world
    q, v, tau = make_inputs(mech, Bl, 101 + rank)
    st = rbd.MechanismState(mech, Bl, tdt)
    st.q.copy_(torch.from_numpy(q).to(tdt)); st.v.copy_(torch.from_numpy(v).to(tdt))
    tau_d = torch.from_numpy(tau).to(tdt).cuda()
    res = rbd.DynamicsResult(mech, Bl, tdt)
    nv = st.nv
    steps = max(5, min(args.steps, 20))

    def timed(fn, sync=None):
        for _ in range(3):
            fn()
        if sync:
            sync()
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if sync:
            sync()
        e1.record()
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return total * steps / (float(t.item()) * 1e-3)

    no_gather = timed(lambda: rbd.dynamics_(res, st, tau_d, want_qd=False))
    out_nccl = torch.empty((world, nv, Bl), dtype=tdt, device="cuda")

    def nccl_step():
        rbd.dynamics_(res, st, tau_d, want_qd=False)
        dist.all_gather_into_tensor(out_nccl, res.vd)
    nccl = timed(nccl_step)
    fused, fused_ok, why, fused_p2p, multicast = None, None, None, None, False
    try:
        g0 = GatheredResult(nv, Bl, tdt, use_multicast=False)          # one store per peer
        fused_p2p = timed(lambda: (dynamics_gather_(g0, st, tau_d), g0.barrier()))
        del g0
        g = GatheredResult(nv, Bl, tdt)                                # NVLS multicast when the box has it
        multicast = bool(g.multicast_ptr)
        fused = timed(lambda: (dynamics_gather_(g, st, tau_d), g.barrier())) if multicast else fused_p2p
        g.barrier(); torch.cuda.synchronize()
        # every GPU must now hold every rank's v̇, bit-identical to what the NCCL path gathered
        ok = bool(torch.equal(g.tensor.view(nv, world, Bl).permute(1, 0, 2), out_nccl))
        okt = torch.tensor([1.0 if ok else 0.0], device="cuda")
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        fused_ok = bool(okt.item() == 1.0)
        specialised = bool(rbd.launch_info().specialised)
    except Exception as e:          # symmetric memory unavailable: the NCCL number stands
        why = f"{type(e).__name__}: {e}"[:200]
        specialised = False
    es = 4 if tdt == torch.float32 else 8
    best = fused if fused is not None else nccl
    return {
        "with_nccl_gather": {
            "value": best, "unit": "evals/s", "total_batch": total, "batch_per_gpu": Bl,
            "method": "fused: the kernel stores v̇ into every GPU's gathered array over NVLink (rbd_dynamics_gather)" if fused is not None
                      else "ncclAllGather after the kernel",
            "fused_gather_value": fused, "fused_gather_p2p_stores_value": fused_p2p, "fused_uses_nvls_multicast": multicast,
            "nccl_allgather_after_kernel_value": nccl, "no_gather_value": no_gather,
            "frac_of_no_gather": best / no_gather, "fused_matches_nccl_bitwise": fused_ok, "fused_unavailable": why,
            "fused_uses_specialised_kernels": specialised,
            "nvlink_bytes_sent_per_gpu_per_step": (world - 1) * nv * Bl * es,
            "nvlink_bytes_received_per_gpu_per_step": (world - 1) * nv * Bl * es,
            "note": "an all-gather of v̇ needs every GPU to RECEIVE (N-1)/N of the 604 MB result per step, so NVLink ingress bounds "
                    "any gather at N=8 near 0.59 ms per 2^22 samples (7.1 G evals/s at 900 GB/s)"},
        "strong_scaling": {"value": no_gather, "unit": "evals/s", "total_batch": total, "batch_per_gpu": Bl,
                           "note": "same total work at every N (config 5 without the gather); the headline `value` is weak scaling"},
    }


def bind_to_gpu_numa_node(local_rank):
    """Run this rank's threads on, and allocate its pinned buffers from, the NUMA node its GPU hangs off (nvidia-smi topo: on the
    8-GPU boxes GPUs 0-3 sit on node 0 and 4-7 on node 1; unbound ranks were measured at 38.7 instead of 62.9 GB/s of PCIe)."""
    info = {"node": None, "cpus": None}
    try:
        import torch
        out = subprocess.run(["nvidia-smi", f"--id={local_rank}", "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        bdf = (out or "").lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        node_path = f"/sys/bus/pci/devices/{bdf}/numa_node"
        node = int(open(node_path).read().strip())
        if node < 0:
            return info
        cpulist = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)          # first-touch policy then places the pinned pages on this node
            info = {"node": node, "cpus": len(cpus)}
    except Exception:
        pass
    return info


def run_reference(args):
    """--impl reference: the reference's own algorithm on the host CPU (oracle port; Julia is not installed)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import rigidbodydynamics.jl_b200 as rbd
    mech = rbd.load_model("atlas", floating=True)
    cores = effective_cores()
    n = 8192 * cores
    q, v, tau = make_inputs(mech, n, 1)
    from oracle import Oracle
    o = Oracle(mech.flatten())
    dt = np.float32 if args.dtype == "f32" else np.float64
    qs, vs, ts = (np.ascontiguousarray(a, dt) for a in (q, v, tau))
    for _ in range(max(1, args.warmup)):
        o.dynamics(qs, vs, ts, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.dynamics(qs, vs, ts, nthreads=cores)
    el = time.perf_counter() - t0
    val = args.steps * n / el
    sample = f"{n} Atlas states per step (bounded sample of the 2^20 batch), {np.dtype(dt).name}, {cores} threads"
    _emit(({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": {"workload": "atlas floating-base dynamics! (CRBA+RNEA+Cholesky) on host CPU", "sample": sample},
        "cpu_baseline": {"value": val, "unit": "evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


_JSON_FD = None


def _claim_stdout():
    """stdout must carry exactly ONE JSON line, but libraries write banners to file descriptor 1 (NCCL prints its version there at
    communicator creation).  Keep a private duplicate of the real stdout for the result and point fd 1 at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1 << 20, help="samples per GPU")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-config5", action="store_true", help="N > 1: skip BASELINE config 5 (2^22 samples in total, result gather timed)")
    ap.add_argument("--no-other", action="store_true", help="skip the secondary configs (fp64, RNEA, CRBA, ext. wrenches)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write v̇ of the last timed step to DIR/vd.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        return run_reference(args)
    jit_cache = private_jit_cache()

    import torch
    import rigidbodydynamics.jl_b200 as rbd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else {"node": None, "cpus": None}
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    mech = rbd.load_model("atlas", floating=True)
    B = args.batch
    tdt = torch.float32 if args.dtype == "f32" else torch.float64
    q, v, tau = make_inputs(mech, B, 1 + rank)
    state = rbd.MechanismState(mech, B, tdt)
    state.q.copy_(torch.from_numpy(q).to(tdt))
    state.v.copy_(torch.from_numpy(v).to(tdt))
    tau_d = torch.from_numpy(tau).to(tdt).cuda()
    result = rbd.DynamicsResult(mech, B, tdt)

    def step():
        rbd.dynamics_(result, state, tau_d, want_qd=False)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(args.warmup):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    t_wall1 = time.time()
    ms = ev0.elapsed_time(ev1)
    dump = output_sample(result.vd) if args.dump_outputs and rank == 0 else None
    # keep the GPU under the same load until the sampler has a few readings inside a loaded window
    t_load_end = t_wall1
    if sampler and (t_wall1 - t_wall0) < 0.6:
        while time.time() - t_wall0 < 0.8:
            step()
        torch.cuda.synchronize()
        t_load_end = time.time()
    clocks = sampler.stop(t_wall0, t_load_end) if sampler else None
    ms_t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms = float(ms_t.item())
    linfo = rbd.launch_info()
    value = world * B * args.steps / (ms * 1e-3)

    # BASELINE config 5 as written: Atlas fp32, 2^22 samples IN TOTAL over the N GPUs (strong scaling), result gather inside the
    # timed region.  Three timings: no gather; the collective the reference design would use (ncclAllGather after the kernel); and
    # this repo's fused gather (the kernel stores v̇ into every GPU's gathered array over NVLink, rbd_dynamics_gather).
    config5 = None
    if dist is not None and not args.no_config5:
        config5 = run_config5(rbd, mech, dist, world, rank, args, tdt)

    # end-to-end through the host-pointer C-ABI entry point: pinned host buffers, copies inside the timed region
    import ctypes
    lib = rbd.load_library()
    hq = torch.from_numpy(q).to(tdt).pin_memory()
    hv = torch.from_numpy(v).to(tdt).pin_memory()
    ht = torch.from_numpy(tau).to(tdt).pin_memory()
    hvd = torch.empty((state.nv, B), dtype=tdt).pin_memory()
    code = rbd._cabi.RBD_F32 if args.dtype == "f32" else rbd._cabi.RBD_F64

    def e2e_step():
        rbd._cabi.check(lib.rbd_dynamics_host(state.handle.ptr, code, B, B, hq.data_ptr(), hv.data_ptr(), ht.data_ptr(),
                                              None, hvd.data_ptr(), None))
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_val = world * B * e2e_steps / float(e2e_t.item())
    es = 4 if args.dtype == "f32" else 8
    e2e_ok = bool(torch.allclose(hvd.cuda(), result.vd, rtol=0, atol=0))

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        bpe = BYTES_PER_EVAL[args.dtype]
        achieved = (B * args.steps / (ms * 1e-3)) * bpe / 1e9       # per GPU
        traffic, traffic_src = None, None
        try:        # DRAM bytes per launch from the committed ncu --set full capture of this exact workload (same kernels, same batch)
            with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
                for name, rec in json.load(f).items():
                    if rec["samples"] == B and args.dtype == "f32":
                        traffic = rec["dram_bytes_read"] + rec["dram_bytes_write"]
                        traffic_src = {"capture": name, "command": rec.get("command"), "bytes_per_sample": traffic / B}
        except (OSError, KeyError, ValueError):
            pass
        out = {
            "metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"atlas floating-base (nq 37, nv 36) dynamics! = ABA, batch {B} per GPU, {args.dtype}",
                       "batch_per_gpu": B, "l2": "inputs (109 rows x batch) exceed the 126 MB L2; no reuse between steps",
                       "parallelism": f"batch-sharded x{world}, no data-path collective"},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "evals/s", "h2d_bytes_per_step": (37 + 36 + 36) * B * es,
                    "d2h_bytes_per_step": 36 * B * es, "steps": e2e_steps, "matches_device_path": e2e_ok, "numa_binding": numa},
            "gpu_launches": args.steps * linfo.kernels_launched,
            "launch": {"grid": linfo.grid, "block": linfo.block, "smem_bytes": linfo.smem_bytes,
                       "blocks_per_sm": linfo.blocks_per_sm},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": B * bpe,
                         "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback 6650 GB/s",
                         "kernels": "model-specialised (NVRTC) pair / unified CTA" if linfo.specialised else "generic kernel pair",
                         "note": "algorithmic bytes/eval x evals/s per GPU; traffic = ncu dram bytes per launch of the same workload "
                                 "(profiles/r2_traffic.json, not measured in this run).  The kernel is bound by instruction supply, not by "
                                 "HBM: the model-specialised program is ~12.4 k warp-instructions per 32 samples (generic: 27.5 k) but "
                                 "streams from L2 at ~1.4 instr/clk/SM (ncu: no_instruction stalls dominate, profiles/r2_jit_aba_*)"},
        }
        # The roofline that actually bounds this kernel: warp-instruction ISSUE (4 schedulers x 1 instruction/clk per SM).  The executed
        # instruction count per 32 samples is ncu's smsp__inst_executed of the specialised program (profiles/r2_jit_aba_*: 12.4 k; the
        # generic kernel pair: 27.5 k, profiles/r1_aba_f32_fast_smem_kernel_2p20_summary.txt) -- a constant of the program, not measured
        # in this run; the clock is the one sampled under load above.
        try:
            if args.dtype == "f32" and clocks and clocks.get("sm_mhz"):
                wi = 12.4e3 if linfo.specialised else 27.5e3
                ipc_peak = 148 * 4 * float(clocks["sm_mhz"]) * 1e6
                issued = value / world / 32.0 * wi
                out["roofline_issue"] = {"bound": "warp-instruction issue", "achieved": issued / 1e9, "peak": ipc_peak / 1e9,
                                         "unit": "G warp-instr/s", "frac": issued / ipc_peak, "warp_instr_per_32_samples": wi,
                                         "evals_per_s_at_peak_issue": ipc_peak / wi * 32.0}
        except Exception:      # a descriptor, never a reason to lose the bench line
            pass
        if config5:
            out["with_nccl_gather"] = config5["with_nccl_gather"]
            out["strong_scaling"] = config5["strong_scaling"]
        if world == 1 and not args.no_other:
            out["other_configs"] = add_rooflines(other_configs(max(5, min(args.steps, 20))), peak)
        if not args.no_cpu and world == 1:
            out["cpu_baseline"] = cpu_baseline(mech, q, v, tau, args.dtype)
            # accuracy of this run against the fp64 oracle on a small sample
            from oracle import Oracle
            o = Oracle(mech.flatten())
            n = 1024
            ref = o.dynamics(q[:, :n], v[:, :n], tau[:, :n])
            got = result.vd[:, :n].double().cpu().numpy()
            scale = np.maximum(1.0, np.abs(ref).max(0))
            out["accuracy"] = {"max_rel_err_vs_fp64_oracle": float((np.abs(got - ref).max(0) / scale).max()), "samples": n}
        _emit(out)
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "vd.npy"), dump.cpu().numpy())
    if dist is not None:
        dist.destroy_process_group()
    if jit_cache is not None:
        jit_cache.cleanup()


if __name__ == "__main__":
    main()

"""TEST INFRASTRUCTURE: runs the device algorithms of csrc/rbd_device.cuh on the CPU (see hostsim.cpp)."""
import ctypes, os, subprocess
import numpy as np
from rigidbodydynamics.jl_b200._cabi import RbdModelDesc, make_desc

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "..", "..", "rigidbodydynamics", "jl_b200", "csrc")
_LIB = os.path.join(_HERE, "libhostsim.so")


def build(force=False):
    srcs = [os.path.join(_HERE, "hostsim.cpp")] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)
                                                   if f.endswith((".cuh", ".h", ".cpp"))]
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", _LIB,
                               os.path.join(_HERE, "hostsim.cpp"), os.path.join(_CSRC, "rbd_model.cpp"),
                               os.path.join(_CSRC, "rbd_codegen.cpp")])
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def info(desc):
    d, keep = make_desc(desc)
    nrows, general, nslots = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    order = (ctypes.c_int * desc.nb)()
    rc = lib().hostsim_info(ctypes.byref(d), ctypes.byref(nrows), ctypes.byref(general), ctypes.byref(nslots), order)
    assert rc == 0, rc
    return dict(nrows=nrows.value, general=general.value, nslots=nslots.value, order=list(order))


def dynamics(desc, q, v, tau=None, wext=None, want_qd=False):
    dt = q.dtype
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q); v = np.ascontiguousarray(v, dt)
    tau = None if tau is None else np.ascontiguousarray(tau, dt)
    wext = None if wext is None else np.ascontiguousarray(wext, dt)
    B = q.shape[1]
    vd = np.empty((desc.nv, B), dt)
    qd = np.empty((desc.nq, B), dt) if want_qd else None
    fn = lib().hostsim_dynamics
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 6
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(v), _p(tau), _p(wext), _p(vd), _p(qd))
    assert rc == 0, rc
    return (vd, qd) if want_qd else vd


def inverse_dynamics(desc, q, v, vd=None, wext=None):
    dt = q.dtype
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q); v = np.ascontiguousarray(v, dt)
    vd = None if vd is None else np.ascontiguousarray(vd, dt)
    wext = None if wext is None else np.ascontiguousarray(wext, dt)
    B = q.shape[1]
    tau = np.empty((desc.nv, B), dt)
    fn = lib().hostsim_inverse_dynamics
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 5
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(v), _p(vd), _p(wext), _p(tau))
    assert rc == 0, rc
    return tau


def mass_matrix(desc, q):
    dt = q.dtype
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q)
    B = q.shape[1]
    M = np.full((desc.nv * desc.nv, B), np.nan, dt)
    fn = lib().hostsim_mass_matrix
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 2
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(M))
    assert rc == 0, rc
    return M


def dynamics_derivatives(desc, q, v, tau=None):
    """csrc/rbd_deriv.cuh on the CPU: (vd [nv, B], dvd_dq [nv*nv, B], dvd_dv [nv*nv, B]), entry (i, j) at row i + j*nv."""
    dt = q.dtype
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q); v = np.ascontiguousarray(v, dt)
    tau = None if tau is None else np.ascontiguousarray(tau, dt)
    B, nv = q.shape[1], desc.nv
    vd = np.empty((nv, B), dt)
    dq = np.zeros((nv * nv, B), dt); dv = np.zeros((nv * nv, B), dt)
    fn = lib().hostsim_derivatives
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 6
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(v), _p(tau), _p(vd), _p(dq), _p(dv))
    assert rc == 0, rc
    return vd, dq, dv


def dynamics_dual(desc, q, v, tau=None):
    """Dual{Float64,6} arrays [rows, B, 7]."""
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q, np.float64); v = np.ascontiguousarray(v, np.float64)
    tau = None if tau is None else np.ascontiguousarray(tau, np.float64)
    B = q.shape[1]
    vd = np.full((desc.nv, B, 7), np.nan)
    fn = lib().hostsim_dynamics_dual
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int64] + [ctypes.c_void_p] * 4
    rc = fn(ctypes.byref(d), B, _p(q), _p(v), _p(tau), _p(vd))
    assert rc == 0, rc
    return vd


def integrate(desc, q, v, tau=None, dt=1e-4, nsteps=1):
    dt_ = q.dtype
    d, keep = make_desc(desc)
    q = np.array(q, dt_, order="C"); v = np.array(v, dt_, order="C")
    tau = None if tau is None else np.ascontiguousarray(tau, dt_)
    fn = lib().hostsim_integrate
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                   ctypes.c_double, ctypes.c_int]
    rc = fn(ctypes.byref(d), 0 if dt_ == np.float32 else 1, q.shape[1], _p(q), _p(v), _p(tau), float(dt), int(nsteps))
    assert rc == 0, rc
    return q, v


KIN_ROWS = ("transforms", "com", "ke", "pe", "momentum", "mrb", "A", "J")


def kinematics(desc, q, v=None, sign=None, want=KIN_ROWS):
    """kin_sample on the CPU; returns the same dict as Oracle.kinematics."""
    dt = q.dtype
    d, keep = make_desc(desc)
    q = np.ascontiguousarray(q); v = None if v is None else np.ascontiguousarray(v, dt)
    B = q.shape[1]
    rows = {"transforms": 12 * desc.nb, "com": 3, "ke": 1, "pe": 1, "momentum": 6, "mrb": 6, "A": 6 * desc.nv, "J": 6 * desc.nv}
    out = {k: (np.full((rows[k], B), np.nan, dt) if k in want else None) for k in KIN_ROWS}
    if v is None:
        out["ke"] = out["momentum"] = out["mrb"] = None
    sg = None if sign is None else np.ascontiguousarray(sign, np.int8)
    if sg is None:
        out["J"] = None
    ptrs = (ctypes.c_void_p * 8)(*[None if out[k] is None else out[k].ctypes.data for k in KIN_ROWS])
    fn = lib().hostsim_kinematics
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                   ctypes.c_void_p]
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(v), _p(sg), ptrs)
    assert rc == 0, rc
    return {k: a for k, a in out.items() if a is not None}


def flags(desc):
    """Per-body flag words (csrc/rbd_types.h BodyFlags) in preorder."""
    d, keep = make_desc(desc)
    out = (ctypes.c_int * desc.nb)()
    rc = lib().hostsim_flags(ctypes.byref(d), out)
    assert rc == 0, rc
    return list(out)


SPEC_STATS = ("nodes_traced", "nodes_live", "add", "mul", "div", "neg", "sincos", "load", "store", "sld", "sst", "stash_rows")


def spec_source(desc, algo="aba", dtype=np.float64, has_in2=True, has_out1=False, flavor=0):
    """Source text + statistics of the model-specialised program csrc/rbd_codegen.cpp generates for this mechanism."""
    d, keep = make_desc(desc)
    fn = lib().hostsim_spec_source
    fn.restype = ctypes.c_void_p
    fn.argtypes = [ctypes.POINTER(RbdModelDesc)] + [ctypes.c_int] * 5 + [ctypes.c_void_p]
    stats = (ctypes.c_int * 12)()
    p = fn(ctypes.byref(d), {"aba": 0, "rnea": 1, "crba": 2, "kin": 3}[algo], 0 if np.dtype(dtype) == np.float32 else 1, int(has_in2),
           int(has_out1), flavor, stats)
    assert p, "specialisation failed"
    src = ctypes.string_at(p).decode()
    lib().hostsim_free.argtypes = [ctypes.c_void_p]
    lib().hostsim_free(p)
    return src, dict(zip(SPEC_STATS, stats))


def spec_kin(mask, sign=None, nb=0):
    """Select the rbd_kinematics variant the next spec_source / SpecProgram(algo="kin") call generates: bit k of ``mask`` = output k of
    KIN_ROWS, ``sign`` = the geometric jacobian's path signs in reference joint order."""
    sg = None if sign is None else np.ascontiguousarray(sign, np.int8)
    lib().hostsim_spec_kin.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int]
    lib().hostsim_spec_kin(int(mask), _p(sg), int(nb))


class SpecProgram:
    """The specialised program compiled for the CPU (g++) -- the same straight-line code the NVRTC kernels run."""

    def __init__(self, desc, algo="aba", dtype=np.float64, has_in2=True, has_out1=False):
        import hashlib, tempfile
        self.desc, self.algo, self.dtype = desc, algo, np.dtype(dtype)
        src, self.stats = spec_source(desc, algo, dtype, has_in2, has_out1, 0)
        tag = hashlib.sha1(src.encode()).hexdigest()[:16]
        d = os.path.join(tempfile.gettempdir(), f"rbd_spec_cpu_{os.getuid()}")      # per user: /tmp is shared
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, f"spec_{tag}.so")
        if not os.path.exists(so):
            cpp = os.path.join(d, f"spec_{tag}.cpp")
            with open(cpp, "w") as f:
                f.write(src)
            subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-ffp-contract=off",
                                   "-I", _CSRC, "-o", so + ".tmp", cpp])
            os.replace(so + ".tmp", so)
        self.fn = ctypes.CDLL(so).rbd_spec_cpu
        self.fn.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_longlong, ctypes.c_void_p] + ([ctypes.c_void_p] if algo == "kin" else [])
        self.has_in2, self.has_out1 = has_in2, has_out1

    def run_kin(self, q, v, rows):
        """rbd_kinematics variant: ``rows`` = list of 8 row counts (0 = output not requested); returns the list of outputs."""
        dt = self.dtype
        q = np.ascontiguousarray(q, dt); v = None if v is None else np.ascontiguousarray(v, dt)
        B = q.shape[1]
        outs = [np.full((r, B), np.nan, dt) if r else None for r in rows]
        sh = np.zeros(self.stats["stash_rows"] + 8, dt)
        es = dt.itemsize
        for b in range(B):
            ko = (ctypes.c_void_p * 8)(*[None if o is None else o.ctypes.data + b * es for o in outs])
            self.fn(q.ctypes.data + b * es, None if v is None else v.ctypes.data + b * es, None, None, None, B, sh.ctypes.data, ko)
        return outs

    def run(self, q, v, in2=None, out0_rows=None, out1_rows=None):
        dt = self.dtype
        q = np.ascontiguousarray(q, dt); v = np.ascontiguousarray(v, dt)
        in2 = None if in2 is None else np.ascontiguousarray(in2, dt)
        B = q.shape[1]
        o0 = np.full((out0_rows or self.desc.nv, B), np.nan, dt)
        o1 = np.full((out1_rows or self.desc.nq, B), np.nan, dt) if self.has_out1 else None
        sh = np.zeros(self.stats["stash_rows"] + 8, dt)
        es = dt.itemsize
        for b in range(B):
            self.fn(q.ctypes.data + b * es, v.ctypes.data + b * es, None if in2 is None else in2.ctypes.data + b * es,
                    o0.ctypes.data + b * es, None if o1 is None else o1.ctypes.data + b * es, B, sh.ctypes.data)
        return (o0, o1) if self.has_out1 else o0


def contact(desc, q, v, cd, s=None):
    """contact_sample (csrc/rbd_kin.cuh) on the CPU for a ``ContactDesc``; returns (wrenches, state_derivatives, state)."""
    d, keep = make_desc(desc)
    st, keep2 = cd.c_struct()
    q = np.ascontiguousarray(q); v = np.ascontiguousarray(v, q.dtype)
    dt, B = q.dtype, q.shape[1]
    ns = cd.nstates
    s = np.zeros((ns, B), dt) if s is None else np.array(s, dt, copy=True, order="C")
    sd = np.full((ns, B), np.nan, dt); wr = np.full((6 * desc.nb, B), np.nan, dt)
    fn = lib().hostsim_contact
    fn.argtypes = [ctypes.POINTER(RbdModelDesc), ctypes.c_int, ctypes.c_int64] + [ctypes.c_void_p] * 6
    rc = fn(ctypes.byref(d), 0 if dt == np.float32 else 1, B, _p(q), _p(v), ctypes.byref(st), _p(s), _p(sd), _p(wr))
    assert rc == 0, rc
    return wr, sd, s

"""CPU ORACLE (test infrastructure, NOT product code): ctypes front-end of oracle/libik_oracle.so.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
PARITY UNPINNED -- see oracle/ik_oracle.h.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from . import urdf_flatten

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

TASK_FRAME, TASK_ALIGN_AXIS, TASK_POSTURE, TASK_COM = 0, 1, 2, 3
POSITION, ORIENTATION, FULL = 0, 1, 2

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class _CModel(C.Structure):
    _fields_ = [("njoints", C.c_int), ("nq", C.c_int), ("nv", C.c_int), ("parent", _ip), ("jtype", _ip),
                ("idx_q", _ip), ("idx_v", _ip), ("placement", _dp), ("axis", _dp), ("lower", _dp), ("upper", _dp),
                ("nframes", C.c_int), ("frame_parent", _ip), ("frame_placement", _dp), ("mass", _dp), ("com", _dp)]


class _CProblem(C.Structure):
    _fields_ = [("ntasks", C.c_int), ("max_priority_level", C.c_int), ("kind", _ip), ("frame", _ip), ("ref", _ip),
                ("type", _ip), ("priority", _ip), ("weight", _dp), ("mask", _dp),
                ("nconstraints", C.c_int), ("c_frame", _ip), ("c_ref", _ip), ("c_type", _ip)]


class _CParams(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("step_length", C.c_double), ("damping", C.c_double),
                ("tolerance", C.c_double)]


def build(force=False):
    so = os.path.join(_HERE, "libik_oracle.so")
    src = os.path.join(_HERE, "ik_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.iko_dls.restype = C.c_int
    return _LIB


_LIB_FMA = None


def lib_fma():
    """The FP64 restatement compiled with fused multiply-adds (-ffp-contract=fast -mfma): same algorithm, other rounding."""
    global _LIB_FMA
    if _LIB_FMA is None:
        build()
        so = os.path.join(_HERE, "libik_oracle_fma.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-C", _HERE, "-s"])
        _LIB_FMA = C.CDLL(so)
    return _LIB_FMA


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _pd(a):
    return a.ctypes.data_as(_dp)


def _pi(a):
    return a.ctypes.data_as(_ip)


class Model:
    def __init__(self, flat):
        self.flat = flat
        self.nq, self.nv, self.njoints, self.nframes = flat["nq"], flat["nv"], flat["njoints"], flat["nframes"]
        flat.setdefault("mass", np.zeros(self.njoints))
        flat.setdefault("com", np.zeros((self.njoints, 3)))
        self._keep = {k: np.ascontiguousarray(flat[k]) for k in
                      ("parent", "jtype", "idx_q", "idx_v", "placement", "axis", "lower", "upper", "frame_parent",
                       "frame_placement")}
        self._keep["mass"] = np.ascontiguousarray(flat["mass"], dtype=np.float64)
        self._keep["com"] = np.ascontiguousarray(flat["com"], dtype=np.float64)
        k = self._keep
        self.c = _CModel(self.njoints, self.nq, self.nv, _pi(k["parent"]), _pi(k["jtype"]), _pi(k["idx_q"]),
                         _pi(k["idx_v"]), _pd(k["placement"]), _pd(k["axis"]), _pd(k["lower"]), _pd(k["upper"]),
                         self.nframes, _pi(k["frame_parent"]), _pd(k["frame_placement"]), _pd(k["mass"]), _pd(k["com"]))

    @classmethod
    def from_urdf(cls, xml_text, free_flyer=True):
        return cls(urdf_flatten.flatten_urdf(xml_text, free_flyer))

    def frame_id(self, name):
        return urdf_flatten.frame_id(self.flat, name)

    def neutral(self):
        q = np.zeros(self.nq)
        for j in range(self.njoints):
            if self.flat["jtype"][j] == urdf_flatten.J_FREEFLYER:
                q[self.flat["idx_q"][j] + 6] = 1.0
        return q

    def fk(self, q):
        out = np.zeros((self.njoints, 12))
        lib().iko_fk(C.byref(self.c), _pd(_d(q)), _pd(out))
        return out

    def frame_placement(self, q, frame):
        oMi = self.fk(q)
        out = np.zeros(12)
        lib().iko_frame_placement(C.byref(self.c), _pd(oMi), C.c_int(frame), _pd(out))
        return out

    def frame_jacobian_local(self, q, frame):
        oMi = self.fk(q)
        Jw = np.zeros((6, self.nv))
        Jf = np.zeros((6, self.nv))
        lib().iko_joint_jacobians(C.byref(self.c), _pd(oMi), _pd(Jw))
        lib().iko_frame_jacobian_local(C.byref(self.c), _pd(oMi), _pd(Jw), C.c_int(frame), _pd(Jf))
        return Jf

    def center_of_mass(self, q):
        """pinocchio::jacobianCenterOfMass: (com [3], Jcom [3, nv]) in the world frame."""
        com = np.zeros(3)
        J = np.zeros((3, self.nv))
        lib().iko_center_of_mass(C.byref(self.c), _pd(_d(q)), _pd(com), _pd(J))
        return com, J

    def integrate(self, q, v):
        out = np.zeros(self.nq)
        lib().iko_integrate(C.byref(self.c), _pd(_d(q)), _pd(_d(v)), _pd(out))
        return out

    def clip(self, q):
        out = _d(q).copy()
        lib().iko_clip(C.byref(self.c), _pd(out))
        return out


class Problem:
    """Mirror of ik::InverseKinematicsProblem restricted to what the oracle needs (problem.hpp:9-206)."""

    def __init__(self, model, max_priority_level=0):
        self.model = model
        self.max_priority_level = max_priority_level
        self.tasks = []
        self.constraints = []
        self._c = None

    def add_frame_constraint(self, frame, ktype=FULL, ref="universe"):
        """FrameConstraint (frame.hpp:333-465): ik::dls keeps the frame's velocity relative to `ref` at zero."""
        self.constraints.append(dict(frame=self._fid(frame), ref=self._fid(ref), type=ktype, dim=6 if ktype == FULL else 3))
        self._c = None
        return len(self.constraints) - 1

    @property
    def c_size(self):
        return sum(x["dim"] for x in self.constraints)

    def constraint_jacobian(self, q):
        Jc = np.zeros((max(self.c_size, 1), self.model.nv))
        lib().iko_constraint_jacobian(C.byref(self.model.c), C.byref(self.c), _pd(_d(q)), _pd(Jc))
        return Jc[:self.c_size]

    def add_frame_task(self, frame, ktype=FULL, ref="universe", priority=0, weight=None):
        f, r = self._fid(frame), self._fid(ref)
        dim = 6 if ktype == FULL else 3
        self.tasks.append(dict(kind=TASK_FRAME, frame=f, ref=r, type=ktype, priority=priority, dim=dim, tsz=12,
                               weight=np.ones(dim) if weight is None else _d(weight), mask=np.zeros(0)))
        self._c = None
        return len(self.tasks) - 1

    def add_align_axis_task(self, frame, axis, ref="universe", priority=0, weight=None):
        f, r = self._fid(frame), self._fid(ref)
        self.tasks.append(dict(kind=TASK_ALIGN_AXIS, frame=f, ref=r, type=axis, priority=priority, dim=1, tsz=3,
                               weight=np.ones(1) if weight is None else _d(weight), mask=np.zeros(0)))
        self._c = None
        return len(self.tasks) - 1

    def add_posture_task(self, nj, priority=0, weight=None, mask=None):
        self.tasks.append(dict(kind=TASK_POSTURE, frame=0, ref=0, type=nj, priority=priority, dim=nj, tsz=nj,
                               weight=np.ones(nj) if weight is None else _d(weight),
                               mask=np.ones(nj) if mask is None else _d(mask)))
        self._c = None
        return len(self.tasks) - 1

    def add_com_task(self, ref="universe", priority=0, weight=None):
        """CentreOfMassTask (centre_of_mass.hpp:14-52): the centre of mass expressed in frame `ref` tracks a 3-vector."""
        self.tasks.append(dict(kind=TASK_COM, frame=0, ref=self._fid(ref), type=0, priority=priority, dim=3, tsz=3,
                               weight=np.ones(3) if weight is None else _d(weight), mask=np.zeros(0)))
        self._c = None
        return len(self.tasks) - 1

    def _fid(self, name):
        if isinstance(name, int):
            return name
        f = self.model.frame_id(name)
        if f >= self.model.nframes:
            raise KeyError("unknown frame %r" % name)
        return f

    @property
    def c(self):
        if self._c is None:
            t = self.tasks
            arr = lambda key: np.array([x[key] for x in t], dtype=np.int32)
            self._keep = dict(kind=arr("kind"), frame=arr("frame"), ref=arr("ref"), type=arr("type"),
                              priority=arr("priority"),
                              weight=_d(np.concatenate([x["weight"] for x in t]) if t else np.zeros(0)),
                              mask=_d(np.concatenate([x["mask"] for x in t] + [np.zeros(1)])))
            k = self._keep
            cs = self.constraints
            carr = lambda key: np.array([x[key] for x in cs] + [0], dtype=np.int32)
            k.update(c_frame=carr("frame"), c_ref=carr("ref"), c_type=carr("type"))
            self._c = _CProblem(len(t), self.max_priority_level, _pi(k["kind"]), _pi(k["frame"]), _pi(k["ref"]),
                                _pi(k["type"]), _pi(k["priority"]), _pd(k["weight"]), _pd(k["mask"]),
                                len(cs), _pi(k["c_frame"]), _pi(k["c_ref"]), _pi(k["c_type"]))
        return self._c

    @property
    def target_size(self):
        return sum(x["tsz"] for x in self.tasks)

    @property
    def rows(self):
        return sum(x["dim"] for x in self.tasks)

    def e_size(self, priority):
        return sum(x["dim"] for x in self.tasks if x["priority"] == priority)

    def evaluate(self, q, targets):
        e = np.zeros(self.rows)
        J = np.zeros((self.rows, self.model.nv))
        lib().iko_evaluate(C.byref(self.model.c), C.byref(self.c), _pd(_d(q)), _pd(_d(targets)), _pd(e), _pd(J))
        return e, J


def params(max_iterations=100, step_length=1.0, damping=1e-2, tolerance=1e-4):
    """Library defaults: common.hpp:61-65, dls.hpp:25, visitor.hpp:19."""
    return _CParams(max_iterations, step_length, damping, tolerance)


def dls(problem, q0, targets, prm=None):
    """ik::dls (dls.cpp:5-78) on one problem.  Returns q, success, iterations, resid, dq."""
    prm = prm or params()
    m = problem.model
    q = np.zeros(m.nq)
    dq = np.zeros(m.nv)
    it = C.c_int(0)
    res = C.c_double(0)
    ok = lib().iko_dls(C.byref(m.c), C.byref(problem.c), C.byref(prm), _pd(_d(q0)), _pd(_d(targets)), _pd(q),
                       C.byref(it), C.byref(res), _pd(dq))
    return q, bool(ok), it.value, res.value, dq


def dls_batch(problem, q0, targets, prm=None, nthreads=1, fma=False):
    """Loop of ik::dls over a batch.  q0 [B, nq], targets [B, target_size] (AoS).  fma=True: the FMA-contracted build."""
    prm = prm or params()
    m = problem.model
    q0 = _d(q0)
    targets = _d(targets)
    B = q0.shape[0]
    assert q0.shape == (B, m.nq) and targets.shape == (B, problem.target_size)
    q = np.zeros((B, m.nq))
    ok = np.zeros(B, dtype=np.uint8)
    it = np.zeros(B, dtype=np.int32)
    res = np.zeros(B)
    (lib_fma() if fma else lib()).iko_dls_batch(C.byref(m.c), C.byref(problem.c), C.byref(prm), C.c_int(B), _pd(q0), _pd(targets),
                                                _pd(q), ok.ctypes.data_as(C.POINTER(C.c_ubyte)), _pi(it), _pd(res),
                                                C.c_int(nthreads))
    return q, ok.astype(bool), it, res


_PIK_LEVELS = "the ik::pik oracle holds IKO_MAX_LEVELS = 8 priority levels: a task has priority 8 or more"


class _CPikParams(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("step_length", C.c_double), ("tolerance", C.c_double),
                ("lam", C.c_double * 8)]


# ---- FP32 build of the same restatement (libik_oracle_f32.so, ik_oracle.c -DIKO_F32) ---------------------------------
_fp = C.POINTER(C.c_float)
_LIB32 = None


class _CModelF(C.Structure):
    _fields_ = [(n, _fp if t is _dp else t) for n, t in _CModel._fields_]


class _CProblemF(C.Structure):
    _fields_ = [(n, _fp if t is _dp else t) for n, t in _CProblem._fields_]


class _CParamsF(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("step_length", C.c_float), ("damping", C.c_float), ("tolerance", C.c_float)]


def lib_f32():
    global _LIB32
    if _LIB32 is None:
        build()
        so = os.path.join(_HERE, "libik_oracle_f32.so")
        if not os.path.exists(so):
            subprocess.check_call(["make", "-C", _HERE, "-s"])
        _LIB32 = C.CDLL(so)
    return _LIB32


def _f32_structs(problem):
    """The model / problem structs of `problem` with every float64 array converted to float32 (returns the structs and the
    arrays they point into, which the caller keeps alive)."""
    m = problem.model
    keep = []

    def conv(struct, cls):
        vals = []
        for (n, t), (_, tf) in zip(struct._fields_, cls._fields_):
            v = getattr(struct, n)
            if t is _dp:
                # the float64 array behind the pointer: look its length up in the owners' keep-alive dicts
                src = next(a for a in list(m._keep.values()) + list(problem._keep.values())
                           if a.dtype == np.float64 and a.ctypes.data == C.cast(v, C.c_void_p).value)
                with np.errstate(over="ignore"):  # +-DBL_MAX limits of the free-flyer become +-inf
                    a32 = np.ascontiguousarray(src, dtype=np.float32)
                keep.append(a32)
                v = a32.ctypes.data_as(_fp)
            vals.append(v)
        return cls(*vals)

    pc = problem.c  # materialises problem._keep
    return conv(m.c, _CModelF), conv(pc, _CProblemF), keep


def _f32_batch(fn, problem, q0, targets, cprm, nthreads):
    cm, cp, keep = _f32_structs(problem)
    m = problem.model
    q0 = np.ascontiguousarray(q0, dtype=np.float32)
    targets = np.ascontiguousarray(targets, dtype=np.float32)
    B = q0.shape[0]
    assert q0.shape == (B, m.nq) and targets.shape == (B, problem.target_size)
    q = np.zeros((B, m.nq), dtype=np.float32)
    ok = np.zeros(B, dtype=np.uint8)
    it = np.zeros(B, dtype=np.int32)
    res = np.zeros(B, dtype=np.float32)
    rc = getattr(lib_f32(), fn)(C.byref(cm), C.byref(cp), C.byref(cprm), C.c_int(B), q0.ctypes.data_as(_fp),
                                targets.ctypes.data_as(_fp), q.ctypes.data_as(_fp), ok.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                _pi(it), res.ctypes.data_as(_fp), C.c_int(nthreads))
    return rc, (q.astype(np.float64), ok.astype(bool), it, res.astype(np.float64))


def dls_batch_f32(problem, q0, targets, prm=None, nthreads=1):
    """ik::dls looped over a batch with number_t = float: every scalar of the restatement (model constants, FK, log6,
    Gram, pivoted LDL^T, integrate, stop test) is single precision.  Returns float64 copies of q / resid."""
    prm = prm or params()
    cprm = _CParamsF(prm.max_iterations, prm.step_length, prm.damping, prm.tolerance)
    return _f32_batch("iko_dls_batch", problem, q0, targets, cprm, nthreads)[1]


class _CPikParamsF(C.Structure):
    _fields_ = [("max_iterations", C.c_int), ("step_length", C.c_float), ("tolerance", C.c_float), ("lam", C.c_float * 8)]


def pik_batch_f32(problem, q0, targets, prm=None, nthreads=1):
    """ik::pik looped over a batch with number_t = float (the FP32 build of the same restatement: SVD damped inverse,
    pivoted QR rank threshold with FLT_EPSILON, projector, integrate).  prm: pik_params(...).  Returns float64 copies."""
    prm = prm or pik_params()
    cprm = _CPikParamsF(prm.max_iterations, prm.step_length, prm.tolerance, (C.c_float * 8)(*prm.lam))
    rc, out = _f32_batch("iko_pik_batch", problem, q0, targets, cprm, nthreads)
    if rc != 0:
        raise ValueError(_PIK_LEVELS)
    return out


def pik_params(max_iterations=100, step_length=1.0, lambdas=None, tolerance=1e-4):
    """pik.hpp:13-18 and pik_data::lambda (pik.hpp:31: 1.0 per priority level)."""
    lambdas = list(lambdas or [])
    if len(lambdas) > 8:
        raise ValueError("the ik::pik oracle holds IKO_MAX_LEVELS = 8 lambdas; got %d" % len(lambdas))
    lam = (C.c_double * 8)(*([1.0] * 8))
    for i, v in enumerate(lambdas):
        lam[i] = float(v)
    return _CPikParams(max_iterations, step_length, tolerance, lam)


def pik(problem, q0, targets, prm=None):
    """ik::pik (pik.cpp:31-96) on one problem.  Returns q, success, iterations, resid, dq."""
    prm = prm or pik_params()
    m = problem.model
    q = np.zeros(m.nq)
    dq = np.zeros(m.nv)
    it = C.c_int(0)
    res = C.c_double(0)
    ok = lib().iko_pik(C.byref(m.c), C.byref(problem.c), C.byref(prm), _pd(_d(q0)), _pd(_d(targets)), _pd(q),
                       C.byref(it), C.byref(res), _pd(dq))
    if ok < 0:
        raise ValueError(_PIK_LEVELS)
    return q, bool(ok), it.value, res.value, dq


def pik_batch(problem, q0, targets, prm=None, nthreads=1):
    """Loop of ik::pik over a batch.  q0 [B, nq], targets [B, target_size] (AoS)."""
    prm = prm or pik_params()
    m = problem.model
    q0 = _d(q0)
    targets = _d(targets)
    B = q0.shape[0]
    assert q0.shape == (B, m.nq) and targets.shape == (B, problem.target_size)
    q = np.zeros((B, m.nq))
    ok = np.zeros(B, dtype=np.uint8)
    it = np.zeros(B, dtype=np.int32)
    res = np.zeros(B)
    rc = lib().iko_pik_batch(C.byref(m.c), C.byref(problem.c), C.byref(prm), C.c_int(B), _pd(q0), _pd(targets), _pd(q),
                             ok.ctypes.data_as(C.POINTER(C.c_ubyte)), _pi(it), _pd(res), C.c_int(nthreads))
    if rc != 0:
        raise ValueError(_PIK_LEVELS)
    return q, ok.astype(bool), it, res


def damp_pseudoinverse(M, lam):
    """damp_pseudoinverse (pik.cpp:5-21): M [m, n] -> [n, m]."""
    M = _d(M)
    m, n = M.shape
    out = np.zeros((n, m))
    lib().iko_damp_pseudoinverse(C.c_int(m), C.c_int(n), _pd(M), C.c_double(lam), _pd(out))
    return out


def rowspace_projector(M):
    """pinv(M) @ M through the restated complete orthogonal decomposition (pik.cpp:59-61).  Returns (P [n, n], rank)."""
    M = _d(M)
    m, n = M.shape
    out = np.zeros((n, n))
    lib().iko_rowspace_projector.restype = C.c_int
    r = lib().iko_rowspace_projector(C.c_int(m), C.c_int(n), _pd(M), _pd(out))
    return out, int(r)


def ldlt_solve(A, b):
    A = _d(A).copy()
    n = A.shape[0]
    x = np.zeros(n)
    lib().iko_ldlt_solve(C.c_int(n), _pd(A), _pd(_d(b)), _pd(x))
    return x


def _unary(name, x, nout):
    out = np.zeros(nout)
    getattr(lib(), name)(_pd(_d(x)), _pd(out))
    return out


def exp3(w):
    return _unary("iko_exp3", w, 9).reshape(3, 3)


def exp6(v):
    return _unary("iko_exp6", v, 12)


def log6(M):
    return _unary("iko_log6", M, 6)


def Jlog6(M):
    return _unary("iko_Jlog6", M, 36).reshape(6, 6)


def log3(R):
    w = np.zeros(3)
    t = C.c_double(0)
    lib().iko_log3(_pd(_d(R).reshape(-1)), _pd(w), C.byref(t))
    return w, t.value


def se3_mul(A, B):
    out = np.zeros(12)
    lib().iko_se3_mul(_pd(_d(A)), _pd(_d(B)), _pd(out))
    return out


def se3_actinv(A, B):
    out = np.zeros(12)
    lib().iko_se3_actinv(_pd(_d(A)), _pd(_d(B)), _pd(out))
    return out


def se3(R=None, p=None):
    R = np.eye(3) if R is None else np.asarray(R, dtype=np.float64).reshape(3, 3)
    p = np.zeros(3) if p is None else np.asarray(p, dtype=np.float64)
    return np.concatenate([R.reshape(-1), p])

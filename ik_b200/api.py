"""Host-side mirror of the reference's task / solver interface (namespace ik), over the C ABI.

Names, argument meaning and failure behaviour follow dazzmo/ik so the parity tests read like tests of the
reference: ``InverseKinematicsProblem`` (ik/ik/problem.hpp:9-206), ``FrameTask`` / ``KinematicType``
(frame.hpp:20,78-200), ``AlignAxisTask`` (frame.hpp:210-319), ``PostureTask`` (posture.hpp:17-86),
``dls_parameters`` (dls.hpp:24-28), ``dls_data`` (dls.hpp:34-65, data.hpp:8-28), ``dls`` (dls.hpp:111-114).
The batched entry points (``dls_batch`` on device tensors, ``dls_batch_host`` on host arrays) are the
extension the reference lacks.  All arithmetic happens in libikb200.so on the GPU; there is no CPU path.
"""
import ctypes as C
import enum
import os

import numpy as np

from . import _capi as capi

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


class KinematicType(enum.IntEnum):  # frame.hpp:20
    Position = 0
    Orientation = 1
    Full = 2


class AlignAxisType(enum.IntEnum):  # frame.hpp:202
    AxisX = 0
    AxisY = 1
    AxisZ = 2


def _as_f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Model:
    """Flattened kinematic tree; stands in for ik::model_t = pinocchio::Model (common.hpp:17)."""

    def __init__(self, handle):
        self._h = handle
        lib = capi.lib
        self.njoints = lib.ikb_model_njoints(handle)
        self.nq = lib.ikb_model_nq(handle)
        self.nv = lib.ikb_model_nv(handle)
        self.nframes = lib.ikb_model_nframes(handle)
        self.names = [lib.ikb_model_joint_name(handle, j).decode() for j in range(self.njoints)]
        self.frame_names = [lib.ikb_model_frame_name(handle, f).decode() for f in range(self.nframes)]
        self.parents = np.zeros(self.njoints, dtype=np.int32)
        self.jtypes = np.zeros(self.njoints, dtype=np.int32)
        self.idx_qs = np.zeros(self.njoints, dtype=np.int32)
        self.idx_vs = np.zeros(self.njoints, dtype=np.int32)
        i32 = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
        capi.check(lib.ikb_model_get_topology(handle, i32(self.parents), i32(self.jtypes), i32(self.idx_qs),
                                              i32(self.idx_vs)), "ikb_model_get_topology")
        self.jointPlacements = np.zeros((self.njoints, 12))
        self.axes = np.zeros((self.njoints, 3))
        capi.check(lib.ikb_model_get_placements(handle, _dptr(self.jointPlacements), _dptr(self.axes)),
                   "ikb_model_get_placements")
        self.frame_parents = np.zeros(self.nframes, dtype=np.int32)
        self.frame_types = np.zeros(self.nframes, dtype=np.int32)
        self.framePlacements = np.zeros((self.nframes, 12))
        capi.check(lib.ikb_model_get_frames(handle, i32(self.frame_parents), i32(self.frame_types),
                                            _dptr(self.framePlacements)), "ikb_model_get_frames")

    def __del__(self):
        if getattr(self, "_h", None) and capi is not None and getattr(capi, "lib", None) is not None:  # (None at interpreter exit)
            capi.lib.ikb_model_free(self._h)
            self._h = None

    @classmethod
    def from_urdf(cls, xml_text, free_flyer=True):
        """pinocchio::urdf::buildModelFromXML(xml, JointModelFreeFlyer(), model) (cassie.cpp:34-35)."""
        data = xml_text.encode() if isinstance(xml_text, str) else xml_text
        h = C.c_void_p()
        capi.check(capi.lib.ikb_model_from_urdf(data, len(data), int(free_flyer), C.byref(h)), "ikb_model_from_urdf")
        return cls(h)

    @classmethod
    def builtin(cls, name, free_flyer=True):
        with open(os.path.join(_DATA, name + ".urdf")) as f:
            return cls.from_urdf(f.read(), free_flyer)

    def getFrameId(self, name):
        """model.getFrameId(name): nframes when the frame does not exist (common.hpp:50)."""
        return capi.lib.ikb_model_frame_id(self._h, name.encode())

    @property
    def lowerPositionLimit(self):
        lo = np.zeros(self.nq)
        capi.check(capi.lib.ikb_model_get_limits(self._h, _dptr(lo), None), "ikb_model_get_limits")
        return lo

    @property
    def upperPositionLimit(self):
        hi = np.zeros(self.nq)
        capi.check(capi.lib.ikb_model_get_limits(self._h, None, _dptr(hi)), "ikb_model_get_limits")
        return hi

    def set_limits(self, lower=None, upper=None):
        lo = _as_f64(lower) if lower is not None else None
        hi = _as_f64(upper) if upper is not None else None
        capi.check(capi.lib.ikb_model_set_limits(self._h, _dptr(lo) if lo is not None else None,
                                                 _dptr(hi) if hi is not None else None), "ikb_model_set_limits")

    def inertias(self):
        """(mass [njoints], centre of mass in the joint frame [njoints, 3]) of the bodies each joint supports."""
        mass, com = np.zeros(self.njoints), np.zeros((self.njoints, 3))
        capi.check(capi.lib.ikb_model_get_inertias(self._h, _dptr(mass), _dptr(com)), "ikb_model_get_inertias")
        return mass, com

    def set_inertias(self, mass, com):
        mass, com = _as_f64(mass), _as_f64(com)
        if mass.shape != (self.njoints,) or com.shape != (self.njoints, 3):
            raise ValueError("inertias: expected mass [%d] and com [%d, 3]" % (self.njoints, self.njoints))
        capi.check(capi.lib.ikb_model_set_inertias(self._h, _dptr(mass), _dptr(com)), "ikb_model_set_inertias")

    def neutral(self):
        q = np.zeros(self.nq)
        capi.check(capi.lib.ikb_model_neutral(self._h, _dptr(q)), "ikb_model_neutral")
        return q


class Task:  # task.hpp:19-57
    def __init__(self, dimension):
        self._dimension = dimension
        self._weighting = np.ones(dimension)

    def dimension(self):
        return self._dimension

    def weighting(self):
        return self._weighting


class FrameTask(Task):  # frame.hpp:78-200
    def __init__(self, model, frame, type=KinematicType.Full, reference_frame="universe"):
        self.type = KinematicType(type)
        super().__init__(6 if self.type == KinematicType.Full else 3)
        self.frame = frame
        self.reference_frame = reference_frame
        self.target = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], dtype=np.float64)  # se3_t::Identity()

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))
    target_size = 12


class FrameConstraint:  # frame.hpp:333-465 -- hard constraint: ik::dls keeps `frame` at rest relative to `reference_frame`
    def __init__(self, model, frame, type=KinematicType.Full, reference_frame="universe"):
        self.type = KinematicType(type)
        self._dim = 6 if self.type == KinematicType.Full else 3
        self.frame = frame
        self.reference_frame = reference_frame
        self.target = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], dtype=np.float64)  # declared, not read by ik::dls

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))

    def dimension(self):
        return self._dim


class AlignAxisTask(Task):  # frame.hpp:210-319
    def __init__(self, model, frame, axis, reference_frame="universe"):
        super().__init__(1)
        self.axis = AlignAxisType(axis)
        self.frame = frame
        self.reference_frame = reference_frame
        self.target = np.zeros(3)

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))
    target_size = 3


class PostureTask(Task):  # posture.hpp:17-86
    def __init__(self, model, nj):
        super().__init__(nj)
        self.nj = nj
        self.target = np.zeros(nj)
        self.mask = np.ones(nj)

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))

    @property
    def target_size(self):
        return self.nj


class CentreOfMassTask(Task):  # centre_of_mass.hpp:14-52
    def __init__(self, model, reference_frame="universe"):
        super().__init__(3)
        self.reference_frame = reference_frame
        self.target = np.zeros(3)  # centre of mass expressed in the reference frame

    create = classmethod(lambda cls, *a, **k: cls(*a, **k))
    target_size = 3


class dls_parameters:  # dls.hpp:24-28 + common.hpp:59-66
    def __init__(self, max_iterations=100, max_time=1.0, step_length=1.0, damping=1e-2, random_restart=False,
                 tolerance=1e-4):
        self.max_iterations = max_iterations
        self.max_time = max_time
        self.step_length = step_length
        self.damping = damping
        self.random_restart = random_restart
        self.tolerance = tolerance  # visitor.hpp:19

    def c(self):
        return capi.DlsParams(self.max_iterations, int(self.random_restart), self.max_time, self.step_length,
                              self.damping, self.tolerance)


class pik_parameters:  # pik.hpp:13-18 + pik_data::lambda (pik.hpp:31)
    def __init__(self, max_iterations=100, damping=1e-2, step_length=1.0, max_time=1.0, lambdas=None, tolerance=1e-4):
        self.max_iterations = max_iterations
        self.damping = damping          # declared by the reference, never read (pik.cpp uses pik_data::lambda)
        self.step_length = step_length
        self.max_time = max_time
        self.lambdas = list(lambdas) if lambdas is not None else []   # per priority level; missing levels: 1.0
        if len(self.lambdas) > 7:
            raise ValueError("ik::pik holds at most 7 priority levels (ikb_pik_params::lambda); got %d lambdas" % len(self.lambdas))
        self.tolerance = tolerance

    def c(self):
        p = capi.PikParams()
        capi.lib.ikb_pik_params_default(C.byref(p))
        p.max_iterations = int(self.max_iterations)
        p.step_length = float(self.step_length)
        p.tolerance = float(self.tolerance)
        for i, v in enumerate(self.lambdas):
            p.lam[i] = float(v)
        return p


class inverse_kinematics_visitor:  # visitor.hpp:7-24
    """The stock stop test runs in the kernel (`tolerance` is its squared-norm threshold).  A subclass that overrides
    should_stop is honoured by dls() / pik(): the iteration loop then runs on the host, one device iteration per step."""
    tolerance = 1e-4

    def should_stop(self, problem, e, dq):
        """visitor.hpp:15-21: e = list of the weighted error vectors per priority level; true when ||e[0]||^2 < 1e-4."""
        return float(np.dot(e[0], e[0])) < self.tolerance


class InverseKinematicsProblem:  # problem.hpp:9-206
    def __init__(self, model, max_priority_level=0):
        self._model = model
        self._max_priority_level = max_priority_level
        self._tasks = []  # (name, task, priority) in insertion order
        self._constraints = []  # (name, FrameConstraint) in insertion order
        self._h = None
        self._device = None
        self._sig = None

    def __del__(self):
        if getattr(self, "_h", None) and capi is not None and getattr(capi, "lib", None) is not None:
            capi.lib.ikb_problem_free(self._h)
            self._h = None

    def model(self):
        return self._model

    def max_priority_level(self):
        return self._max_priority_level

    def _add(self, name, task, priority):
        if self._h is not None:
            raise RuntimeError("problem already finalized (device constants are immutable)")
        if priority > self._max_priority_level:
            raise IndexError("Maximum priority level exceeded!")  # problem.hpp:162-163
        self._tasks.append((name, task, priority))
        return task

    def add_frame_constraint(self, name, constraint):  # problem.hpp:107-118
        if self._h is not None:
            raise RuntimeError("problem already finalized (device constants are immutable)")
        self._constraints.append((name, constraint))
        return constraint

    def get_all_constraints(self):  # problem.hpp:167-169
        return [c for _, c in self._constraints]

    def add_frame_task(self, name, task, priority=0):  # problem.hpp:55-66
        return self._add(name, task, priority)

    def add_align_axis_task(self, name, task, priority=0):  # problem.hpp:94-105
        return self._add(name, task, priority)

    def add_posture_task(self, name, task, priority=0):  # problem.hpp:134-145
        return self._add(name, task, priority)

    def add_centre_of_mass_task(self, task, priority=0):  # problem.hpp:121-128 (one per problem, no name)
        self._com_task = self._add("centre_of_mass", task, priority)
        return task

    def get_centre_of_mass_task(self):  # problem.hpp:130-132
        return getattr(self, "_com_task", None)

    def _get(self, name, cls):
        for n, t, _ in self._tasks:
            if n == name and isinstance(t, cls):
                return t
        raise KeyError("%s %r does not exist" % (cls.__name__, name))  # the reference indexes out of range here

    def get_frame_task(self, name):  # problem.hpp:79-81
        return self._get(name, FrameTask)

    def get_align_axis_task(self, name):
        return self._get(name, AlignAxisTask)

    def get_posture_task(self, name):
        return self._get(name, PostureTask)

    def get_all_tasks(self, priority):  # problem.hpp:160-165
        if priority > self._max_priority_level:
            raise IndexError("Maximum priority level exceeded!")
        return [t for _, t, p in self._tasks if p == priority]

    def e_size(self, priority):  # problem.hpp:34-40
        return sum(t.dimension() for t in self.get_all_tasks(priority))

    def c_size(self):  # problem.hpp:47-53
        return sum(c.dimension() for _, c in self._constraints)

    @property
    def target_size(self):
        return sum(t.target_size for _, t, _ in self._tasks)

    def target_offset(self, task):
        off = 0
        for _, t, _ in self._tasks:
            if t is task:
                return off
            off += t.target_size
        raise KeyError("task is not part of this problem")

    def gather_targets(self):
        """Flatten the tasks' public ``target`` members (frame.hpp:189) into one per-problem target vector."""
        parts = [_as_f64(t.target).reshape(-1) for _, t, _ in self._tasks]
        return np.concatenate(parts) if parts else np.zeros(0)

    def _build_handle(self, device):
        """Create the C-ABI problem handle; device=None stops before ikb_problem_finalize (host-only handle)."""
        lib = capi.lib
        h = C.c_void_p()
        capi.check(lib.ikb_problem_create(self._model._h, self._max_priority_level, C.byref(h)), "ikb_problem_create")
        try:
            m = self._model
            for name, t, prio in self._tasks:
                w = _as_f64(t.weighting())
                if isinstance(t, PostureTask):
                    mask = _as_f64(t.mask)
                    capi.check_index(lib.ikb_problem_add_posture_task(h, t.nj, prio, _dptr(w), _dptr(mask)),
                                     "ikb_problem_add_posture_task")
                    continue
                if isinstance(t, CentreOfMassTask):
                    r = m.getFrameId(t.reference_frame)
                    if r >= m.nframes:
                        raise KeyError("centre of mass task: unknown frame %r" % (t.reference_frame,))
                    capi.check_index(lib.ikb_problem_add_com_task(h, r, prio, _dptr(w)), "ikb_problem_add_com_task")
                    continue
                f, r = m.getFrameId(t.frame), m.getFrameId(t.reference_frame)
                if f >= m.nframes or r >= m.nframes:
                    raise KeyError("task %r: unknown frame %r / %r" % (name, t.frame, t.reference_frame))
                if isinstance(t, FrameTask):
                    capi.check_index(lib.ikb_problem_add_frame_task(h, f, int(t.type), r, prio, _dptr(w)),
                                     "ikb_problem_add_frame_task")
                else:
                    capi.check_index(lib.ikb_problem_add_align_axis_task(h, f, int(t.axis), r, prio, _dptr(w)),
                                     "ikb_problem_add_align_axis_task")
            for name, c in self._constraints:
                f, r = m.getFrameId(c.frame), m.getFrameId(c.reference_frame)
                if f >= m.nframes or r >= m.nframes:
                    raise KeyError("constraint %r: unknown frame %r / %r" % (name, c.frame, c.reference_frame))
                capi.check_index(lib.ikb_problem_add_frame_constraint(h, f, int(c.type), r), "ikb_problem_add_frame_constraint")
            if device is not None:
                capi.check(lib.ikb_problem_finalize(h, device), "ikb_problem_finalize")
        except Exception:
            lib.ikb_problem_free(h)
            raise
        return h

    def specialisation(self):
        """Name of the compiled topology-specialised kernel matching this problem, or None (host-only query)."""
        h = self._build_handle(None)
        try:
            n = capi.lib.ikb_problem_specialisation(h)
            return n.decode() if n else None
        finally:
            capi.lib.ikb_problem_free(h)

    # ---- device side ----
    def _signature(self):
        """Everything ikb_problem_finalize bakes into the handle: the task list, row weights, posture masks, joint limits.
        The reference reads `task->weighting()` and `mask` at every evaluation (data.cpp:49-50, posture.hpp:52) and the
        limits at every clamp (common.hpp:54-55), so edits between solves must take effect."""
        parts = [np.asarray(self._model.lowerPositionLimit, dtype=np.float64).tobytes(),
                 np.asarray(self._model.upperPositionLimit, dtype=np.float64).tobytes()]
        for name, t, prio in self._tasks:
            parts.append(("%s|%s|%d" % (name, type(t).__name__, prio)).encode())
            parts.append(_as_f64(t.weighting()).tobytes())
            if isinstance(t, PostureTask):
                parts.append(_as_f64(t.mask).tobytes())
        parts.append(str(len(self._constraints)).encode())
        return b"".join(parts)

    def finalize(self, device=0):
        if self._h is not None:
            if device is not None and self._device is not None and device != self._device:
                raise ValueError("problem is finalized on cuda:%d; its buffers / tensors must live there (got cuda:%d)"
                                 % (self._device, device))
            if self._signature() == self._sig:
                return self
            # weights / masks / limits were edited since the handle was built: rebuild it (queues created from the old
            # handle keep solving the old problem -- create them after the last edit)
            capi.lib.ikb_problem_free(self._h)
            self._h = None
            device = self._device
        self._h = self._build_handle(device)
        self._device = device
        self._sig = self._signature()
        return self

    def status_string(self):
        """Note on the kernel selection (ikb_problem_status_string): why a near-miss of a compiled specialisation fell back
        to the table-driven kernel; "" when there is nothing to say."""
        s = capi.lib.ikb_problem_status_string(self._h) if self._h is not None else b""
        return s.decode() if s else ""

    @property
    def compact_target_size(self):
        """Scalars per problem of the compact wire format of the targets (IKB_TARGETS_COMPACT, include/ikb200.h)."""
        h = self._h if self._h is not None else self._build_handle(None)
        try:
            return int(capi.lib.ikb_problem_compact_target_size(h))
        finally:
            if h is not self._h:
                capi.lib.ikb_problem_free(h)

    def compact_targets(self, targets):
        """SE3 target records [B, tsz] (AoS) -> compact records [B, csz]: per FrameTask Full = unit quaternion (x, y, z, w)
        + translation, Position = translation (the rotation must be the identity, FrameTask's default target),
        Orientation = quaternion; other tasks unchanged."""
        targets = np.asarray(targets, dtype=np.float64)
        parts, off = [], 0
        for _, t, _ in self._tasks:
            n = int(np.asarray(t.target).size)
            blk = targets[:, off:off + n]
            off += n
            if isinstance(t, FrameTask):
                R, tr = blk[:, :9].reshape(-1, 3, 3), blk[:, 9:12]
                if t.type == KinematicType.Position:
                    if not np.allclose(R, np.eye(3)[None], atol=0):
                        raise ValueError("compact Position targets carry no rotation: the SE3 target's rotation must be the identity")
                    parts.append(tr)
                elif t.type == KinematicType.Orientation:
                    parts.append(_rot_to_quat(R))
                else:
                    parts.append(np.concatenate([_rot_to_quat(R), tr], axis=1))
            else:
                parts.append(blk)
        return np.ascontiguousarray(np.concatenate(parts, axis=1))

    def kernel_name(self, dtype="f64"):
        n = capi.lib.ikb_problem_kernel_name(self._h, _DT[dtype][0])
        return n.decode() if n else None


_DT = {"f64": (capi.F64, np.float64), "f32": (capi.F32, np.float32)}


def _rot_to_quat(R):
    """Rotation matrices [B, 3, 3] -> unit quaternions [B, 4] (x, y, z, w), w >= 0 (Shepperd's method, vectorised)."""
    R = np.asarray(R, dtype=np.float64)
    B = R.shape[0]
    q = np.zeros((B, 4))
    tr = R[:, 0, 0] + R[:, 1, 1] + R[:, 2, 2]
    cand = np.stack([R[:, 0, 0], R[:, 1, 1], R[:, 2, 2], tr], axis=1)
    k = cand.argmax(axis=1)
    for i in range(3):
        m = k == i
        if not m.any():
            continue
        j, l = (i + 1) % 3, (i + 2) % 3
        s_ = np.sqrt(np.maximum(1.0 + R[m, i, i] - R[m, j, j] - R[m, l, l], 0)) * 2
        q[m, i] = 0.25 * s_
        q[m, j] = (R[m, j, i] + R[m, i, j]) / s_
        q[m, l] = (R[m, l, i] + R[m, i, l]) / s_
        q[m, 3] = (R[m, l, j] - R[m, j, l]) / s_
    m = k == 3
    if m.any():
        s_ = np.sqrt(np.maximum(tr[m] + 1.0, 0)) * 2
        q[m, 3] = 0.25 * s_
        q[m, 0] = (R[m, 2, 1] - R[m, 1, 2]) / s_
        q[m, 1] = (R[m, 0, 2] - R[m, 2, 0]) / s_
        q[m, 2] = (R[m, 1, 0] - R[m, 0, 1]) / s_
    q *= np.where(q[:, 3:4] < 0, -1.0, 1.0)
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def _host_io(problem, q0, targets, dtype, layout, out, compact=False, outputs=("q", "success", "iters", "resid")):
    """ikb_batch_io over HOST arrays.  layout "soa": q0 [nq, B], targets [tsz, B]; "aos": q0 [B, nq], targets [B, tsz]; a
    q0 of shape (nq,) is ONE initial guess for the whole batch (batch_stride = 0).  compact: `targets` holds the compact
    wire format (csz scalars per problem).  outputs: which of success / iters / resid come back (q always does).
    Returns (io, B, result dict, keep-alive tuple)."""
    code, npdt = _DT[dtype]
    nq = problem.model().nq
    tsz = problem.compact_target_size if compact else problem.target_size
    assert q0.dtype == npdt and targets.dtype == npdt and q0.flags.c_contiguous and targets.flags.c_contiguous
    if layout == "soa":
        B = targets.shape[1]
        assert targets.shape == (tsz, B)
        strides = lambda k: (B, 1)
        qshape = (nq, B)
    else:
        B = targets.shape[0]
        assert targets.shape == (B, tsz)
        strides = lambda k: (1, k)
        qshape = (B, nq)
    q0_strides = (1, 0) if q0.ndim == 1 else strides(nq)
    assert q0.shape == ((nq,) if q0.ndim == 1 else qshape)
    out = out or {}

    def buf(key, shape, dt):
        if key != "q" and key not in outputs:
            return None
        a = out.get(key)
        if a is None:
            a = np.empty(shape, dtype=dt)
        assert a.shape == shape and a.dtype == dt and a.flags.c_contiguous, "output %r: wrong shape / dtype / layout" % key
        return a

    q = buf("q", qshape, npdt)
    success, iters, resid = buf("success", (B,), np.uint8), buf("iters", (B,), np.int32), buf("resid", (B,), npdt)
    ptr = lambda a: a.ctypes.data if a is not None else None
    io = capi.BatchIO(q0.ctypes.data, *q0_strides, targets.ctypes.data, *strides(tsz), q.ctypes.data, *strides(nq),
                      ptr(success), ptr(iters), ptr(resid), capi.TARGETS_COMPACT if compact else capi.TARGETS_SE3, 0)
    res = dict(q=q, success=success, iters=iters, resid=resid)
    return io, B, res, (q0, targets, res)


class dls_data:  # dls.hpp:34-65 / data.hpp:8-28
    def __init__(self, problem):
        m = problem.model()
        rows = sum(int(t.dimension()) for _, t, _ in problem._tasks)
        self.success = False
        self.q = np.zeros(m.nq)
        self.dq = np.zeros(m.nv)            # problem_data::dq: the last step direction computed (dls.cpp:52)
        self.e = np.zeros(rows)             # stacked weighted task errors of the last evaluation (data.hpp:24, dls.cpp:18-24)
        self.J = np.zeros((rows, m.nv))     # stacked weighted task Jacobian of the last evaluation
        self.iterations = 0  # dls_info::iterations (dls.hpp:71-74), never filled by the reference
        self.residual = 0.0


def _solve_one(problem, q0, prm, pik_prm=None, want=True):
    m = problem.model()
    rows = sum(int(t.dimension()) for _, t, _ in problem._tasks)
    q0 = _as_f64(q0)
    tg = _as_f64(problem.gather_targets())
    q, dq, e, J = np.zeros(m.nq), np.zeros(m.nv), np.zeros(rows), np.zeros((rows, m.nv))
    ok, it, res = C.c_int(0), C.c_int(0), C.c_double(0)
    aux = (_dptr(dq), _dptr(e), _dptr(J)) if want else (None, None, None)
    if pik_prm is None:
        capi.check(capi.lib.ikb_dls_solve_ex(problem._h, C.byref(prm), _dptr(q0), _dptr(tg), _dptr(q), C.byref(ok), C.byref(it),
                                             C.byref(res), *aux), "ikb_dls_solve_ex")
    else:
        capi.check(capi.lib.ikb_pik_solve_ex(problem._h, C.byref(pik_prm), _dptr(q0), _dptr(tg), _dptr(q), C.byref(ok), C.byref(it),
                                             C.byref(res), *aux), "ikb_pik_solve_ex")
    return q, bool(ok.value), it.value, res.value, dq, e, J


def _stepped(problem, q0, data, visitor, p, pik):
    """A visitor that OVERRIDES should_stop (visitor.hpp:15-21 is virtual-by-convention in the reference): the loop of
    dls.cpp:14-74 runs on the host, one device iteration (evaluate, dq, integrate, clamp) per step, and the user's stop
    test sees e and dq exactly where the reference calls it (dls.cpp:61)."""
    q = _as_f64(q0).copy()
    data.success = False
    levels = problem.max_priority_level() + 1
    row_level = np.concatenate([np.full(int(t.dimension()), prio) for _, t, prio in sorted(problem._tasks, key=lambda x: x[2])])
    for it in range(p.max_iterations):
        if pik:
            one = pik_parameters(max_iterations=1, step_length=p.step_length, lambdas=p.lambdas, tolerance=-1.0)
            qn, _, _, res, dq, e, J = _solve_one(problem, q, None, one.c())
        else:
            one = dls_parameters(max_iterations=1, step_length=p.step_length, damping=p.damping, tolerance=-1.0)
            qn, _, _, res, dq, e, J = _solve_one(problem, q, one.c())
        data.dq, data.e, data.J, data.residual, data.iterations = dq, e, J, res, it
        if visitor.should_stop(problem, [e[row_level == l] for l in range(levels)], dq):   # dls.cpp:61-64
            data.success = True
            data.q = q
            return q
        q = qn
    data.iterations = p.max_iterations
    data.q = q
    return q


def dls(problem, q0, data=None, visitor=None, p=None):
    """vector_t ik::dls(problem, q0, data, visitor, p) (dls.hpp:111-114): one FP64 solve on the GPU.  `data` receives what
    the reference leaves in dls_data: success, q, dq, e, J (data.hpp:15-28).  A visitor whose class overrides should_stop
    is honoured (host-stepped loop); the stock visitor's test runs in the kernel with its `tolerance`."""
    problem.finalize(problem._device if problem._device is not None else 0)
    p = p or dls_parameters()
    data = data if data is not None else dls_data(problem)
    if visitor is not None and type(visitor).should_stop is not inverse_kinematics_visitor.should_stop:
        return _stepped(problem, q0, data, visitor, p, False)
    if visitor is not None:
        p = dls_parameters(max_iterations=p.max_iterations, step_length=p.step_length, damping=p.damping, tolerance=visitor.tolerance)
    q, ok, it, res, dq, e, J = _solve_one(problem, q0, p.c())
    data.q, data.success, data.iterations, data.residual, data.dq, data.e, data.J = q, ok, it, res, dq, e, J
    return q


def dls_batch_host(problem, q0, targets, p=None, dtype="f64", layout="soa", out=None, compact=False,
                   outputs=("q", "success", "iters", "resid")):
    """Batched ik::dls on HOST arrays (numpy, ideally pinned): H2D + solve + D2H inside the call.

    layout "soa": q0 [nq, B], targets [tsz, B]; "aos": q0 [B, nq], targets [B, tsz]; q0 of shape (nq,) = one initial guess
    for the whole batch.  compact=True: `targets` is the compact wire format (InverseKinematicsProblem.compact_targets).
    Returns dict(q, success, iters, resid) in the same layout (None for outputs not asked for).  ``out`` may hold
    preallocated result arrays."""
    problem.finalize(problem._device if problem._device is not None else 0)
    p = p or dls_parameters()
    code, npdt = _DT[dtype]
    q0 = np.ascontiguousarray(q0, dtype=npdt)
    targets = np.ascontiguousarray(targets, dtype=npdt)
    io, B, res, _ = _host_io(problem, q0, targets, dtype, layout, out, compact, outputs)
    prm = p.c()
    capi.check(capi.lib.ikb_dls_solve_batch_host(problem._h, code, C.byref(prm), B, C.byref(io)),
               "ikb_dls_solve_batch_host")
    return res


def dls_batch(problem, q0, targets, p=None, out=None, stream=None):
    """Batched ik::dls on DEVICE tensors (torch, SoA): q0 [nq, B], targets [tsz, B], float64 or float32.

    Enqueues on ``stream`` (default: torch's current stream) and returns without synchronising.
    Returns dict(q [nq,B], success [B] uint8, iters [B] int32, resid [B])."""
    import torch

    p = p or dls_parameters()
    nq, tsz = problem.model().nq, problem.target_size
    assert q0.is_cuda and targets.is_cuda and q0.dtype == targets.dtype and q0.device == targets.device
    problem.finalize(q0.device.index or 0)   # raises when the problem lives on another device
    dtype = "f64" if q0.dtype == torch.float64 else "f32"
    B = q0.shape[1]
    assert q0.shape == (nq, B) and targets.shape == (tsz, B) and q0.is_contiguous() and targets.is_contiguous()
    out = out or {}
    for k, shape, dt in (("q", (nq, B), q0.dtype), ("success", (B,), torch.uint8), ("iters", (B,), torch.int32), ("resid", (B,), q0.dtype)):
        o = out.get(k)
        if o is not None and not (o.device == q0.device and tuple(o.shape) == shape and o.dtype == dt and o.is_contiguous()):
            raise ValueError("out[%r] must be a contiguous %s tensor of shape %s on %s" % (k, dt, shape, q0.device))
    q = out.get("q") if out.get("q") is not None else torch.empty((nq, B), dtype=q0.dtype, device=q0.device)
    success = out.get("success") if out.get("success") is not None else torch.empty(B, dtype=torch.uint8, device=q0.device)
    iters = out.get("iters") if out.get("iters") is not None else torch.empty(B, dtype=torch.int32, device=q0.device)
    resid = out.get("resid") if out.get("resid") is not None else torch.empty(B, dtype=q0.dtype, device=q0.device)
    io = capi.BatchIO(q0.data_ptr(), B, 1, targets.data_ptr(), B, 1, q.data_ptr(), B, 1, success.data_ptr(),
                      iters.data_ptr(), resid.data_ptr())
    s = stream if stream is not None else torch.cuda.current_stream(q0.device).cuda_stream
    prm = p.c()
    capi.check(capi.lib.ikb_dls_solve_batch(problem._h, _DT[dtype][0], C.byref(prm), B, C.byref(io), C.c_void_p(s)),
               "ikb_dls_solve_batch")
    return dict(q=q, success=success, iters=iters, resid=resid)


def pik_batch(problem, q0, targets, p=None, out=None, stream=None):
    """Batched ik::pik (pik.cpp:31-96) on DEVICE tensors; arguments and results as dls_batch."""
    import torch

    p = p or pik_parameters()
    nq, tsz = problem.model().nq, problem.target_size
    assert q0.is_cuda and targets.is_cuda and q0.dtype == targets.dtype
    problem.finalize(q0.device.index or 0)
    dtype = "f64" if q0.dtype == torch.float64 else "f32"
    B = q0.shape[1]
    assert q0.shape == (nq, B) and targets.shape == (tsz, B) and q0.is_contiguous() and targets.is_contiguous()
    out = out or {}
    q = out.get("q") if out.get("q") is not None else torch.empty((nq, B), dtype=q0.dtype, device=q0.device)
    success = out.get("success") if out.get("success") is not None else torch.empty(B, dtype=torch.uint8, device=q0.device)
    iters = out.get("iters") if out.get("iters") is not None else torch.empty(B, dtype=torch.int32, device=q0.device)
    resid = out.get("resid") if out.get("resid") is not None else torch.empty(B, dtype=q0.dtype, device=q0.device)
    io = capi.BatchIO(q0.data_ptr(), B, 1, targets.data_ptr(), B, 1, q.data_ptr(), B, 1, success.data_ptr(),
                      iters.data_ptr(), resid.data_ptr())
    s = stream if stream is not None else torch.cuda.current_stream(q0.device).cuda_stream
    prm = p.c()
    capi.check(capi.lib.ikb_pik_solve_batch(problem._h, _DT[dtype][0], C.byref(prm), B, C.byref(io), C.c_void_p(s)),
               "ikb_pik_solve_batch")
    return dict(q=q, success=success, iters=iters, resid=resid)


def pik_batch_host(problem, q0, targets, p=None, dtype="f64"):
    """Batched ik::pik on HOST arrays, AoS: q0 [B, nq], targets [B, tsz]."""
    problem.finalize(problem._device or 0)
    p = p or pik_parameters()
    code, npdt = _DT[dtype]
    nq, tsz = problem.model().nq, problem.target_size
    q0 = np.ascontiguousarray(q0, dtype=npdt)
    targets = np.ascontiguousarray(targets, dtype=npdt)
    B = q0.shape[0]
    assert q0.shape == (B, nq) and targets.shape == (B, tsz)
    q = np.empty((B, nq), dtype=npdt)
    success, iters, resid = np.empty(B, dtype=np.uint8), np.empty(B, dtype=np.int32), np.empty(B, dtype=npdt)
    io = capi.BatchIO(q0.ctypes.data, 1, nq, targets.ctypes.data, 1, tsz, q.ctypes.data, 1, nq, success.ctypes.data,
                      iters.ctypes.data, resid.ctypes.data)
    prm = p.c()
    capi.check(capi.lib.ikb_pik_solve_batch_host(problem._h, code, C.byref(prm), B, C.byref(io)), "ikb_pik_solve_batch_host")
    return dict(q=q, success=success, iters=iters, resid=resid)


class pik_data(dls_data):  # pik.hpp:27-49: the user-owned per-solve record (P, da, lambda live in the kernel / parameters)
    pass


def pik(problem, q0, data=None, visitor=None, p=None):
    """vector_t ik::pik(problem, q0, data, visitor, p) (pik.hpp:51-54): one problem, targets from the tasks' `target`
    members; `data` receives success, q, dq, e, J like dls()."""
    problem.finalize(problem._device if problem._device is not None else 0)
    p = p or pik_parameters()
    data = data if data is not None else pik_data(problem)
    if visitor is not None and type(visitor).should_stop is not inverse_kinematics_visitor.should_stop:
        return _stepped(problem, q0, data, visitor, p, True)
    if visitor is not None:
        p = pik_parameters(max_iterations=p.max_iterations, step_length=p.step_length, lambdas=p.lambdas, tolerance=visitor.tolerance)
    q, ok, it, res, dq, e, J = _solve_one(problem, q0, None, p.c())
    data.q, data.success, data.iterations, data.residual, data.dq, data.e, data.J = q, ok, it, res, dq, e, J
    return q


class SolveQueue:
    """Pipelined stream of batches (ikb_queue_*, include/ikb200.h): up to ``depth`` batches in flight, ``merge``
    consecutive batches per kernel pair (the ~0.7 ms straggler chain is paid once per group), host-buffer copies of one
    group beside the kernels of its neighbours.  Results are those of dls_batch / dls_batch_host (bit for bit in FP64 when
    both take the same kernels, to rounding otherwise; see include/ikb200.h).

        queue = ik.SolveQueue(problem, depth=8, merge=4)
        tickets = [queue.submit(q0_k, targets_k, out=out_k) for ...]     # device tensors (torch, SoA)
        queue.wait(tickets[0]); ... ; queue.drain()
    """

    def __init__(self, problem, depth=8, merge=4, device=0):
        problem.finalize(problem._device if problem._device is not None else device)
        self._problem = problem
        self._h = C.c_void_p()
        capi.check(capi.lib.ikb_queue_create(problem._h, depth, merge, C.byref(self._h)), "ikb_queue_create")
        self._keep = {}  # ticket -> buffers that must outlive the batch

    def __del__(self):
        if getattr(self, "_h", None) and capi is not None and getattr(capi, "lib", None) is not None:
            capi.lib.ikb_queue_free(self._h)
            self._h = None

    def submit(self, q0, targets, p=None, out=None, in_stream=None):
        """Device tensors q0 [nq, B], targets [tsz, B]; inputs must be ready in ``in_stream`` order (default: torch's
        current stream).  Returns (ticket, dict(q, success, iters, resid)); the outputs are valid after wait(ticket)."""
        import torch

        problem = self._problem
        p = p or dls_parameters()
        nq, tsz = problem.model().nq, problem.target_size
        dtype = "f64" if q0.dtype == torch.float64 else "f32"
        B = q0.shape[1]
        assert q0.is_cuda and targets.is_cuda and q0.dtype == targets.dtype
        assert q0.shape == (nq, B) and targets.shape == (tsz, B) and q0.is_contiguous() and targets.is_contiguous()
        out = out or {}
        q = out.get("q") if out.get("q") is not None else torch.empty((nq, B), dtype=q0.dtype, device=q0.device)
        success = out.get("success") if out.get("success") is not None else torch.empty(B, dtype=torch.uint8, device=q0.device)
        iters = out.get("iters") if out.get("iters") is not None else torch.empty(B, dtype=torch.int32, device=q0.device)
        resid = out.get("resid") if out.get("resid") is not None else torch.empty(B, dtype=q0.dtype, device=q0.device)
        io = capi.BatchIO(q0.data_ptr(), B, 1, targets.data_ptr(), B, 1, q.data_ptr(), B, 1, success.data_ptr(),
                          iters.data_ptr(), resid.data_ptr())
        s = in_stream if in_stream is not None else torch.cuda.current_stream(q0.device).cuda_stream
        prm = p.c()
        t = capi.check_index(capi.lib.ikb_queue_submit(self._h, _DT[dtype][0], C.byref(prm), B, C.byref(io), C.c_void_p(s)),
                             "ikb_queue_submit")
        res = dict(q=q, success=success, iters=iters, resid=resid)
        self._keep[t] = (q0, targets, res)
        self._prune(t)
        return t, res

    def submit_host(self, q0, targets, p=None, dtype="f64", layout="soa", out=None, compact=False,
                    outputs=("q", "success", "iters", "resid")):
        """Host arrays (numpy; pinned -- ikb_host_alloc -- for the copies to overlap), arguments as dls_batch_host."""
        p = p or dls_parameters()
        io, B, res, keep = _host_io(self._problem, q0, targets, dtype, layout, out, compact, outputs)
        prm = p.c()
        t = capi.check_index(capi.lib.ikb_queue_submit_host(self._h, _DT[dtype][0], C.byref(prm), B, C.byref(io)), "ikb_queue_submit_host")
        self._keep[t] = keep
        self._prune(t)
        return t, res

    def _prune(self, t):
        # buffers of batches that left the pipeline long ago (callers that only use wait_on_stream never pop them)
        for old in [k for k in self._keep if k < t - 64]:
            del self._keep[old]

    def wait(self, ticket):
        capi.check(capi.lib.ikb_queue_wait(self._h, ticket), "ikb_queue_wait")
        return self._keep.pop(ticket, (None, None, None))[2]

    def wait_on_stream(self, ticket, stream=None):
        import torch

        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        capi.check(capi.lib.ikb_queue_wait_on_stream(self._h, ticket, C.c_void_p(s)), "ikb_queue_wait_on_stream")

    def flush(self):
        capi.check(capi.lib.ikb_queue_flush(self._h), "ikb_queue_flush")

    def drain(self):
        capi.check(capi.lib.ikb_queue_drain(self._h), "ikb_queue_drain")
        self._keep.clear()


class MultiGPU:
    """Several GPUs behind one handle (ikb_multi_*, include/ikb200.h): a HOST batch is cut into contiguous slices
    [r B / G, (r + 1) B / G) (SURVEY 8e), slice r is staged, solved and read back on device r -- all devices concurrently
    under the calling thread -- and the results land in the caller's arrays: no gather, no collective.

        multi = ik.MultiGPU(problem, devices=[0, 1, 2, 3])
        out = multi.dls_batch_host(q0, targets)                  # blocking
        t, out = multi.submit_host(q0_k, targets_k); ...; multi.wait(t)   # pipelined, as SolveQueue
    """

    def __init__(self, problem, devices=None, depth=4, merge=1):
        if devices is None:
            devices = list(range(capi.lib.ikb_device_count()))
        self._problem = problem
        self.devices = list(devices)
        h = problem._h if problem._h is not None else problem._build_handle(None)
        self._h = C.c_void_p()
        dev = np.asarray(self.devices, dtype=np.int32)
        try:
            rc = capi.lib.ikb_multi_create(h, dev.ctypes.data_as(C.POINTER(C.c_int32)), len(dev), depth, merge, C.byref(self._h))
            if rc != capi.OK:
                capi.lib.ikb_multi_free(self._h)
                self._h = None
                capi.check(rc, "ikb_multi_create")
        finally:
            if h is not problem._h:
                capi.lib.ikb_problem_free(h)
        self._keep = {}

    def __del__(self):
        if getattr(self, "_h", None) and capi is not None and getattr(capi, "lib", None) is not None:
            capi.lib.ikb_multi_free(self._h)
            self._h = None

    def kernel_name(self, index=0, dtype="f64"):
        n = capi.lib.ikb_problem_kernel_name(capi.lib.ikb_multi_problem(self._h, index), _DT[dtype][0])
        return n.decode() if n else None

    def submit_host(self, q0, targets, p=None, dtype="f64", layout="soa", out=None, compact=False,
                    outputs=("q", "success", "iters", "resid")):
        p = p or dls_parameters()
        io, B, res, keep = _host_io(self._problem, q0, targets, dtype, layout, out, compact, outputs)
        prm = p.c()
        t = capi.check_index(capi.lib.ikb_multi_submit_host(self._h, _DT[dtype][0], C.byref(prm), B, C.byref(io)), "ikb_multi_submit_host")
        self._keep[t] = keep
        for old in [k for k in self._keep if k < t - 64]:
            del self._keep[old]
        return t, res

    def wait(self, ticket):
        capi.check(capi.lib.ikb_multi_wait(self._h, ticket), "ikb_multi_wait")
        return self._keep.pop(ticket, (None, None, None))[2]

    def drain(self):
        capi.check(capi.lib.ikb_multi_drain(self._h), "ikb_multi_drain")
        self._keep.clear()

    def dls_batch_host(self, q0, targets, p=None, dtype="f64", layout="soa", out=None, compact=False,
                       outputs=("q", "success", "iters", "resid")):
        npdt = _DT[dtype][1]
        t, res = self.submit_host(np.ascontiguousarray(q0, dtype=npdt), np.ascontiguousarray(targets, dtype=npdt), p, dtype, layout,
                                  out, compact, outputs)
        self.wait(t)
        return res


def fk_batch(problem, q, frames, out=None, stream=None):
    """Batched framesForwardKinematics (data.cpp:28-29) on device tensors: q [nq, B] -> [len(frames)*12, B]."""
    import torch

    m = problem.model()
    problem.finalize(q.device.index or 0)
    ids = np.array([m.getFrameId(f) if isinstance(f, str) else int(f) for f in frames], dtype=np.int32)
    if (ids >= m.nframes).any():
        raise KeyError("unknown frame in %r" % (frames,))
    B = q.shape[1]
    dtype = "f64" if q.dtype == torch.float64 else "f32"
    if out is None:
        out = torch.empty((len(ids) * 12, B), dtype=q.dtype, device=q.device)
    s = stream if stream is not None else torch.cuda.current_stream(q.device).cuda_stream
    capi.check(capi.lib.ikb_fk_batch(problem._h, _DT[dtype][0], B, C.c_void_p(q.data_ptr()), B, 1, len(ids),
                                     ids.ctypes.data_as(C.POINTER(C.c_int32)), C.c_void_p(out.data_ptr()),
                                     C.c_void_p(s)), "ikb_fk_batch")
    return out


def kernel_launch_count():
    return int(capi.lib.ikb_kernel_launch_count())

"""CPU ORACLE for URDF `continuous` joints (test infrastructure, NOT product code).

The oracle in oracle/ restates the reference's path for the joint types it was written for and stays as it is.  This module
extends that restatement to Pinocchio's unbounded revolute joint (JointModelRevoluteUnbounded{X,Y,Z} /
RevoluteUnboundedUnaligned, SpecialOrthogonalOperation<2>) without touching it: `build()` copies oracle/ik_oracle.{c,h}
into build/oracle_continuous/, splices in the rules below (every splice must match its anchor exactly once, so a change of
the base file fails loudly instead of silently dropping a rule) and compiles the same three variants as oracle/Makefile
(FP64, FP32, FP64 with fused multiply-adds).  For a model without continuous joints the derived library computes exactly
what the base one does.  The URDF side (`flatten_urdf`) is restated on top of oracle/urdf_flatten.py.

Switches restated, so that a reader who has Pinocchio can check them one by one:
  * nq = 2, nv = 1, q = (cos theta, sin theta); the neutral configuration is (1, 0);
  * aligned X / Y / Z when the URDF axis isApprox a unit vector (the revolute joints' test), else unaligned with the axis
    normalised; types RUBX/RUBY/RUBZ/unaligned = 10..13, the revolute type with the same axis + 8;
  * calc builds the rotation about the axis from c = q[0], s = q[1] AS GIVEN (no sin / cos evaluated, no renormalisation);
    motion subspace and Jacobian column are the revolute joint's with that axis;
  * integrate: w = v[0], (c', s') = (cos w c - sin w s, sin w c + cos w s), then (c', s') *= (3 - (c'^2 + s'^2)) / 2;
  * limits: the URDF parser gives both entries -1.01 / +1.01 and ignores <limit lower/upper>.  This one is restated from
    memory of Pinocchio's parsers/urdf/model.cpp and could not be checked against its source; the clamp over all nq
    (reference common.hpp:53-56) runs on the two entries as on every other one.
"""
import ctypes as C
import os
import subprocess
import xml.etree.ElementTree as ET

import numpy as np

from oracle import oracle as O
from oracle import urdf_flatten as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "build", "oracle_continuous")
J_CONTINUOUS = (10, 11, 12, 13)   # = J_RX .. J_REV_UNALIGNED + 8

_H_SPLICES = [(
    "IKO_J_PX = 6, IKO_J_PY = 7, IKO_J_PZ = 8, IKO_J_PRIS_UNALIGNED = 9 };",
    "IKO_J_PX = 6, IKO_J_PY = 7, IKO_J_PZ = 8, IKO_J_PRIS_UNALIGNED = 9,\n"
    "       IKO_J_RUBX = 10, IKO_J_RUBY = 11, IKO_J_RUBZ = 12, IKO_J_RUB_UNALIGNED = 13 };")]

_C_SPLICES = [
    # the axis of a continuous joint is that of the revolute joint of the same kind
    ("        case IKO_J_RX: case IKO_J_PX: a[0] = 1; break;\n"
     "        case IKO_J_RY: case IKO_J_PY: a[1] = 1; break;\n"
     "        case IKO_J_RZ: case IKO_J_PZ: a[2] = 1; break;",
     "        case IKO_J_RX: case IKO_J_PX: case IKO_J_RUBX: a[0] = 1; break;\n"
     "        case IKO_J_RY: case IKO_J_PY: case IKO_J_RUBY: a[1] = 1; break;\n"
     "        case IKO_J_RZ: case IKO_J_PZ: case IKO_J_RUBZ: a[2] = 1; break;"),
    # calc: (c, s) as given
    ("/* joint transform M_j(q) (Pinocchio Joint*::calc) */",
     "static int is_cont(int t) { return t >= IKO_J_RUBX && t <= IKO_J_RUB_UNALIGNED; }\n\n"
     "/* joint transform M_j(q) (Pinocchio Joint*::calc).  Continuous (RevoluteUnbounded): c = q[0], s = q[1] as given. */"),
    ("    } else if (t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) {\n"
     "        const double s = sin(qj[0]), c = cos(qj[0]);\n"
     "        if (t == IKO_J_RX) { M[4] = c; M[5] = -s; M[7] = s; M[8] = c; }\n"
     "        else if (t == IKO_J_RY) { M[0] = c; M[2] = s; M[6] = -s; M[8] = c; }\n"
     "        else if (t == IKO_J_RZ) { M[0] = c; M[1] = -s; M[3] = s; M[4] = c; }",
     "    } else if ((t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) || is_cont(t)) {\n"
     "        const double s = is_cont(t) ? qj[1] : sin(qj[0]), c = is_cont(t) ? qj[0] : cos(qj[0]);\n"
     "        if (t == IKO_J_RX || t == IKO_J_RUBX) { M[4] = c; M[5] = -s; M[7] = s; M[8] = c; }\n"
     "        else if (t == IKO_J_RY || t == IKO_J_RUBY) { M[0] = c; M[2] = s; M[6] = -s; M[8] = c; }\n"
     "        else if (t == IKO_J_RZ || t == IKO_J_RUBZ) { M[0] = c; M[1] = -s; M[3] = s; M[4] = c; }"),
    # world Jacobian column: the revolute one about the same axis
    ("        } else if (t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) {\n"
     "            double a[3], z[3], pxz[3];",
     "        } else if ((t >= IKO_J_RX && t <= IKO_J_REV_UNALIGNED) || is_cont(t)) {\n"
     "            double a[3], z[3], pxz[3];"),
    # integrate: SpecialOrthogonalOperation<2>::integrate_impl
    ("            for (int i = 0; i < 4; ++i) qout[iq + 3 + i] = quat[i] * alpha;\n"
     "        } else {",
     "            for (int i = 0; i < 4; ++i) qout[iq + 3 + i] = quat[i] * alpha;\n"
     "        } else if (is_cont(m->jtype[j])) {\n"
     "            const double ca = q[iq], sa = q[iq + 1], w = v[iv];\n"
     "            const double cw = cos(w), sw = sin(w);\n"
     "            const double c1 = cw * ca - sw * sa, s1 = sw * ca + cw * sa;\n"
     "            const double n2 = c1 * c1 + s1 * s1, alpha = (3 - n2) / 2;\n"
     "            qout[iq] = c1 * alpha;\n"
     "            qout[iq + 1] = s1 * alpha;\n"
     "        } else {"),
]

_VARIANTS = {"f64": [], "f32": ["-DIKO_F32", "-fsingle-precision-constant"], "fma": ["-ffp-contract=fast", "-mfma"]}
_LIBS = {}


def _splice(text, splices, what):
    for old, new in splices:
        if text.count(old) != 1:
            raise RuntimeError("continuous oracle: anchor not found exactly once in %s:\n%s" % (what, old))
        text = text.replace(old, new)
    return text


def build():
    """Derive and compile the three libraries when oracle/ik_oracle.{c,h} or this module are newer than them."""
    os.makedirs(OUT, exist_ok=True)
    srcs = [os.path.join(ROOT, "oracle", f) for f in ("ik_oracle.c", "ik_oracle.h")] + [os.path.abspath(__file__)]
    sos = {v: os.path.join(OUT, "libik_oracle_continuous_%s.so" % v) for v in _VARIANTS}
    newest = max(os.path.getmtime(s) for s in srcs)
    if all(os.path.exists(so) and os.path.getmtime(so) >= newest for so in sos.values()):
        return sos
    for name, splices in (("ik_oracle.h", _H_SPLICES), ("ik_oracle.c", _C_SPLICES)):
        with open(os.path.join(ROOT, "oracle", name)) as f:
            text = _splice(f.read(), splices, name)
        with open(os.path.join(OUT, name), "w") as f:
            f.write(text)
    base = ["gcc", "-O3", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-Wno-unused-parameter", "-ffp-contract=off", "-shared"]
    for v, flags in _VARIANTS.items():
        subprocess.check_call(base + flags + ["-o", sos[v], os.path.join(OUT, "ik_oracle.c"), "-lm", "-lpthread"])
    return sos


def lib(variant="f64"):
    if variant not in _LIBS:
        _LIBS[variant] = C.CDLL(build()[variant])
    return _LIBS[variant]


def flatten_urdf(xml_text, free_flyer=True):
    """oracle/urdf_flatten.flatten_urdf with `continuous` joints: flattened as the revolute joint with the same axis (same
    traversal, placements and axis test), then retyped (+8), given two configuration entries bounded by +-1.01 and the
    configuration offsets recounted."""
    root = ET.fromstring(xml_text)
    cont = set()
    for j in root.findall("joint"):
        if j.get("type") == "continuous":
            cont.add(j.get("name"))
            j.set("type", "revolute")
    f = U.flatten_urdf(ET.tostring(root, encoding="unicode"), free_flyer)
    lower, upper, idx_q, nq = [], [], [0], 0
    for j in range(1, f["njoints"]):
        a = int(f["idx_q"][j])
        n = 7 if f["jtype"][j] == U.J_FREEFLYER else 1
        idx_q.append(nq)
        if f["names"][j] in cont:
            f["jtype"][j] += 8
            lower += [-1.01, -1.01]
            upper += [1.01, 1.01]
            nq += 2
        else:
            lower += list(f["lower"][a:a + n])
            upper += list(f["upper"][a:a + n])
            nq += n
    f.update(nq=nq, idx_q=np.array(idx_q, dtype=np.int32), lower=np.array(lower), upper=np.array(upper))
    return f


class Model(O.Model):
    """oracle.Model on the derived library."""

    @classmethod
    def from_urdf(cls, xml_text, free_flyer=True):
        return cls(flatten_urdf(xml_text, free_flyer))

    def neutral(self):
        q = super().neutral()
        for j in range(self.njoints):
            if self.flat["jtype"][j] in J_CONTINUOUS:
                q[self.flat["idx_q"][j]] = 1.0   # (cos, sin) = (1, 0)
        return q

    def fk(self, q):
        out = np.zeros((self.njoints, 12))
        lib().iko_fk(C.byref(self.c), O._pd(O._d(q)), O._pd(out))
        return out

    def frame_placement(self, q, frame):
        out = np.zeros(12)
        lib().iko_frame_placement(C.byref(self.c), O._pd(self.fk(q)), C.c_int(frame), O._pd(out))
        return out

    def frame_jacobian_local(self, q, frame):
        oMi = self.fk(q)
        Jw, Jf = np.zeros((6, self.nv)), np.zeros((6, self.nv))
        lib().iko_joint_jacobians(C.byref(self.c), O._pd(oMi), O._pd(Jw))
        lib().iko_frame_jacobian_local(C.byref(self.c), O._pd(oMi), O._pd(Jw), C.c_int(frame), O._pd(Jf))
        return Jf

    def integrate(self, q, v):
        out = np.zeros(self.nq)
        lib().iko_integrate(C.byref(self.c), O._pd(O._d(q)), O._pd(O._d(v)), O._pd(out))
        return out


class Problem(O.Problem):
    """oracle.Problem on the derived library."""

    def evaluate(self, q, targets):
        e, J = np.zeros(self.rows), np.zeros((self.rows, self.model.nv))
        lib().iko_evaluate(C.byref(self.model.c), C.byref(self.c), O._pd(O._d(q)), O._pd(O._d(targets)), O._pd(e), O._pd(J))
        return e, J


def problem_like(problem, omodel):
    """oracle.bridge.oracle_problem_like for a Model of this module."""
    from oracle.bridge import oracle_problem_like
    base = oracle_problem_like(problem, omodel)
    p = Problem(omodel, base.max_priority_level)
    p.tasks, p.constraints = base.tasks, base.constraints
    return p


def _batch(fn, variant, problem, q0, targets, prm, nthreads):
    m = problem.model
    q0, targets = O._d(q0), O._d(targets)
    B = q0.shape[0]
    assert q0.shape == (B, m.nq) and targets.shape == (B, problem.target_size)
    q, ok, it, res = np.zeros((B, m.nq)), np.zeros(B, dtype=np.uint8), np.zeros(B, dtype=np.int32), np.zeros(B)
    rc = getattr(lib(variant), fn)(C.byref(m.c), C.byref(problem.c), C.byref(prm), C.c_int(B), O._pd(q0), O._pd(targets),
                                   O._pd(q), ok.ctypes.data_as(C.POINTER(C.c_ubyte)), O._pi(it), O._pd(res), C.c_int(nthreads))
    return rc, (q, ok.astype(bool), it, res)


def dls_batch(problem, q0, targets, prm=None, nthreads=1, fma=False):
    """oracle.dls_batch on the derived library (fma=True: its FMA-contracted build)."""
    return _batch("iko_dls_batch", "fma" if fma else "f64", problem, q0, targets, prm or O.params(), nthreads)[1]


def pik_batch(problem, q0, targets, prm=None, nthreads=1, fma=False):
    """oracle.pik_batch on the derived library (fma=True: its FMA-contracted build)."""
    rc, out = _batch("iko_pik_batch", "fma" if fma else "f64", problem, q0, targets, prm or O.pik_params(), nthreads)
    if rc != 0:
        raise ValueError(O._PIK_LEVELS)
    return out


def dls_batch_f32(problem, q0, targets, prm=None, nthreads=1):
    """oracle.dls_batch_f32 on the derived library: the same restatement with every scalar a float."""
    prm = prm or O.params()
    cm, cp, keep = O._f32_structs(problem)
    m = problem.model
    q0 = np.ascontiguousarray(q0, dtype=np.float32)
    targets = np.ascontiguousarray(targets, dtype=np.float32)
    B = q0.shape[0]
    q, ok, it, res = np.zeros((B, m.nq), dtype=np.float32), np.zeros(B, dtype=np.uint8), np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.float32)
    cprm = O._CParamsF(prm.max_iterations, prm.step_length, prm.damping, prm.tolerance)
    lib("f32").iko_dls_batch(C.byref(cm), C.byref(cp), C.byref(cprm), C.c_int(B), q0.ctypes.data_as(O._fp),
                             targets.ctypes.data_as(O._fp), q.ctypes.data_as(O._fp), ok.ctypes.data_as(C.POINTER(C.c_ubyte)),
                             O._pi(it), res.ctypes.data_as(O._fp), C.c_int(nthreads))
    return q.astype(np.float64), ok.astype(bool), it, res.astype(np.float64)

#!/usr/bin/env python3
"""Generate a topology-specialised DLS IK kernel body (CUDA C++) for one (robot, task list) pair.

    python tools/gen_kernel.py <flat_model.json> <spec.json> <out.cuh>

The generic kernel (ik_b200/csrc/dls_generic.cuh) walks the kinematic tree through tables and keeps its
per-problem scratch in local memory.  For the benchmark robots that is 50x away from the FP64 roofline, so the
hot path is specialised: this script unrolls the reference's evaluate -> solve iteration (dls.cpp:14-64,
data.cpp:25-58, frame.hpp:37-62,152-182) for a FIXED tree and FIXED frame-task list into straight-line code:

* joint placements are compile-time constants, folded into the arithmetic (exact zeros / ones of the URDF vanish);
* only joints that support a task frame are visited, only structurally non-zero Jacobian entries exist;
* the task Jacobian never materialises the 6 x nv frame Jacobian: with M1 = A R_f^T, M2 = B R_f^T (A, B the blocks
  of Jlog6(tMf)) a revolute column is  top = -(M1 ((p_j - p_f) x z_j) + M2 z_j),  bottom = -(M1 z_j);
* the non-zero entries of the weighted task Jacobian go to a per-thread strip of shared memory (slot k of thread t
  at sJ[k * BLOCK + t]: conflict-free), the Gram matrix is accumulated from them into REGISTERS (packed lower
  triangle, fully unrolled), factorised there (LDL^T) and the step dq = -J^T y re-reads the strip once.

* the damped normal equations (dls.cpp:39-53) never materialise the Gram matrix either: it is accumulated block column
  by block column (width W) into registers straight from the strip, each block column is updated left-looking from
  the factor columns already stored, factorised in registers (LDL^T, no pivoting: G is SPD thanks to the damping) and
  written to a second strip; the right-hand side rides along as an extra row, so the forward substitution and the
  D^-1 scaling come for free and only the back substitution re-reads the factor.

The emitted struct is consumed by dls_spec.cuh (thread-per-problem persistent kernel with lane refill) and -- being
__host__ __device__ -- by the CPU unit-test harness.  Supported: free-flyer or fixed base; RX/RY/RZ/unaligned
revolute and prismatic joints; FrameTask (Position / Orientation / Full) with the `universe` reference frame.
Anything else runs on the generic kernel.
"""
import json
import re
import sys

J_UNIVERSE, J_FF, J_RX, J_RY, J_RZ, J_RU, J_PX, J_PY, J_PZ, J_PU = range(10)
POSITION, ORIENTATION, FULL = 0, 1, 2


# ------------------------------------------------------------------------------------------------------------
# tiny symbolic layer: a value is a python float (compile-time constant) or a str (name of a `const T` variable)
# ------------------------------------------------------------------------------------------------------------
class Emitter:
    def __init__(self, prefix=""):
        self.lines = []
        self.n = 0
        self.indent = "        "
        self.prefix = prefix  # keeps the temporaries of interleaved emitters apart

    def comment(self, text):
        self.lines.append("%s// %s" % (self.indent, text))

    def raw(self, text):
        self.lines.append(self.indent + text)

    def var(self, expr, hint="t"):
        """Materialise an expression string as a named const variable."""
        name = "%s%s_%d" % (self.prefix, hint, self.n)
        self.n += 1
        self.lines.append("%sconst T %s = %s;" % (self.indent, name, expr))
        return name


def is_const(x):
    return isinstance(x, (int, float))


def lit(x):
    if is_const(x):
        return "T(%r)" % float(x)
    return x


def neg(E, a, hint="n"):
    if is_const(a):
        return -a
    return E.var("-%s" % a, hint)


def sop(E, terms, hint="t", add=None):
    """Signed sum of products: terms are (a, b) or (a, b, sign) with sign = +1/-1; result = sum sign*a*b (+ add).
    Constant-folds, drops zero terms, strips unit factors; returns a float or the name of a (new) variable."""
    const_part = 0.0
    parts = []  # (sign, coeff or None, var expression)
    if add is not None:
        if is_const(add):
            const_part += add
        else:
            parts.append((1, None, add))
    for term in terms:
        a, b = term[0], term[1]
        sign = term[2] if len(term) > 2 else 1
        if is_const(a) and is_const(b):
            const_part += sign * a * b
            continue
        if is_const(b):
            a, b = b, a
        if is_const(a):
            if a == 0:
                continue
            if a < 0:
                a, sign = -a, -sign
            parts.append((sign, None if a == 1.0 else a, b))
        else:
            parts.append((sign, None, "%s * %s" % (a, b)))
    if not parts:
        return const_part
    if len(parts) == 1 and parts[0][0] == 1 and parts[0][1] is None and " " not in parts[0][2] and const_part == 0:
        return parts[0][2]  # plain alias, no new variable
    expr = ""
    for k, (sign, coeff, body) in enumerate(parts):
        body = body if coeff is None else "%s * %s" % (lit(coeff), body)
        if k == 0:
            expr = body if sign > 0 else "-" + (body if " " not in body else "(%s)" % body)
        else:
            expr += " %s %s" % ("+" if sign > 0 else "-", body)
    if const_part != 0:
        expr += (" + %s" % lit(const_part)) if const_part > 0 else (" - %s" % lit(-const_part))
    return E.var(expr, hint)


def matmul(E, A, B, hint="m"):
    return [sop(E, [(A[3 * i + k], B[3 * k + j]) for k in range(3)], hint) for i in range(3) for j in range(3)]


def matvec(E, R, v, hint="v", add=None):
    return [sop(E, [(R[3 * i + k], v[k]) for k in range(3)], hint, None if add is None else add[i]) for i in range(3)]


def _cross_comp(E, a, b, i, hint):
    """component i of a x b"""
    j, k = (i + 1) % 3, (i + 2) % 3
    return sop(E, [(a[j], b[k]), (a[k], b[j], -1)], hint)


def sub3(E, a, b, hint="d"):
    out = []
    for x, y in zip(a, b):
        if is_const(x) and is_const(y):
            out.append(x - y)
        elif is_const(y) and y == 0:
            out.append(x)
        else:
            out.append(E.var("%s - %s" % (lit(x), lit(y)), hint))
    return out


def arr(E, name, vals):
    E.raw("const T %s[%d] = {%s};" % (name, len(vals), ", ".join(lit(v) for v in vals)))


# ------------------------------------------------------------------------------------------------------------
# generator
# ------------------------------------------------------------------------------------------------------------
class Generator:
    def __init__(self, model, spec):
        self.m = model
        self.spec = spec
        self.joints = model["joints"]
        self.frames = {f["name"]: f for f in model["frames"]}
        self.nq, self.nv = model["nq"], model["nv"]
        self.tasks = []
        row = 0
        toff = 0
        self.rows_p0 = 0
        # tasks are listed in STACKED order: priority level, then insertion order (dls.cpp:18-24)
        prios = [int(t.get("priority", 0)) for t in spec["tasks"]]
        if prios != sorted(prios):
            raise ValueError("spec tasks must be listed in stacked (priority) order")
        for t in spec["tasks"]:
            kind = t.get("kind", "frame")
            if kind == "posture":  # PostureTask (posture.hpp:17-86): the last nj coordinates, no frame
                nj = int(t["nj"])
                universe = self.frames["universe"]
                self.tasks.append(dict(frame=universe, kind=kind, ktype=nj, dim=nj, row=row, toff=toff, tsize=nj, chain=[],
                                       name="posture(%d)" % nj, ref=universe, ref_name="universe", priority=int(t.get("priority", 0))))
                if int(t.get("priority", 0)) == 0:
                    self.rows_p0 += nj
                row += nj
                toff += nj
                continue
            f = self.frames[t["frame"]]
            if kind == "frame":
                ktype = {"position": POSITION, "orientation": ORIENTATION, "full": FULL}[t["type"]]
                dim = 6 if ktype == FULL else 3
                tsize = 12
            elif kind == "align":  # AlignAxisTask (frame.hpp:210-319): one row, target = the axis to align with (3 scalars)
                ktype = {"x": 0, "y": 1, "z": 2}[t["axis"]]
                dim = 1
                tsize = 3
            else:
                raise ValueError("unsupported task kind %r (PostureTask runs on the generic kernel)" % kind)
            ref = self.frames[t.get("reference", "universe")]
            chain = []
            j = f["parent"]
            while j > 0:
                chain.append(j)
                j = self.joints[j]["parent"]
            chain.reverse()
            self.tasks.append(dict(frame=f, kind=kind, ktype=ktype, dim=dim, row=row, toff=toff, tsize=tsize, chain=chain,
                                   name=t["frame"], ref=ref, ref_name=t.get("reference", "universe"),
                                   priority=int(t.get("priority", 0))))
            if int(t.get("priority", 0)) == 0:
                self.rows_p0 += dim
            row += dim
            toff += tsize
        self.rows = row
        self.tsz = toff
        self.slots = {}  # (row, col) -> slot index
        # mirror mode (gen_evaluate_mirrored): while the body of task A is emitted for the pair (A, B), quantities that
        # differ between the two sides are emitted as side-dependent variables
        self.mir = None
        # role-local configuration registers (arrow specs): global q index -> index into the role's own T q[NQL]
        self.qmap = None
        # spec "fold_task" (gen_fold): slot / row -> name of the register that holds the fold task's Jacobian entry / error
        self.jreg = None
        self.ereg = None

    def ql(self, iq):
        """register index of configuration scalar iq in the code being emitted (role-local for arrow specs)"""
        return self.qmap[iq] if self.qmap is not None else iq

    def slot(self, row, col):
        key = (row, col)
        if key not in self.slots:
            self.slots[key] = len(self.slots)
        return self.slots[key]

    # ---- FK of one joint (memoised) ----
    def fk_joint(self, E, j, world):
        """Emit the world placement of joint j; returns dict(R=[9], p=[3], z=[3] axis in world)."""
        if j in world:
            return world[j]
        jt = self.joints[j]
        par = jt["parent"]
        P = self.mirror_placement(E, j, jt["placement"])
        PR, Pp = P[:9], P[9:]
        if par > 0:
            pw = self.fk_joint(E, par, world)
            parR, parp = pw["R"], pw["p"]
        else:
            parR, parp = [1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0], [0.0, 0.0, 0.0]
        E.comment("joint %d %s (type %d, parent %d)" % (j, jt["name"], jt["type"], par))
        t = jt["type"]
        iq = jt["idx_q"]
        A = matmul(E, parR, PR, "A%d" % j)
        p = matvec(E, parR, Pp, "p%d" % j, add=parp)
        if t == J_FF:
            E.raw("T Rq%d[9];" % j)
            E.raw("quat_to_rot(q[%d], q[%d], q[%d], q[%d], Rq%d);" % (self.ql(iq + 3), self.ql(iq + 4), self.ql(iq + 5), self.ql(iq + 6), j))
            Rq = ["Rq%d[%d]" % (j, k) for k in range(9)]
            R = matmul(E, A, Rq, "R%d" % j)
            p = matvec(E, A, ["q[%d]" % self.ql(iq + k) for k in range(3)], "p%d" % j, add=p)
            w = dict(R=R, p=p, z=None, type=t)
        elif t in (J_RX, J_RY, J_RZ, J_RU):
            E.raw("T s%d, c%d;" % (j, j))
            E.raw("sincos_(%s, &s%d, &c%d);" % (self.qref(j, iq), j, j))
            s, c = "s%d" % j, "c%d" % j
            if t == J_RU:
                a = jt["axis"]
                v = E.var("T(1) - %s" % c, "v%d" % j)
                Rj = [sop(E, [(a[0] * a[0], v)], "r", c), sop(E, [(a[0] * a[1], v), (-a[2], s)], "r"),
                      sop(E, [(a[0] * a[2], v), (a[1], s)], "r"),
                      sop(E, [(a[0] * a[1], v), (a[2], s)], "r"), sop(E, [(a[1] * a[1], v)], "r", c),
                      sop(E, [(a[1] * a[2], v), (-a[0], s)], "r"),
                      sop(E, [(a[0] * a[2], v), (-a[1], s)], "r"), sop(E, [(a[1] * a[2], v), (a[0], s)], "r"),
                      sop(E, [(a[2] * a[2], v)], "r", c)]
                R = matmul(E, A, Rj, "R%d" % j)
                z = matvec(E, A, a, "z%d" % j)
            else:
                # A * Rot(axis, q): the axis column is unchanged, the other two mix with (c, s)
                k = {J_RX: 0, J_RY: 1, J_RZ: 2}[t]
                u, v2 = (k + 1) % 3, (k + 2) % 3  # Rot maps e_u -> c e_u + s e_v, e_v -> -s e_u + c e_v
                R = [None] * 9
                for i in range(3):
                    R[3 * i + k] = A[3 * i + k]
                    R[3 * i + u] = sop(E, [(A[3 * i + u], c), (A[3 * i + v2], s)], "R%d" % j)
                    R[3 * i + v2] = sop(E, [(A[3 * i + v2], c), (A[3 * i + u], s, -1)], "R%d" % j)
                z = [A[k], A[3 + k], A[6 + k]]
            w = dict(R=R, p=p, z=z, type=t)
        elif t in (J_PX, J_PY, J_PZ, J_PU):
            a = jt["axis"] if t == J_PU else [1.0 if i == t - J_PX else 0.0 for i in range(3)]
            z = matvec(E, A, a, "z%d" % j)
            p = [sop(E, [(z[i], self.qref(j, iq))], "p%d" % j, p[i]) for i in range(3)]
            w = dict(R=A, p=p, z=z, type=t)
        else:
            raise ValueError("unsupported joint type %d" % t)
        world[j] = w
        return w

    # ---- mirrored tasks ----
    def qref(self, j, iq):
        """Expression of the configuration scalar of (revolute / prismatic) joint j."""
        if self.mir and j in self.mir["jmap"]:
            return "qm%d" % j
        return "q[%d]" % self.ql(iq)

    def mirror_placement(self, E, j, P):
        """Placement of joint j; in mirror mode entries that differ on the other side become side-dependent variables."""
        if not (self.mir and j in self.mir["jmap"]):
            return P
        PB = self.joints[self.mir["jmap"][j]]["placement"]
        out = []
        for i, (a, b) in enumerate(zip(P, PB)):
            if a == b:
                out.append(a)
            else:
                if (a == 0) != (b == 0) or abs(a) == 1.0 or abs(b) == 1.0:
                    raise ValueError("mirror: joint %d placement entry %d has a different structure on the two sides" % (j, i))
                out.append(E.var("side ? %s : %s" % (lit(b), lit(a)), "pm%d_" % j))
        return out

    def gen_evaluate_mirrored(self, ta, tb):
        """ONE evaluate body for two tasks that are mirror images of each other (Cassie's feet): same chain structure, same
        task type, placements equal up to a few entries.  `side` = 0 evaluates task ta, 1 task tb: the entries that differ
        are side-dependent variables, the joint coordinates are selected once, and the row / slot / target offsets of the
        other side are folded into the base pointers of the strips.  Both warp roles then run the SAME instructions -- in
        lock step they share every instruction line they fetch (the kernels are instruction-fetch bound)."""
        A, B = self.tasks[ta], self.tasks[tb]
        if (A["kind"], A["ktype"], A["dim"], A["tsize"], len(A["chain"]), A["ref_name"]) != \
                (B["kind"], B["ktype"], B["dim"], B["tsize"], len(B["chain"]), B["ref_name"]):
            raise ValueError("mirror: tasks %d and %d differ in shape" % (ta, tb))
        if A["frame"]["placement"] != B["frame"]["placement"] or not self.is_universe(A["ref"]):
            raise ValueError("mirror: frame placements differ / moving reference frame")
        jmap = {}
        for ja, jb in zip(A["chain"], B["chain"]):
            if ja != jb:
                if self.joints[ja]["type"] != self.joints[jb]["type"] or self.joints[ja]["type"] in (J_RU, J_PU, J_FF):
                    raise ValueError("mirror: joints %d / %d differ in type" % (ja, jb))
                pa, pb = self.joints[ja]["parent"], self.joints[jb]["parent"]
                if not (pa == pb or jmap.get(pa) == pb):
                    raise ValueError("mirror: joints %d / %d hang off different parents" % (ja, jb))
                jmap[ja] = jb
        E = Emitter()
        E.comment("side 0: task %d (%s), side 1: task %d (%s)" % (ta, A["name"], tb, B["name"]))
        for ja, jb in jmap.items():
            if self.qmap is not None:   # role-local registers: both sides keep the joint at the same index
                if self.qmap_b[self.joints[jb]["idx_q"]] != self.qmap[self.joints[ja]["idx_q"]]:
                    raise ValueError("mirror: joints %d / %d sit in different local registers" % (ja, jb))
                E.raw("const T qm%d = q[%d];" % (ja, self.qmap[self.joints[ja]["idx_q"]]))
            else:
                E.raw("const T qm%d = side ? q[%d] : q[%d];" % (ja, self.joints[jb]["idx_q"], self.joints[ja]["idx_q"]))
        for i in range(A["dim"]):
            E.raw("const T wm%d = side ? c.weight[%d] : c.weight[%d];" % (i, B["row"] + i, A["row"] + i))
        s0 = len(self.slots)
        self.mir = dict(jmap=jmap, row=A["row"], toff=A["toff"])
        body = Emitter()
        self.gen_task(body, ta, {})
        self.mir = None
        nA = len(self.slots) - s0
        # the other side's Jacobian entries take the same slots, nA further on
        for (r, cidx), k in list(self.slots.items()):
            if k >= s0:
                if cidx < 6 and self.joints[A["chain"][0]]["type"] == J_FF:
                    cb = cidx  # free-flyer columns are shared
                else:
                    ja = next(j for j in A["chain"] if self.joints[j]["idx_v"] == cidx)
                    cb = self.joints[jmap.get(ja, ja)]["idx_v"]
                self.slots[(r - A["row"] + B["row"], cb)] = k + nA
        E.raw("const S sJm{sJ.base + side * (%d * S::kStride)};  // the other side's slots" % nA)
        E.raw("const S sEm{sE.base + side * (%d * S::kStride)};  // ... rows" % (B["row"] - A["row"]))
        E.raw("const S tgm{tg.base + side * (%d * S::kStride)};  // ... target pose" % (B["toff"] - A["toff"]))
        E.lines.extend(body.lines)
        return E.lines

    def gen_evaluate(self, task_ids):
        """evaluate_w<k>(): FK of the joints supporting the tasks of one warp role, their weighted error rows (-> strip sE)
        and the non-zero entries of their weighted Jacobian rows (-> strip sJ)."""
        E = Emitter()
        world = {}
        inter = [g for g in self.spec.get("interleave", []) if all(t in task_ids for t in g)]
        done = set()
        for cnt, ti in enumerate(task_ids):
            if ti in done:
                continue
            if cnt > 0:
                E.raw("IKB_PHASE_FENCE();")
            grp = next((g for g in inter if ti in g), None)
            if grp is None:
                self.gen_task(E, ti, world)
                done.add(ti)
                continue
            # Independent tasks with the same shape (Cassie's two legs): emit them in lock step, statement by statement, so
            # that ptxas sees two independent dependency chains side by side (a lone warp per scheduler has no other
            # source of latency hiding).  Joints common to their chains are emitted once, up front.
            common = set(self.tasks[grp[0]]["chain"])
            for t in grp[1:]:
                common &= set(self.tasks[t]["chain"])
            for j in sorted(common):
                self.fk_joint(E, j, world)
            subs = []
            for k, t in enumerate(grp):
                Ek = Emitter(prefix="%c" % (ord("a") + k))
                wk = dict(world)
                self.gen_task(Ek, t, wk)
                subs.append((Ek, wk))
                done.add(t)
            n = max(len(Ek.lines) for Ek, _ in subs)
            for i in range(n):
                for Ek, _ in subs:
                    if i < len(Ek.lines):
                        E.lines.append(Ek.lines[i])
            for _, wk in subs:
                world.update(wk)
        return E.lines

    def frame_world(self, E, f, world, hint):
        """World placement (R[9], p[3]) of model frame f = placement of its parent joint times the frame placement."""
        jf = f["parent"]
        if jf > 0:
            w = self.fk_joint(E, jf, world)
            jR, jp = w["R"], w["p"]
        else:
            jR, jp = [1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0], [0.0, 0.0, 0.0]
        FP = f["placement"]
        return matmul(E, jR, FP[:9], "R" + hint), matvec(E, jR, FP[9:], "p" + hint, add=jp)

    def is_universe(self, f):
        return f["parent"] == 0 and f["placement"] == [1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0, 0, 0, 0]

    def gen_task(self, E, ti, world):
        """Error rows and Jacobian non-zeros of task ti (FK of its chain memoised in `world`)."""
        if self.tasks[ti]["kind"] == "align":
            return self.gen_align_task(E, ti, world)
        if self.tasks[ti]["kind"] == "posture":
            return self.gen_posture_task(E, ti)
        if True:
            task = self.tasks[ti]
            f = task["frame"]
            E.comment("==== task %d: frame %s, %s, reference %s ====" % (ti, task["name"], ["Position", "Orientation", "Full"][task["ktype"]],
                                                                        task["ref_name"]))
            FP = f["placement"]
            ident = FP == [1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0, 0, 0, 0]
            Rf, pf = self.frame_world(E, f, world, "f")
            n = ti
            toff = task["toff"]
            E.raw("T Rt%d[9], pt%d[3];" % (n, n))
            tgn, sEn, sJn = ("tgm", "sEm", "sJm") if self.mir else ("tg", "sE", "sJ")
            wexpr = (lambda r: "wm%d" % (r - task["row"])) if self.mir else (lambda r: "c.weight[%d]" % r)
            if self.is_universe(task["ref"]):
                E.raw("for (int k = 0; k < 9; ++k) Rt%d[k] = %s[%d + k];" % (n, tgn, toff))
                E.raw("for (int k = 0; k < 3; ++k) pt%d[k] = %s[%d + k];" % (n, tgn, toff + 9))
            else:
                # oMt = oMr * target (frame.hpp:46-47).  The reference frame moves with q but compute_jacobian does not
                # differentiate it (frame.hpp:169-181, SURVEY 8a note) -- neither does this code.
                Rr, pr = self.frame_world(E, task["ref"], world, "r")
                arr(E, "Rr%d" % n, Rr)
                arr(E, "pr%d" % n, pr)
                E.raw("T Rg%d[9], pg%d[3];" % (n, n))
                E.raw("for (int k = 0; k < 9; ++k) Rg%d[k] = tg[%d + k];" % (n, toff))
                E.raw("for (int k = 0; k < 3; ++k) pg%d[k] = tg[%d + k];" % (n, toff + 9))
                E.raw("se3_mul(Rr%d, pr%d, Rg%d, pg%d, Rt%d, pt%d);" % (n, n, n, n, n, n))
            arr(E, "Rf%d" % n, Rf)
            arr(E, "pf%d" % n, pf)
            # fMt = oMf^-1 * oMt  (frame.hpp:48-50, universe reference => oMt = target)
            E.raw("T Re%d[9], d%d[3], pe%d[3], w%d[3], th%d, st%d, ct%d, lin%d[3];" % (n, n, n, n, n, n, n, n))
            E.raw("mat3T_mul(Rf%d, Rt%d, Re%d);" % (n, n, n))
            E.raw("for (int k = 0; k < 3; ++k) d%d[k] = pt%d[k] - pf%d[k];" % (n, n, n))
            E.raw("rotT_vec(Rf%d, d%d, pe%d);" % (n, n, n))
            E.raw("log3(Re%d, w%d, th%d, st%d, ct%d);" % (n, n, n, n, n))
            E.raw("const LogCoeffs<T> lc%d = log_coeffs(th%d, st%d, ct%d);" % (n, n, n, n))
            E.raw("log6_from(w%d, lc%d, pe%d, lin%d);" % (n, n, n, n))
            # tMf = fMt^-1: rotation Re^T (log3 = -w, same angle), translation Rt^T (pf - pt)
            E.raw("T nw%d[3] = {-w%d[0], -w%d[1], -w%d[2]}, nd%d[3] = {-d%d[0], -d%d[1], -d%d[2]}, p2%d[3], A%dm[9], B%dm[9];"
                  % (n, n, n, n, n, n, n, n, n, n, n))
            E.raw("rotT_vec(Rt%d, nd%d, p2%d);" % (n, n, n))
            E.raw("jlog6_blocks(nw%d, th%d, lc%d, p2%d, A%dm, B%dm);" % (n, n, n, n, n, n))
            kt, row = task["ktype"], task["row"]
            # error rows, weighted (data.cpp:49)
            src = {POSITION: ["lin%d[%d]" % (n, i) for i in range(3)], ORIENTATION: ["w%d[%d]" % (n, i) for i in range(3)],
                   FULL: ["lin%d[%d]" % (n, i) for i in range(3)] + ["w%d[%d]" % (n, i) for i in range(3)]}[kt]
            for i, s in enumerate(src):
                if self.jreg is not None:   # fold task: the weighted error stays in a register (fold_publish stores it)
                    self.ereg[row + i] = E.var("%s * %s" % (wexpr(row + i), s), "ev")
                    continue
                E.raw("%s.set(%d, %s * %s);" % (sEn, row + i, wexpr(row + i), s))
            top = kt in (POSITION, FULL)
            bot = kt in (ORIENTATION, FULL)
            brow = row + (3 if kt == FULL else 0)
            A = ["A%dm[%d]" % (n, k) for k in range(9)]
            Bm = ["B%dm[%d]" % (n, k) for k in range(9)]

            def store(r, col, val):
                k = self.slot(r, col)
                if self.jreg is not None:   # fold task: the entry never leaves the registers
                    self.jreg[k] = E.var("%s * %s" % (wexpr(r), lit(val)), "jv")
                    return
                E.raw("%s.set(%d, %s * %s);  // J[%d][%d]" % (sJn, k, wexpr(r), lit(val), r, col))

            chain = task["chain"]
            ff_self = ident and len(chain) == 1 and self.joints[chain[0]]["type"] == J_FF
            if ff_self:
                # frame == the free-flyer joint frame: Jf_LOCAL = I6, J = -Jlog6 = -[[A, B], [0, A]]
                iv = self.joints[chain[0]]["idx_v"]
                for i in range(3):
                    for k in range(3):
                        if top:
                            store(row + i, iv + k, E.var("-%s" % A[3 * i + k], "j"))
                            store(row + i, iv + 3 + k, E.var("-%s" % Bm[3 * i + k], "j"))
                        if bot:
                            store(brow + i, iv + 3 + k, E.var("-%s" % A[3 * i + k], "j"))
                return
            # M1 = A Rf^T, M2 = B Rf^T
            RfT = [Rf[3 * j_ + i] for i in range(3) for j_ in range(3)]
            M1 = matmul(E, A, RfT, "M1_")
            M2 = matmul(E, Bm, RfT, "M2_") if top else None
            for j in chain:
                w = world[j] if j in world else self.fk_joint(E, j, world)
                jt = self.joints[j]
                iv = jt["idx_v"]
                if jt["type"] == J_FF:
                    dpf = sub3(E, w["p"], pf, "dp")
                    for k in range(3):
                        rk = [w["R"][k], w["R"][3 + k], w["R"][6 + k]]
                        m1r = matvec(E, M1, rk, "m1r")
                        if top:
                            for i in range(3):
                                store(row + i, iv + k, neg(E, m1r[i]))
                            cx = [_cross_comp(E, dpf, rk, i, "cx") for i in range(3)]
                            m1c = matvec(E, M1, cx, "m1c")
                            m2r = matvec(E, M2, rk, "m2r")
                            for i in range(3):
                                store(row + i, iv + 3 + k, E.var("-(%s + %s)" % (lit(m1c[i]), lit(m2r[i])), "j"))
                        if bot:
                            for i in range(3):
                                store(brow + i, iv + 3 + k, neg(E, m1r[i]))
                elif jt["type"] in (J_RX, J_RY, J_RZ, J_RU):
                    z = w["z"]
                    m1z = matvec(E, M1, z, "m1z")
                    if top:
                        dpf = sub3(E, w["p"], pf, "dp")
                        cx = [_cross_comp(E, dpf, z, i, "cx") for i in range(3)]
                        m1c = matvec(E, M1, cx, "m1c")
                        m2z = matvec(E, M2, z, "m2z")
                        for i in range(3):
                            store(row + i, iv, E.var("-(%s + %s)" % (lit(m1c[i]), lit(m2z[i])), "j"))
                    if bot:
                        for i in range(3):
                            store(brow + i, iv, neg(E, m1z[i]))
                else:  # prismatic: world column [z; 0]
                    if top:
                        m1z = matvec(E, M1, w["z"], "m1z")
                        for i in range(3):
                            store(row + i, iv, neg(E, m1z[i]))

    def gen_posture_task(self, E, ti):
        """PostureTask (posture.hpp:47-66): e = (q.bottomRows(nj) - target) .* mask, J.rightCols(nj) = I (the reference does
        not apply the mask to J); both weighted by the task's row weights (data.cpp:49-50)."""
        task = self.tasks[ti]
        nj, row, toff = task["dim"], task["row"], task["toff"]
        E.comment("==== task %d: posture of the last %d coordinates ====" % (ti, nj))
        for i in range(nj):
            E.raw("sE.set(%d, c.weight[%d] * ((q[%d] - tg[%d]) * c.mask[%d]));" % (row + i, row + i, self.nq - nj + i, toff + i, row + i))
            E.raw("sJ.set(%d, c.weight[%d]);  // J[%d][%d]" % (self.slot(row + i, self.nv - nj + i), row + i, row + i, self.nv - nj + i))

    def gen_align_task(self, E, ti, world):
        """AlignAxisTask (frame.hpp:246-299): e = 1 - r . t^,  J = -(r x t^)^T R_rMf Jf_LOCAL.bottomRows(3), with r the
        aligned axis of the frame expressed in the reference frame and t^ the normalised target."""
        task = self.tasks[ti]
        f = task["frame"]
        n, toff, row, ax = ti, task["toff"], task["row"], task["ktype"]
        E.comment("==== task %d: align axis %s of frame %s, reference %s ====" % (ti, "xyz"[ax], task["name"], task["ref_name"]))
        Rf, pf = self.frame_world(E, f, world, "f")
        arr(E, "Rf%d" % n, Rf)
        if self.is_universe(task["ref"]):
            E.raw("T Rm%d[9];" % n)
            E.raw("for (int k = 0; k < 9; ++k) Rm%d[k] = Rf%d[k];" % (n, n))
        else:
            Rr, _ = self.frame_world(E, task["ref"], world, "r")
            arr(E, "Rr%d" % n, Rr)
            E.raw("T Rm%d[9];" % n)
            E.raw("mat3T_mul(Rr%d, Rf%d, Rm%d);  // rotation of rMf = oMr^-1 oMf" % (n, n, n))
        E.raw("const T rv%d[3] = {Rm%d[%d], Rm%d[%d], Rm%d[%d]};" % (n, n, ax, n, 3 + ax, n, 6 + ax))
        E.raw("T tn%d[3] = {tg[%d], tg[%d], tg[%d]};" % (n, toff, toff + 1, toff + 2))
        E.raw("const T nn%d = sqrt_(dot3(tn%d, tn%d));" % (n, n, n))
        E.raw("for (int k = 0; k < 3; ++k) tn%d[k] = tn%d[k] / nn%d;  // target.normalized()" % (n, n, n))
        E.raw("sE.set(%d, c.weight[%d] * (T(1) - dot3(rv%d, tn%d)));" % (row, row, n, n))
        E.raw("T rxt%d[3], r3%d[3], u%d[3];" % (n, n, n))
        E.raw("cross3(rv%d, tn%d, rxt%d);" % (n, n, n))
        E.raw("rotT_vec(Rm%d, rxt%d, r3%d);   // (r x t)^T R_rMf" % (n, n, n))
        E.raw("rot_vec(Rf%d, r3%d, u%d);      // ... times Rf^T w_j for every column: (Rf r3) . w_j" % (n, n, n))
        u = ["u%d[%d]" % (n, k) for k in range(3)]
        for j in task["chain"]:
            w = world[j] if j in world else self.fk_joint(E, j, world)
            jt = self.joints[j]
            iv = jt["idx_v"]
            if jt["type"] == J_FF:
                for k in range(3):  # angular columns only: world column [p x R e_k; R e_k]
                    rk = [w["R"][k], w["R"][3 + k], w["R"][6 + k]]
                    d = sop(E, [(u[i], rk[i]) for i in range(3)], "al")
                    E.raw("sJ.set(%d, c.weight[%d] * -(%s));  // J[%d][%d]" % (self.slot(row, iv + 3 + k), row, lit(d), row, iv + 3 + k))
            elif jt["type"] in (J_RX, J_RY, J_RZ, J_RU):
                d = sop(E, [(u[i], w["z"][i]) for i in range(3)], "al")
                E.raw("sJ.set(%d, c.weight[%d] * -(%s));  // J[%d][%d]" % (self.slot(row, iv), row, lit(d), row, iv))
            # prismatic joints have no angular part

    def gen_presolve(self, P):
        """The leading P x P block of the factorisation, which involves only the task rows of the SOLVER role itself: Gram
        entries, LDL^T of the block and the first P entries of D^-1 L^-1 e.  The solver role runs this right after its own
        evaluate, while the other roles are still evaluating theirs (its tasks are cheaper), i.e. off the critical path.
        Results go to the factor strip (L, d at their usual slots; yp at slot YOFF + j)."""
        M = self.rows
        ind = "        "
        L = []
        nstrict = M * (M - 1) // 2

        def Lidx(i, k):
            return i * (i - 1) // 2 + k

        order, pos = self.order, self.pos  # elimination order: position -> task row, and back
        col_rows = {}
        for (r, c) in self.slots:
            if pos[r] < P:
                col_rows.setdefault(c, []).append(pos[r])
        for c in col_rows:
            col_rows[c].sort()
        nfma = 0
        L.append(ind + "IKB_PHASE_FENCE();  // the J / e entries below were written by this very thread")
        for j in range(P):
            for i in range(j, P):
                L.append(ind + "T g_%d_%d = %s;" % (i, j, "damping2" if i == j else "T(0)"))
            L.append(ind + "T g_e_%d = sE.get(%d);" % (j, order[j]))
        for c in sorted(col_rows):
            rs = col_rows[c]
            L.append(ind + "{  // J column %d" % c)
            for i in rs:
                L.append(ind + "    const T a%d = sJ.get(%d);" % (i, self.slots[(order[i], c)]))
            for j in rs:
                for i in rs:
                    if i >= j:
                        L.append(ind + "    g_%d_%d += a%d * a%d;" % (i, j, i, j))
                        nfma += 1
            L.append(ind + "}")
        for j in range(P):
            L.append(ind + "sL.set(%d, g_%d_%d);" % (nstrict + j, j, j))
            L.append(ind + "const T inv_%d = rcp_(g_%d_%d);" % (j, j, j))
            for i in range(j + 1, P):
                L.append(ind + "const T l_%d_%d = g_%d_%d * inv_%d;" % (i, j, i, j, j))
                L.append(ind + "sL.set(%d, l_%d_%d);" % (Lidx(i, j), i, j))
            L.append(ind + "sL.set(%d, g_e_%d * inv_%d);  // yp[%d]" % (self.yoff + j, j, j, j))
            for j2 in range(j + 1, P):
                for i in range(j2, P):
                    L.append(ind + "g_%d_%d -= l_%d_%d * g_%d_%d;" % (i, j2, i, j, j2, j))
                    nfma += 1
                L.append(ind + "g_e_%d -= (g_e_%d * inv_%d) * g_%d_%d;" % (j2, j, j, j2, j))
        L.append(ind + "IKB_PHASE_FENCE();")
        self.presolve_fma = nfma
        return L

    def gen_solve(self, W, P=0):
        """y = (J J^T + damping^2 I)^-1 e  (dls.cpp:39-41,53) -- fused Gram / blocked left-looking LDL^T / substitutions.

        Strip sL layout: strictly-lower L[i][k] at i*(i-1)/2 + k, then d[k] at M*(M-1)/2 + k.
        P > 0: the leading P x P block (and yp[0..P)) has been produced by gen_presolve; the first block column is then
        columns 0..P-1 restricted to the rows below the block."""
        M = self.rows
        ind = "        "
        L = []
        nstrict = M * (M - 1) // 2

        def Lidx(i, k):
            return i * (i - 1) // 2 + k

        order, pos = self.order, self.pos  # elimination order (the SOLVER role's rows first when it presolves): every
        col_rows = {}                       # index below is a POSITION in that order; order[i] is the task row
        for (r, c) in self.slots:
            col_rows.setdefault(c, []).append(pos[r])
        for c in col_rows:
            col_rows[c].sort()
        nfma = 0
        L.append(ind + "T e[%d], yp[%d];  // yp = D^-1 L^-1 e, produced as the extra row of the factorisation" % (M, M))
        L.append(ind + "#pragma unroll")
        if order == list(range(M)):
            L.append(ind + "for (int i = 0; i < %d; ++i) e[i] = sE.get(i);" % M)
        else:
            L.pop()  # the #pragma unroll
            for i in range(M):
                L.append(ind + "e[%d] = sE.get(%d);" % (i, order[i]))
        L.append(ind + "T res = T(0);")
        for r in range(self.rows_p0):
            L.append(ind + "res += e[%d] * e[%d];  // visitor.hpp:19 (priority-0 rows, in task-row order)" % (pos[r], pos[r]))
        L.append(ind + "IKB_PHASE_FENCE();  // sE may alias the factor strip: every e is in a register from here on")
        if P > 0:
            # ---- block column 0..P-1, rows P..M-1, against the pre-factorised P x P block ----
            L.append(ind + "#pragma unroll")
            L.append(ind + "for (int j = 0; j < %d; ++j) yp[j] = sL.get(%d + j);  // from presolve" % (P, self.yoff))
            L.append(ind + "IKB_PHASE_FENCE();")
            L.append(ind + "// ---- block column 0..%d (rows %d..%d; the diagonal block comes from presolve) ----" % (P - 1, P, M - 1))
            for j in range(P):
                for i in range(P, M):
                    L.append(ind + "T g_%d_%d = T(0);" % (i, j))
            for c in sorted(col_rows):
                rs = col_rows[c]
                bj = [j for j in rs if j < P]
                lo = [i for i in rs if i >= P]
                if not bj or not lo:
                    continue
                L.append(ind + "{  // J column %d" % c)
                for i in bj + lo:
                    L.append(ind + "    const T a%d = sJ.get(%d);" % (i, self.slots[(order[i], c)]))
                for j in bj:
                    for i in lo:
                        L.append(ind + "    g_%d_%d += a%d * a%d;" % (i, j, i, j))
                        nfma += 1
                L.append(ind + "}")
            for j in range(P):
                L.append(ind + "{  // column %d" % j)
                L.append(ind + "    const T d%d = sL.get(%d), pinv%d = rcp_(d%d);" % (j, nstrict + j, j, j))
                for i in range(P, M):
                    L.append(ind + "    const T l_%d_%d = g_%d_%d * pinv%d;" % (i, j, i, j, j))
                    L.append(ind + "    sL.set(%d, l_%d_%d);" % (Lidx(i, j), i, j))
                for j2 in range(j + 1, P):
                    L.append(ind + "    const T pv_%d_%d = sL.get(%d) * d%d;  // L[%d][%d] d[%d]" % (j2, j, Lidx(j2, j), j, j2, j, j))
                    for i in range(P, M):
                        L.append(ind + "    g_%d_%d -= l_%d_%d * pv_%d_%d;" % (i, j2, i, j, j2, j))
                        nfma += 1
                L.append(ind + "}")
        starts = list(range(P, M, W)) if P > 0 else list(range(0, M, W))
        for j0 in starts:
            j1 = min(j0 + W, M)
            blk = list(range(j0, j1))
            L.append(ind + "IKB_PHASE_FENCE();")
            L.append(ind + "// ---- block column %d..%d ----" % (j0, j1 - 1))
            for j in blk:
                for i in range(j, M):
                    L.append(ind + "T g_%d_%d = %s;" % (i, j, "damping2" if i == j else "T(0)"))
                L.append(ind + "T g_e_%d = e[%d];" % (j, j))
            # Gram part: G[i][j] = sum_c J[i][c] J[j][c]
            for c in sorted(col_rows):
                rs = col_rows[c]
                bj = [j for j in rs if j0 <= j < j1]
                if not bj:
                    continue
                need = [i for i in rs if i >= bj[0]]
                L.append(ind + "{  // J column %d" % c)
                for i in need:
                    L.append(ind + "    const T a%d = sJ.get(%d);" % (i, self.slots[(order[i], c)]))
                for j in bj:
                    for i in need:
                        if i >= j:
                            L.append(ind + "    g_%d_%d += a%d * a%d;" % (i, j, i, j))
                            nfma += 1
                L.append(ind + "}")
            # left-looking update from the factor columns k < j0
            for k in range(j0):
                L.append(ind + "{  // minus column %d of the factor" % k)
                L.append(ind + "    const T dk = sL.get(%d);" % (nstrict + k))
                for i in range(j0, M):
                    L.append(ind + "    const T l%d = sL.get(%d);" % (i, Lidx(i, k)))
                for j in blk:
                    L.append(ind + "    const T v%d = l%d * dk;" % (j, j))
                for j in blk:
                    for i in range(j, M):
                        L.append(ind + "    g_%d_%d -= l%d * v%d;" % (i, j, i, j))
                        nfma += 1
                    L.append(ind + "    g_e_%d -= yp[%d] * v%d;" % (j, k, j))
                L.append(ind + "}")
            # factorise the block column in registers
            for j in blk:
                L.append(ind + "sL.set(%d, g_%d_%d);" % (nstrict + j, j, j))
                L.append(ind + "const T inv_%d = rcp_(g_%d_%d);" % (j, j, j))
                for i in range(j + 1, M):
                    L.append(ind + "const T l_%d_%d = g_%d_%d * inv_%d;" % (i, j, i, j, j))
                    L.append(ind + "sL.set(%d, l_%d_%d);" % (Lidx(i, j), i, j))
                L.append(ind + "yp[%d] = g_e_%d * inv_%d;" % (j, j, j))
                for j2 in range(j + 1, j1):
                    for i in range(j2, M):
                        L.append(ind + "g_%d_%d -= l_%d_%d * g_%d_%d;" % (i, j2, i, j, j2, j))
                        nfma += 1
                    L.append(ind + "g_e_%d -= yp[%d] * g_%d_%d;" % (j2, j, j2, j))
        # back substitution y = L^-T yp, column oriented
        L.append(ind + "IKB_PHASE_FENCE();")
        L.append(ind + "// ---- back substitution ----")
        for k in range(M - 1, -1, -1):
            for i in range(k):
                L.append(ind + "yp[%d] -= sL.get(%d) * yp[%d];" % (i, Lidx(k, i), k))
                nfma += 1
        for i in range(M):
            L.append(ind + "y[%d] = yp[%d];" % (order[i], i))
        L.append(ind + "return res;")
        self.solve_fma = nfma
        return L

    def gen_solve_parallel(self, W, R, solver):
        """The same factorisation as gen_solve, distributed over the R warp roles of a group (one code list per role).

        Block column kb (columns j0..j1-1): the rows of the diagonal block belong to role kb % R for this column, the rows
        below it to role (i % R) (cyclic), the right-hand-side row to role `solver`.
          phase 1  every role accumulates Gram + left-looking updates for its rows; the diagonal owner factorises the W x W
                   block in registers and publishes it (L entries, pivots d) in the strip              -> sync
          phase 2  every role eliminates its sub-diagonal rows against the published block (W(W-1)/2 + W loads), writes
                   its L entries; the solver role does the same for the rhs row (forward substitution)   -> sync
        After the last block column the solver role back-substitutes (serial) -- y ends in its registers.
        All roles execute the same sequence of sync() calls."""
        M = self.rows
        ind = "        "
        nstrict = M * (M - 1) // 2

        def Lidx(i, k):
            return i * (i - 1) // 2 + k

        col_rows = {}
        for (r, c) in self.slots:
            col_rows.setdefault(c, []).append(r)
        for c in col_rows:
            col_rows[c].sort()
        codes = [[] for _ in range(R)]
        nfma = [0] * R
        rolled = int(self.spec.get("rolled_update", 0))  # 0 = unrolled; n = `#pragma unroll n` on the loop over factor columns
        for role in range(R):
            L = codes[role]
            if role == solver:
                L.append(ind + "T e[%d], yp[%d];" % (M, M))
                L.append(ind + "#pragma unroll")
                L.append(ind + "for (int i = 0; i < %d; ++i) e[i] = sE.get(i);" % M)
            L.append(ind + "sync();  // e is in the solver's registers: the strip slots it aliased may be overwritten now")
        nblk = (M + W - 1) // W
        for kb in range(nblk):
            j0, j1 = kb * W, min(kb * W + W, M)
            blk = list(range(j0, j1))
            downer = kb % R
            for role in range(R):
                L = codes[role]
                own = [i for i in range(j1, M) if i % R == role]
                rows = (blk if role == downer else []) + own  # matrix rows this role accumulates in this block column
                has_e = role == solver
                L.append(ind + "// ---- block column %d..%d: rows %s%s ----" % (j0, j1 - 1, rows, " + rhs" if has_e else ""))
                L.append(ind + "IKB_PHASE_FENCE();")
                pairs = [(i, j) for j in blk for i in rows if i >= j]
                for (i, j) in pairs:
                    L.append(ind + "T g_%d_%d = %s;" % (i, j, "damping2" if i == j else "T(0)"))
                if has_e:
                    for j in blk:
                        L.append(ind + "T g_e_%d = e[%d];" % (j, j))
                # Gram part
                for c in sorted(col_rows):
                    rs = col_rows[c]
                    bj = [j for j in rs if j0 <= j < j1]
                    mine = [i for i in rs if i in rows]
                    use = [(i, j) for j in bj for i in mine if i >= j]
                    if not use:
                        continue
                    need = sorted(set([i for i, _ in use] + [j for _, j in use]))
                    L.append(ind + "{  // J column %d" % c)
                    for i in need:
                        L.append(ind + "    const T a%d = sJ.get(%d);" % (i, self.slots[(i, c)]))
                    for (i, j) in use:
                        L.append(ind + "    g_%d_%d += a%d * a%d;" % (i, j, i, j))
                        nfma[role] += 1
                    L.append(ind + "}")
                # left-looking update from factor columns k < j0
                if (rows or has_e) and rolled and j0 > 0:
                    # ONE loop body for all factor columns k < j0 (run-time k: the strip addresses advance by a stride, the
                    # accumulators keep their registers); same operations in the same order as the unrolled form below, so
                    # the results are bit-identical -- only the code is j0 times smaller.  yp[k] comes from the strip (the
                    # solver role publishes it there in phase 2), because a register array cannot take a run-time index.
                    L.append(ind + "#pragma unroll %d" % rolled)
                    L.append(ind + "for (int k = 0; k < %d; ++k) {  // minus column k of the factor" % j0)
                    L.append(ind + "    const S sK{sL.base + k * S::kStride};")
                    L.append(ind + "    const T dk = sK.get(%d);" % nstrict)
                    for i in sorted(set(rows) | set(blk)):
                        L.append(ind + "    const T l%d = sK.get(%d);" % (i, Lidx(i, 0)))
                    for j in blk:
                        L.append(ind + "    const T v%d = l%d * dk;" % (j, j))
                    for (i, j) in pairs:
                        L.append(ind + "    g_%d_%d -= l%d * v%d;" % (i, j, i, j))
                        nfma[role] += j0
                    if has_e:
                        L.append(ind + "    const T ypk = sK.get(%d);" % (nstrict + M))
                        for j in blk:
                            L.append(ind + "    g_e_%d -= ypk * v%d;" % (j, j))
                    L.append(ind + "}")
                elif rows or has_e:
                    for k in range(j0):
                        L.append(ind + "{  // minus column %d of the factor" % k)
                        L.append(ind + "    const T dk = sL.get(%d);" % (nstrict + k))
                        for i in sorted(set(rows) | set(blk)):
                            L.append(ind + "    const T l%d = sL.get(%d);" % (i, Lidx(i, k)))
                        for j in blk:
                            L.append(ind + "    const T v%d = l%d * dk;" % (j, j))
                        for (i, j) in pairs:
                            L.append(ind + "    g_%d_%d -= l%d * v%d;" % (i, j, i, j))
                            nfma[role] += 1
                        if has_e:
                            for j in blk:
                                L.append(ind + "    g_e_%d -= yp[%d] * v%d;" % (j, k, j))
                        L.append(ind + "}")
                if role == downer:
                    # factorise the diagonal block in registers and publish it
                    for j in blk:
                        L.append(ind + "sL.set(%d, g_%d_%d);" % (nstrict + j, j, j))
                        L.append(ind + "const T inv_%d = rcp_(g_%d_%d);" % (j, j, j))
                        for i in range(j + 1, j1):
                            L.append(ind + "const T l_%d_%d = g_%d_%d * inv_%d;" % (i, j, i, j, j))
                            L.append(ind + "sL.set(%d, l_%d_%d);" % (Lidx(i, j), i, j))
                        for j2 in range(j + 1, j1):
                            for i in range(j2, j1):
                                L.append(ind + "g_%d_%d -= l_%d_%d * g_%d_%d;" % (i, j2, i, j, j2, j))
                                nfma[role] += 1
                L.append(ind + "sync();  // diagonal block %d..%d published" % (j0, j1 - 1))
                # phase 2: sub-diagonal rows (and the rhs row) against the published block
                if own or has_e:
                    L.append(ind + "{")
                    for j in blk:
                        L.append(ind + "    const T pd%d = sL.get(%d), pinv%d = rcp_(pd%d);" % (j, nstrict + j, j, j))
                        for j2 in range(j + 1, j1):
                            L.append(ind + "    const T pv_%d_%d = sL.get(%d) * pd%d;  // L[%d][%d] d[%d]" % (j2, j, Lidx(j2, j), j, j2, j, j))
                    for j in blk:
                        for i in own:
                            L.append(ind + "    const T l_%d_%d = g_%d_%d * pinv%d;" % (i, j, i, j, j))
                            L.append(ind + "    sL.set(%d, l_%d_%d);" % (Lidx(i, j), i, j))
                            for j2 in range(j + 1, j1):
                                L.append(ind + "    g_%d_%d -= l_%d_%d * pv_%d_%d;" % (i, j2, i, j, j2, j))
                                nfma[role] += 1
                        if has_e:
                            L.append(ind + "    yp[%d] = g_e_%d * pinv%d;" % (j, j, j))
                            if rolled:
                                L.append(ind + "    sL.set(%d, yp[%d]);" % (nstrict + M + j, j))
                            for j2 in range(j + 1, j1):
                                L.append(ind + "    g_e_%d -= yp[%d] * pv_%d_%d;" % (j2, j, j2, j))
                    L.append(ind + "}")
                L.append(ind + "sync();  // block column %d..%d of the factor complete" % (j0, j1 - 1))
        L = codes[solver]
        L.append(ind + "// ---- back substitution (solver role) ----")
        for k in range(M - 1, -1, -1):
            for i in range(k):
                L.append(ind + "yp[%d] -= sL.get(%d) * yp[%d];" % (i, Lidx(k, i), k))
                nfma[solver] += 1
        L.append(ind + "#pragma unroll")
        L.append(ind + "for (int i = 0; i < %d; ++i) y[i] = yp[i];" % M)
        self.psolve_fma = nfma
        return codes

    def gen_solve_uniform(self, R, solver):
        """The distributed factorisation with ONE body for all R warp roles (spec "uniform_solve").

        The fetch of the role-specific bodies of gen_solve_parallel is what bounds the humanoid kernel (ncu: no_instruction
        is the top stall): here every role runs the SAME instructions on rows picked by its run-time role index r, so the
        warps of a group -- kept in step by the barriers -- share every fetched line.
          phase 0  (role-specific, small) Gram: role r accumulates the task blocks {r,r}, {r,r+1}, {r,r+2} (indices mod R; the
                   R(R-1)/2 off-diagonal blocks are exactly the pairs at cyclic distance 1 and 2 for R = 5) of
                   G = J J^T + damping^2 I into the factor strip: strictly-lower entries in place, the diagonal in its own
                   M slots (DI), e in the right-hand-side slots (RHS; Spec::EOFF points there)            -> sync
          block column kb = 0..M/R-1 (width R, columns j0..j0+R-1), every role:
                   rows r+R*m, m > kb, are its own; the R x R diagonal block is computed redundantly by everybody (same
                   instructions on the same values: identical bits), so there is no publish/consume barrier inside a
                   block column.  Left-looking loop over the finished factor columns k < j0 (run-time k), the diagonal block
                   factorised in registers, own rows eliminated against it and stored; the solver role also carries the
                   rhs row, the pivots d and -- AFTER the barrier, because everybody reads the block's Gram entries from
                   those very slots -- the L entries inside the diagonal block                                -> sync
        One barrier per block column (M/R + 1 in all) instead of two per 2 columns.  Back substitution: solver role."""
        M = self.rows
        if M % R or len(self.tasks) != R or any(t["dim"] != M // R for t in self.tasks):
            raise ValueError("uniform_solve needs R tasks of M/R rows each")
        ind = "        "
        nstrict = M * (M - 1) // 2
        DF, RHS, DI = nstrict, nstrict + M, nstrict + 2 * M
        NB, W = M // R, R
        TD = M // R  # rows per task

        def Lidx(i, k):
            return i * (i - 1) // 2 + k

        row_cols = {}
        for (r, c) in self.slots:
            row_cols.setdefault(r, set()).add(c)
        # ---- phase 0: Gram, per role ----
        roll_gram = bool(self.spec.get("rolled_gram", True))
        grams, grams_blocks = [], []
        nf_gram = [0] * R
        for role in range(R):
            L = []
            blocks = [(role, role)]
            if self.spec.get("gram_blocks"):  # explicit (balanced) assignment of the off-diagonal task blocks: [[ta, tb], ...] per role
                blocks += [(max(a, b), min(a, b)) for a, b in self.spec["gram_blocks"][role]]
            else:
                for d in (1, 2):
                    o = (role + d) % R
                    if o != role and (max(role, o), min(role, o)) not in blocks:
                        blocks.append((max(role, o), min(role, o)))
                if R != 5:
                    raise ValueError("uniform_solve: the default Gram block assignment is written for 5 roles")
            for (ta, tb) in blocks:
                ra = list(range(self.tasks[ta]["row"], self.tasks[ta]["row"] + TD))
                rb = list(range(self.tasks[tb]["row"], self.tasks[tb]["row"] + TD))
                pairs = [(i, j) for i in ra for j in rb if i >= j]
                L.append(ind + "{  // Gram block (task %d, task %d)" % (ta, tb))
                for (i, j) in pairs:
                    L.append(ind + "    T g_%d_%d = %s;" % (i, j, "damping2" if i == j else "T(0)"))
                cols = sorted(set().union(*[row_cols.get(i, set()) for i in ra]) & set().union(*[row_cols.get(j, set()) for j in rb]))
                # Runs of consecutive columns that involve the same rows, with slots affine in the column, become ONE rolled
                # loop (run-time column, one shifted strip per distinct slot stride): the same FMAs in the same order,
                # a third of the code -- the Gram phase is instruction-fetch bound (DESIGN.md 4.1).
                def col_use(c):
                    return [(i, j) for (i, j) in pairs if c in row_cols.get(i, ()) and c in row_cols.get(j, ())]
                runs, k0 = [], 0
                while k0 < len(cols):
                    c0 = cols[k0]
                    use0 = col_use(c0)
                    need0 = sorted(set([i for i, _ in use0] + [j for _, j in use0]))
                    k1 = k0 + 1
                    stride = None
                    while roll_gram and k1 < len(cols) and cols[k1] == cols[k1 - 1] + 1 and col_use(cols[k1]) == use0:
                        st = {i: self.slots[(i, cols[k1])] - self.slots[(i, cols[k1 - 1])] for i in need0}
                        if stride is None:
                            stride = st
                        if st != stride:
                            break
                        k1 += 1
                    runs.append((cols[k0:k1], use0, need0, stride))
                    k0 = k1
                for (rc, use, need, stride) in runs:
                    if not use:
                        continue
                    if len(rc) == 1:
                        c = rc[0]
                        L.append(ind + "    {  // J column %d" % c)
                        for i in need:
                            L.append(ind + "        const T a%d = sJ.get(%d);" % (i, self.slots[(i, c)]))
                        for (i, j) in use:
                            L.append(ind + "        g_%d_%d += a%d * a%d;" % (i, j, i, j))
                            nf_gram[role] += 1
                        L.append(ind + "    }")
                        continue
                    L.append(ind + "    #pragma unroll 1")
                    L.append(ind + "    for (int k = 0; k < %d; ++k) {  // J columns %d..%d" % (len(rc), rc[0], rc[-1]))
                    for st in sorted(set(stride.values())):
                        L.append(ind + "        const S sC%d{sJ.base + k * %d * S::kStride};" % (st, st))
                    for i in need:
                        L.append(ind + "        const T a%d = sC%d.get(%d);" % (i, stride[i], self.slots[(i, rc[0])]))
                    for (i, j) in use:
                        L.append(ind + "        g_%d_%d += a%d * a%d;" % (i, j, i, j))
                        nf_gram[role] += len(rc)
                    L.append(ind + "    }")
                for (i, j) in pairs:
                    L.append(ind + "    sL.set(%d, g_%d_%d);" % (DI + i if i == j else Lidx(i, j), i, j))
                L.append(ind + "}")
            grams.append(L)
            grams_blocks.append(blocks)
        owned = sorted(b for role in range(R) for b in grams_blocks[role])
        if owned != sorted((a, b) for a in range(R) for b in range(a + 1)):
            raise ValueError("uniform_solve: the Gram blocks must be assigned exactly once each")
        # ---- block columns: one body, run-time role r ----
        L = []
        nf = 0
        L.append(ind + "const int r = role;")
        for m in range(1, NB):
            L.append(ind + "const S sO%d{sL.base + ((r + %d) * (r + %d) / 2) * S::kStride};  // own row r + %d: L[r + %d][.]" %
                     (m, R * m, R * m - 1, R * m, R * m))
        for kb in range(NB):
            j0 = kb * W
            own = list(range(kb + 1, NB))
            tri = [(a, b) for b in range(W) for a in range(b, W)]
            L.append(ind + "// ---- block column %d..%d ----" % (j0, j0 + W - 1))
            L.append(ind + "IKB_PHASE_FENCE();")
            if kb == NB - 1:
                L.append(ind + "if (r == %d) {  // nobody owns rows below the last block: the solver role alone" % solver)
            for (a, b) in tri:
                L.append(ind + "T d%d_%d_%d = sL.get(%d);" % (kb, a, b, DI + j0 + a if a == b else Lidx(j0 + a, j0 + b)))
            for m in own:
                for b in range(W):
                    L.append(ind + "T o%d_%d_%d = sO%d.get(%d);" % (kb, m, b, m, j0 + b))
            for b in range(W):
                L.append(ind + "T e%d_%d = T(0);" % (kb, b))
            L.append(ind + "if (r == %d) {" % solver)
            for b in range(W):
                L.append(ind + "    e%d_%d = sL.get(%d);" % (kb, b, RHS + j0 + b))
            L.append(ind + "}")
            if j0 > 0:
                L.append(ind + "#pragma unroll %d" % int(self.spec.get("rolled_update", 2) or 2))
                L.append(ind + "for (int k = 0; k < %d; ++k) {  // minus column k of the factor" % j0)
                L.append(ind + "    const S sK{sL.base + k * S::kStride};")
                L.append(ind + "    const T dk = sK.get(%d);" % DF)
                for a in range(W):
                    L.append(ind + "    const T l%d = sK.get(%d);" % (a, Lidx(j0 + a, 0)))
                for b in range(W):
                    L.append(ind + "    const T v%d = l%d * dk;" % (b, b))
                for (a, b) in tri:
                    L.append(ind + "    d%d_%d_%d -= l%d * v%d;" % (kb, a, b, a, b))
                nf += j0 * len(tri)
                for m in own:
                    L.append(ind + "    const T lo%d = sO%d.get(k);" % (m, m))
                    for b in range(W):
                        L.append(ind + "    o%d_%d_%d -= lo%d * v%d;" % (kb, m, b, m, b))
                    nf += j0 * W
                L.append(ind + "    if (r == %d) {" % solver)
                L.append(ind + "        const T le = sK.get(%d);" % RHS)
                for b in range(W):
                    L.append(ind + "        e%d_%d -= le * v%d;" % (kb, b, b))
                L.append(ind + "    }")
                L.append(ind + "}")
            # the diagonal block, in registers (every role: identical bits)
            for b in range(W):
                L.append(ind + "const T inv%d_%d = rcp_(d%d_%d_%d);" % (kb, b, kb, b, b))
                for a in range(b + 1, W):
                    L.append(ind + "const T l%d_%d_%d = d%d_%d_%d * inv%d_%d;" % (kb, a, b, kb, a, b, kb, b))
                for b2 in range(b + 1, W):
                    for a in range(b2, W):
                        L.append(ind + "d%d_%d_%d -= l%d_%d_%d * d%d_%d_%d;" % (kb, a, b2, kb, a, b, kb, b2, b))
                        nf += 1
            # own rows against the block
            for m in own:
                for b in range(W):
                    L.append(ind + "{ const T lo = o%d_%d_%d * inv%d_%d; sO%d.set(%d, lo);" % (kb, m, b, kb, b, m, j0 + b))
                    for b2 in range(b + 1, W):
                        L.append(ind + "  o%d_%d_%d -= lo * d%d_%d_%d;" % (kb, m, b2, kb, b2, b))
                        nf += 1
                    L.append(ind + "}")
            L.append(ind + "if (r == %d) {  // pivots and the rhs row (forward substitution rides along)" % solver)
            for b in range(W):
                L.append(ind + "    sL.set(%d, d%d_%d_%d);" % (DF + j0 + b, kb, b, b))
            for b in range(W):
                L.append(ind + "    { const T yb = e%d_%d * inv%d_%d; sL.set(%d, yb);" % (kb, b, kb, b, RHS + j0 + b))
                for b2 in range(b + 1, W):
                    L.append(ind + "      e%d_%d -= yb * d%d_%d_%d;" % (kb, b2, kb, b2, b))
                L.append(ind + "    }")
            L.append(ind + "}")
            if kb < NB - 1:
                L.append(ind + "sync();  // block column %d..%d of the factor complete; everybody has read the block's Gram entries" % (j0, j0 + W - 1))
            L.append(ind + "if (r == %d) {" % solver)
            for b in range(W):
                for a in range(b + 1, W):
                    L.append(ind + "    sL.set(%d, l%d_%d_%d);" % (Lidx(j0 + a, j0 + b), kb, a, b))
            L.append(ind + "}")
            if kb == NB - 1:
                L.append(ind + "}")
        L.append(ind + "if (r == %d) {  // ---- back substitution (solver role) ----" % solver)
        L.append(ind + "    T yp[%d];" % M)
        L.append(ind + "    #pragma unroll")
        L.append(ind + "    for (int i = 0; i < %d; ++i) yp[i] = sL.get(%d + i);" % (M, RHS))
        for k in range(M - 1, -1, -1):
            for i in range(k):
                L.append(ind + "    yp[%d] -= sL.get(%d) * yp[%d];" % (i, Lidx(k, i), k))
                nf += 1
        L.append(ind + "    #pragma unroll")
        L.append(ind + "    for (int i = 0; i < %d; ++i) sL.set(%d + i, yp[i]);  // y for step_role() of every role" % (M, RHS))
        L.append(ind + "    #pragma unroll")
        L.append(ind + "    for (int i = 0; i < %d; ++i) y[i] = yp[i];" % M)
        L.append(ind + "}")
        self.usolve_fma = (nf_gram, nf)
        self.rhs_off = RHS
        return grams, L

    def tmem_batch(self, lines, strip, ind):
        """Spec "tmem_j": the Jacobian reads of a block of generated lines become one getn() per run of consecutive slots,
        issued at the top of the block -- a few tcgen05.ld and ONE wait per run (TStrip::getn) instead of a load and a wait
        per entry.  The same values reach the same expressions."""
        if not self.spec.get("tmem_j"):
            return lines
        pat = re.compile(r"\b%s\.get\((-?\d+)\)" % strip)
        runs = []
        for k in sorted({int(k) for ln in lines for k in pat.findall(ln)}):
            if runs and runs[-1][0] + runs[-1][1] == k:
                runs[-1][1] += 1
            else:
                runs.append([k, 1])
        head, name = [], {}
        for k0, n in runs:
            nm = "jb%d" % k0 if k0 >= 0 else "jbm%d" % -k0
            head.append(ind + "T %s[%d];" % (nm, n))
            head.append(ind + "%s.getn(%d, %s);" % (strip, k0, nm))
            for i in range(n):
                name[k0 + i] = "%s[%d]" % (nm, i)
        return head + [pat.sub(lambda mt: name[int(mt.group(1))], ln) for ln in lines]

    def gen_solve_arrow(self, groups, solver, fold=None):
        """Spec "arrow_solve": the step WITHOUT the dense M x M factorisation, for task sets whose Jacobian is "bordered block
        diagonal": a few columns (the free-flyer; joints that several limbs' tasks share) are touched by several warp
        roles, every other column by ONE role only.  With U_a / C_a the shared / private columns of role a's rows,
        G = J J^T + l^2 I = blockdiag(D_a) + U U^T, D_a = C_a C_a^T + l^2 I, and the step dq = -J^T G^-1 e is

            s = -dq_shared = (l^2 I + sum_a l^2 U_a^T D_a^-1 U_a)^-1  sum_a l^2 U_a^T D_a^-1 e_a      (k x k, k = #shared columns)
            y_a = D_a^-1 (e_a - U_a s),   dq_private(a) = -C_a^T y_a                                  (role-local)

        (the push-through / Woodbury identity; it is the SAME dq as dls.cpp:52-53 up to rounding, and -- written with the
        l^2 factor on both sides -- well scaled: a role without private columns contributes U^T U and U^T e, no 1 / l^2).
        Work per role: one m_a x m_a LDL^T (m_a = its rows) and k_a + 1 substitutions; then, identically in every role, the
        k x k system.  ONE group barrier (the contributions are published) instead of one or two per block column, and
        no role waits for another one's factor columns.
          phase 1  role a, reading ONLY its own rows of J and e (so it follows the role's evaluate without a barrier):
                   D_a, its LDL^T, X = D_a^-1 U_a column by column, S'_a = l^2 U_a^T X, t'_a = l^2 X^T e_a -> published   -> sync
          phase 2  every role, same code: C = l^2 I + sum S'_a, b = sum t'_a, LDL^T, s = C^-1 b
          phase 3  role a with private columns: y_a = D_a^-1 (e_a - U_a s) -> its own (dead) factor slots; the solver role stores s.
        step_role() then takes dq_shared = -s and its private columns from y (gen_step_roles_arrow).
        Strip layout (sL): e (M, written by evaluate, never overwritten) | s (k) | per role: published S'_a, t'_a and, for a
        role with private columns, the factor of D_a (whose slots finally carry y_a).  A role WITHOUT private columns
        publishes into its own Jacobian slots instead (nobody else reads them, and it has them in registers by then).
        Roles of a mirrored task pair share one body (`side` rebases the strips), as their evaluate does.
        `fold`: index of the group that is the spec's "fold_task" (no warp role of its own, see gen_fold): its contributions
        are published from registers by gen_fold, in the factor strip; the warp role of group k is then k - 1."""
        M = self.rows
        R = len(groups)
        ind = "        "
        role_rows = [[self.tasks[t]["row"] + i for t in sorted(g) for i in range(self.tasks[t]["dim"])] for g in groups]
        row_role = {r: k for k, rows in enumerate(role_rows) for r in rows}
        col_roles = {}
        for (r, c) in self.slots:
            col_roles.setdefault(c, set()).add(row_role[r])
        shared = sorted(c for c, rs in col_roles.items() if len(rs) > 1)
        ks = len(shared)
        if ks == 0 or ks > 12:
            raise ValueError("arrow_solve: %d shared columns (needs 1..12)" % ks)
        spos = {c: i for i, c in enumerate(shared)}
        KK = ks * (ks + 1) // 2
        per = KK + ks

        def Sidx(i, j):
            return i * (i + 1) // 2 + j

        def has(r, c):
            return (r, c) in self.slots

        privs = [sorted(c for c, rs in col_roles.items() if rs == {k}) for k in range(R)]
        ushs = [[c for c in shared if any(has(r, c) for r in role_rows[k])] for k in range(R)]
        # ---- strip layout ----
        SOFF = M
        off = M + ks
        # "arrow_common_once": the joints common to all roles (the free-flyer) are stepped by the solver role alone, which
        # publishes their new coordinates here; the other roles fetch them behind the barrier at the top of the next trip
        # "arrow_fac_regs": the factor of D_a and y_a stay in the role's registers between the phases (few rows per role)
        fac_regs = bool(self.spec.get("arrow_fac_regs", False))
        self.arrow_qc = None      # one set of slots every role reads (factor in registers), or ...
        self.arrow_mail = None    # ... role -> slots of its own copy ("mailbox": the role's factor slots and e rows, which are
        #                               private to it and dead between the second barrier and its next evaluate -- no extra slots)
        ncq = 0
        if self.spec.get("arrow_common_once", True):
            chains_ = [sorted(set(j for t in g for j in self.tasks[t]["chain"])) for g in groups]
            ncq = len(self.joint_cols(sorted(set.intersection(*[set(ch) for ch in chains_])))[1])
            if ncq and fac_regs:
                self.arrow_qc = off
                off += ncq
        y_regs = fac_regs
        pub = {}     # role -> ("J", [slots]) | ("L", base)
        facb = {}    # role -> base of its factor (m (m + 1) / 2 slots) in sL
        for k in range(R):
            own = sorted(self.slots[(r, c)] for (r, c) in self.slots if row_role[r] == k)
            if not privs[k] and len(own) >= per and self.spec.get("arrow_pub_in_j", True) and not self.spec.get("tmem_j") and k != fold:
                pub[k] = ("J", own[:per])
            else:
                pub[k] = ("L", off)
                off += per
            if privs[k]:
                m = len(role_rows[k])
                facb[k] = off
                if not fac_regs:
                    off += m * (m + 1) // 2
        nfact = off
        mmax = max([len(role_rows[k]) for k in range(R) if privs[k]] or [1])
        if ncq and not fac_regs:
            mail = {}
            for k in range(R):
                if k == solver or k == fold:
                    continue
                m = len(role_rows[k])
                own = ([facb[k] + i for i in range(m * (m + 1) // 2)] if privs[k] else []) + list(role_rows[k])   # (e row r sits in slot r)
                if self.spec.get("arrow_cap_solo"):
                    # the solver role alone reads the published contributions, before the second barrier of psolve(); the
                    # factor and e are still being read by the role's phase 3 when the solver role steps
                    own = [pub[k][1] + i for i in range(per)] if pub[k][0] == "L" else []
                if len(own) < ncq:
                    mail = None
                    break
                mail[k] = own[:ncq]
            if mail is not None and (not privs[solver] or fold is not None):
                self.arrow_mail = {k - (fold is not None): v for k, v in mail.items()}   # keyed by warp role
                y_regs = True      # (y must not sit in the factor slots: the solver role fills the mailboxes while the others step)
        self.arrow_y = {}   # row -> sL slot of y[row] (rows of roles with private columns)

        def pub_at(k, idx):
            kind, where = pub[k]
            return ("sJ", where[idx]) if kind == "J" else ("sL", where + idx)

        entries = {}   # (ci, cj) -> roles that publish it ; ('t', ci) -> roles
        nf = [0] * R

        def emit_role(k, dJ=0, dR=0, dL=0):
            """(phase 1, phase 3) of role k; strip indices are emitted minus (dJ, dR, dL) and go through the rebased strips
            sJr / sEr / sLr, so that a mirrored role can run the body of its partner."""
            rows = role_rows[k]
            m = len(rows)
            priv, ush = privs[k], ushs[k]
            L, F = [], []

            def jget(r, c):
                return "sJr.get(%d)" % (self.slots[(r, c)] - dJ)

            def pset(idx, expr):
                strip, at = pub_at(k, idx)
                return ind + ("sJr.set(%d, %s);" % (at - dJ, expr) if strip == "sJ" else "sLr.set(%d, %s);" % (at - dL, expr))

            for i, r in enumerate(rows):
                L.append(ind + "const T e%d = sEr.get(%d);" % (i, r - dR))

            def u(i, c):   # expression of U_a[i][c] (None = structural zero); loads are emitted per column
                return "u%d_%d" % (i, spos[c]) if has(rows[i], c) else None

            if not priv:
                # D_a = l^2 I: l^2 U^T D^-1 U = U^T U, l^2 U^T D^-1 e = U^T e -- no division by the damping
                for c in ush:
                    for i in range(m):
                        if has(rows[i], c):
                            L.append(ind + "const T u%d_%d = %s;" % (i, spos[c], jget(rows[i], c)))
                L.append(ind + "IKB_PHASE_FENCE();   // every entry is in registers: the slots may be overwritten")
                for a_, c in enumerate(ush):
                    for c2 in ush[:a_ + 1]:
                        terms = ["%s * %s" % (u(i, c), u(i, c2)) for i in range(m) if u(i, c) and u(i, c2)]
                        if terms:
                            L.append(pset(Sidx(spos[c], spos[c2]), " + ".join(terms)))
                            entries.setdefault((spos[c], spos[c2]), set()).add(k)
                            nf[k] += len(terms)
                    terms = ["%s * e%d" % (u(i, c), i) for i in range(m) if u(i, c)]
                    L.append(pset(KK + spos[c], " + ".join(terms)))
                    entries.setdefault(("t", spos[c]), set()).add(k)
                    nf[k] += len(terms)
                return L, F
            # ---- D_a = C_a C_a^T + l^2 I ----
            for i in range(m):
                for j in range(i + 1):
                    L.append(ind + "T d%d_%d = %s;" % (i, j, "damping2" if i == j else "T(0)"))
            for pc, c in enumerate(priv):
                need = [i for i in range(m) if has(rows[i], c)]
                L.append(ind + "{  // private column #%d" % pc)
                blk = []
                for i in need:
                    blk.append(ind + "    const T a%d = %s;" % (i, jget(rows[i], c)))
                for i in need:
                    for j in need:
                        if i >= j:
                            blk.append(ind + "    d%d_%d += a%d * a%d;" % (i, j, i, j))
                            nf[k] += 1
                L.extend(self.tmem_batch(blk, "sJr", ind + "    "))
                L.append(ind + "}")
            # ---- LDL^T in registers (SPD thanks to the damping: no pivoting) ----
            fi = 0
            fac_l, fac_inv = {}, {}
            for j in range(m):
                L.append(ind + "const T inv%d = rcp_(d%d_%d);" % (j, j, j))
                fac_inv[j] = fi if fac_regs else facb[k] + fi
                L.append(ind + ("fac[%d] = inv%d;" % (fi, j) if fac_regs else "sLr.set(%d, inv%d);" % (fac_inv[j] - dL, j)))
                fi += 1
                for i in range(j + 1, m):
                    L.append(ind + "const T l%d_%d = d%d_%d * inv%d;" % (i, j, i, j, j))
                    fac_l[(i, j)] = fi if fac_regs else facb[k] + fi
                    L.append(ind + ("fac[%d] = l%d_%d;" % (fi, i, j) if fac_regs else "sLr.set(%d, l%d_%d);" % (fac_l[(i, j)] - dL, i, j)))
                    fi += 1
                for j2 in range(j + 1, m):
                    for i in range(j2, m):
                        L.append(ind + "d%d_%d -= l%d_%d * d%d_%d;" % (i, j2, i, j, j2, j))
                        nf[k] += 1

            def solve_lines(out, rhs, x, lname=lambda i, j: "l%d_%d" % (i, j), iname=lambda j: "inv%d" % j):
                """x = D_a^-1 rhs : forward substitution, D^-1, back substitution; rhs[i] = expression or None (zero)."""
                z = []
                for i in range(m):
                    terms = ["%s * %s" % (lname(i, j), z[j]) for j in range(i) if z[j]]
                    if rhs[i] is None and not terms:
                        z.append(None)
                        continue
                    nm = "%sz%d" % (x, i)
                    out.append(ind + "const T %s = %s%s;" % (nm, rhs[i] if rhs[i] is not None else "T(0)", "".join(" - " + t for t in terms)))
                    nf[k] += len(terms)
                    z.append(nm)
                w = [None] * m
                for i in range(m - 1, -1, -1):
                    terms = ["%s * %s" % (lname(j, i), w[j]) for j in range(i + 1, m) if w[j]]
                    if z[i] is None and not terms:
                        continue
                    nm = "%s%d" % (x, i)
                    base = "%s * %s" % (z[i], iname(i)) if z[i] else "T(0)"
                    out.append(ind + "const T %s = %s%s;" % (nm, base, "".join(" - " + t for t in terms)))
                    nf[k] += len(terms) + 1
                    w[i] = nm
                return w

            # One shared column at a time (short live ranges: x_c lives only inside its block, the other columns' entries are
            # re-read from the strip): x_c = D_a^-1 u_c, then S'[c][c2] = l^2 x_c . u_c2 for c2 <= c (D_a^-1 is symmetric) and
            # t'[c] = l^2 x_c . e_a -- so D_a^-1 e_a is never formed.
            for a_, c in enumerate(ush):
                L.append(ind + "IKB_PHASE_FENCE();")
                L.append(ind + "{  // shared column %d" % c)
                L0 = L
                L = []
                for i in range(m):
                    if has(rows[i], c):
                        L.append(ind + "const T u%d_%d = %s;" % (i, spos[c], jget(rows[i], c)))
                x = solve_lines(L, [u(i, c) for i in range(m)], "x%d_" % spos[c])
                for c2 in ush[:a_ + 1]:
                    terms = ["%s * %s" % (x[i], u(i, c2) if c2 == c else jget(rows[i], c2))
                             for i in range(m) if x[i] and has(rows[i], c2)]
                    if terms:
                        L.append(pset(Sidx(spos[c], spos[c2]), "damping2 * (%s)" % " + ".join(terms)))
                        entries.setdefault((spos[c], spos[c2]), set()).add(k)
                        nf[k] += len(terms)
                terms = ["%s * e%d" % (x[i], i) for i in range(m) if x[i]]
                L.append(pset(KK + spos[c], "damping2 * (%s)" % (" + ".join(terms) if terms else "T(0)")))
                entries.setdefault(("t", spos[c]), set()).add(k)
                nf[k] += len(terms)
                L = L0 + self.tmem_batch(L, "sJr", ind)
                L.append(ind + "}")
            # ---- phase 3: y_a = D_a^-1 (e_a - U_a s) ----
            for i in range(m):
                terms = ["%s * s[%d]" % (jget(rows[i], c), spos[c]) for c in ush if has(rows[i], c)]
                F.append(ind + "const T r%d = sEr.get(%d)%s;" % (i, rows[i] - dR, "".join(" - " + t for t in terms)))
                nf[k] += len(terms)
            for (i, j), idx in sorted(fac_l.items()):
                F.append(ind + ("const T fl%d_%d = fac[%d];" % (i, j, idx) if fac_regs else "const T fl%d_%d = sLr.get(%d);" % (i, j, idx - dL)))
            for j, idx in sorted(fac_inv.items()):
                F.append(ind + ("const T fi%d = fac[%d];" % (j, idx) if fac_regs else "const T fi%d = sLr.get(%d);" % (j, idx - dL)))
            w = solve_lines(F, ["r%d" % i for i in range(m)], "y_", lname=lambda i, j: "fl%d_%d" % (i, j), iname=lambda j: "fi%d" % j)
            F[:] = self.tmem_batch(F, "sJr", ind)
            if y_regs:
                for i in range(m):
                    F.append(ind + "y[%d] = %s;" % (i, w[i] if w[i] else "T(0)"))
                    self.arrow_y[rows[i]] = ("reg", i)
                return L, F
            F.append(ind + "IKB_PHASE_FENCE();   // the factor is in registers: its slots now carry y")
            for i in range(m):
                F.append(ind + "sLr.set(%d, %s);" % (facb[k] + i - dL, w[i] if w[i] else "T(0)"))
                self.arrow_y[rows[i]] = facb[k] + i
            return L, F

        # mirrored pairs: (role a, role b) whose bodies are identical up to constant strip offsets
        mirror_of = {}    # role b -> (role a, dJ, dR, dL)
        for pair in self.spec.get("mirror", []):
            ra = next((k for k, g in enumerate(groups) if list(g) == [pair[0]]), None)
            rb = next((k for k, g in enumerate(groups) if list(g) == [pair[1]]), None)
            if ra is None or rb is None or not privs[ra] or not privs[rb] or pub[ra][0] != "L" or pub[rb][0] != "L":
                continue
            try:
                dJ = self.slots[(role_rows[rb][0], shared[0])] - self.slots[(role_rows[ra][0], shared[0])]
            except KeyError:
                continue
            dR = role_rows[rb][0] - role_rows[ra][0]
            dL = pub[rb][1] - pub[ra][1]
            save = (dict(entries), list(nf), dict(self.arrow_y))
            try:
                same = emit_role(ra) == emit_role(rb, dJ, dR, dL)
            except KeyError:
                same = False
            entries.clear()
            entries.update(save[0])
            nf[:] = save[1]
            self.arrow_y = save[2]
            if same:
                mirror_of[rb] = (ra, dJ, dR, dL)
        locals_, finishes = [], []
        for k in range(R):
            if k == fold:
                if privs[k] or pub[k][0] != "L":
                    raise ValueError("fold_task: its rows must touch shared columns only")
                self.fold_pub = self.gen_fold_publish(role_rows[k], ushs[k], has, spos, KK, pub[k][1], R - 1)
                for key in self.fold_pub[1]:
                    entries.setdefault(key, set()).add(k)
                nf[k] = self.fold_pub[2]
                locals_.append([])
                finishes.append([])
                continue
            hdr = ind + "// role %d: rows %s, private columns %s, shared columns %s" % (k, role_rows[k], privs[k], ushs[k])
            L, F = emit_role(k)
            locals_.append([hdr] + L)
            finishes.append(F)
        # ---- phase 2: the k x k system, identical in every role ----
        Cc = []

        def pget(k, idx):
            strip, at = pub_at(k, idx)
            return "%s.get(%d)" % (strip, at)

        for i in range(ks):
            for j in range(i + 1):
                terms = [pget(k, Sidx(i, j)) for k in sorted(entries.get((i, j), []))]
                Cc.append(ind + "T c%d_%d = %s%s;" % (i, j, "damping2" if i == j else "T(0)", "".join(" + " + t for t in terms)))
            terms = [pget(k, KK + i) for k in sorted(entries.get(("t", i), []))]
            Cc.append(ind + "const T b%d = %s;" % (i, " + ".join(terms) if terms else "T(0)"))
        for j in range(ks):
            Cc.append(ind + "const T ci%d = rcp_(c%d_%d);" % (j, j, j))
            for i in range(j + 1, ks):
                Cc.append(ind + "const T cl%d_%d = c%d_%d * ci%d;" % (i, j, i, j, j))
            for j2 in range(j + 1, ks):
                for i in range(j2, ks):
                    Cc.append(ind + "c%d_%d -= cl%d_%d * c%d_%d;" % (i, j2, i, j, j2, j))
        for i in range(ks):
            Cc.append(ind + "const T cz%d = b%d%s;" % (i, i, "".join(" - cl%d_%d * cz%d" % (i, j, j) for j in range(i))))
        for i in range(ks - 1, -1, -1):
            Cc.append(ind + "s[%d] = cz%d * ci%d%s;" % (i, i, i, "".join(" - cl%d_%d * s[%d]" % (j, i, j) for j in range(i + 1, ks))))
        self.arrow = dict(shared=shared, spos=spos, soff=SOFF, ks=ks, nfact=nfact, fma=nf, mirror_of=mirror_of,
                          pub=pub, facb=facb, fac_regs=fac_regs, y_regs=y_regs, nfac=mmax * (mmax + 1) // 2 if fac_regs else 1, my=mmax)
        self.rhs_off = 0
        return locals_, Cc, finishes

    def gen_fold_publish(self, rows, ush, has, spos, KK, off, nw):
        """Spec "fold_task": the contributions of the fold task's rows to the shared-column system (U^T U and U^T e -- the rows
        have no private columns, so D = l^2 I cancels), with the SAME terms in the same order as a warp role of its own
        publishes them (gen_solve_arrow, branch `not priv`), but straight from the registers of the fold task's evaluation,
        which every warp role runs.  The rows are cut into nw consecutive runs, run w belonging to warp role w: the role
        stores the weighted errors of its rows, and an entry is published by the role that owns the last row among its
        terms (Cassie's pelvis: role 0 the 18 entries of the position rows, role 1 the 9 that also involve the orientation
        rows -- 54 FMAs each).  Returns (lines per warp role, published entries, FMAs)."""
        m = len(rows)
        own = {r: i * nw // m for i, r in enumerate(rows)}
        code = [[] for _ in range(nw)]
        keys, nfma = [], 0
        for r in rows:
            code[own[r]].append("sE.set(%d, %s);" % (r, self.ereg[r]))

        def u(i, c):
            return self.jreg[self.slots[(rows[i], c)]]

        for a_, c in enumerate(ush):
            for c2 in ush[:a_ + 1]:
                idx = [i for i in range(m) if has(rows[i], c) and has(rows[i], c2)]
                if idx:
                    at = off + spos[c] * (spos[c] + 1) // 2 + spos[c2]
                    code[own[rows[idx[-1]]]].append("sE.set(%d, %s);" % (at, " + ".join("%s * %s" % (u(i, c), u(i, c2)) for i in idx)))
                    keys.append((spos[c], spos[c2]))
                    nfma += len(idx)
            idx = [i for i in range(m) if has(rows[i], c)]
            code[own[rows[idx[-1]]]].append("sE.set(%d, %s);" % (off + KK + spos[c], " + ".join("%s * %s" % (u(i, c), self.ereg[rows[i]]) for i in idx)))
            keys.append(("t", spos[c]))
            nfma += len(idx)
        return code, keys, nfma

    def gen_step_roles_arrow(self, groups, solver):
        """step_role() of spec "arrow_solve": dq of a shared column is -s (from the strip), a private column's comes from the
        role's own rows of y; the joints common to all roles (the free-flyer) are stepped by everybody, redundantly."""
        A = self.arrow
        chains = [sorted(set(j for t in g for j in self.tasks[t]["chain"])) for g in groups]
        common = sorted(set.intersection(*[set(ch) for ch in chains]))
        covered = set(j for ch in chains for j in ch)
        loose = [j for j, jt in enumerate(self.joints) if jt["type"] != J_UNIVERSE and j not in covered]
        ind = "        "

        def dq_lines(cols, ind_):
            L = []
            for c in cols:
                if c in A["spos"]:
                    L.append(ind_ + "dq[%d] = -s[%d];" % (c, A["spos"][c]))
                else:
                    L.extend(self.gen_dq([c], ind_)[1:])
            return L

        ccols, cqs = self.joint_cols(common)
        self.qmap = self.qmaps[0] if self.qmaps else None      # the common joints sit in the same registers in every role
        C = [ind + "IKB_PHASE_FENCE();"] + dq_lines(ccols, ind) + self.gen_integrate(common, ind)
        roles, qsets = [], []
        for k, ch in enumerate(chains):
            own = [j for j in ch if j not in common] + (loose if k == solver else [])
            cols, qs = self.joint_cols(own)
            self.qmap = self.qmaps[k] if self.qmaps else None
            self.ymap = {r: v[1] for r, v in self.arrow_y.items() if isinstance(v, tuple)} or None   # y in the role's registers
            # (one run per column: the whole role's block at once would hold 2 x 21 more registers across the step)
            dq = [b for ln in dq_lines(cols, ind + "    ") for b in self.tmem_batch([ln], "sJ", ind + "    ")]
            roles.append(dq + self.gen_integrate(own, ind + "    "))
            qsets.append(qs + (cqs if k == solver else []))
        self.qmap = None
        self.ymap = None
        self.arrow_common = (cqs, ccols)
        return C, roles, qsets

    def gen_dq(self, cols=None, ind="        "):
        L = []
        L.append(ind + "IKB_PHASE_FENCE();")
        for c in (range(self.nv) if cols is None else cols):
            rs = sorted(r for (r, cc) in self.slots if cc == c)
            if not rs:
                L.append(ind + "dq[%d] = T(0);" % c)
                continue
            ymap = getattr(self, "ymap", None)
            expr = " + ".join("sJ.get(%d) * y[%d]" % (self.slots[(r, c)], ymap[r] if ymap else r) for r in rs)
            L.append(ind + "dq[%d] = -(%s);" % (c, expr))
        return L

    def joint_cols(self, joints):
        """velocity columns / configuration entries of a set of joints"""
        cols, qs = [], []
        for j in joints:
            jt = self.joints[j]
            nvj, nqj = (6, 7) if jt["type"] == J_FF else (1, 1)
            cols.extend(range(jt["idx_v"], jt["idx_v"] + nvj))
            qs.extend(range(jt["idx_q"], jt["idx_q"] + nqj))
        return cols, qs

    def gen_step_roles(self, groups, solver):
        """Distributed step (spec "uniform_solve"): after the solve every role takes dq = -J^T y and the manifold step
        (dls.cpp:52,67-71) on the coordinates ITS evaluate reads -- the joints common to all roles (the free-flyer) by
        everybody, redundantly and with the same instructions; the rest of its chains by the role alone -- instead of the
        solver role doing all of it while the others wait.  Returns (common code, per-role code, per-role q entries)."""
        chains = [sorted(set(j for t in g for j in self.tasks[t]["chain"])) for g in groups]
        common = sorted(set.intersection(*[set(ch) for ch in chains]))
        covered = set(j for ch in chains for j in ch)
        loose = [j for j, jt in enumerate(self.joints) if jt["type"] != J_UNIVERSE and j not in covered]
        ind = "        "
        ccols, cqs = self.joint_cols(common)
        C = self.gen_dq(ccols, ind) + self.gen_integrate(common, ind)
        roles, qsets = [], []
        for k, ch in enumerate(chains):
            own = [j for j in ch if j not in common] + (loose if k == solver else [])
            cols, qs = self.joint_cols(own)
            roles.append(self.gen_dq(cols, ind + "    ") + self.gen_integrate(own, ind + "    "))
            qsets.append(qs + (cqs if k == solver else []))
        return C, roles, qsets

    def gen_integrate(self, joints=None, ind="        "):
        """pinocchio::integrate (dls.cpp:67-68) + clamp (common.hpp:53-56), joint by joint."""
        L = []
        for j, jt in enumerate(self.joints):
            if jt["type"] == J_UNIVERSE or (joints is not None and j not in joints):
                continue
            iq, iv = jt["idx_q"], jt["idx_v"]
            if jt["type"] == J_FF:
                L.append(ind + "{")
                L.append(ind + "    T v6[6], R0[9];")
                L.append(ind + "    for (int k = 0; k < 6; ++k) v6[k] = step * dq[%d + k];" % iv)
                L.append(ind + "    quat_to_rot(q[%d], q[%d], q[%d], q[%d], R0);" % (self.ql(iq + 3), self.ql(iq + 4), self.ql(iq + 5), self.ql(iq + 6)))
                if [self.ql(iq + k) for k in range(7)] != list(range(self.ql(iq), self.ql(iq) + 7)):
                    raise ValueError("free-flyer coordinates must be contiguous in the local registers")
                L.append(ind + "    integrate_freeflyer(R0, &q[%d], &q[%d], v6);" % (self.ql(iq), self.ql(iq + 3)))
                L.append(ind + "}")
            else:
                L.append(ind + "q[%d] += step * dq[%d];" % (self.ql(iq), iv))
        if joints is not None:
            for k in self.joint_cols(joints)[1]:
                L.append(ind + "q[%d] = min_(c.upper[%d], max_(q[%d], c.lower[%d]));" % (self.ql(k), k, self.ql(k), k))
            return L
        L.append(ind + "#pragma unroll")
        L.append(ind + "for (int k = 0; k < %d; ++k) q[k] = min_(c.upper[k], max_(q[k], c.lower[k]));" % self.nq)
        return L

    def signature(self):
        """C++ initialisers used by matches(): the specialisation is only valid for exactly this tree / task list."""
        used = sorted(set(j for t in self.tasks for j in t["chain"]))
        return used

    def emit(self, struct_name, display_name):
        groups = self.spec.get("warp_groups") or [list(range(len(self.tasks)))]
        # "fold_task": a task whose rows touch only the columns shared by all roles (Cassie's pelvis pose: the free-flyer) and
        # that has no warp role of its own -- every role evaluates it in registers and publishes its share of the task's
        # contributions to the shared-column system (gen_fold_publish).  The solve sees it as a group of its own (`units`).
        fold = self.spec.get("fold_task")
        folds = [fold] if fold is not None else []
        units = [folds] + groups if folds else groups
        wsh = len(folds)   # group k of `units` is warp role k - wsh
        if sorted(t for g in units for t in g) != list(range(len(self.tasks))):
            raise ValueError("warp_groups (and fold_task) must partition the task list")
        solver = int(self.spec.get("solver_warp", 0))
        # mirrored task pairs (each alone in its warp role) share ONE evaluate body
        mirrors = {}   # role index -> (shared body id, side)
        shared = []    # bodies
        for pair in self.spec.get("mirror", []):
            ta, tb = pair
            ra = next(k for k, g in enumerate(groups) if g == [ta])
            rb = next(k for k, g in enumerate(groups) if g == [tb])
            mirrors[ra] = (len(shared), 0)
            mirrors[rb] = (len(shared), 1)
            shared.append(None)
        arrow = bool(self.spec.get("arrow_solve")) and len(groups) > 1
        if folds and not (arrow and self.tasks[fold]["kind"] == "frame"):
            raise ValueError("fold_task needs arrow_solve, two or more warp roles and a frame task")
        self.qmaps = None
        nql = self.nq
        if arrow and self.spec.get("local_q", True):
            # Role-local configuration registers: a role keeps only the coordinates its evaluate reads (and its step_role
            # writes) -- the joints common to all roles first (same registers in every role), then its own chains; mirrored
            # roles keep corresponding joints in the same registers, so their shared body needs no select.  (With one
            # T q[NQ] for all roles every coordinate is live in every warp: 2 NQ registers in FP64.)
            chains = [sorted(set(j for t in g + folds for j in self.tasks[t]["chain"])) for g in groups]
            common = sorted(set.intersection(*[set(ch) for ch in chains]))
            if folds and not set(self.tasks[fold]["chain"]) <= set(common):
                raise ValueError("fold_task: its chain must be common to all warp roles")
            covered = set(j for ch in chains for j in ch)
            loose = [j for j, jt in enumerate(self.joints) if jt["type"] != J_UNIVERSE and j not in covered]
            self.qmaps = []
            for k, ch in enumerate(chains):
                mp = {}
                for j in common + [j for j in ch if j not in common] + (loose if k == solver else []):
                    for iq in self.joint_cols([j])[1]:
                        mp[iq] = len(mp)
                self.qmaps.append(mp)
            nql = max(len(mp) for mp in self.qmaps)
        fold_ev = None
        if folds:
            # first, so that its (never stored) Jacobian entries take the first slots and every warp role's slots follow
            self.qmap = self.qmaps[0] if self.qmaps else None   # (its coordinates sit in the same registers in every role)
            self.jreg, self.ereg = {}, {}
            Ef = Emitter(prefix="f")
            self.gen_task(Ef, fold, {})
            fold_ev = Ef.lines
            self.fold_regs = (self.jreg, self.ereg)
            self.jreg = self.ereg = None
        evs = []
        for k, g in enumerate(groups):
            self.qmap = self.qmaps[k] if self.qmaps else None
            if k in mirrors:
                bid, side = mirrors[k]
                if side == 0:
                    pair = self.spec["mirror"][bid]
                    rb = next(r for r, v in mirrors.items() if v == (bid, 1))
                    self.qmap_b = self.qmaps[rb] if self.qmaps else None
                    shared[bid] = self.gen_evaluate_mirrored(pair[0], pair[1])
                evs.append(None)
            else:
                evs.append(self.gen_evaluate(g))
        self.qmap = None
        dq = self.gen_dq()
        integ = self.gen_integrate()
        rows, nslot = self.rows, len(self.slots)
        # presolve: the solver role factorises the leading block of its own task rows before the first barrier
        P = 0
        self.order = list(range(rows))
        self.pos = list(range(rows))
        if self.spec.get("presolve") and len(groups) > 1 and not self.spec.get("parallel_solve"):
            own_rows = [self.tasks[t]["row"] + i for t in sorted(groups[solver]) for i in range(self.tasks[t]["dim"])]
            P = len(own_rows)
            # the solver role's rows are eliminated first (a symmetric permutation of the normal equations)
            self.order = own_rows + [r for r in range(rows) if r not in own_rows]
            self.pos = [self.order.index(r) for r in range(rows)]
        nstrict = rows * (rows - 1) // 2
        self.eoff = P * (P - 1) // 2 if P else 0          # e lives where rows >= P of L will go (written after e was read)
        self.yoff = self.eoff + rows                        # yp[0..P) of presolve
        if P and self.yoff + P > nstrict:
            raise ValueError("presolve: the factor strip cannot hold e and yp beside the leading block")
        presolve = self.gen_presolve(P) if P else []
        solve = self.gen_solve(int(self.spec.get("block_width", 4)), P)
        used = self.signature()
        nfact = max(rows * (rows + 1) // 2, rows + self.nq)  # the factor strip also carries e (M) and the stepped q (NQ)
        uniform = bool(self.spec.get("uniform_solve")) and bool(self.spec.get("parallel_solve")) and len(groups) > 1
        if arrow:
            uniform = False
            if folds:
                self.jreg, self.ereg = self.fold_regs
            arrow_code = self.gen_solve_arrow(units, solver + wsh, 0 if folds else None)
            self.jreg = self.ereg = None
            nfact = max(self.arrow["nfact"], rows + self.nq)   # layout: see gen_solve_arrow
            self.eoff = 0
        if uniform:
            nfact = nstrict + 3 * rows                        # L | d | rhs (e, then yp) | Gram diagonal (gen_solve_uniform)
            self.eoff = nstrict + rows
        elif self.spec.get("rolled_update") and self.spec.get("parallel_solve") and len(groups) > 1:
            nfact += rows                                     # ... and yp for the rolled left-looking loops (gen_solve_parallel)
        out = []
        out.append("// GENERATED by tools/gen_kernel.py -- do not edit.  Specialisation: %s" % display_name)
        out.append("// rows=%d nv=%d nq=%d non-zero Jacobian entries=%d solve FMAs=%d warp roles=%d" %
                   (rows, self.nv, self.nq, nslot, self.solve_fma, len(groups)))
        out.append("#pragma once")
        out.append('#include "../se3_math.cuh"')
        out.append('#include "../spec_common.hpp"')
        out.append("namespace ikb {")
        out.append("struct %s {" % struct_name)
        out.append("    static constexpr int NQ = %d, NV = %d, M = %d, M0 = %d, TSZ = %d, NSLOT = %d, NFACT = %d;" %
                   (self.nq, self.nv, rows, self.rows_p0, self.tsz, nslot, nfact))
        out.append("    // NQL: configuration registers per thread (arrow specs: a role keeps only the coordinates it reads and steps)")
        out.append("    static constexpr int NQL = %d;" % nql)
        out.append("    // MY: entries of y a role keeps between psolve() and step_role() (arrow specs with the factor in registers: its own rows)")
        out.append("    static constexpr int MY = %d;" % (self.arrow["my"] if arrow and self.arrow["y_regs"] else rows))
        out.append("    // warp roles: the tasks are split over NWARPS warps that evaluate concurrently; role SOLVER solves")
        out.append("    static constexpr int NWARPS = %d, SOLVER = %d;" % (len(groups), solver))
        out.append("    // PSOLVE: distribute the factorisation over the roles (pays off for large M; for M = 12 the ~7 extra group")
        out.append("    // barriers cost more than the shorter critical path saves -- measured, DESIGN.md 4.1)")
        out.append("    static constexpr bool PSOLVE = %s;" % ("true" if (self.spec.get("parallel_solve") or arrow) and len(groups) > 1 else "false"))
        out.append("    // DSTEP: after psolve() y sits in the strip and every role steps its own coordinates (step_role / store_q)")
        out.append("    static constexpr bool DSTEP = %s;" % ("true" if (uniform or arrow) else "false"))
        out.append("    // ARROW: psolve() is the bordered-block-diagonal step (gen_solve_arrow); the serial solve() is not laid out for its strip")
        out.append("    static constexpr bool ARROW = %s;" % ("true" if arrow else "false"))
        # Jacobian slots per role (every slot belongs to the role that evaluates its row; a role's slots are consecutive)
        row_role_ = {self.tasks[t]["row"] + i: k for k, g in enumerate(groups) for t in g for i in range(self.tasks[t]["dim"])}
        # (the fold task's entries are never stored: they belong to no role's slots)
        jslots = [sorted(sl for (r, c_), sl in self.slots.items() if row_role_.get(r) == k) for k in range(len(groups))]
        contiguous = all(js == list(range(js[0], js[0] + len(js))) for js in jslots if js)
        tmemj = bool(arrow and self.spec.get("tmem_j") and contiguous)
        out.append("    // TMEMJ: every role reads and writes only its own rows of J, and this spec asks the FP64 kernel to keep them in")
        out.append("    // tensor memory (tmem_scratch.cuh, TStrip) instead of shared memory; j_first / j_count: a role's slots")
        out.append("    static constexpr bool TMEMJ = %s;" % ("true" if tmemj else "false"))
        out.append("    static constexpr int j_first(int role) { return %s; }" %
                   " : ".join(["role == %d ? %d" % (k, js[0] if js else 0) for k, js in enumerate(jslots)] + ["0"]))
        out.append("    static constexpr int j_count(int role) { return %s; }" %
                   " : ".join(["role == %d ? %d" % (k, len(js)) for k, js in enumerate(jslots)] + ["0"]))
        # QSTAGE: NQ consecutive Jacobian slots that are dead, for a problem that has CONVERGED, from the barrier inside psolve()
        # to the next evaluate -- the rows of a role that publishes its contributions in the factor strip (not in its own
        # Jacobian slots) and reads its rows afterwards only to step.  The kernel stages the configuration of the slot's NEXT
        # problem there one trip ahead (dls_spec.cuh, kPrefetch); -1: no such run of slots.
        qstage = -1
        if arrow and contiguous and not tmemj and not self.spec.get("arrow_cap_solo"):
            for k, js in enumerate(jslots):
                if k != solver and self.arrow["pub"][k][0] == "L" and len(js) >= self.nq:
                    qstage = js[0]
                    break
        out.append("    // QSTAGE: first of NQ Jacobian slots where the kernel may stage the next problem's configuration (-1: none)")
        out.append("    static constexpr int QSTAGE = %d;" % qstage)
        out.append("    // CAPSOLO: psolve() ends behind a barrier of its own (the shared-column system is solved by the SOLVER role alone)")
        out.append("    static constexpr bool CAPSOLO = %s;" % ("true" if arrow and self.spec.get("arrow_cap_solo") else "false"))
        out.append("    // PRE: leading rows whose P x P factor block the SOLVER role computes in presolve(), before the first barrier;")
        out.append("    // EOFF: slot of the factor strip where e starts (rows >= PRE of L, written only after e has been read)")
        out.append("    static constexpr int PRE = %d, EOFF = %d;" % (P, self.eoff))
        out.append('    static const char *name() { return "%s"; }' % display_name)
        for k, (g, ev) in enumerate(zip(groups, evs)):
            names = ", ".join("%s %s" % (self.tasks[t]["name"], ("align-" + "xyz"[self.tasks[t]["ktype"]]) if self.tasks[t]["kind"] == "align"
                                         else "" if self.tasks[t]["kind"] == "posture"
                                         else ["Position", "Orientation", "Full"][self.tasks[t]["ktype"]]) for t in g)
            out.append("    // ---- role %d: %s ----" % (k, names))
            out.append("    // copy this role's target poses into the strip sT")
            out.append("    template <typename T, typename S>")
            out.append("    static IKB_HD void load_targets_w%d(const T *tg, long long es, const S &sT) {" % k)
            spans = [(self.tasks[t]["toff"], self.tasks[t]["toff"] + self.tasks[t]["tsize"]) for t in g]
            for t in folds:   # the fold task's target: its own share (every role reads all of it behind the barrier at the top of a trip)
                t0, n = self.tasks[t]["toff"], self.tasks[t]["tsize"]
                spans.append((t0 + k * n // len(groups), t0 + (k + 1) * n // len(groups)))
            for a_, b_ in spans:
                out.append("#pragma unroll")
                out.append("        for (int k = %d; k < %d; ++k) sT.copy_in(k, tg + k * es);  // asynchronous: strip_copies_wait() before evaluate" % (a_, b_))
            out.append("    }")
            if ev is None:
                continue
            out.append("    // FK + task errors (-> sE) + weighted task Jacobian non-zeros (-> sJ)")
            out.append("    template <typename T, typename S>")
            out.append("    static IKB_HD void evaluate_w%d(const T (&q)[NQL], const S &tg, const SpecConsts<T, NQ, M> &c, const S &sJ, const S &sE) {" % k)
            out.extend(ev)
            out.append("    }")
        if folds:
            out.append("    // ---- fold task %d (%s): every role evaluates it in registers; role k stores its share of the rows / contributions ----" %
                       (fold, self.tasks[fold]["name"]))
            out.append("    template <typename T, typename S>")
            out.append("    static IKB_HD void evaluate_f(const int role, const T (&q)[NQL], const S &tg, const SpecConsts<T, NQ, M> &c, const S &sE) {")
            out.extend(fold_ev)
            for k, code in enumerate(self.fold_pub[0]):
                out.append("        if (role == %d) {" % k)
                out.extend("            " + ln for ln in code)
                out.append("        }")
            out.append("    }")
        for bid, body in enumerate(shared):
            out.append("    // ---- shared by the roles of the mirrored tasks %s (side = 0 / 1) ----" % (self.spec["mirror"][bid],))
            out.append("    template <typename T, typename S>")
            out.append("    static IKB_HD void evaluate_m%d(const int side, const T (&q)[NQL], const S &tg, const SpecConsts<T, NQ, M> &c, const S &sJ, const S &sE) {" % bid)
            out.extend(body)
            out.append("    }")
        out.append("    // role dispatch (warp-uniform)")
        out.append("    template <typename T, typename S>")
        out.append("    static IKB_HD void load_targets(int role, const T *tg, long long es, const S &sT) {")
        for k in range(len(groups)):
            out.append("        if (role == %d) load_targets_w%d(tg, es, sT);" % (k, k))
        out.append("    }")
        out.append("    template <typename T, typename S>")
        out.append("    static IKB_HD void evaluate(int role, const T (&q)[NQL], const S &tg, const SpecConsts<T, NQ, M> &c, const S &sJ, const S &sE) {")
        if folds:
            out.append("        evaluate_f(role, q, tg, c, sE);")
        for k in range(len(groups)):
            if k not in mirrors:
                out.append("        if (role == %d) evaluate_w%d(q, tg, c, sJ, sE);" % (k, k))
        for bid in range(len(shared)):
            ra, rb = [k for k, v in sorted(mirrors.items()) if v[0] == bid]
            out.append("        if (role == %d || role == %d) evaluate_m%d(role == %d ? 1 : 0, q, tg, c, sJ, sE);  // one copy of the code for both" % (ra, rb, bid, rb))
        out.append("    }")
        out.append("    // leading PRE x PRE block of the factorisation (solver role, right after its own evaluate)")
        out.append("    template <typename T, typename S>")
        out.append("    static IKB_HD void presolve(const S &sJ, const S &sL, const S &sE, T damping2) {")
        out.extend(presolve)
        out.append("    }")
        out.append("    // y = (J J^T + damping^2 I)^-1 e: fused Gram + blocked LDL^T (factor -> strip sL) + substitutions.")
        out.append("    // Reads e from sE (may alias the start of sL), returns ||e[0..M0)||^2 (the stop-test quantity, visitor.hpp:19).")
        if not arrow:   # (an arrow spec's strip has no room for the dense factor; its step is psolve())
            out.append("    template <typename T, typename S>")
            out.append("    static IKB_HD T solve(const S &sJ, const S &sL, const S &sE, T damping2, T (&y)[M]) {")
            out.extend(solve)
            out.append("    }")
        if uniform:
            grams, ubody = self.gen_solve_uniform(len(groups), solver)
            out.append("    // The same solve distributed over the warp roles with ONE factorisation body (see gen_solve_uniform).")
            out.append("    // FMAs: Gram per role %s, factorisation + back substitution %d" % self.usolve_fma)
            for k, code in enumerate(grams):
                out.append("    template <typename T, typename S>")
                out.append("    static IKB_HD void ugram_w%d(const S &sJ, const S &sL, T damping2) {" % k)
                out.extend(code)
                out.append("    }")
            out.append("    template <typename T, typename S, typename SYNC>")
            out.append("    static IKB_HD void psolve(int role, const S &sJ, const S &sL, const S &sE, T damping2, T (&y)[M], SYNC &sync) {")
            for k in range(len(groups)):
                out.append("        if (role == %d) ugram_w%d(sJ, sL, damping2);" % (k, k))
            out.append("        sync();  // the normal equations are in the strip")
            out.extend(ubody)
            out.append("    }")
        if arrow:
            locals_, cap, finishes = arrow_code
            A = self.arrow
            out.append("    // Bordered-block-diagonal step (see gen_solve_arrow): shared columns %s; FMAs per role %s" % (A["shared"], A["fma"]))
            out.append("    // strip sL: e [0, %d) | s [%d, %d) | published contributions %s | factors / y %s" %
                       (rows, A["soff"], A["soff"] + A["ks"], {k: v if v[0] == "L" else "own J slots" for k, v in A["pub"].items()}, A["facb"]))
            partner = {ra: rb for rb, (ra, _, _, _) in A["mirror_of"].items()}
            nu, su = len(units), solver + wsh   # (groups of the solve and the SOLVER role's group; role of group k: k - wsh)
            for k in range(nu):
                if k in A["mirror_of"] or k < wsh:
                    continue   # runs the body of its mirror partner / the fold task publishes from its evaluate
                if k in partner:
                    _, dJ, dR, dL = A["mirror_of"][partner[k]]
                    sig = "const int side, "
                    reb = ["        const S sJr{sJ.base + side * (%d * S::kStride)}, sEr{sE.base + side * (%d * S::kStride)}, sLr{sL.base + side * (%d * S::kStride)};"
                           % (dJ, dR, dL)]
                    nm = "m%d" % k
                else:
                    sig = ""
                    reb = ["        const S &sJr = sJ, &sEr = sE, &sLr = sL;"]
                    nm = "w%d" % k
                out.append("    template <typename T, typename S>")
                out.append("    static IKB_HD void arrow_local_%s(%sconst S &sJ, const S &sL, const S &sE, T damping2, T (&fac)[%d]) {" % (nm, sig, A["nfac"]))
                out.extend(reb)
                out.extend(locals_[k])
                out.append("    }")
                if finishes[k]:
                    out.append("    template <typename T, typename S>")
                    out.append("    static IKB_HD void arrow_finish_%s(%sconst S &sJ, const S &sL, const S &sE, const T (&s)[%d], const T (&fac)[%d], T (&y)[MY]) {" % (nm, sig, A["ks"], A["nfac"]))
                    out.extend(reb)
                    out.extend(finishes[k])
                    out.append("    }")

            def call(fn, k, args):
                if k in A["mirror_of"]:
                    return "%s_m%d(1, %s)" % (fn, A["mirror_of"][k][0], args)
                if k in partner:
                    return "%s_m%d(0, %s)" % (fn, k, args)
                return "%s_w%d(%s)" % (fn, k, args)

            out.append("    // phase 1 reads only the role's own rows of J and e: no barrier between evaluate() and psolve().  `hook` runs")
            out.append("    // right after the one barrier (all of e is visible and stays intact): the kernel's stop test and ticket prefetch.")
            out.append("    template <typename T, typename S, typename SYNC, typename HOOK>")
            out.append("    static IKB_HD void psolve(int role, const S &sJ, const S &sL, const S &sE, T damping2, T (&y)[MY], SYNC &sync, HOOK &hook) {")
            out.append("        T s[%d], fac[%d];" % (A["ks"], A["nfac"]))
            for k in range(nu):
                if k in A["mirror_of"] or k < wsh:
                    continue
                cond = "role == %d || role == %d" % (k - wsh, partner[k] - wsh) if k in partner else "role == %d" % (k - wsh)
                fn = "arrow_local_m%d(role == %d ? 1 : 0, sJ, sL, sE, damping2, fac)" % (k, partner[k] - wsh) if k in partner else "arrow_local_w%d(sJ, sL, sE, damping2, fac)" % k
                out.append("        if (%s) %s;" % (cond, fn))
            out.append("        sync();  // every role's contribution to the shared-column system is in the strip")
            out.append("        hook();")
            s_storer = None
            if self.spec.get("arrow_cap_solo"):
                if folds:
                    raise ValueError("fold_task: arrow_cap_solo is not supported")
                # the small system on the solver role alone (the others wait at a second barrier instead of repeating it)
                out.append("        if (role == %d) {" % solver)
                out.extend(cap)
                out.append("#pragma unroll")
                out.append("            for (int i = 0; i < %d; ++i) sL.set(%d + i, s[i]);" % (A["ks"], A["soff"]))
                out.append("        }")
                out.append("        sync();  // s, ||e||^2 and the next ticket are visible: the kernel needs no barrier behind psolve()")
                out.append("        if (role != %d) {" % solver)
                out.append("#pragma unroll")
                out.append("            for (int i = 0; i < %d; ++i) s[i] = sL.get(%d + i);" % (A["ks"], A["soff"]))
                out.append("        }")
            elif not finishes[su] and any(finishes[k] for k in range(nu) if k != su) and self.spec.get("arrow_solver_skips_cap", True):
                # The SOLVER role has no rows of its own to finish (no private columns): it needs s only for its step, which
                # reads it from the strip behind the next barrier.  It skips the shared-column system, so its time between the
                # two barriers belongs to the stop test, the ticket and the staged refill (dls_spec.cuh, kPrefetch) -- latency
                # that used to sit in front of 400 instructions the other roles were running too.
                s_storer = [k for k in range(nu) if k != su and finishes[k] and k not in A["mirror_of"]][0] - wsh
                out.append("        if (role != %d) {" % solver)
                out.extend("    " + ln for ln in cap)
                out.append("        }")
            else:
                out.extend(cap)
            out.append("        IKB_PHASE_FENCE();")
            for k in range(nu):
                if k in A["mirror_of"] or not finishes[k]:
                    continue
                cond = "role == %d || role == %d" % (k - wsh, partner[k] - wsh) if k in partner else "role == %d" % (k - wsh)
                fn = "arrow_finish_m%d(role == %d ? 1 : 0, sJ, sL, sE, s, fac, y)" % (k, partner[k] - wsh) if k in partner else "arrow_finish_w%d(sJ, sL, sE, s, fac, y)" % k
                out.append("        if (%s) %s;" % (cond, fn))
            if not self.spec.get("arrow_cap_solo"):
                out.append("        if (role == %d) {" % (s_storer if s_storer is not None else solver))
                out.append("#pragma unroll")
                out.append("            for (int i = 0; i < %d; ++i) sL.set(%d + i, s[i]);" % (A["ks"], A["soff"]))
                out.append("        }")
            out.append("        (void)y;")
            out.append("        (void)fac;")
            out.append("    }")
        psolve = [] if (uniform or arrow) else self.gen_solve_parallel(int(self.spec.get("parallel_block_width", self.spec.get("block_width", 4))), len(groups), solver)
        out.append("    // The same solve distributed over the warp roles (cyclic row ownership; see gen_solve_parallel): every role")
        out.append("    // calls psolve(role, ...) with a group barrier `sync`; y is produced in the SOLVER role's registers only.")
        if not (uniform or arrow):
            out.append("    // FMAs per role: %s" % self.psolve_fma)
        for k, code in enumerate(psolve):
            out.append("    template <typename T, typename S, typename SYNC>")
            out.append("    static IKB_HD void psolve_w%d(const S &sJ, const S &sL, const S &sE, T damping2, T (&y)[M], SYNC &sync) {" % k)
            out.extend(code)
            out.append("    }")
        if not (uniform or arrow):
            out.append("    template <typename T, typename S, typename SYNC>")
            out.append("    static IKB_HD void psolve(int role, const S &sJ, const S &sL, const S &sE, T damping2, T (&y)[M], SYNC &sync) {")
            for k in range(len(groups)):
                out.append("        if (role == %d) psolve_w%d(sJ, sL, sE, damping2, y, sync);" % (k, k))
            out.append("    }")
        out.append("    // dq = -J^T y from the strip (dls.cpp:52)")
        out.append("    template <typename T, typename S>")
        out.append("    static IKB_HD void step_direction(const S &sJ, const T (&y)[M], T (&dq)[NV]) {")
        out.extend(dq)
        out.append("    }")
        out.append("    // q <- clamp(integrate(q, step*dq))")
        out.append("    template <typename T>")
        out.append("    static IKB_HD void integrate(T (&q)[NQ], const T (&dq)[NV], T step, const SpecConsts<T, NQ, M> &c) {")
        out.extend(integ)
        out.append("    }")
        if uniform or arrow:
            C, roles, qsets = self.gen_step_roles_arrow([g + folds for g in groups], solver) if arrow else self.gen_step_roles(groups, solver)
            out.append("    // Distributed step (see gen_step_roles): y from the strip; common joints by every role, the others by their role.")
            out.append("    template <typename T, typename S>")
            yreg = arrow and self.arrow["y_regs"]
            out.append("    static IKB_HD void step_role(int role, const S &sJ, const S &sL, T (&q)[NQL], T step, const SpecConsts<T, NQ, M> &c%s) {" %
                       (", const T (&y)[MY]" if yreg else ""))
            out.append("        T dq[NV];" if yreg else "        T y[M], dq[NV];")
            if not arrow:
                out.append("        #pragma unroll")
                out.append("        for (int i = 0; i < M; ++i) y[i] = sL.get(%d + i);" % self.rhs_off)
            if arrow:
                out.append("        T s[%d];" % self.arrow["ks"])
                out.append("        #pragma unroll")
                out.append("        for (int i = 0; i < %d; ++i) s[i] = sL.get(%d + i);" % (self.arrow["ks"], self.arrow["soff"]))
            once = arrow and (self.arrow_qc is not None or self.arrow_mail is not None)
            if once:   # the common joints: the solver role alone, which publishes the stepped coordinates (fetch_common)
                out.append("        if (role == %d) {" % solver)
                out.extend(C)
                for i, iq in enumerate(self.arrow_common[0]):
                    src = "q[%d]" % (self.qmaps[solver][iq] if self.qmaps else iq)
                    if self.arrow_qc is not None:
                        out.append("            sL.set(%d, %s);" % (self.arrow_qc + i, src))
                    else:
                        for k in sorted(self.arrow_mail):
                            out.append("            sL.set(%d, %s);  // role %d's copy" % (self.arrow_mail[k][i], src, k))
                out.append("        }")
            else:
                out.extend(C)
            for k, code in enumerate(roles):
                out.append("        if (role == %d) {" % k)
                if arrow and not yreg:   # y of the role's own rows (phase 3 left it in the role's factor slots)
                    for t in sorted(groups[k]):
                        for i in range(self.tasks[t]["dim"]):
                            r = self.tasks[t]["row"] + i
                            if r in self.arrow_y:
                                out.append("            y[%d] = sL.get(%d);" % (r, self.arrow_y[r]))
                out.extend(code)
                out.append("        }")
            out.append("    }")
            out.append("    // the entries of q a role owns (its step_role keeps exactly these current), written to the result")
            out.append("    template <typename T>")
            out.append("    static IKB_HD void store_q(int role, const T (&q)[NQL], T *dst, long long es) {")
            for k, qs in enumerate(qsets):
                out.append("        if (role == %d) {" % k)
                for iq in sorted(qs):
                    out.append("            dst[%d * es] = q[%d];" % (iq, self.qmaps[k][iq] if self.qmaps else iq))
                out.append("        }")
            out.append("    }")
        out.append("    // QCOMMON: the coordinates common to all roles are stepped by the SOLVER role alone; after the barrier at the top of")
        out.append("    // the next trip the other roles copy them from the strip (fetch_common)")
        once = arrow and (self.arrow_qc is not None or self.arrow_mail is not None)
        out.append("    static constexpr bool QCOMMON = %s;" % ("true" if once else "false"))
        out.append("    template <typename T, typename S>")
        out.append("    static IKB_HD void fetch_common(int role, const S &sL, T (&q)[NQL]) {")
        if once and self.arrow_qc is not None:
            out.append("        if (role != %d) {" % solver)
            for i, iq in enumerate(self.arrow_common[0]):
                out.append("            q[%d] = sL.get(%d);" % (self.qmaps[0][iq] if self.qmaps else iq, self.arrow_qc + i))
            out.append("        }")
        elif once:
            for k in sorted(self.arrow_mail):
                out.append("        if (role == %d) {" % k)
                for i, iq in enumerate(self.arrow_common[0]):
                    out.append("            q[%d] = sL.get(%d);" % (self.qmaps[0][iq] if self.qmaps else iq, self.arrow_mail[k][i]))
                out.append("        }")
        out.append("    }")
        out.append("    // the configuration of a problem into a role's registers (arrow specs: only the coordinates the role keeps)")
        out.append("    template <typename T>")
        out.append("    static IKB_HD void load_q(int role, const T *src, long long es, T (&q)[NQL]) {")
        if self.qmaps:
            for k, mp in enumerate(self.qmaps):
                out.append("        if (role == %d) {" % k)
                for iq, l in sorted(mp.items()):
                    out.append("            q[%d] = src[%d * es];" % (l, iq))
                for l in range(len(mp), nql):
                    out.append("            q[%d] = T(0);" % l)
                out.append("        }")
        else:
            out.append("#pragma unroll")
            out.append("        for (int k = 0; k < NQ; ++k) q[k] = src[k * es];")
        out.append("    }")
        # signature data for matches()
        out.append("    // ---- signature (host): the tree and task list this code was generated for ----")
        out.append("    static constexpr int NJOINTS = %d, NTASKS = %d;" % (len(self.joints), len(self.tasks)))
        out.append("    static const int *sig_parent() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(j["parent"]) for j in self.joints))
        out.append("    static const int *sig_type() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(j["type"]) for j in self.joints))
        out.append("    static const int *sig_used() { static const int v[] = {%s, -1}; return v; }" % ", ".join(map(str, used)))
        pl = []
        for j in self.joints:
            pl.extend(j["placement"])
            pl.extend(j["axis"])
        out.append("    static const double *sig_placement() { static const double v[] = {%s}; return v; }" %
                   ", ".join(repr(float(x)) for x in pl))
        inv = sorted(self.slots.items(), key=lambda kv: kv[1])
        out.append("    // (row, col) of every strip slot, for tests that rebuild the dense task Jacobian")
        out.append("    static const int *slot_rc() { static const int v[] = {%s}; return v; }" %
                   ", ".join("%d, %d" % rc for rc, _ in inv))
        out.append("    static const int *sig_task_type() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(t["ktype"]) for t in self.tasks))
        out.append("    // task kind (0 frame, 1 align-axis, 2 posture; sig_task_type is the axis / the number of coordinates for those)")
        out.append("    static const int *sig_task_kind() { static const int v[] = {%s}; return v; }" %
                   ", ".join({"frame": "0", "align": "1", "posture": "2"}[t["kind"]] for t in self.tasks))
        out.append("    static const int *sig_task_ref_joint() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(t["ref"]["parent"]) for t in self.tasks))
        rpl = []
        for t in self.tasks:
            rpl.extend(t["ref"]["placement"])
        out.append("    static const double *sig_task_ref_placement() { static const double v[] = {%s}; return v; }" %
                   ", ".join(repr(float(x)) for x in rpl))
        out.append("    static const int *sig_task_priority() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(t["priority"]) for t in self.tasks))
        out.append("    static const int *sig_task_joint() { static const int v[] = {%s}; return v; }" %
                   ", ".join(str(t["frame"]["parent"]) for t in self.tasks))
        fpl = []
        for t in self.tasks:
            fpl.extend(t["frame"]["placement"])
        out.append("    static const double *sig_task_placement() { static const double v[] = {%s}; return v; }" %
                   ", ".join(repr(float(x)) for x in fpl))
        out.append("};")
        out.append("}  // namespace ikb")
        # The Jacobian strip has a type of its own (SJ): the kernel may keep it in tensor memory (TStrip, tmem_scratch.cuh)
        # while the other strips are shared memory.  Every function that takes sJ gets the extra template parameter.
        import re
        for i, ln in enumerate(out):
            if "const S &sJ" in ln and "static IKB_HD" in ln:
                out[i] = ln.replace("const S &sJ", "const SJ &sJ")
                j = i - 1
                while not out[j].lstrip().startswith("template <"):
                    j -= 1
                if "typename SJ" not in out[j]:
                    if "const S &" not in out[i] and " S " not in out[i]:   # sJ was the only strip: S is no longer deducible
                        out[j] = out[j].replace("typename S>", "typename SJ>").replace("typename S,", "typename SJ,", 1)
                    else:
                        out[j] = (out[j].replace("typename S>", "typename S, typename SJ>") if "typename S>" in out[j]
                                  else out[j].replace("typename S,", "typename S, typename SJ,", 1))
            ln = out[i]
            ln = re.sub(r"const S sJm\{sJ\.base \+ side \* \((\d+) \* S::kStride\)\}", r"const SJ sJm{sJ.base + side * (\1 * SJ::kStride)}", ln)
            ln = re.sub(r"const S sJr\{sJ\.base \+ side \* \((-?\d+) \* S::kStride\)\}, ", r"const SJ sJr{sJ.base + side * (\1 * SJ::kStride)}; const S ", ln)
            ln = ln.replace("const S &sJr = sJ, &sEr = sE, &sLr = sL;", "const SJ &sJr = sJ; const S &sEr = sE, &sLr = sL;")
            ln = re.sub(r"const S sC(\d+)\{sJ\.base \+ k \* (\d+) \* S::kStride\}", r"const SJ sC\1{sJ.base + k * \2 * SJ::kStride}", ln)
            out[i] = ln
        return "\n".join(out) + "\n"


def main():
    model = json.load(open(sys.argv[1]))
    spec = json.load(open(sys.argv[2]))
    g = Generator(model, spec)
    text = g.emit(spec["struct"], spec["name"])
    with open(sys.argv[3], "w") as f:
        f.write(text)
    print("gen_kernel: %s -> %s (%d rows, %d Jacobian slots, %d lines)" % (spec["name"], sys.argv[3], g.rows, len(g.slots),
                                                                           text.count("\n")))


if __name__ == "__main__":
    main()

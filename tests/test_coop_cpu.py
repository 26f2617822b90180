"""The table-driven team-per-problem kernel (ik_b200/csrc/dls_coop.cuh) on the CPU: tests/cpu_harness/coop_harness.cpp
runs the kernel's own __host__ __device__ source with the lanes of a team as fibers, on a problem blob filled by the
product's host code, and this file compares it with the oracle -- first evaluation (e, J), flags, iteration counts, q --
for every task kind, both broadcast variants (warp shuffle / shared memory), ik::dls with FrameConstraints and ik::pik.
Test scaffolding only: nothing here is linked into libikb200.so and the product has no CPU path."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ik_b200 as ik
from ik_b200 import workloads as W
from oracle import oracle as O
from tests import pik_cases as PC
from tests.common import make_workload, oracle_model, oracle_problem_like, urdf_text

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def _pd(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def _pi(a):
    return a.ctypes.data_as(_ip)


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(ROOT, "build", "cpu_harness")
    os.makedirs(out, exist_ok=True)
    src = os.path.join(ROOT, "tests", "cpu_harness", "coop_harness.cpp")
    so = os.path.join(out, "libcoop_harness.so")
    deps = [src] + [os.path.join(ROOT, "ik_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "ik_b200", "csrc"))
                    if f.endswith((".cuh", ".hpp", ".cpp"))]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-ffp-contract=off", "-o", so, src])
    return C.CDLL(so)


def coop_solve(lib, pb, urdf, free_flyer, q0, tg, prm=None, f32=False, shfl=True, pik_lambdas=None):
    """Run the batch through the harness.  prm: O.params(...).  Returns q, ok, iters, resid, e_first, J_first, size class."""
    m = pb.model()
    prm = prm or O.params()
    kinds, frames, refs, types, prios, wts, masks = [], [], [], [], [], [], []
    for _, t, prio in pb._tasks:
        if isinstance(t, ik.FrameTask):
            kinds.append(0); frames.append(m.getFrameId(t.frame)); refs.append(m.getFrameId(t.reference_frame)); types.append(int(t.type))
        elif isinstance(t, ik.AlignAxisTask):
            kinds.append(1); frames.append(m.getFrameId(t.frame)); refs.append(m.getFrameId(t.reference_frame)); types.append(int(t.axis))
        elif isinstance(t, ik.CentreOfMassTask):
            kinds.append(3); frames.append(0); refs.append(m.getFrameId(t.reference_frame)); types.append(0)
        else:
            kinds.append(2); frames.append(0); refs.append(0); types.append(t.nj)
            masks.append(np.asarray(t.mask, dtype=np.float64))
        prios.append(prio)
        wts.append(np.asarray(t.weighting(), dtype=np.float64))
    cons = pb.get_all_constraints()
    cf = np.array([m.getFrameId(c.frame) for c in cons] + [0], dtype=np.int32)
    cr = np.array([m.getFrameId(c.reference_frame) for c in cons] + [0], dtype=np.int32)
    ct = np.array([int(c.type) for c in cons] + [0], dtype=np.int32)
    ai = lambda x: np.array(x, dtype=np.int32)
    kinds, frames, refs, types, prios = map(ai, (kinds, frames, refs, types, prios))
    wts = np.ascontiguousarray(np.concatenate(wts))
    masks = np.ascontiguousarray(np.concatenate(masks + [np.zeros(1)]))
    q0 = np.ascontiguousarray(q0, dtype=np.float64)
    tg = np.ascontiguousarray(tg, dtype=np.float64)
    B = q0.shape[0]
    rows = sum(int(t.dimension()) for _, t, _ in pb._tasks)
    q = np.zeros((B, m.nq))
    ok, it = np.zeros(B, dtype=np.int32), np.zeros(B, dtype=np.int32)
    res, e0, J0 = np.zeros(B), np.zeros(rows), np.zeros((rows, m.nv))
    lam = np.ones(8)
    if pik_lambdas is not None:
        lam[:len(pik_lambdas)] = pik_lambdas
    lo, hi = np.ascontiguousarray(m.lowerPositionLimit), np.ascontiguousarray(m.upperPositionLimit)
    cls = C.c_int(-1)
    xml = urdf_text(urdf).encode()
    rc = lib.coop_solve(xml, C.c_int(1 if free_flyer else 0), C.c_int(pb.max_priority_level()), C.c_int(len(kinds)), _pi(kinds),
                        _pi(frames), _pi(refs), _pi(types), _pi(prios), _pd(wts), _pd(masks), C.c_int(len(cons)), _pi(cf), _pi(cr),
                        _pi(ct), _pd(lo), _pd(hi), C.c_int(1 if f32 else 0), C.c_int(1 if shfl else 0),
                        C.c_int(0 if pik_lambdas is None else 1), _pd(lam), C.c_int(prm.max_iterations), C.c_double(prm.step_length),
                        C.c_double(prm.damping), C.c_double(prm.tolerance), C.c_int(B), _pd(q0), _pd(tg), _pd(q), _pi(ok), _pi(it),
                        _pd(res), _pd(e0), _pd(J0), C.byref(cls))
    assert rc == 0
    return q, ok.astype(bool), it, res, e0, J0, cls.value


def _check(lib, pb, urdf, ff, q0, tg, prm=None, oprm=None, shfl=True, qtol=1e-8, converged_only=False, cls=None):
    om = oracle_model(urdf, free_flyer=ff)
    om.flat["lower"][:] = pb.model().lowerPositionLimit
    om.flat["upper"][:] = pb.model().upperPositionLimit
    om = O.Model(om.flat)
    opb = oracle_problem_like(pb, om)
    q_ref, ok_ref, it_ref, res_ref = O.dls_batch(opb, q0, tg, oprm or O.params())
    q, ok, it, res, e0, J0, c = coop_solve(lib, pb, urdf, ff, q0, tg, oprm, shfl=shfl)
    if cls is not None:
        assert c == cls
    e_ref, J_ref = opb.evaluate(q0[0], tg[0])[:2]
    assert np.abs(e0 - e_ref).max() < 1e-12
    assert np.abs(J0 - np.asarray(J_ref).reshape(J0.shape)).max() < 1e-11
    assert (ok == ok_ref).all() and (it == it_ref).all()
    sel = ok if converged_only else np.ones_like(ok)
    assert np.abs(q - q_ref)[sel].max() < qtol
    assert np.abs(res - res_ref)[ok].max(initial=0) < 1e-10
    return q, ok, it


@pytest.mark.parametrize("shfl", [True, False])
@pytest.mark.parametrize("params", ["defaults", "demo"])
def test_cassie_feet_pelvis(lib, shfl, params):
    pb = W.cassie_feet_pelvis_problem()
    om = oracle_model("cassie")
    q0, tg, _ = make_workload(pb, om, 24 if params == "defaults" else 6, standing=W.CASSIE_STANDING)
    oprm = O.params() if params == "defaults" else O.params(200, 0.1, 0.1)
    _check(lib, pb, "cassie", True, q0, tg, oprm=oprm, shfl=shfl, cls=1)


def test_cassie_demo_tasks_moving_reference_and_align_axis(lib):
    pb = W.cassie_demo_problem()
    om = oracle_model("cassie")
    q0, tg, _ = make_workload(pb, om, 16, seed=31, standing=W.CASSIE_STANDING)
    _check(lib, pb, "cassie", True, q0, tg, qtol=1e-7, converged_only=True, cls=1)


def test_cassie_demo_with_posture_on_level_1(lib):
    pb = W.cassie_demo_posture_problem()
    om = oracle_model("cassie")
    q0, tg, _ = make_workload(pb, om, 8, seed=57, standing=W.CASSIE_STANDING)
    _check(lib, pb, "cassie", True, q0, tg, converged_only=True, cls=3)   # 26 rows on the Cassie tree: the 30-row class with the small-tree scratch, a warp per problem


@pytest.mark.parametrize("shfl", [True, False])
def test_humanoid(lib, shfl):
    pb = W.humanoid_problem()
    om = oracle_model("humanoid")
    q0, tg, _ = make_workload(pb, om, 4 if shfl else 8, seed=5, start="near")
    _check(lib, pb, "humanoid", True, q0, tg, shfl=shfl, cls=2)


def test_manipulator_and_ur5(lib):
    pb = W.manipulator_problem()
    om = oracle_model("manipulator", free_flyer=False)
    q0, tg, _ = make_workload(pb, om, 24, seed=11, start="near")
    _check(lib, pb, "manipulator", False, q0, tg, cls=0)
    m = ik.Model.builtin("ur5", free_flyer=False)
    pb = ik.InverseKinematicsProblem(m, 1)
    t_ori = ik.FrameTask(m, "ee_link", ik.KinematicType.Orientation)
    t_pos = ik.FrameTask(m, "tool0", ik.KinematicType.Position)
    t_pos.weighting()[:] = [1.0, 0.5, 2.0]
    pb.add_frame_task("ori", t_ori, 1)
    pb.add_frame_task("pos", t_pos, 0)
    m.set_limits(np.maximum(m.lowerPositionLimit, -3.0), np.minimum(m.upperPositionLimit, 3.0))
    om = oracle_model("ur5", free_flyer=False)
    om.flat["lower"][:] = m.lowerPositionLimit
    om.flat["upper"][:] = m.upperPositionLimit
    om = O.Model(om.flat)
    q0, tg, _ = make_workload(pb, om, 24, seed=21, start="near")
    _check(lib, pb, "ur5", False, q0, tg, converged_only=True, cls=0)


def test_f32_build_is_close(lib):
    pb = W.cassie_feet_pelvis_problem()
    om = oracle_model("cassie")
    opb = oracle_problem_like(pb, om)
    q0, tg, _ = make_workload(pb, om, 32, standing=W.CASSIE_STANDING)
    q_ref, ok_ref, it_ref, _ = O.dls_batch(opb, q0, tg)
    q, ok, it, res, _, _, _ = coop_solve(lib, pb, "cassie", True, q0, tg, f32=True)
    same = (it == it_ref) & ok & ok_ref
    assert same.mean() > 0.9 and np.percentile(np.abs(q - q_ref)[same].max(axis=1), 90) < 1e-4


@pytest.mark.parametrize("ref", ["universe", "pelvis"])
@pytest.mark.parametrize("ktype", ["Full", "Position"])
def test_frame_constraint_projection(lib, ktype, ref):
    """dq <- (I - Jc^+ Jc) dq (dls.cpp:26-34,44-52) with the cooperative rank-revealing QR (lane <-> column)."""
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Full))
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position))
    pb.add_frame_constraint("fr", ik.FrameConstraint(m, "RightFootFront", getattr(ik.KinematicType, ktype), ref))
    om = oracle_model("cassie")
    B = 8
    q0, tg, _ = make_workload(pb, om, B, seed=91, standing=W.CASSIE_STANDING)
    s0 = W.standing_configuration(m, W.CASSIE_STANDING)
    lf = om.frame_placement(s0, om.frame_id("LeftFootFront"))[9:]
    rng = np.random.default_rng(3)
    tg[:, :9] = np.eye(3).reshape(-1)
    tg[:, 9:12] = rng.uniform(-0.03, 0.03, (B, 3))
    tg[:, 21:24] = lf + rng.uniform(-0.05, 0.05, (B, 3))
    _check(lib, pb, "cassie", True, q0, tg, oprm=O.params(max_iterations=60, step_length=0.5), qtol=1e-7)


def test_centre_of_mass_task(lib):
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position))
    com = pb.add_centre_of_mass_task(ik.CentreOfMassTask(m, "universe"))
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position))
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Orientation))
    com.weighting()[:] = [2.0, 2.0, 0.5]
    om = oracle_model("cassie")
    B = 10
    q0, tg, qstar = make_workload(pb, om, B, seed=17, standing=W.CASSIE_STANDING)
    off = pb.target_offset(com)
    for b in range(B):
        tg[b, off:off + 3] = om.center_of_mass(qstar[b])[0]
    _check(lib, pb, "cassie", True, q0, tg, qtol=1e-7, converged_only=True)


@pytest.mark.parametrize("lambdas", [[1e-2, 1e-1], [1.0, 1.0]])
def test_pik_priority_recursion(lib, lambdas):
    """ik::pik (pik.cpp:31-96): demo task set on level 0, posture on level 1; the step of every level is one damped solve
    on the team's registers, the projector update one cooperative row-space basis."""
    pb = W.cassie_demo_posture_problem()
    om = oracle_model("cassie")
    opb = oracle_problem_like(pb, om)
    B = 6
    q0, tg, _ = make_workload(pb, om, B, seed=57, standing=W.CASSIE_STANDING)
    mi = 30
    q_ref, ok_ref, it_ref, res_ref = O.pik_batch(opb, q0, tg, O.pik_params(mi, 1.0, lambdas))
    q, ok, it, res, _, _, _ = coop_solve(lib, pb, "cassie", True, q0, tg, O.params(max_iterations=mi), pik_lambdas=lambdas)
    assert (ok == ok_ref).all() and (it == it_ref).all()
    assert np.abs(q - q_ref).max() < 1e-7 and np.abs(res - res_ref).max() < 1e-9


_PIK_LEVEL_CASES = {"three": (PC.cassie_three, 3), "seven": (PC.cassie_seven, 1), "empty_middle": (PC.cassie_gap, 1),
                    "rank_deficient_middle": (PC.cassie_rank_deficient, 3), "max_priority_20": (lambda: PC.cassie_three(20), 3),
                    "humanoid_three": (PC.humanoid_three, 2), "arm_empty_middle": (PC.arm_gap, 0)}


@pytest.mark.parametrize("lambdas", [[1e-2, 1e-1, 1.0], []])
@pytest.mark.parametrize("case", sorted(_PIK_LEVEL_CASES))
def test_pik_beyond_two_levels(lib, case, lambdas):
    """ik::pik with three to seven levels: the row-space bases of several levels stacked in the scratch and the projection
    of J_i over all of them (J_i P, P = I - sum w w^T), an empty level between two used ones, the rank-revealing basis of
    a rank-deficient middle level, max_priority_level 20 with tasks on levels 0-2 (the level table holds 7), and every
    size class of the kernel (TEAM = 8, 16, 32 on the Cassie and the 32-joint tree tables).  [] = default lambdas 1.0."""
    make, cls = _PIK_LEVEL_CASES[case]
    c = make()
    _, opb = c.oracle()
    B = 6
    mi, tol = c.stop(40)
    q0, tg = c.workload(B, seed=23)
    q_ref, ok_ref, it_ref, res_ref = O.pik_batch(opb, q0, tg, O.pik_params(mi, 1.0, lambdas, tol))
    q, ok, it, res, _, _, c_cls = coop_solve(lib, c.pb, c.urdf, c.free_flyer, q0, tg, O.params(max_iterations=mi, tolerance=tol),
                                             pik_lambdas=lambdas)
    assert c_cls == cls
    assert (ok == ok_ref).all() and (it == it_ref).all()
    assert np.abs(q - q_ref).max() < 1e-7 and np.abs(res - res_ref).max() < 1e-9


@pytest.mark.parametrize("case", ["three", "seven", "rank_deficient_middle"])
def test_pik_warp_neighbour_with_more_rounds_changes_nothing(lib, case):
    """Teams of 8 or 16 lanes share a warp, so the loops of the row-space basis and the projection run as many trips as
    the largest rank in the warp (coop_warp_rounds): a neighbour's level of higher rank, or a team without a problem, must
    not stall or change this team.  The harness plays such a neighbour (three more trips in every such loop); the results
    are bit for bit those of a lone team."""
    c = _PIK_LEVEL_CASES[case][0]()
    q0, tg = c.workload(4, seed=29)
    runs = []
    for extra in (0, 3):
        lib.coop_set_neighbour_extra(C.c_int(extra))
        try:
            runs.append(coop_solve(lib, c.pb, c.urdf, c.free_flyer, q0, tg, O.params(max_iterations=20), pik_lambdas=[1e-2, 1e-1, 1.0]))
        finally:
            lib.coop_set_neighbour_extra(C.c_int(0))
    assert all(np.array_equal(a, b) for a, b in zip(runs[0][:4], runs[1][:4]))

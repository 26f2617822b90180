"""URDF `continuous` joints (Pinocchio's RevoluteUnbounded: q = (cos, sin), one velocity coordinate) without a GPU: the two
flatteners, the C ABI's model and problem rules, the oracle from first principles, the oracle's continuous arm against the
same arm declared revolute, the table-driven kernel's own source (tests/cpu_harness/coop_harness.cpp) and a generated
plugin body against the oracle."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import ik_b200 as ik
from ik_b200 import _capi as capi
from ik_b200 import specialise as S
from ik_b200 import workloads as W
from oracle import oracle as O
from tests import continuous_cases as CC
from tests import continuous_oracle as CO
from tests import test_coop_cpu as TC
from tests.test_coop_cpu import lib  # noqa: F401  (fixture: the coop harness)
from tests.test_device_code_cpu import _spec_solve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_kernel as G  # noqa: E402

FLATTEN_CASES = {"arm": (CC.arm_urdf(), False), "arm_free_flyer": (CC.arm_urdf(), True), "ur5_unaligned": (CC.ur5_urdf(), False)}


@pytest.mark.parametrize("name", sorted(FLATTEN_CASES))
def test_flatteners_agree(name):
    xml, ff = FLATTEN_CASES[name]
    m, f = ik.Model.from_urdf(xml, ff), CO.flatten_urdf(xml, ff)
    assert m.nq == f["nq"] and m.nv == f["nv"] and m.nq > m.nv
    assert np.array_equal(m.jtypes, f["jtype"]) and np.array_equal(m.parents, f["parent"])
    assert np.array_equal(m.idx_qs, f["idx_q"]) and np.array_equal(m.idx_vs, f["idx_v"])
    assert np.array_equal(m.lowerPositionLimit, f["lower"]) and np.array_equal(m.upperPositionLimit, f["upper"])
    assert np.abs(m.jointPlacements - f["placement"]).max() <= 1e-15 and np.abs(m.axes - f["axis"]).max() <= 1e-15
    assert m.frame_names == f["frame_names"] and np.abs(m.framePlacements - f["frame_placement"]).max() <= 1e-15
    cont = [j for j in range(m.njoints) if m.jtypes[j] in W.J_CONTINUOUS]
    assert len(cont) == (6 if name.startswith("ur5") else 4)
    for j in cont:   # nq 2, limits +-1.01 whatever <limit> says
        iq = int(m.idx_qs[j])
        assert m.lowerPositionLimit[iq:iq + 2].tolist() == [-1.01, -1.01] and m.upperPositionLimit[iq:iq + 2].tolist() == [1.01, 1.01]
    if name.startswith("ur5"):
        assert [int(t) for t in m.jtypes[1:]] == [12, 11, 11, 11, 13, 11]
        assert np.allclose(m.axes[5], [0, 0.6, 0.8])
    nq = m.neutral()
    assert all(nq[int(m.idx_qs[j])] == 1.0 and nq[int(m.idx_qs[j]) + 1] == 0.0 for j in cont)
    assert np.array_equal(nq, CO.Model(f).neutral())


def _desc(m, jtype=None):
    i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
    keep = dict(parent=i32(m.parents), jtype=i32(m.jtypes if jtype is None else jtype), pl=np.ascontiguousarray(m.jointPlacements),
                ax=np.ascontiguousarray(m.axes), lo=m.lowerPositionLimit, hi=m.upperPositionLimit,
                fp=i32(m.frame_parents), fpl=np.ascontiguousarray(m.framePlacements))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    d = capi.ModelDesc(m.njoints, ip(keep["parent"]), ip(keep["jtype"]), dp(keep["pl"]), dp(keep["ax"]), dp(keep["lo"]), dp(keep["hi"]),
                       None, m.nframes, ip(keep["fp"]), dp(keep["fpl"]), None)
    return d, keep


def test_model_from_desc_round_trips_and_refuses_unknown_types():
    m = ik.Model.from_urdf(CC.ur5_urdf(), False)
    d, keep = _desc(m)
    h = C.c_void_p()
    capi.check(capi.lib.ikb_model_from_desc(C.byref(d), C.byref(h)), "ikb_model_from_desc")
    m2 = ik.Model(h)
    assert (m2.nq, m2.nv) == (m.nq, m.nv) == (12, 6)
    assert np.array_equal(m2.jtypes, m.jtypes) and np.array_equal(m2.idx_qs, m.idx_qs) and np.array_equal(m2.idx_vs, m.idx_vs)
    assert np.array_equal(m2.lowerPositionLimit, m.lowerPositionLimit) and np.array_equal(m2.neutral(), m.neutral())
    bad = m.jtypes.copy()
    bad[2] = 14
    d, keep = _desc(m, bad)
    assert capi.lib.ikb_model_from_desc(C.byref(d), C.byref(h)) == capi.ERR_INVALID_ARG


def test_planar_and_floating_joints_stay_refused():
    for kind in ("planar", "floating"):
        xml = CC.arm_urdf().replace('<joint name="arm2_joint" type="revolute">', '<joint name="arm2_joint" type="%s">' % kind)
        with pytest.raises(capi.IkbError, match="not supported"):
            ik.Model.from_urdf(xml, False)
        with pytest.raises(ValueError, match="unsupported joint type"):
            CO.flatten_urdf(xml, False)


def _posture_status(xml, nj):
    m = ik.Model.from_urdf(xml, False)
    p = C.c_void_p()
    capi.check(capi.lib.ikb_problem_create(m._h, 0, C.byref(p)), "ikb_problem_create")
    try:
        return capi.lib.ikb_problem_add_posture_task(p, nj, 0, None, None), capi.lib.ikb_last_error().decode()
    finally:
        capi.lib.ikb_problem_free(p)


def test_posture_task_over_a_continuous_tail_is_refused():
    rc, msg = _posture_status(CC.arm_urdf(), 1)   # arm7_joint is continuous
    assert rc == -4 and "continuous" in msg and "arm7_joint" in msg
    rc, _ = _posture_status(CC.derive_urdf("manipulator", ("arm1_joint", "arm3_joint"), widen=100.0), 4)   # tail: joints 4-7, revolute
    assert rc >= 0
    rc, msg = _posture_status(CC.derive_urdf("manipulator", ("arm1_joint", "arm3_joint"), widen=100.0), 5)
    assert rc == -4 and "arm3_joint" in msg


def _single_joint_model(kind, axis):
    xml = ('<robot name="one"><link name="a"/><link name="b"/><joint name="j" type="%s"><parent link="a"/><child link="b"/>'
           '<origin xyz="0.1 -0.2 0.3" rpy="0.3 -0.5 0.7"/><axis xyz="%s"/><limit lower="-10" upper="10"/></joint>'
           '<joint name="t" type="fixed"><parent link="b"/><child link="c"/><origin xyz="0.4 0.1 -0.2" rpy="0.1 0.2 0.3"/></joint>'
           '<link name="c"/></robot>') % (kind, axis)
    return CO.Model.from_urdf(xml, False)


@pytest.mark.parametrize("axis", ["1 0 0", "0 1 0", "0 0 1", "0.3 -0.4 0.5"])
def test_oracle_continuous_joint_from_first_principles(axis):
    cont, rev = _single_joint_model("continuous", axis), _single_joint_model("revolute", axis)
    assert cont.nq == 2 and cont.nv == 1 and cont.flat["jtype"][1] == rev.flat["jtype"][1] + 8
    f = cont.frame_id("c")
    rng = np.random.default_rng(5)
    for th in rng.uniform(-np.pi, np.pi, 20):
        qc = np.array([np.cos(th), np.sin(th)])
        assert np.abs(cont.frame_placement(qc, f) - rev.frame_placement(np.array([th]), f)).max() <= 1e-15   # FK, to 1e-15
        w = rng.uniform(-2, 2)
        q1 = cont.integrate(qc, np.array([w]))                                                               # SO(2) integrate
        assert abs(np.angle(np.exp(1j * (np.arctan2(q1[1], q1[0]) - th - w)))) < 1e-14
        assert abs(np.hypot(*q1) - 1) < 1e-15
        J = cont.frame_jacobian_local(qc, f)                                                                 # Jacobian vs FD along q (+) eps v
        eps = 1e-6
        Mp, Mm = (cont.frame_placement(cont.integrate(qc, np.array([s * eps])), f) for s in (1, -1))
        fd = (O.log6(O.se3_actinv(cont.frame_placement(qc, f), Mp)) - O.log6(O.se3_actinv(cont.frame_placement(qc, f), Mm))) / (2 * eps)
        assert np.abs(J[:, 0] - fd).max() < 1e-8
        assert np.abs(J - rev.frame_jacobian_local(np.array([th]), f)).max() < 1e-15
    # calc takes (c, s) as given: a pair off the unit circle is not renormalised
    qc = np.array([0.6, 0.6])
    R = cont.frame_placement(qc, cont.frame_id("b"))[:9].reshape(3, 3)
    assert abs(np.linalg.det(R) - 1) > 1e-2


def same_robot_solves(B=600, seed=3):
    """Oracle ik::dls on the widened all-revolute arm and on the continuous arm from corresponding starts."""
    cont, rev = CC.case_a(True), CC.case_a(False)
    q0c, tg, _ = cont.workload(B, seed)
    q0r = q0c[:, [0, 2, 3, 5, 6, 8, 9]].copy()   # arm1..7: continuous at q entries 0, 3, 6, 9 (cos), revolute 2, 5, 8
    for k, iq in enumerate((0, 3, 6, 9)):
        q0r[:, 2 * k] = np.arctan2(q0c[:, iq + 1], q0c[:, iq])
    q0c = CC.to_continuous(rev.model, cont.model, q0r)
    rr = CO.dls_batch(rev.opb, q0r, tg, nthreads=os.cpu_count() or 1)
    rc = CO.dls_batch(cont.opb, q0c, tg, nthreads=os.cpu_count() or 1)
    return cont, rev, rr, rc


def test_revolute_and_continuous_arm_are_the_same_robot():
    """The two declarations of the Gen3-like arm solve the same problems: equal flags and step counts apart from a small,
    pinned fraction (different rounding of a chaotic iteration), and equal joint angles on converged problems."""
    cont, rev, (qr, okr, itr, _), (qc, okc, itc, _) = same_robot_solves()
    agree = (okr == okc) & (itr == itc)
    print("revolute vs continuous arm: %d / %d problems differ in flags or step counts" % ((~agree).sum(), agree.size))
    assert agree.mean() >= 0.98
    ang = CC.angles(cont.model, qc)
    for k, j in enumerate((1, 3, 5, 7)):
        d = np.angle(np.exp(1j * (ang[:, j] - qr[:, 2 * (k)])))
        assert np.abs(d[agree & okr]).max() < 1e-9
    assert okr.mean() > 0.9


def _harness_check(lib, case, B, shfl, pik=False, qtol=1e-8, monkeypatch=None):  # noqa: F811
    monkeypatch.setattr(TC, "urdf_text", lambda xml: xml)   # the harness takes the URDF text itself
    q0, tg, _ = case.workload(B, seed=41)
    if pik:
        prm = O.params(max_iterations=40)
        q_ref, ok_ref, it_ref, res_ref = CO.pik_batch(case.opb, q0, tg, O.pik_params(40, 1.0, [1e-2, 1e-1]))
        q, ok, it, res, e0, J0, cls = TC.coop_solve(lib, case.pb, case.xml, case.free_flyer, q0, tg, prm, shfl=shfl,
                                                    pik_lambdas=[1e-2, 1e-1])
    else:
        q_ref, ok_ref, it_ref, res_ref = CO.dls_batch(case.opb, q0, tg)
        q, ok, it, res, e0, J0, cls = TC.coop_solve(lib, case.pb, case.xml, case.free_flyer, q0, tg, shfl=shfl)
    e_ref, J_ref = case.opb.evaluate(q0[0], tg[0])
    assert np.abs(e0 - e_ref).max() < 1e-12 and np.abs(J0 - J_ref).max() < 1e-11
    assert (ok == ok_ref).all() and (it == it_ref).all()
    sel = ok if pik else np.ones_like(ok)   # ik::pik: unconverged problems wander far on the widened revolute joints
    assert np.abs(q - q_ref)[sel].max() < qtol and np.abs(res - res_ref)[ok].max(initial=0) < 1e-10
    return cls


@pytest.mark.parametrize("shfl", [True, False])
@pytest.mark.parametrize("name,cls", [("a", 0), ("b", 1), ("c", 0), ("d", 0)])
def test_table_driven_kernel_on_the_cpu_harness(lib, monkeypatch, name, cls, shfl):  # noqa: F811
    """(a) Gen3-like arm, fixed base; (b) on a free-flyer; (c) all-continuous UR5 with an unaligned axis, weighted Position
    + Orientation on two levels; (d) the arm of (a) under ik::pik.  nq exceeds nv by 4 / 4 / 6 / 4 and every case keeps the
    size class its tree, nv and rows give (NQ = nv + 4 still holds q)."""
    case = CC.CASES[name]()
    assert _harness_check(lib, case, 16, shfl, pik=name == "d", monkeypatch=monkeypatch) == cls


def test_table_driven_kernel_f32_is_close(lib, monkeypatch):  # noqa: F811
    monkeypatch.setattr(TC, "urdf_text", lambda xml: xml)
    case = CC.case_a()
    q0, tg, _ = case.workload(32, seed=43)
    q_ref, ok_ref, it_ref, _ = CO.dls_batch(case.opb, q0, tg)
    q, ok, it, _, _, _, _ = TC.coop_solve(lib, case.pb, case.xml, False, q0, tg, f32=True)
    same = (it == it_ref) & ok & ok_ref
    assert same.mean() > 0.8 and np.percentile(np.abs(q - q_ref)[same].max(axis=1), 90) < 1e-4


@pytest.fixture(scope="module")
def plugin_lib():
    """tests/cpu_harness/spec_plugin_harness.cpp around the generated body of case (a)"""
    case = CC.case_a()
    mj, sj = S.model_json(case.model), S.spec_json(case.pb, "cont_arm")
    out = os.path.join(ROOT, "build", "cpu_harness")
    os.makedirs(out, exist_ok=True)
    header = os.path.join(out, "spec_cont_arm.cuh")
    with open(header, "w") as f:
        f.write(G.Generator(mj, sj).emit(sj["struct"], sj["name"]))
    so = os.path.join(out, "libspec_plugin_harness.so")
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-fPIC", "-shared", "-pthread", "-x", "c++", "-ffp-contract=off",
                           "-I" + os.path.join(ROOT, "ik_b200", "csrc", "gen"), '-DIKB_PLUGIN_HEADER="%s"' % header,
                           "-DIKB_PLUGIN_STRUCT=" + sj["struct"], "-o", so,
                           os.path.join(ROOT, "tests", "cpu_harness", "spec_plugin_harness.cpp")])
    return case, C.CDLL(so)


def test_generated_plugin_body_matches_oracle(plugin_lib):
    case, lib = plugin_lib
    q0, tg, _ = case.workload(64, seed=47)
    prm = O.params()
    q_ref, ok_ref, it_ref, res_ref = CO.dls_batch(case.opb, q0, tg, prm)
    q, ok, it, res, _ = _spec_solve(lib, "plugin", "f64", case.pb, q0, tg, prm)
    assert (ok == ok_ref).all() and (it == it_ref).all()
    assert np.abs(q - q_ref).max() < 1e-8 and np.abs(res - res_ref).max() < 1e-10


def test_generator_refuses_options_that_assume_one_scalar_per_joint():
    case = CC.case_a()
    mj = S.model_json(case.model)
    for opt in ({"mirror": [[0, 0]]}, {"fold_task": 0}, {"tmem_j": True}):
        with pytest.raises(ValueError, match="continuous"):
            G.Generator(mj, S.spec_json(case.pb, "x", **opt))


def test_workloads_of_continuous_joints():
    m = CC.case_c().model
    qs = W.sample_configurations(m, 64, seed=9)
    q0 = W.near_start(m, qs, seed=9)
    for j in range(1, m.njoints):
        iq = int(m.idx_qs[j])
        assert np.allclose(np.hypot(qs[:, iq], qs[:, iq + 1]), 1, atol=1e-15)
        d = np.angle(np.exp(1j * (np.arctan2(q0[:, iq + 1], q0[:, iq]) - np.arctan2(qs[:, iq + 1], qs[:, iq]))))
        assert np.abs(d).max() <= 0.3 + 1e-12 and np.abs(d).max() > 0.2


def test_continuous_oracle_is_the_base_oracle_on_other_joints():
    """tests/continuous_oracle.py derives its library from oracle/ik_oracle.c: on a robot without continuous joints it must
    compute exactly what the base library computes (flattening, evaluation, the whole ik::dls loop), bit for bit."""
    from oracle.bridge import oracle_model, oracle_problem_like, urdf_text
    pb = W.manipulator_problem()
    om = oracle_model("manipulator", free_flyer=False)
    cm = CO.Model.from_urdf(urdf_text("manipulator"), False)
    for k in ("jtype", "idx_q", "idx_v", "lower", "upper", "placement", "axis", "frame_placement"):
        assert np.array_equal(cm.flat[k], om.flat[k]), k
    q0, tg, _ = CC.Case(urdf_text("manipulator"), False, lambda m: [("tool", ik.FrameTask(m, "tool", ik.KinematicType.Full), 0)]).workload(64, 5)
    base = O.dls_batch(oracle_problem_like(pb, om), q0, tg)
    derived = CO.dls_batch(CO.problem_like(pb, cm), q0, tg)
    assert all(np.array_equal(a, b) for a, b in zip(base, derived))
    assert np.array_equal(O.dls_batch(oracle_problem_like(pb, om), q0, tg, fma=True)[0],
                          CO.dls_batch(CO.problem_like(pb, cm), q0, tg, fma=True)[0])

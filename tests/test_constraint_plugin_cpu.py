"""Generated straight-line code for problems with FrameConstraints, without a GPU: the body tools/gen_kernel.py emits for a
constraint list compiled with g++ (tests/cpu_harness/spec_constraint_harness.cpp) against the oracle -- one evaluation (e, J,
Jc, the projected step and the rank of Jc) and whole ik::dls solves in FP64 and FP32 -- the generator's refusals, and the
matching of a compiled plugin (in a child interpreter: a loaded plugin stays registered for the whole process)."""
import ctypes as C
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import ik_b200 as ik
from ik_b200 import specialise as S
from ik_b200 import workloads as W
from oracle import oracle as O
from oracle.bridge import oracle_frame_poses, urdf_text
from tests import continuous_cases as CC
from tests import continuous_oracle as CO
from tests.test_device_code_cpu import _spec_solve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_kernel as G  # noqa: E402

CASSIE_PRM = dict(max_iterations=60, step_length=0.5)   # as test_gpu_parity.test_frame_constraint_null_space_projection


class Case:
    """(URDF, free-flyer, problem) with its oracle problem and a workload whose targets the constraints leave reachable."""

    def __init__(self, xml, free_flyer, make, targets, prm=None):
        self.xml, self.free_flyer, self.prm = xml, free_flyer, prm or {}
        self.model = ik.Model.from_urdf(xml, free_flyer)
        self.pb = make(self.model)
        om = CO.Model.from_urdf(xml, free_flyer)
        om.flat["lower"][:] = self.model.lowerPositionLimit
        om.flat["upper"][:] = self.model.upperPositionLimit
        self.om = CO.Model(om.flat)
        self.opb = CO.problem_like(self.pb, self.om)
        self._targets = targets

    def workload(self, B, seed):
        return self._targets(self, B, seed)

    def constraint_jacobian(self, q):
        Jc = np.zeros((self.pb.c_size(), self.model.nv))
        CO.lib().iko_constraint_jacobian(C.byref(self.om.c), C.byref(self.opb.c), O._pd(O._d(q)), O._pd(Jc))
        return Jc


def _planted_targets(case, B, seed):
    """Standing start; pelvis at the identity moved by up to 3 cm, the left foot within 5 cm of where it stands (the draw of
    test_gpu_parity.test_frame_constraint_null_space_projection)."""
    s0 = W.standing_configuration(case.model, W.CASSIE_STANDING)
    q0 = np.tile(s0, (B, 1))
    lf = case.om.frame_placement(s0, case.om.frame_id("LeftFootFront"))[9:]
    rng = np.random.default_rng(seed)
    tg = np.zeros((B, case.pb.target_size))
    tg[:, :9] = np.eye(3).reshape(-1)
    tg[:, 9:12] = rng.uniform(-0.03, 0.03, (B, 3))
    tg[:, 12:21] = np.eye(3).reshape(-1)
    tg[:, 21:24] = lf + rng.uniform(-0.05, 0.05, (B, 3))
    return q0, tg


def _stance_targets(case, B, seed):
    s0 = W.standing_configuration(case.model, W.CASSIE_STANDING)
    return np.tile(s0, (B, 1)), W.cassie_stance_targets(case.pb, B, seed)


def _arm_targets(pinned):
    """Warm start near a sampled q*; the tool target comes from q0 with the joints past the first `pinned` moved to q*'s
    values, so that a solution keeps the constrained frame where it starts."""
    def make(case, B, seed):
        m = case.model
        qstar = W.sample_configurations(m, B, seed)
        q0 = W.near_start(m, qstar, seed)
        q1 = q0.copy()
        first = int(m.idx_qs[pinned + 1])
        q1[:, first:] = qstar[:, first:]
        poses = oracle_frame_poses(case.om, q1, W.task_frames(case.pb))
        return q0, W.targets_from_frame_poses(case.pb, poses, q1)
    return make


def _arm(frame, ktype, cframe, cktype):
    def make(m):
        pb = ik.InverseKinematicsProblem(m, 0)
        pb.add_frame_task("tool", ik.FrameTask(m, frame, ktype))
        pb.add_frame_constraint("c", ik.FrameConstraint(m, cframe, cktype))
        return pb
    return make


CASES = {
    # (a) pelvis Full + LeftFootFront Position tasks, RightFootFront Position constraint
    "cassie": lambda: Case(urdf_text("cassie"), True, W.cassie_constraint_problem, _planted_targets, CASSIE_PRM),
    # (b) the same with a Full constraint relative to the moving pelvis frame
    "cassie_pelvis": lambda: Case(urdf_text("cassie"), True, lambda m: W.cassie_constraint_problem(m, ik.KinematicType.Full, "pelvis"),
                                  _planted_targets, CASSIE_PRM),
    # (c) pelvis Full task, both feet pinned by Full constraints: 12 constraint rows
    "stance": lambda: Case(urdf_text("cassie"), True, W.cassie_stance_problem, _stance_targets, CASSIE_PRM),
    # (d) fixed-base UR5: the forearm frame moves with the first three joints only, so Jc (6 rows) has rank 3
    "ur5": lambda: Case(urdf_text("ur5"), False, _arm("tool0", ik.KinematicType.Position, "forearm_link", ik.KinematicType.Full),
                        _arm_targets(3)),
    # (e) the all-continuous UR5: (cos, sin) coordinates, the upper arm's position pinned (3 rows over 2 columns)
    "ur5_continuous": lambda: Case(CC.ur5_urdf(), False, _arm("tool0", ik.KinematicType.Position, "upper_arm_link", ik.KinematicType.Position),
                                   _arm_targets(2)),
}
# harness builds: (case, warp roles)
BUILDS = {"cassie": ("cassie", 1), "cassie_2roles": ("cassie", 2), "cassie_pelvis": ("cassie_pelvis", 1), "stance": ("stance", 1),
          "stance_2roles": ("stance", 2), "ur5": ("ur5", 1), "ur5_continuous": ("ur5_continuous", 1)}


@pytest.fixture(scope="module")
def harness():
    """Every build's generated body around tests/cpu_harness/spec_constraint_harness.cpp, compiled in parallel."""
    out = os.path.join(ROOT, "build", "cpu_harness")
    os.makedirs(out, exist_ok=True)
    cases = {k: make() for k, make in CASES.items()}

    def build(key):
        case, roles = BUILDS[key]
        c = cases[case]
        mj, sj = S.model_json(c.model), S.spec_json(c.pb, "con_" + key, roles=roles)
        header = os.path.join(out, "spec_con_%s.cuh" % key)
        with open(header, "w") as f:
            f.write(G.Generator(mj, sj).emit(sj["struct"], sj["name"]))
        so = os.path.join(out, "libspec_con_%s.so" % key)
        subprocess.check_call(["g++", "-O1", "-std=c++20", "-fPIC", "-shared", "-pthread", "-x", "c++", "-ffp-contract=off",
                               "-I" + os.path.join(ROOT, "ik_b200", "csrc", "gen"), '-DIKB_PLUGIN_HEADER="%s"' % header,
                               "-DIKB_PLUGIN_STRUCT=" + sj["struct"], "-o", so,
                               os.path.join(ROOT, "tests", "cpu_harness", "spec_constraint_harness.cpp")])
        return key, (c, C.CDLL(so))

    with ThreadPoolExecutor(max_workers=min(len(BUILDS), os.cpu_count() or 1)) as ex:
        return dict(ex.map(build, sorted(BUILDS)))


def _ceval(lib, pb, q, tg, y):
    m = pb.model()
    w = np.ascontiguousarray(np.concatenate([t.weighting() for _, t, _ in pb._tasks]))
    M, mc = len(w), pb.c_size()
    e, J, Jc, dq = np.zeros(M), np.zeros(M * m.nv), np.zeros(mc * m.nv), np.zeros(m.nv)
    pd = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rank = lib.h_spec_plugin_ceval(pd(w), pd(np.ascontiguousarray(q)), pd(np.ascontiguousarray(tg)), pd(np.ascontiguousarray(y)),
                                   pd(e), pd(J), pd(Jc), pd(dq))
    return e, J.reshape(M, m.nv), Jc.reshape(mc, m.nv), dq, rank


@pytest.mark.parametrize("key", sorted(BUILDS))
def test_evaluation_and_projection_match_oracle(harness, key):
    """e, J and Jc of the generated body, the projected step (I - P) (-J^T y) with P, r = O.rowspace_projector(Jc), and
    the rank, at random configurations (the constraint's frame anywhere) and random y."""
    case, lib = harness[key]
    _, tg = case.workload(16, seed=5)
    qs = W.sample_configurations(case.model, 16, seed=6)
    rng = np.random.default_rng(7)
    worst, ranks = 0.0, set()
    for b in range(16):
        y = rng.standard_normal(case.opb.rows)
        e, J, Jc, dq, rank = _ceval(lib, case.pb, qs[b], tg[b], y)
        e_ref, J_ref = case.opb.evaluate(qs[b], tg[b])
        Jc_ref = case.constraint_jacobian(qs[b])
        P, r = O.rowspace_projector(Jc_ref)
        dq_ref = -(np.eye(case.model.nv) - P) @ (J_ref.T @ y)
        worst = max(worst, np.abs(e - e_ref).max(), np.abs(J - J_ref).max(), np.abs(Jc - Jc_ref).max(), np.abs(dq - dq_ref).max())
        assert rank == r, (b, rank, r)
        ranks.add(r)
    print("%s: max |e, J, Jc, dq - oracle| = %.2e, ranks %s" % (key, worst, sorted(ranks)))
    assert worst < 1e-12
    if key in ("ur5", "ur5_continuous"):   # structurally rank-deficient: the forearm moves with 3 joints, the upper arm's
        assert ranks == {{"ur5": 3, "ur5_continuous": 1}[key]}   # origin (on the shoulder-lift axis) with one


@pytest.mark.parametrize("key", sorted(BUILDS))
def test_whole_solves_match_oracle(harness, key):
    """ik::dls to the end on 200 problems, one and two warp roles: flags and step counts identical to the oracle's"""
    case, lib = harness[key]
    q0, tg = case.workload(200, seed=11)
    prm = O.params(**case.prm)
    q_ref, ok_ref, it_ref, res_ref = CO.dls_batch(case.opb, q0, tg, prm, nthreads=os.cpu_count() or 1)
    q, ok, it, res, _ = _spec_solve(lib, "plugin", "f64", case.pb, q0, tg, prm)
    print("%s: converged %.3f, iters %.1f, |dq| max %.2e" % (key, ok_ref.mean(), it_ref.mean(), np.abs(q - q_ref).max()))
    assert (ok == ok_ref).all() and (it == it_ref).all()
    assert np.abs(q - q_ref).max() < 1e-9 and np.abs(res - res_ref).max() < 1e-10
    assert ok_ref.mean() > (0.7 if key.startswith("stance") else 0.8)


@pytest.mark.parametrize("key", ["cassie", "stance", "ur5_continuous"])
def test_f32_spread_is_bounded_by_the_f32_oracle(harness, key):
    case, lib = harness[key]
    q0, tg = case.workload(200, seed=17)
    prm = O.params(**case.prm)
    q64, ok64, it64, _ = CO.dls_batch(case.opb, q0, tg, prm, nthreads=os.cpu_count() or 1)
    stats = {}
    q32 = _spec_solve(lib, "plugin", "f32", case.pb, q0, tg, prm)[:3]
    for label, (q, ok, it) in (("oracle f32", CO.dls_batch_f32(case.opb, q0, tg, prm)[:3]), ("generated f32", q32)):
        both = ok & ok64 & (it == it64)
        err = np.abs(q - q64).max(axis=1)[both]
        stats[label] = dict(flags=(ok == ok64).mean(), p99=np.percentile(err, 99) if err.size else 0.0)
        print("%s %s vs oracle f64: flags agree %.4f, |dq| p99 %.2e" % (key, label, stats[label]["flags"], stats[label]["p99"]))
    assert stats["generated f32"]["flags"] >= stats["oracle f32"]["flags"] - 0.02
    assert stats["generated f32"]["p99"] <= 10 * stats["oracle f32"]["p99"] + 1e-6


def test_pinned_foot_stays_put(harness):
    """(c): both feet stay within 2 mm of where they stand while the pelvis moves to its target"""
    case, lib = harness["stance"]
    q0, tg = case.workload(40, seed=19)
    q, ok, _, _, _ = _spec_solve(lib, "plugin", "f64", case.pb, q0, tg, O.params(**case.prm))
    assert ok.mean() > 0.7
    for frame in ("LeftFootFront", "RightFootFront"):
        f = case.om.frame_id(frame)
        for b in range(40):
            d = case.om.frame_placement(q[b], f) - case.om.frame_placement(q0[b], f)
            assert np.abs(d).max() < 2e-3


# ---- generator ----

def _gen(case, roles=1, **options):
    return G.Generator(S.model_json(case.model), S.spec_json(case.pb, "x", roles=roles, **options))


@pytest.mark.parametrize("option", [{"arrow_solve": True}, {"mirror": [[0, 1]]}, {"fold_task": 0}, {"tmem_j": True},
                                    {"uniform_solve": True}, {"parallel_solve": True}, {"presolve": True},
                                    {"interleave": [[0, 1]]}])
def test_generator_refuses_options_constraints_break(option):
    case = CASES["cassie"]()
    with pytest.raises(ValueError, match="%s.*FrameConstraints" % list(option)[0]):
        _gen(case, roles=2, **option)


def test_generator_refuses_com_task_and_too_many_constraints():
    m = W.cassie_model()
    pb = W.cassie_constraint_problem(m)
    pb.add_centre_of_mass_task(ik.CentreOfMassTask(m))
    with pytest.raises(ValueError, match="centre-of-mass"):
        G.Generator(S.model_json(m), S.spec_json(pb, "x"))
    mj, sj = S.model_json(m), S.spec_json(W.cassie_stance_problem(m), "x")
    sj["constraints"].append({"frame": "pelvis", "type": "position", "reference": "universe"})   # 15 rows
    with pytest.raises(ValueError, match="12 constraint rows"):
        G.Generator(mj, sj)
    sj["constraints"] = [{"frame": "pelvis", "type": "position", "reference": "universe"}] * 5
    with pytest.raises(ValueError, match="at most 4"):
        G.Generator(mj, sj)


def test_constraint_columns_and_strip_layout():
    """U: the columns of joints that move the frame or the reference frame, not both; Jc dense over U behind the task
    slots, counted in NSLOT, which spec_launch (SpecLaunch restated) turns into bytes per problem."""
    case = CASES["cassie_pelvis"]()
    g = _gen(case)
    src = g.emit("SpecX", "x")
    rf = case.model.frame_parents[case.model.frame_names.index("RightFootFront")]
    leg = []
    j = rf
    while case.model.jtypes[j] != W.J_FREEFLYER:
        leg.append(int(case.model.idx_vs[j]))
        j = case.model.parents[j]
    assert g.ucols == sorted(leg)   # the free-flyer moves both the foot and the pelvis: its columns cancel
    assert "MC = 6, NU = %d, CSLOT = %d;" % (len(leg), len(g.slots)) in src
    assert "NSLOT = %d," % (len(g.slots) + 6 * len(leg)) in src
    st = CASES["stance"]()
    gs = _gen(st)
    ssrc = gs.emit("SpecX", "x")
    nu = len(gs.ucols)
    assert set(range(6)) <= set(gs.ucols) and "MC = 12, NU = %d" % nu in ssrc
    L = S.spec_launch(ssrc, 8)
    nslot, nfact, tsz = len(gs.slots) + 12 * nu, gs.rows * (gs.rows + 1) // 2, 12
    assert L["per_problem"] == (nslot + max(nfact, gs.rows + gs.nq) + tsz + 1) * 8 + 8


def test_builtin_specs_emit_no_constraint_code():
    """Every built-in specification regenerates to the header the build made from it, with no constraint member."""
    for name in sorted(os.listdir(os.path.join(ROOT, "ik_b200", "specs"))):
        stem = name[:-5]
        built = os.path.join(ROOT, "ik_b200", "csrc", "gen", stem + ".cuh")
        flat = os.path.join(ROOT, "build", "models", stem + ".json")
        if not (os.path.exists(built) and os.path.exists(flat)):
            pytest.skip("the library has not been built")
        spec = json.load(open(os.path.join(ROOT, "ik_b200", "specs", name)))
        text = G.Generator(json.load(open(flat)), spec).emit(spec["struct"], spec["name"])
        assert text == open(built).read(), stem
        assert "CSLOT" not in text and "sig_con_" not in text and "project(" not in text


# ---- matching ----

_MATCH_PROBE = r"""
import sys
sys.path.insert(0, %(root)r)
from concurrent.futures import ThreadPoolExecutor
import ik_b200 as ik
from ik_b200 import specialise as S
from ik_b200 import workloads as W
K = ik.KinematicType
m = W.cassie_model()
print("before:", W.cassie_constraint_problem(m).specialisation())
with ThreadPoolExecutor(2) as ex:
    sos = list(ex.map(lambda a: S.build_plugin(*a, out_dir=%(out)r), [(W.cassie_constraint_problem(m), "con_match_a"),
                                                                       (W.cassie_stance_problem(m), "con_match_c")]))
for so in sos:
    S.load_plugin(so)

def planted(ctype=K.Position, frame="RightFootFront", ref="universe"):
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", K.Full))
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", K.Position))
    if ctype is not None:
        pb.add_frame_constraint("c", ik.FrameConstraint(m, frame, ctype, ref))
    return pb

def stance(order):
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", K.Full))
    for f in order:
        pb.add_frame_constraint(f, ik.FrameConstraint(m, f, K.Full))
    return pb

print("own:", planted().specialisation())
print("no constraint:", planted(None).specialisation())
print("other type:", planted(K.Full).specialisation())
print("other frame:", planted(frame="LeftFootFront").specialisation())
print("other reference:", planted(ref="pelvis").specialisation())
print("stance:", stance(["LeftFootFront", "RightFootFront"]).specialisation())
print("stance swapped:", stance(["RightFootFront", "LeftFootFront"]).specialisation())
print("feet+pelvis:", W.cassie_feet_pelvis_problem(m).specialisation())
"""


def test_plugin_matching(tmp_path):
    """Plugins compiled for (a) and (c) match their own problems only: not without the constraint, with another constraint
    type, frame or reference frame, or with the constraints in another order; the built-in specialisations still match
    theirs, and before any plugin is loaded a constraint problem has no specialisation (the table-driven kernel)."""
    r = subprocess.run([sys.executable, "-c", _MATCH_PROBE % {"root": ROOT, "out": str(tmp_path)}], capture_output=True, text=True,
                       cwd=ROOT)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    for line in ("before: None", "own: con_match_a", "no constraint: None", "other type: None", "other frame: None",
                 "other reference: None", "stance: con_match_c", "stance swapped: None", "feet+pelvis: cassie_feet_pelvis"):
        assert line in r.stdout, line

"""Generated straight-line code for problems with a CentreOfMassTask, without a GPU: the body tools/gen_kernel.py emits for a
com task compiled with g++ (tests/cpu_harness/spec_plugin_harness.cpp) against the oracle -- one evaluation (e, J) and
whole ik::dls solves in FP64, FP32 and with the role-distributed solve -- the generator's refusals and slot layout, and the
matching of a compiled plugin (in a child interpreter: a loaded plugin stays registered for the whole process)."""
import ctypes as C
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
from oracle.bridge import urdf_text
from tests import continuous_cases as CC
from tests import continuous_oracle as CO
from tests.test_device_code_cpu import _spec_solve

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_kernel as G  # noqa: E402

# A small arm with every kind of velocity column a com task has: a prismatic joint, a revolute joint about an axis off the
# coordinate axes, and a last revolute joint whose link carries no mass (no com column for it; the tool's task uses it).
SLIDER_URDF = """<robot name="slider">
  <link name="base"/>
  <link name="carriage"><inertial><origin xyz="0.05 -0.02 0.1" rpy="0 0 0"/><mass value="2.5"/></inertial></link>
  <link name="arm"><inertial><origin xyz="0.2 0.03 -0.04" rpy="0.1 0.2 0.3"/><mass value="1.2"/></inertial></link>
  <link name="hand"/>
  <link name="tool"/>
  <joint name="slide" type="prismatic"><parent link="base"/><child link="carriage"/><origin xyz="0.1 0 0.2" rpy="0 0 0.3"/>
    <axis xyz="1 0 0"/><limit lower="-0.5" upper="0.5"/></joint>
  <joint name="tilt" type="revolute"><parent link="carriage"/><child link="arm"/><origin xyz="0 0.1 0.3" rpy="0.2 0 0"/>
    <axis xyz="0.48 0.6 0.64"/><limit lower="-2.5" upper="2.5"/></joint>
  <joint name="wrist" type="revolute"><parent link="arm"/><child link="hand"/><origin xyz="0.4 0 0" rpy="0 0 0"/>
    <axis xyz="0 0 1"/><limit lower="-2.5" upper="2.5"/></joint>
  <joint name="tool_joint" type="fixed"><parent link="hand"/><child link="tool"/><origin xyz="0.1 0.05 0" rpy="0 0 0"/></joint>
</robot>"""


class Case:
    """(URDF, free-flyer, task list) with its product problem, oracle problem and workload."""

    def __init__(self, xml, free_flyer, tasks, standing=None, com_weights=None):
        self.xml, self.standing = xml, standing
        self.model = ik.Model.from_urdf(xml, free_flyer)
        self.pb = tasks(self.model)
        if com_weights is not None:
            self.pb.get_centre_of_mass_task().weighting()[:] = com_weights
        om = CO.Model.from_urdf(xml, free_flyer)
        om.flat["lower"][:] = self.model.lowerPositionLimit
        om.flat["upper"][:] = self.model.upperPositionLimit
        self.om = CO.Model(om.flat)
        self.opb = CO.problem_like(self.pb, self.om)

    def centre_of_mass(self, q):
        """the oracle's world centre of mass at q (iko_center_of_mass of the library that knows continuous joints)"""
        com, J = np.zeros(3), np.zeros((3, self.model.nv))
        CO.lib().iko_center_of_mass(C.byref(self.om.c), O._pd(O._d(q)), O._pd(com), O._pd(J))
        return com

    def workload(self, B, seed):
        """(q0, targets, q*): frame targets from the oracle's FK of q*, the com target from the oracle's centre of mass at q*
        (W.com_targets), warm or standing start"""
        from oracle.bridge import oracle_frame_poses
        qstar = W.sample_configurations(self.model, B, seed)
        poses = oracle_frame_poses(self.om, qstar, W.task_frames(self.pb))
        tg = W.targets_from_frame_poses(self.pb, poses, qstar)
        W.com_targets(self.pb, tg, np.array([self.centre_of_mass(q) for q in qstar]), poses)
        if self.standing is not None:
            q0 = np.tile(W.standing_configuration(self.model, self.standing), (B, 1))
        else:
            q0 = W.near_start(self.model, qstar, seed)
        return q0, tg, qstar


def _tool_and_com(frame, ktype=ik.KinematicType.Position):
    def make(m):
        pb = ik.InverseKinematicsProblem(m, 0)
        pb.add_frame_task("tool", ik.FrameTask(m, frame, ktype))
        pb.add_centre_of_mass_task(ik.CentreOfMassTask(m))
        return pb
    return make


CASES = {
    "cassie": lambda: Case(urdf_text("cassie"), True, W.cassie_com_problem, W.CASSIE_STANDING, [2.0, 2.0, 0.5]),
    "cassie_lf": lambda: Case(urdf_text("cassie"), True, lambda m: W.cassie_com_problem(m, "LeftFootFront"), W.CASSIE_STANDING),
    "ur5": lambda: Case(urdf_text("ur5"), False, _tool_and_com("tool0"), com_weights=[1.0, 0.5, 2.0]),
    "ur5_continuous": lambda: Case(CC.ur5_urdf(), False, _tool_and_com("tool0")),
    "slider": lambda: Case(SLIDER_URDF, False, _tool_and_com("tool")),
}
# harness builds: (case, warp roles)
BUILDS = {"cassie": ("cassie", 1), "cassie_2roles": ("cassie", 2), "cassie_lf": ("cassie_lf", 1), "ur5": ("ur5", 1),
          "ur5_continuous": ("ur5_continuous", 1), "slider": ("slider", 1)}


@pytest.fixture(scope="module")
def harness():
    """Every build's generated body around tests/cpu_harness/spec_plugin_harness.cpp, compiled in parallel."""
    out = os.path.join(ROOT, "build", "cpu_harness")
    os.makedirs(out, exist_ok=True)
    cases = {k: make() for k, make in CASES.items()}

    def build(key):
        case, roles = BUILDS[key]
        c = cases[case]
        mj, sj = S.model_json(c.model), S.spec_json(c.pb, "com_" + key, roles=roles)
        header = os.path.join(out, "spec_com_%s.cuh" % key)
        with open(header, "w") as f:
            f.write(G.Generator(mj, sj).emit(sj["struct"], sj["name"]))
        so = os.path.join(out, "libspec_com_%s.so" % key)
        subprocess.check_call(["g++", "-O1", "-std=c++20", "-fPIC", "-shared", "-pthread", "-x", "c++", "-ffp-contract=off",
                               "-I" + os.path.join(ROOT, "ik_b200", "csrc", "gen"), '-DIKB_PLUGIN_HEADER="%s"' % header,
                               "-DIKB_PLUGIN_STRUCT=" + sj["struct"], "-o", so,
                               os.path.join(ROOT, "tests", "cpu_harness", "spec_plugin_harness.cpp")])
        return key, (c, C.CDLL(so))

    with ThreadPoolExecutor(max_workers=min(len(BUILDS), os.cpu_count() or 1)) as ex:
        return dict(ex.map(build, sorted(BUILDS)))


def _eval(lib, pb, q, tg):
    m = pb.model()
    w = np.ascontiguousarray(np.concatenate([t.weighting() for _, t, _ in pb._tasks]))
    M = len(w)
    e, J = np.zeros(M), np.zeros(M * m.nv)
    pd = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    lib.h_spec_plugin_eval(pd(w), pd(np.ascontiguousarray(q)), pd(np.ascontiguousarray(tg)), pd(e), pd(J))
    return e, J.reshape(M, m.nv)


@pytest.mark.parametrize("key", sorted(BUILDS))
def test_evaluation_matches_oracle(harness, key):
    """e and the weighted task Jacobian of the generated body at random configurations (away from the targets' q*)."""
    case, lib = harness[key]
    _, tg, _ = case.workload(16, seed=5)
    qs = W.sample_configurations(case.model, 16, seed=6)
    worst = 0.0
    for b in range(16):
        e, J = _eval(lib, case.pb, qs[b], tg[b])
        e_ref, J_ref = case.opb.evaluate(qs[b], tg[b])
        worst = max(worst, np.abs(e - e_ref).max(), np.abs(J - J_ref).max())
    print("%s: max |e - e_ref|, |J - J_ref| = %.2e" % (key, worst))
    assert worst < 1e-12


@pytest.mark.parametrize("name", sorted(CASES))
def test_com_targets_are_reached_at_the_sampled_configurations(name):
    """W.com_targets: at q* the oracle's centre-of-mass rows of e vanish (universe and moving reference frames alike)."""
    case = CASES[name]()
    _, tg, qstar = case.workload(8, seed=3)
    com = case.pb.get_centre_of_mass_task()
    row = sum(t.dimension() for _, t, _ in case.pb._tasks[:[t for _, t, _ in case.pb._tasks].index(com)])
    for b in range(8):
        e, _ = case.opb.evaluate(qstar[b], tg[b])
        assert np.abs(e[row:row + 3]).max() < 1e-12 and np.abs(e).max() < 1e-9


@pytest.mark.parametrize("key", ["cassie", "cassie_2roles", "ur5", "ur5_continuous", "slider"])
def test_whole_solves_match_oracle(harness, key):
    """ik::dls to the end on 300 problems: the one-role solve (_d) and, with two roles, the role-distributed one (_pd)"""
    case, lib = harness[key]
    q0, tg, _ = case.workload(300, seed=11)
    prm = O.params()
    q_ref, ok_ref, it_ref, res_ref = CO.dls_batch(case.opb, q0, tg, prm, nthreads=os.cpu_count() or 1)
    for variant in ("f64", "f64p"):
        q, ok, it, res, _ = _spec_solve(lib, "plugin", variant, case.pb, q0, tg, prm)
        print("%s %s: converged %.3f, |dq| max %.2e" % (key, variant, ok_ref.mean(), np.abs(q - q_ref).max()))
        assert (ok == ok_ref).all() and (it == it_ref).all()
        assert np.abs(q - q_ref).max() < 1e-9 and np.abs(res - res_ref)[ok].max(initial=0) < 1e-10
    assert ok_ref.mean() > 0.8


def test_moving_reference_first_steps_match_oracle(harness):
    """Relative to the moving LeftFootFront frame the reference does not differentiate the frame's own motion, the iteration
    wanders chaotically: the first 6 steps are compared (as in test_gpu_parity.test_centre_of_mass_task)."""
    case, lib = harness["cassie_lf"]
    q0, tg, _ = case.workload(200, seed=13)
    prm = O.params(max_iterations=6)
    q_ref, ok_ref, it_ref, _ = CO.dls_batch(case.opb, q0, tg, prm)
    q, ok, it, _, _ = _spec_solve(lib, "plugin", "f64", case.pb, q0, tg, prm)
    assert (ok == ok_ref).all() and (it == it_ref).all() and np.abs(q - q_ref).max() < 1e-9


@pytest.mark.parametrize("key", ["cassie", "slider"])
def test_f32_spread_is_bounded_by_the_f32_oracle(harness, key):
    case, lib = harness[key]
    q0, tg, _ = case.workload(300, seed=17)
    prm = O.params()
    q64, ok64, it64, _ = CO.dls_batch(case.opb, q0, tg, prm)
    stats = {}
    q32 = _spec_solve(lib, "plugin", "f32", case.pb, q0, tg, prm)[:3]
    for label, (q, ok, it) in (("oracle f32", CO.dls_batch_f32(case.opb, q0, tg, prm)[:3]), ("generated f32", q32)):
        both = ok & ok64 & (it == it64)
        err = np.abs(q - q64).max(axis=1)[both]
        stats[label] = dict(flags=(ok == ok64).mean(), p99=np.percentile(err, 99) if err.size else 0.0)
        print("%s %s vs oracle f64: flags agree %.4f, |dq| p99 %.2e" % (key, label, stats[label]["flags"], stats[label]["p99"]))
    assert stats["generated f32"]["flags"] >= stats["oracle f32"]["flags"] - 0.02
    assert stats["generated f32"]["p99"] <= 10 * stats["oracle f32"]["p99"] + 1e-6


# ---- generator ----

def _gen(case, roles=1, **options):
    return G.Generator(S.model_json(case.model), S.spec_json(case.pb, "x", roles=roles, **options))


@pytest.mark.parametrize("option", [{"arrow_solve": True}, {"mirror": [[0, 2]]}, {"fold_task": 3}, {"tmem_j": True},
                                    {"uniform_solve": True}, {"parallel_solve": True}, {"presolve": True},
                                    {"interleave": [[0, 2]]}])
def test_generator_refuses_options_a_com_task_breaks(option):
    case = CASES["cassie"]()
    with pytest.raises(ValueError, match="%s.*centre-of-mass" % list(option)[0]):
        _gen(case, roles=2, **option)


@pytest.mark.parametrize("roles", [1, 2])
def test_one_and_two_role_specs_generate(roles):
    case = CASES["cassie"]()
    g = _gen(case, roles)
    src = g.emit("SpecX", "x")
    assert "static constexpr int NQ = 23, NV = 22, M = 12" in src and ("NWARPS = %d" % roles) in src
    assert "sig_inertia()" in src and "sig_task_kind() { static const int v[] = {0, 3, 0, 0}" in src
    com_cols = sorted(set(c for (r, c) in g.slots if 3 <= r < 6))
    assert com_cols == list(range(22))   # every Cassie link carries mass: every velocity coordinate moves the centre of mass


def test_joints_without_subtree_mass_get_no_slots():
    case = CASES["slider"]()
    g = _gen(case)
    g.emit("SpecX", "x")   # (slots are assigned while the body is emitted)
    wrist = case.model.names.index("wrist")
    iv = int(case.model.idx_vs[wrist])
    assert g.com_joints() == [1, 2]
    com_slots = [(r, c) for (r, c) in g.slots if 3 <= r < 6]
    assert sorted(set(c for _, c in com_slots)) == [0, 1] and all(c != iv for _, c in com_slots)
    assert any(c == iv for (r, c) in g.slots if r < 3)   # the tool's task still has the wrist's column


def test_frame_task_specs_emit_no_inertia():
    case = Case(urdf_text("cassie"), True, W.cassie_feet_pelvis_problem)
    src = _gen(case).emit("SpecX", "x")
    assert "sig_inertia" not in src


def test_launch_that_does_not_fit_is_a_readable_error():
    src = ("static constexpr int NQ = 7, NV = 6, M = 200, M0 = 200, TSZ = 600, NSLOT = 1200, NFACT = 20100;\n"
           "static constexpr int NQL = 7;\nstatic constexpr int NWARPS = 1, SOLVER = 0;\nstatic constexpr bool ARROW = false;\n")
    with pytest.raises(ValueError, match="does not fit in shared memory"):
        S.check_launch_fits(src, "huge")
    small = src.replace("NFACT = 20100", "NFACT = 100").replace("NSLOT = 1200", "NSLOT = 100")
    S.check_launch_fits(small, "small")
    with pytest.raises(ValueError, match="too many warp roles"):
        S.check_launch_fits(small.replace("NWARPS = 1", "NWARPS = 13"), "wide")
    # the numbers the kernel's SpecLaunch gives the Cassie com plugin: 2 176 B per problem, 3 groups (96 problems) per SM
    case = CASES["cassie"]()
    L = S.spec_launch(_gen(case).emit("SpecX", "x"), 8)
    assert (L["per_problem"], L["groups"]) == (2176, 3)


# ---- matching ----

_MATCH_PROBE = r"""
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np
import ik_b200 as ik
from ik_b200 import specialise as S
from ik_b200 import workloads as W
from tests.test_com_plugin_cpu import CASES
case = CASES["ur5"]()
S.load_plugin(S.build_plugin(case.pb, "ur5_com_match_test", out_dir=%(out)r))
print("plugin:", CASES["ur5"]().pb.specialisation())
m = ik.Model.from_urdf(case.xml, False)
mass, com = m.inertias()
mass[3] *= 1.5
m.set_inertias(mass, com)
pb = ik.InverseKinematicsProblem(m, 0)
pb.add_frame_task("tool", ik.FrameTask(m, "tool0", ik.KinematicType.Position))
pb.add_centre_of_mass_task(ik.CentreOfMassTask(m))
pb.get_centre_of_mass_task().weighting()[:] = [1.0, 0.5, 2.0]
print("other inertias:", pb.specialisation())
print("feet+pelvis:", W.cassie_feet_pelvis_problem().specialisation())
"""


def test_plugin_matching(tmp_path):
    """A plugin compiled for the UR5's com task list matches that problem, not the same list on a model whose inertias
    differ in one mass, and leaves the built-in specialisations alone."""
    r = subprocess.run([sys.executable, "-c", _MATCH_PROBE % {"root": ROOT, "out": str(tmp_path)}], capture_output=True, text=True,
                       cwd=ROOT)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "plugin: ur5_com_match_test" in r.stdout
    assert "other inertias: None" in r.stdout
    assert "feet+pelvis: cassie_feet_pelvis" in r.stdout

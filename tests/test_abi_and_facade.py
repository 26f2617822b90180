"""The drop-in boundary: the C-ABI shared library exports every entry point include/ikb200.h declares, its host-only
calls behave as documented, the solve entry points FAIL LOUDLY without a GPU (no CPU fallback), and the C++ facade
(include/ik/*.hpp, the reference's class names) compiles against it.  GPU: the facade demo -- the reference's only
caller, ik_ros/src/cassie.cpp, minus ROS -- runs and agrees with the oracle."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import ik_b200 as ik
from ik_b200 import _capi as capi
from ik_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "ik_b200", "libikb200.so")
DEMO = os.path.join(ROOT, "build", "cassie_ik_demo")


def _has_gpu():
    return capi.lib.ikb_device_count() > 0


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "ikb200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(ikb_[a-z0-9_]+)\s*\(", header)))
    assert len(declared) >= 35
    lib = C.CDLL(LIB)
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing


def test_version_and_defaults():
    assert capi.lib.ikb_version() == 200
    p = capi.DlsParams()
    capi.lib.ikb_dls_params_default(C.byref(p))
    # common.hpp:61-65, dls.hpp:25, visitor.hpp:19
    assert (p.max_iterations, p.step_length, p.damping, p.tolerance, p.max_time) == (100, 1.0, 1e-2, 1e-4, 1.0)


def test_unknown_frame_and_bad_priority_are_hard_errors():
    m = W.cassie_model()
    assert m.getFrameId("no_such_frame") == m.nframes  # model.getFrameId semantics (common.hpp:50)
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("x", ik.FrameTask(m, "no_such_frame"))
    with pytest.raises(KeyError):
        pb.specialisation()
    h = C.c_void_p()
    capi.check(capi.lib.ikb_problem_create(m._h, 0, C.byref(h)), "create")
    try:
        assert capi.lib.ikb_problem_add_frame_task(h, 1, 2, 0, 3, None) == -1  # priority > max_priority_level
        assert b"priority" in capi.lib.ikb_last_error()
        assert capi.lib.ikb_problem_add_frame_task(h, 10 ** 6, 2, 0, 0, None) == -3  # IKB_ERR_UNKNOWN_FRAME
    finally:
        capi.lib.ikb_problem_free(h)


def test_problem_sizes_follow_the_reference():
    pb = W.cassie_feet_pelvis_problem()
    h = pb._build_handle(None)
    try:
        lib = capi.lib
        assert lib.ikb_problem_num_tasks(h) == 3 and lib.ikb_problem_rows(h) == 12 and lib.ikb_problem_e_size(h, 0) == 12
        assert [lib.ikb_problem_task_dim(h, t) for t in range(3)] == [6, 3, 3]  # frame.hpp:100-107
        assert lib.ikb_problem_target_size(h) == 36
        assert [lib.ikb_problem_task_target_offset(h, t) for t in range(3)] == [0, 12, 24]
    finally:
        capi.lib.ikb_problem_free(h)


def test_model_inertias_follow_the_urdf_and_the_oracle():
    """CentreOfMassTask needs Pinocchio's model.inertias: per joint, the mass / centre of mass of the bodies it carries
    (links behind fixed joints folded into their supporting joint).  The product's URDF parser against the oracle's."""
    from tests.common import oracle_model
    for name, ff in (("cassie", True), ("ur5", False)):
        m = ik.Model.builtin(name, free_flyer=ff)
        om = oracle_model(name, ff)
        mass, com = m.inertias()
        assert mass.shape == (m.njoints,) and np.allclose(mass, om.flat["mass"], rtol=0, atol=1e-12)
        assert np.allclose(com, np.reshape(om.flat["com"], (-1, 3)), rtol=0, atol=1e-12)
    m = W.cassie_model()
    mass, com = m.inertias()
    assert abs(mass[1:].sum() - 34.676752) < 1e-9  # sum of the <mass value=...> entries of the fixture
    # a model without mass cannot carry the task (hard error, not a division by zero on the device)
    m.set_inertias(np.zeros_like(mass), com)
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_centre_of_mass_task(ik.CentreOfMassTask(m))
    with pytest.raises(RuntimeError, match="mass"):
        pb.specialisation()
    m.set_inertias(mass, com)
    assert pb.specialisation() is None and pb.get_centre_of_mass_task().dimension() == 3 and pb.target_size == 3


@pytest.mark.skipif(_has_gpu(), reason="checks the no-GPU failure mode")
def test_solve_fails_loudly_without_a_gpu():
    pb = W.cassie_feet_pelvis_problem()
    with pytest.raises(RuntimeError, match="no CUDA device|CUDA"):
        pb.finalize(0)


def _build_demo():
    os.makedirs(os.path.dirname(DEMO), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "cassie_ik_demo.cpp"), "-L" + os.path.join(ROOT, "ik_b200"),
                           "-likb200", "-Wl,-rpath," + os.path.join(ROOT, "ik_b200"), "-o", DEMO])


def test_cpp_facade_compiles_and_links():
    """include/ik/*.hpp under the reference's include paths; without a GPU the demo must stop at finalize."""
    _build_demo()
    if not _has_gpu():
        r = subprocess.run([DEMO, os.path.join(ROOT, "ik_b200", "data", "cassie.urdf"), "1"], capture_output=True, text=True)
        assert r.returncode == 1 and "no CUDA device" in r.stderr


@pytest.mark.gpu
def test_cpp_facade_demo_matches_oracle():
    """The reference's demo loop (moving-reference foot task + pelvis pose + axis alignment, warm-started, demo
    parameters) through the C++ facade equals the oracle tick by tick."""
    from oracle import oracle as O
    from tests.common import oracle_model

    _build_demo()
    ticks = 6
    r = subprocess.run([DEMO, os.path.join(ROOT, "ik_b200", "data", "cassie.urdf"), str(ticks)], capture_output=True,
                       text=True, check=True)
    lines = [l.split() for l in r.stdout.splitlines() if l.startswith("tick")]
    assert len(lines) == ticks
    om = oracle_model("cassie")
    opb = O.Problem(om, 1)
    opb.add_frame_task("LeftFootFront", O.POSITION, "pelvis", 0)
    opb.add_frame_task("pelvis", O.FULL, "universe", 0)
    opb.add_align_axis_task("LeftFootFront", 1, "universe", 0)
    q = om.neutral()
    prm = O.params(200, 1e-1, 1e-1)
    for k, l in enumerate(lines):
        t = 0.02 * k
        tg = np.concatenate([np.eye(3).reshape(-1), [0.0, 0.1, -0.6 + 0.2 * np.sin(0.5 * t)],
                             np.eye(3).reshape(-1), np.zeros(3), [1.0, 0.0, 0.0]])
        q, ok, it, res, _ = O.dls(opb, q, tg, prm)
        assert int(l[3]) == int(ok) and int(l[5]) == it
        assert abs(float(l[7]) - res) < 1e-9
        assert np.abs(np.array([float(x) for x in l[9:13]]) - q[7:11]).max() < 1e-6
    assert len([l for l in r.stdout.splitlines() if l.startswith("batch")]) == 4
    assert "queue: 3 of 3 merged batches identical" in r.stdout
    assert "sharded batch identical 1" in r.stdout       # ik::dls_batch(..., devices) through ikb_multi_*
    dl = [l.split() for l in r.stdout.splitlines() if l.startswith("data:")][0]
    assert int(dl[2]) == 10 and int(dl[4]) == 220 and float(dl[6]) < 1e-15      # dls_data::e / J of the last evaluation
    assert int(dl[13]) == 1 and int(dl[15]) != int(dl[8]) and float(dl[17]) < 5e-2   # the overridden should_stop decided
    # ik::pik through the facade (cassie.cpp:114-124): same problem, demo parameters, lambda = 1 per level
    pl = [l.split() for l in r.stdout.splitlines() if l.startswith("pik ")][0]
    tgp = np.concatenate([np.eye(3).reshape(-1), [0.0, 0.1, -0.6], np.eye(3).reshape(-1), np.zeros(3), [1.0, 0.0, 0.0]])
    qp, okp, itp, resp, _ = O.pik(opb, om.neutral(), tgp, O.pik_params(max_iterations=200, step_length=1.0, lambdas=[1.0, 1.0]))
    assert int(pl[2]) == int(okp) and int(pl[4]) == itp and abs(float(pl[6]) - resp) < 1e-9
    assert np.abs(np.array([float(x) for x in pl[8:12]]) - qp[7:11]).max() < 1e-6
    # ik::dls with a FrameConstraint through the facade (frame.hpp:333-465, dls.cpp:26-34,44-52)
    cl = [l.split() for l in r.stdout.splitlines() if l.startswith("constraint ")][0]
    opc = O.Problem(om, 0)
    opc.add_frame_task("pelvis", O.FULL, "universe", 0)
    opc.add_frame_constraint("RightFootFront", O.FULL, "universe")
    qc, okc, itc, resc, _ = O.dls(opc, om.neutral(), O.se3(p=[0.0, 0.01, -0.02]), O.params(step_length=0.5))
    assert int(cl[2]) == 6 and int(cl[4]) == int(okc) and int(cl[6]) == itc and abs(float(cl[8]) - resc) < 1e-9
    assert np.abs(np.array([float(x) for x in cl[10:14]]) - qc[7:11]).max() < 1e-6
    # CentreOfMassTask through the facade (centre_of_mass.hpp:14-52)
    bl = [l.split() for l in r.stdout.splitlines() if l.startswith("com ")][0]
    opm = O.Problem(om, 0)
    opm.add_com_task("universe", 0)
    opm.add_frame_task("pelvis", O.ORIENTATION, "universe", 0)
    qb, okb, itb, resb, _ = O.dls(opm, om.neutral(), np.concatenate([[0.02, 0.01, -0.25], O.se3()]), O.params(step_length=0.5))
    assert int(bl[2]) == 6 and int(bl[4]) == int(okb) and int(bl[6]) == itb and abs(float(bl[8]) - resb) < 1e-9
    assert np.abs(np.array([float(x) for x in bl[10:14]]) - qb[[0, 1, 2, 7]]).max() < 1e-6


def test_facade_eigen_branch_compiles(tmp_path):
    """include/ik/ik.hpp offers Eigen-shaped overloads where <Eigen/Core> exists (the reference's environment,
    common.hpp:23-38).  Eigen is not installed in this image, so the branch is compiled against tests/eigen_stub -- a
    syntax / overload-resolution check, not a numerical one."""
    src = tmp_path / "eig.cpp"
    src.write_text("""
#include <type_traits>
#include <utility>
#include "ik/ik.hpp"
#ifndef IK_HAVE_EIGEN
#error "the Eigen branch was not taken"
#endif
int main() {
    Eigen::Matrix3d R; Eigen::Vector3d p;
    ik::se3_t t(R, p);
    (void)t.rotation_eigen(); (void)t.translation_eigen();
    ik::model_t m;
    if (false) {
        ik::InverseKinematicsProblem pb(m, 0);
        ik::dls_data d(pb);
        Eigen::VectorXd q0(3);
        Eigen::VectorXd q = ik::dls(pb, q0, d);
        (void)d.e_eigen(0); (void)d.J_eigen(0); (void)d.dq_eigen(); (void)d.q_eigen(); (void)q;
    }
    return 0;
}
""")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "tests", "eigen_stub"), "-c", str(src), "-o", str(tmp_path / "eig.o")])


_PLUGIN_PROBE = """
import os, sys
sys.path.insert(0, %(root)r)
import ik_b200 as ik
from ik_b200 import _capi as capi
from ik_b200 import specialise as SP

m = ik.Model.builtin("ur5", free_flyer=False)
pb = ik.InverseKinematicsProblem(m, 0)
pb.add_frame_task("tool", ik.FrameTask(m, "tool0", ik.KinematicType.Full))
assert pb.specialisation() is None
so = SP.build_plugin(pb, "ur5_pose_plugin")
assert os.path.exists(so) and SP.build_plugin(pb, "ur5_pose_plugin") == so      # cached by content hash
SP.load_plugin(so)
SP.load_plugin(so)                                                             # idempotent
assert pb.specialisation() == "ur5_pose_plugin"
other = ik.InverseKinematicsProblem(m, 0)
other.add_frame_task("tool", ik.FrameTask(m, "tool0", ik.KinematicType.Position))
assert other.specialisation() is None
assert capi.lib.ikb_load_specialisation(b"/nonexistent/plugin.so") == capi.ERR_INVALID_ARG
print("REGISTERED")
"""


def test_plugin_specialisation_builds_and_registers():
    """ik_b200.specialise (host side, no GPU needed: nvcc cross-compiles): generator -> nvcc -> plugin .so ->
    ikb_load_specialisation; the host-only query then names the plugin for a problem built from the same URDF, and a
    problem with another task list still has none.  A loaded plugin stays registered until its process exits, so this
    runs in a process of its own: other tests build the same UR5 problem and expect the table-driven kernel for it."""
    r = subprocess.run([sys.executable, "-c", _PLUGIN_PROBE % {"root": ROOT}], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0 and "REGISTERED" in r.stdout, r.stdout + r.stderr

"""ik::pik problems beyond two priority levels, shared by the oracle, CPU-harness and GPU tests: three and seven levels,
an empty level between two used ones, a rank-deficient middle level, a max_priority_level far above the highest used
level, on the Cassie, humanoid and 7-DoF arm trees (one per size class of the table-driven kernel)."""
import numpy as np

import ik_b200 as ik
from ik_b200 import workloads as W
from tests.common import make_workload, oracle_model, oracle_problem_like

# Cassie's 16 revolutes; the two spring joints masked out, as in the reference demo's posture task
_CASSIE_POSTURE_MASK = [1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, 1, 1, 0, 1]


class Case:
    """One problem: `levels` = rows per priority level 0 .. highest used, `deficient` = levels whose J_i P loses rank.
    steps: the stop test reads level 0 only, and where level 0 is met after a step or two the lower levels would hardly
    be iterated -- such cases run exactly `steps` steps (tolerance -1) and compare the iterate, converged or not."""

    def __init__(self, name, pb, urdf, free_flyer=True, start="standing", levels=(), deficient=(), shift=None, steps=None):
        self.name, self.pb, self.urdf, self.free_flyer, self.start = name, pb, urdf, free_flyer, start
        self.levels, self.deficient, self.shift, self.steps = tuple(levels), set(deficient), shift, steps
        assert sum(self.levels) == sum(int(t.dimension()) for _, t, _ in pb._tasks)

    def stop(self, max_iterations):
        """(max_iterations, tolerance) of a solve of this case."""
        return (self.steps, -1.0) if self.steps else (max_iterations, 1e-4)

    def oracle(self):
        om = oracle_model(self.urdf, free_flyer=self.free_flyer)
        return om, oracle_problem_like(self.pb, om)

    def workload(self, B, seed):
        om, _ = self.oracle()
        q0, tg, _ = make_workload(self.pb, om, B, seed=seed, standing=W.CASSIE_STANDING if self.urdf == "cassie" else None,
                                  start=self.start)
        if self.shift is not None:   # (task name, offset): a lower level asks for what a higher one fixes, elsewhere
            name, d = self.shift
            off = self.pb.target_offset(self.pb.get_frame_task(name))
            tg[:, off + 9:off + 12] += d
        return q0, tg


def _posture(m, nj, prio, pb):
    t = ik.PostureTask(m, nj)
    t.mask[:] = _CASSIE_POSTURE_MASK[16 - nj:]
    t.weighting()[:] = 0.05
    pb.add_posture_task("posture", t, prio)


def cassie_three(max_priority_level=2):
    """L0 pelvis Full + LeftFootFront Position, L1 RightFootFront Position + AlignAxis, L2 masked posture: 29 rows."""
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, max_priority_level)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Full), 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 0)
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position), 1)
    pb.add_align_axis_task("align", ik.AlignAxisTask(m, "LeftFootFront", ik.AlignAxisType.AxisY), 1)
    _posture(m, 16, 2, pb)
    name = "cassie_three" if max_priority_level == 2 else "cassie_three_max%d" % max_priority_level
    return Case(name, pb, "cassie", levels=(9, 4, 16))


def cassie_gap():
    """Pelvis Full on level 0, both foot Positions on level 2, level 1 empty, max_priority_level 3: 12 rows."""
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 3)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Full), 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 2)
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position), 2)
    return Case("cassie_gap", pb, "cassie", levels=(6, 0, 6), steps=12)


def cassie_rank_deficient():
    """L0 pelvis Full + LeftFootFront Position; L1 the same foot shifted 5 cm + RightFootFront Position, so J_1 P loses
    rank (singular values ~1 ... ~0.03, ~1e-15) while the right foot keeps it well conditioned (Eigen's rank threshold is
    relative to the largest pivot: a level that is redundant through and through is rounding noise whose rank no two
    implementations agree on); L2 posture of the last 15 coordinates: 30 rows."""
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 2)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Full), 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 0)
    pb.add_frame_task("fl2", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 1)
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position), 1)
    _posture(m, 15, 2, pb)
    return Case("cassie_rank_deficient", pb, "cassie", levels=(9, 6, 15), deficient=(1,), shift=("fl2", 0.05))


def cassie_seven():
    """One task per level, seven levels in 11 rows: LeftFootFront Position on level 0, RightFootFront Position on level 2,
    AlignAxis tasks on five distinct frame / axis pairs on levels 1, 3, 4, 5, 6."""
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 6)
    A = ik.AlignAxisType
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 0)
    pb.add_align_axis_task("a1", ik.AlignAxisTask(m, "LeftFootFront", A.AxisX), 1)
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position), 2)
    pb.add_align_axis_task("a3", ik.AlignAxisTask(m, "pelvis", A.AxisZ), 3)
    pb.add_align_axis_task("a4", ik.AlignAxisTask(m, "RightFootFront", A.AxisY), 4)
    pb.add_align_axis_task("a5", ik.AlignAxisTask(m, "pelvis", A.AxisX), 5)
    pb.add_align_axis_task("a6", ik.AlignAxisTask(m, "LeftFootFront", A.AxisZ), 6)
    return Case("cassie_seven", pb, "cassie", levels=(3, 1, 3, 1, 1, 1, 1))


def humanoid_three():
    """Humanoid: torso_root Full on level 0, both legs Full on level 1, both arms Full on level 2: 30 rows."""
    m = ik.Model.builtin("humanoid", free_flyer=True)
    pb = ik.InverseKinematicsProblem(m, 2)
    pb.add_frame_task("root", ik.FrameTask(m, "torso_root", ik.KinematicType.Full), 0)
    for ee, prio in (("lleg_effector", 1), ("rleg_effector", 1), ("larm_effector", 2), ("rarm_effector", 2)):
        pb.add_frame_task(ee, ik.FrameTask(m, ee, ik.KinematicType.Full), prio)
    return Case("humanoid_three", pb, "humanoid", start="near", levels=(6, 12, 12), steps=12)


def arm_gap():
    """7-DoF arm: tool Position on level 0, level 1 empty, tool Orientation on level 2: 6 rows."""
    m = ik.Model.builtin("manipulator", free_flyer=False)
    pb = ik.InverseKinematicsProblem(m, 2)
    pb.add_frame_task("pos", ik.FrameTask(m, "tool", ik.KinematicType.Position), 0)
    pb.add_frame_task("ori", ik.FrameTask(m, "tool", ik.KinematicType.Orientation), 2)
    return Case("arm_gap", pb, "manipulator", free_flyer=False, start="near", levels=(3, 0, 3), steps=12)


def numpy_pik_step(e, J, levels, lambdas):
    """One ik::pik step (pik.cpp:43-62) with numpy: dq = 0, P = I; per level i with rows: Jb = J_i P,
    dq -= V diag(s / (lambda_i^2 + s^2)) U^T (e_i - J_i dq), P -= pinv(Jb) Jb.  Returns dq and dq after every level.
    The rank cut of pinv sits in the gap between the kept singular values (>= 1e-2 here) and those that are rounding
    noise of an exactly redundant row (~1e-15): numpy's default cut lies at the noise level itself, Eigen's pivot
    threshold (eps min(m, n) max pivot) just above it."""
    nv = J.shape[1]
    dq, P, row, after = np.zeros(nv), np.eye(nv), 0, []
    for lvl, mi in enumerate(levels):
        if mi:
            ei, Ji, lam = e[row:row + mi], J[row:row + mi], lambdas[lvl]
            Jb = Ji @ P
            U, s, Vt = np.linalg.svd(Jb, full_matrices=False)
            dq = dq - (Vt.T * (s / (lam * lam + s * s))) @ U.T @ (ei - Ji @ dq)
            P = P - np.linalg.pinv(Jb, rcond=1e-10) @ Jb
            row += mi
        after.append(dq.copy())
    return dq, after

"""Robots with URDF `continuous` joints, derived from the bundled URDFs, and their workloads (shared by the CPU and GPU
tests of continuous joints and tools/continuous_bench.py).

* the 7-DoF arm with its revolute limits widened to +-100 rad (they never bind) and joints 1/3/5/7 continuous -- the
  layout of a Kinova Gen3 -- on a fixed base or on a free-flyer; the all-revolute arm with the same widened limits is the
  same robot, so its workloads map onto the continuous one by theta -> (cos theta, sin theta);
* the UR5 with all six joints continuous and wrist_2's axis turned off the coordinate axes (an unaligned joint).
"""
import re

import numpy as np

import ik_b200 as ik
from ik_b200 import workloads as W
from oracle.bridge import oracle_frame_poses, urdf_text
from tests import continuous_oracle as CO

ARM_CONTINUOUS = ("arm1_joint", "arm3_joint", "arm5_joint", "arm7_joint")
UR5_JOINTS = ("shoulder_pan_joint", "shoulder_lift_joint", "elbow_joint", "wrist_1_joint", "wrist_2_joint", "wrist_3_joint")
UR5_TILTED_AXIS = {"wrist_2_joint": "0 0.6 0.8"}


def derive_urdf(name, continuous=(), widen=None, axes=None):
    """The bundled URDF `name` with the listed revolute joints declared continuous, every <limit> widened to +-widen and
    the axes of `axes` (joint -> "x y z") replaced."""
    xml = urdf_text(name)
    for j in continuous:
        xml, n = re.subn(r'(<joint name="%s" type=")revolute(")' % re.escape(j), r"\1continuous\2", xml)
        assert n == 1, j
    if widen is not None:
        xml = re.sub(r'<limit lower="[^"]*" upper="[^"]*"', '<limit lower="%r" upper="%r"' % (-widen, widen), xml)
    for j, ax in (axes or {}).items():
        xml, n = re.subn(r'(<joint name="%s"[^>]*>.*?<axis xyz=")[^"]*(")' % re.escape(j), r"\g<1>%s\2" % ax, xml, flags=re.S)
        assert n == 1, j
    return xml


def arm_urdf(continuous=True):
    return derive_urdf("manipulator", ARM_CONTINUOUS if continuous else (), widen=100.0)


def ur5_urdf():
    return derive_urdf("ur5", UR5_JOINTS, axes=UR5_TILTED_AXIS)


class Case:
    """One (URDF, task list) with its product problem and oracle problem."""

    def __init__(self, xml, free_flyer, tasks, max_priority=0):
        self.xml, self.free_flyer = xml, free_flyer
        self.model = ik.Model.from_urdf(xml, free_flyer)
        self.pb = ik.InverseKinematicsProblem(self.model, max_priority)
        for name, task, prio in tasks(self.model):
            self.pb.add_frame_task(name, task, prio)
        self.om = CO.Model.from_urdf(xml, free_flyer)
        self.om.flat["lower"][:] = self.model.lowerPositionLimit
        self.om.flat["upper"][:] = self.model.upperPositionLimit
        self.om = CO.Model(self.om.flat)
        self.opb = CO.problem_like(self.pb, self.om)

    def workload(self, B, seed=12345, b0=0):
        """(q0, targets, q*) AoS float64: targets = oracle FK of q*, warm start near q*."""
        qstar = W.sample_configurations(self.model, B, seed, b0)
        poses = oracle_frame_poses(self.om, qstar, W.task_frames(self.pb))
        return W.near_start(self.model, qstar, seed, b0), W.targets_from_frame_poses(self.pb, poses, qstar), qstar


def _tool_full(m):
    return [("tool", ik.FrameTask(m, "tool", ik.KinematicType.Full), 0)]


def _tool_two_levels(m):
    return [("pos", ik.FrameTask(m, "tool", ik.KinematicType.Position), 0),
            ("ori", ik.FrameTask(m, "tool", ik.KinematicType.Orientation), 1)]


def _ur5_weighted(m):
    pos = ik.FrameTask(m, "tool0", ik.KinematicType.Position)
    pos.weighting()[:] = [1.0, 0.5, 2.0]
    ori = ik.FrameTask(m, "ee_link", ik.KinematicType.Orientation)
    ori.weighting()[:] = [0.5, 1.0, 1.5]
    return [("pos", pos, 0), ("ori", ori, 1)]


def case_a(continuous=True):
    """the Gen3-like arm on a fixed base, the tool's pose"""
    return Case(arm_urdf(continuous), False, _tool_full)


def case_b():
    """the same arm on a free-flyer"""
    return Case(arm_urdf(), True, _tool_full)


def case_c():
    """the all-continuous UR5 with one unaligned axis, weighted Position on level 0 and Orientation on level 1"""
    return Case(ur5_urdf(), False, _ur5_weighted, 1)


def case_d():
    """the arm of (a) for ik::pik: the tool's Position on level 0, its Orientation on level 1"""
    return Case(arm_urdf(), False, _tool_two_levels, 1)


CASES = {"a": case_a, "b": case_b, "c": case_c, "d": case_d}


def to_continuous(rev_model, cont_model, q):
    """Map configurations [B, nq] of the all-revolute arm onto the continuous one: theta -> (cos theta, sin theta)."""
    out = np.zeros((q.shape[0], cont_model.nq))
    for j in range(1, rev_model.njoints):
        a, c = int(rev_model.idx_qs[j]), int(cont_model.idx_qs[j])
        if cont_model.jtypes[j] in W.J_CONTINUOUS:
            out[:, c], out[:, c + 1] = np.cos(q[:, a]), np.sin(q[:, a])
        else:
            n = 7 if rev_model.jtypes[j] == W.J_FREEFLYER else 1
            out[:, c:c + n] = q[:, a:a + n]
    return out


def angles(model, q):
    """atan2(s, c) of every continuous joint of `model` in configurations q [B, nq] -> [B, njoints] (NaN elsewhere)."""
    out = np.full((q.shape[0], model.njoints), np.nan)
    for j in range(1, model.njoints):
        if model.jtypes[j] in W.J_CONTINUOUS:
            iq = int(model.idx_qs[j])
            out[:, j] = np.arctan2(q[:, iq + 1], q[:, iq])
    return out

"""Synthetic IK workloads of BASELINE.json (SURVEY.md 8d), generated identically for the CPU oracle and the GPU.

Per problem b (counter-based SplitMix64 keyed by (seed, b, k), so any shard of a batch can be generated
independently): a reachable configuration q* with revolute joints uniform inside the URDF limits, continuous
joints at an angle uniform in [-pi, pi) (q = (cos, sin)), base position uniform in [-0.2, 0.2]^3 m and base
orientation exp3(u), u uniform in [-0.3, 0.3]^3 rad; the task
targets are the task frames' placements at q* expressed in ``universe``.  Position tasks get the target
(Identity, p) -- the reference's FrameTask keeps ``target`` at se3_t::Identity() and callers only set the
translation (ik_ros/src/cassie.cpp:95-96).  The initial guess is the SRDF standing pose with an identity base.
"""
import numpy as np

from .api import (AlignAxisTask, AlignAxisType, CentreOfMassTask, FrameConstraint, FrameTask, InverseKinematicsProblem,
                  KinematicType, Model, PostureTask)

# cassie-description/srdf/cassie.srdf:22-39 (group_state "default"), in model joint order
CASSIE_STANDING = [0.0045, 0.0, 0.4973, -1.1997, 0.0, 1.4267, 0.0, -1.5968,
                   -0.0045, 0.0, 0.4973, -1.1997, 0.0, 1.4267, 0.0, -1.5968]

J_FREEFLYER = 1
J_CONTINUOUS = (10, 11, 12, 13)   # IKB_J_RUBX .. IKB_J_RUB_UNALIGNED: q = (cos theta, sin theta)

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x):
    """SplitMix64 finaliser on uint64 arrays."""
    with np.errstate(over="ignore"):
        z = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


def uniform01(seed, b, k):
    """Deterministic U[0,1) for problem index array ``b`` and stream index ``k``."""
    with np.errstate(over="ignore"):
        key = splitmix64(np.uint64(seed) + np.uint64(0x632BE59BD9B4E019) * np.uint64(k + 1))
        x = splitmix64(key ^ (b.astype(np.uint64) * np.uint64(0xD1342543DE82EF95)))
    return (x >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def sample_configurations(model, B, seed=12345, b0=0, margin=0.0):
    """q* [B, nq] as described in the module docstring (problem indices b0 .. b0+B-1)."""
    b = np.arange(b0, b0 + B, dtype=np.uint64)
    q = np.zeros((B, model.nq))
    lo, hi = model.lowerPositionLimit, model.upperPositionLimit
    k = 0
    for j in range(1, model.njoints):
        iq = int(model.idx_qs[j])
        if model.jtypes[j] == J_FREEFLYER:
            for i in range(3):
                q[:, iq + i] = -0.2 + 0.4 * uniform01(seed, b, k)
                k += 1
            u = np.stack([-0.3 + 0.6 * uniform01(seed, b, k + i) for i in range(3)], axis=1)
            k += 3
            th = np.linalg.norm(u, axis=1)
            s = np.where(th > 1e-12, np.sin(th / 2) / np.maximum(th, 1e-300), 0.5)
            q[:, iq + 3:iq + 6] = u * s[:, None]
            q[:, iq + 6] = np.cos(th / 2)
        elif model.jtypes[j] in J_CONTINUOUS:   # theta ~ U[-pi, pi): a continuous joint has no limits to sample inside
            th = -np.pi + 2 * np.pi * uniform01(seed, b, k)
            k += 1
            q[:, iq], q[:, iq + 1] = np.cos(th), np.sin(th)
        else:
            w = hi[iq] - lo[iq]
            q[:, iq] = lo[iq] + margin * w + (1 - 2 * margin) * w * uniform01(seed, b, k)
            k += 1
    return q


def standing_configuration(model, standing=None):
    q0 = model.neutral()
    if standing is not None:
        q0[model.nq - len(standing):] = standing
    return q0


def near_start(model, qstar, seed=12345, b0=0, radius=0.3):
    """Warm-start initial guesses (the reference's only caller warm-starts every solve, ik_ros/src/cassie.cpp:112):
    revolute joints = q* + U[-radius, radius] clipped to the limits, continuous joints at the angle of q* plus
    U[-radius, radius], floating base at the identity.  Used for the robots that have no SRDF standing pose; starting the serial arm at its singular zero configuration with full
    undamped-ish steps gives chaotic trajectories on which no two floating-point implementations agree."""
    B = qstar.shape[0]
    b = np.arange(b0, b0 + B, dtype=np.uint64)
    q0 = np.tile(model.neutral(), (B, 1))
    lo, hi = model.lowerPositionLimit, model.upperPositionLimit
    k = 1000
    for j in range(1, model.njoints):
        iq = int(model.idx_qs[j])
        if model.jtypes[j] == J_FREEFLYER:
            continue
        d = -radius + 2 * radius * uniform01(seed, b, k)
        k += 1
        if model.jtypes[j] in J_CONTINUOUS:   # perturb the angle of (cos, sin); the pair stays a unit vector, nothing to clip
            th = np.arctan2(qstar[:, iq + 1], qstar[:, iq]) + d
            q0[:, iq], q0[:, iq + 1] = np.cos(th), np.sin(th)
        else:
            q0[:, iq] = np.minimum(hi[iq], np.maximum(lo[iq], qstar[:, iq] + d))
    return q0


def cassie_model():
    return Model.builtin("cassie", free_flyer=True)


def cassie_feet_pelvis_problem(model=None):
    """BASELINE.json configs 1-3: pelvis pose (Full) + both foot-front positions, all in ``universe``."""
    model = model or cassie_model()
    pb = InverseKinematicsProblem(model, 0)
    pb.add_frame_task("pelvis", FrameTask(model, "pelvis", KinematicType.Full))
    pb.add_frame_task("fl", FrameTask(model, "LeftFootFront", KinematicType.Position))
    pb.add_frame_task("fr", FrameTask(model, "RightFootFront", KinematicType.Position))
    return pb


def humanoid_problem(model=None, root_task=True):
    """BASELINE.json config 4: 4 end-effector poses (Full) (+ root pose) on the 32-DoF humanoid: 24 / 30 rows."""
    model = model or Model.builtin("humanoid", free_flyer=True)
    pb = InverseKinematicsProblem(model, 0)
    if root_task:
        pb.add_frame_task("root", FrameTask(model, "torso_root", KinematicType.Full))
    for ee in ("lleg_effector", "rleg_effector", "larm_effector", "rarm_effector"):
        pb.add_frame_task(ee, FrameTask(model, ee, KinematicType.Full))
    return pb


def manipulator_problem(model=None):
    """BASELINE.json config 5: one Full frame task on the fixed-base 7-DoF arm."""
    model = model or Model.builtin("manipulator", free_flyer=False)
    pb = InverseKinematicsProblem(model, 0)
    pb.add_frame_task("tool", FrameTask(model, "tool", KinematicType.Full))
    return pb


def cassie_demo_problem(model=None):
    """The task set of the reference's own demo (ik_ros/src/cassie.cpp:43-81): LeftFootFront Position relative to the
    moving ``pelvis`` frame, pelvis Full in ``universe``, AlignAxisTask on the foot's y axis.  10 task rows."""
    model = model or cassie_model()
    pb = InverseKinematicsProblem(model, 1)
    pb.add_frame_task("fl", FrameTask(model, "LeftFootFront", KinematicType.Position, "pelvis"))
    pb.add_frame_task("pelvis", FrameTask(model, "pelvis", KinematicType.Full))
    pb.add_align_axis_task("align", AlignAxisTask(model, "LeftFootFront", AlignAxisType.AxisY))
    return pb


def cassie_demo_posture_problem(model=None):
    """The demo's full declared task set (cassie.cpp:43-81 with the commented-out posture line enabled): cassie_demo_problem
    plus a PostureTask on the 16 revolutes at priority level 1, spring joints masked out, weight 0.05.  26 task rows."""
    model = model or cassie_model()
    pb = cassie_demo_problem(model)
    posture = PostureTask(model, model.nq - 7)
    posture.mask[:] = [1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, 1, 1, 0, 1]
    posture.weighting()[:] = 0.05
    pb.add_posture_task("posture", posture, 1)
    return pb


def cassie_com_problem(model=None, reference="universe"):
    """Cassie balancing: LeftFootFront Position, the centre of mass (CentreOfMassTask in `reference`), RightFootFront Position
    and the pelvis Orientation, all on level 0 -- 12 task rows.  Set the centre-of-mass target with com_targets()."""
    model = model or cassie_model()
    pb = InverseKinematicsProblem(model, 0)
    pb.add_frame_task("fl", FrameTask(model, "LeftFootFront", KinematicType.Position))
    pb.add_centre_of_mass_task(CentreOfMassTask(model, reference))
    pb.add_frame_task("fr", FrameTask(model, "RightFootFront", KinematicType.Position))
    pb.add_frame_task("pelvis", FrameTask(model, "pelvis", KinematicType.Orientation))
    return pb


def cassie_constraint_problem(model=None, ktype=KinematicType.Position, reference="universe"):
    """Cassie with a planted foot: pelvis Full and LeftFootFront Position tasks (9 task rows), RightFootFront held in place
    relative to `reference` by a FrameConstraint of type `ktype` (ik::dls projects every step onto its null space)."""
    model = model or cassie_model()
    pb = InverseKinematicsProblem(model, 0)
    pb.add_frame_task("pelvis", FrameTask(model, "pelvis", KinematicType.Full))
    pb.add_frame_task("fl", FrameTask(model, "LeftFootFront", KinematicType.Position))
    pb.add_frame_constraint("fr", FrameConstraint(model, "RightFootFront", ktype, reference))
    return pb


def cassie_stance_problem(model=None, reference="universe"):
    """Cassie in double stance: a pelvis Full task (6 rows) with both feet pinned relative to `reference` by Full
    FrameConstraints -- 12 constraint rows, the most a problem may have.  Draw its targets with cassie_stance_targets()."""
    model = model or cassie_model()
    pb = InverseKinematicsProblem(model, 0)
    pb.add_frame_task("pelvis", FrameTask(model, "pelvis", KinematicType.Full))
    pb.add_frame_constraint("fl", FrameConstraint(model, "LeftFootFront", KinematicType.Full, reference))
    pb.add_frame_constraint("fr", FrameConstraint(model, "RightFootFront", KinematicType.Full, reference))
    return pb


def cassie_stance_targets(problem, B, seed=12345, b0=0):
    """Pelvis targets [B, tsz] that the pinned feet of cassie_stance_problem() leave reachable from the standing pose: the
    standing pelvis placement (identity, at the origin) moved by U[-0.01, 0.01]^3 m and turned by exp3(u), u uniform in
    [-0.01, 0.01]^3 rad (problem indices b0 .. b0+B-1).  With both feet held, pelvis moves of a few centimetres are mostly
    out of reach: ik::dls converges on about 80 % of these draws in 60 half steps, on 5 % of +-3 cm / +-0.05 rad ones."""
    b = np.arange(b0, b0 + B, dtype=np.uint64)
    tg = np.zeros((B, problem.target_size))
    off = problem.target_offset(problem.get_frame_task("pelvis"))
    u = np.stack([-0.01 + 0.02 * uniform01(seed, b, 3 + i) for i in range(3)], axis=1)
    th = np.maximum(np.linalg.norm(u, axis=1), 1e-300)[:, None, None]
    K = np.zeros((B, 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -u[:, 2], u[:, 1], -u[:, 0]
    K -= K.transpose(0, 2, 1)
    R = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * (K @ K)
    tg[:, off:off + 9] = R.reshape(B, 9)
    tg[:, off + 9:off + 12] = np.stack([-0.01 + 0.02 * uniform01(seed, b, i) for i in range(3)], axis=1)
    return tg


def com_targets(problem, targets, coms, poses=None):
    """Set the target of the problem's CentreOfMassTask in `targets` [B, tsz] (in place; returned): coms [B, 3] are the world
    centres of mass at the configurations q* the other targets come from (the oracle's center_of_mass, say), expressed here
    in the task's reference frame, whose world placement poses[frame] [B, 12] supplies (task_frames lists it), so that q*
    reaches every target."""
    task = problem.get_centre_of_mass_task()
    if task is None:
        return targets
    c = np.asarray(coms, dtype=np.float64)
    if task.reference_frame != "universe":
        Mr = poses[task.reference_frame]
        c = np.einsum("bji,bj->bi", Mr[:, :9].reshape(-1, 3, 3), c - Mr[:, 9:12])
    off = problem.target_offset(task)
    targets[:, off:off + 3] = c
    return targets


def frame_task_list(problem):
    return [(t, problem.target_offset(t)) for _, t, _ in problem._tasks if isinstance(t, FrameTask)]


def _rel(Mr, Mf):
    """Mr^-1 * Mf for [B, 12] placements (R row-major 9 + p 3)."""
    Rr, Rf = Mr[:, :9].reshape(-1, 3, 3), Mf[:, :9].reshape(-1, 3, 3)
    R = np.einsum("bji,bjk->bik", Rr, Rf)
    p = np.einsum("bji,bj->bi", Rr, Mf[:, 9:12] - Mr[:, 9:12])
    return np.concatenate([R.reshape(-1, 9), p], axis=1)


def targets_from_frame_poses(problem, poses, qstar=None):
    """poses: dict frame name -> [B, 12] world placements at q* (task frames and their reference frames).  Returns targets
    [B, tsz] (AoS) that q* satisfies exactly: frame tasks get the frame's placement relative to the reference frame,
    align-axis tasks the frame's own axis (scaled by 2: the task normalises it, frame.hpp:264)."""
    B = next(iter(poses.values())).shape[0]
    tg = np.zeros((B, problem.target_size))
    for _, t, _ in problem._tasks:
        off = problem.target_offset(t)
        if isinstance(t, FrameTask):
            M = poses[t.frame] if t.reference_frame == "universe" else _rel(poses[t.reference_frame], poses[t.frame])
            if t.type == KinematicType.Full:
                tg[:, off:off + 12] = M
            else:
                tg[:, off:off + 9] = np.eye(3).reshape(-1)
                if t.type == KinematicType.Position:
                    tg[:, off + 9:off + 12] = M[:, 9:12]
                else:
                    tg[:, off:off + 9] = M[:, :9]
        elif isinstance(t, AlignAxisTask):
            M = poses[t.frame] if t.reference_frame == "universe" else _rel(poses[t.reference_frame], poses[t.frame])
            tg[:, off:off + 3] = 2.0 * M[:, :9].reshape(-1, 3, 3)[:, :, int(t.axis)]
        elif isinstance(t, PostureTask) and qstar is not None:
            tg[:, off:off + t.nj] = qstar[:, problem.model().nq - t.nj:]   # the posture the other targets come from
    return tg


def task_frames(problem):
    """Frames whose placements targets_from_frame_poses and com_targets need."""
    names = []
    for _, t, _ in problem._tasks:
        if isinstance(t, (FrameTask, AlignAxisTask, CentreOfMassTask)):
            for n in (t.reference_frame,) if isinstance(t, CentreOfMassTask) else (t.frame, t.reference_frame):
                if n != "universe" and n not in names:
                    names.append(n)
    return names

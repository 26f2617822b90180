"""Table-driven path A/B on one GPU: thread-per-problem local-memory kernel (IKB_GENERIC_LEGACY=1, dls_generic.cuh) vs the
team-per-problem kernel (dls_coop.cuh) with the pivot column broadcast by warp shuffle (IKB_COOP_SHFL=1) or through
shared memory (=0).  Workloads: Cassie feet+pelvis forced off its specialisation, + FrameConstraint, CentreOfMassTask,
ik::pik on the demo task set, humanoid (262,144) and manipulator (1,048,576) forced off theirs.  CUDA-event timing."""
import os, sys
import numpy as np
sys.path.insert(0, os.getcwd())
import torch
import ik_b200 as ik
from ik_b200 import workloads as W

SCALE = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
VARIANTS = sys.argv[2].split(",") if len(sys.argv) > 2 else ["legacy", "shfl", "smem"]
dev = torch.device("cuda:0")
os.environ["IKB_FORCE_GENERIC"] = "1"


def set_variant(v):
    os.environ["IKB_GENERIC_LEGACY"] = "1" if v == "legacy" else "0"
    os.environ["IKB_COOP_SHFL"] = "1" if v == "shfl" else "0"


def workload(make, B, start, com=None):
    pb = make()
    pb.finalize(0)
    m = pb.model()
    names = W.task_frames(pb)
    qstar = W.sample_configurations(m, B, 12345)
    poses_t = torch.cat([ik.fk_batch(pb, torch.tensor(qstar[i:i + 65536].T.copy(), device=dev), names) for i in range(0, B, 65536)], dim=1)
    poses = {n: poses_t[12 * i:12 * i + 12].T.cpu().numpy() for i, n in enumerate(names)}
    tg = W.targets_from_frame_poses(pb, poses, qstar)
    if com is not None:
        tg[:, pb.target_offset(com(pb)):pb.target_offset(com(pb)) + 3] = qstar[:, :3] + [0.0, 0.0, -0.15]
    q0 = np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (B, 1)) if start == "standing" else W.near_start(m, qstar)
    return torch.tensor(q0.T.copy(), device=dev), torch.tensor(tg.T.copy(), device=dev)


def run(name, make, B, start, solve=None, com=None, legacy_ok=True):
    B = max(1024, int(B * SCALE))
    solve = solve or (lambda p, q, t: ik.dls_batch(p, q, t))
    set_variant("smem")
    q0, tg = workload(make, B, start, com)
    ref = None
    for v in VARIANTS:
        if v == "legacy" and not legacy_ok:
            continue
        set_variant(v)
        pb = make()
        pb.finalize(0)
        out = solve(pb, q0, tg)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            out = solve(pb, q0, tg)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        conv = out["success"].sum().item()
        note = ""
        if ref is None:
            ref = {k: x.clone() for k, x in out.items()}
        else:
            agree = ((ref["success"] == out["success"]) & (ref["iters"] == out["iters"]))
            dq = (ref["q"] - out["q"]).abs().max(dim=0).values[agree & out["success"].bool()].max().item()
            note = "vs %s: agree %.6f max|dq| %.1e" % (VARIANTS[0], agree.float().mean().item(), dq)
        print("%-34s %-6s %-30s B=%-8d %9.3f ms %8.2f M solves/s conv %.4f iters %.2f  %s" % (
            name, v, pb.kernel_name(), B, ms, conv / ms / 1e3, conv / B, out["iters"].float().mean().item(), note), flush=True)


def com_pb():
    m = W.cassie_model()
    pb = ik.InverseKinematicsProblem(m, 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position))
    pb.add_centre_of_mass_task(ik.CentreOfMassTask(m))
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position))
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Orientation))
    return pb


run("cassie feet+pelvis", W.cassie_feet_pelvis_problem, 65536, "standing")
run("cassie demo tasks", W.cassie_demo_problem, 65536, "standing")
run("cassie demo + posture (26 rows)", W.cassie_demo_posture_problem, 65536, "standing")
run("cassie + FrameConstraint", W.cassie_constraint_problem, 65536, "standing")
run("cassie CentreOfMassTask", com_pb, 65536, "standing", com=lambda pb: pb.get_centre_of_mass_task())
prm = ik.pik_parameters(lambdas=[1e-2, 1e-1])
run("ik::pik demo + posture (2 levels)", W.cassie_demo_posture_problem, 65536, "standing", solve=lambda p, q, t: ik.pik_batch(p, q, t, prm))
run("humanoid", W.humanoid_problem, 262144, "near")
run("manipulator", W.manipulator_problem, 1048576, "near")

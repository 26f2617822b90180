"""Kernel-level timing of the Cassie FP64 queue workload (bench.py's headline arm: 65 536 problems per batch, merge 8,
24 batches in flight) with torch.profiler: per kernel name, the number of launches and their durations.  The merged
BULK launch is `dls_spec_kernel<Spec, double, GROUPS, 1, true>`; GROUPS x NWARPS warps run on each SM.

    python tools/bulk_kernel_profile.py [TREE] [--steps 48]

TREE (default: this checkout) is the repository tree whose built ik_b200 is imported, so that two builds can be timed
by the same script.  Prints a table; writes nothing."""
import argparse
import os
import sys

ap = argparse.ArgumentParser()
ap.add_argument("tree", nargs="?", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--steps", type=int, default=48)
ap.add_argument("--batch", type=int, default=65536)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.tree))

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import ik_b200 as ik  # noqa: E402
from ik_b200 import workloads as W  # noqa: E402

assert torch.cuda.is_available(), "needs a GPU"
dev = torch.device("cuda:0")
pb = W.cassie_feet_pelvis_problem()
pb.finalize(0)
m = pb.model()
B = args.batch
sets = []
for s in range(4):
    qstar = W.sample_configurations(m, B, seed=100 + s)
    names = W.task_frames(pb)
    poses_t = ik.fk_batch(pb, torch.tensor(qstar.T.copy(), device=dev), names)
    poses = {n: poses_t[12 * i:12 * i + 12].T.cpu().numpy() for i, n in enumerate(names)}
    tg = W.targets_from_frame_poses(pb, poses)
    q0 = np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (B, 1))
    sets.append((torch.tensor(q0.T.copy(), device=dev), torch.tensor(tg.T.copy(), device=dev)))
prm = ik.dls_parameters()
queue = ik.SolveQueue(pb, 24, 8, 0)


def run(steps):
    for k in range(steps):
        queue.submit(*sets[k % len(sets)], prm)
    queue.drain()
    torch.cuda.synchronize()


run(16)   # warm-up: module load, the carried-straggler path
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    run(args.steps)
rows = {}
for e in prof.events():
    if e.device_type.name != "CUDA" or "dls_" not in e.name:
        continue
    rows.setdefault(e.name, []).append(e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3)
print("device %s, %d steps of %d problems" % (torch.cuda.get_device_name(0), args.steps, B))
print("%6s %9s %9s %9s %9s  kernel" % ("calls", "total ms", "mean ms", "min ms", "max ms"))
for name, d in sorted(rows.items(), key=lambda kv: -sum(kv[1])):
    d = np.array(d)
    print("%6d %9.3f %9.3f %9.3f %9.3f  %s" % (len(d), d.sum(), d.mean(), d.min(), d.max(), name[:160]))

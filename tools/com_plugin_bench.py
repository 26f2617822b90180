"""Cassie balancing task list (W.cassie_com_problem: feet positions, centre of mass in `universe`, pelvis orientation) at
65,536 problems on one GPU: generated plugin with one warp role, with two round-robin roles, and the table-driven kernel
(IKB_FORCE_GENERIC=1), alternating in one run.  CUDA events around each solve, L2 overwritten before every timed launch,
median of 7 rounds.  Prints the card, its power limit and SM clock, each path's time and rate, what bounds the plugin's
occupancy (problems per SM from the strips' shared memory and the register budget), and how the outputs agree.

    python tools/com_plugin_bench.py [B]

The plugins are compiled into a temporary directory (nvcc, a few minutes).  A process can select only the first plugin that
matches a problem, so the two-role plugin is generated for a copy of the model whose massless `universe` joint carries
another centre-of-mass entry: nothing reads it (the centre of mass starts at joint 1), but spec_matches compares it
(dls_spec.cuh), so each plugin matches its own problem -- the kernel_name() asserts below check that it does.  Running
each plugin in a process of its own would lose the alternation, which is what makes the timings comparable."""
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import ik_b200 as ik  # noqa: E402
from ik_b200 import specialise as S  # noqa: E402
from ik_b200 import workloads as W  # noqa: E402
from oracle.bridge import oracle_model  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
ROUNDS = 7
dev = torch.device("cuda:0")


def card():
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return "card: %s, %d SMs; nvidia-smi (name, power limit, SM clock, max SM clock): %s" % (props.name, props.multi_processor_count, smi)


def tagged_model(tag):
    m = W.cassie_model()
    mass, com = m.inertias()
    assert mass[0] == 0.0
    com[0] = [0.0, 0.0, tag]
    m.set_inertias(mass, com)
    return m


def occupancy(header):
    """problems per SM of the FP64 throughput launch (specialise.spec_launch, which restates dls_spec.cuh SpecLaunch)"""
    L = S.spec_launch(header, 8)
    return "%d B of strips per problem: %d groups fit in shared memory, %d in the register budget -> %d problems per SM" % (
        L["per_problem"], L["by_smem"], L["by_regs"], 32 * L["groups"])


def main():
    print(card(), flush=True)
    tmp = tempfile.mkdtemp(prefix="ikb_com_bench_")
    problems = {}
    for label, roles, tag in (("plugin 1 role", 1, 0.0), ("plugin 2 roles", 2, 1.0)):
        pb = W.cassie_com_problem(tagged_model(tag))
        name = "cassie_com_bench_%d" % roles
        S.load_plugin(S.build_plugin(pb, name, out_dir=tmp, roles=roles))
        pb = W.cassie_com_problem(tagged_model(tag))
        pb.finalize(0)
        assert pb.kernel_name() == name, pb.kernel_name()
        with open(os.path.join(tmp, "spec_%s.cuh" % name)) as f:
            print("%-16s %s" % (label, occupancy(f.read())), flush=True)
        problems[label] = pb
    os.environ["IKB_FORCE_GENERIC"] = "1"
    pbg = W.cassie_com_problem()
    pbg.finalize(0)
    os.environ.pop("IKB_FORCE_GENERIC")
    problems["table-driven"] = pbg

    m = pbg.model()
    qstar = W.sample_configurations(m, B, 12345)
    names = W.task_frames(pbg)
    poses_t = ik.fk_batch(pbg, torch.tensor(qstar.T.copy(), device=dev), names)
    poses = {n: poses_t[12 * i:12 * i + 12].T.cpu().numpy() for i, n in enumerate(names)}
    om = oracle_model("cassie")   # the centre of mass at q* from the oracle's iko_center_of_mass
    coms = np.array([om.center_of_mass(q)[0] for q in qstar])
    tg = W.com_targets(pbg, W.targets_from_frame_poses(pbg, poses, qstar), coms, poses)
    q0 = np.tile(W.standing_configuration(m, W.CASSIE_STANDING), (B, 1))
    q0_d, tg_d = torch.tensor(q0.T.copy(), device=dev), torch.tensor(tg.T.copy(), device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # twice the 126 MB of L2

    times = {k: [] for k in problems}
    outs = {}
    for k, pb in problems.items():   # warm-up (module load, smem opt-in)
        outs[k] = ik.dls_batch(pb, q0_d, tg_d)
    torch.cuda.synchronize()
    order = list(problems)
    for r in range(ROUNDS):
        for k in (order if r % 2 == 0 else order[::-1]):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[k] = ik.dls_batch(problems[k], q0_d, tg_d)
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    for k, pb in problems.items():
        ms = float(np.median(times[k]))
        o = outs[k]
        conv = o["success"].float().mean().item()
        print("%-16s %-34s B=%d  %8.3f ms (min %.3f, max %.3f)  %7.2f M solves/s  converged %.4f  mean iters %.2f" % (
            k, pb.kernel_name(), B, ms, min(times[k]), max(times[k]), B / ms / 1e3, conv, o["iters"].float().mean().item()), flush=True)
    ref = outs["table-driven"]
    for k in ("plugin 1 role", "plugin 2 roles"):
        o = outs[k]
        agree = (o["success"] == ref["success"]) & (o["iters"] == ref["iters"])
        both = agree & ref["success"].bool()
        dq = (o["q"] - ref["q"]).abs().max(dim=0).values[both]
        print("  %s vs table-driven: flags and step counts agree on %d of %d problems; converged on both: |dq| max %.2e, p99.9 %.2e" % (
            k, int(agree.sum().item()), B, dq.max().item(), torch.quantile(dq, 0.999).item()), flush=True)
    t = {k: float(np.median(v)) for k, v in times.items()}
    print("speed-up over the table-driven kernel: plugin 1 role %.2fx, plugin 2 roles %.2fx" % (
        t["table-driven"] / t["plugin 1 role"], t["table-driven"] / t["plugin 2 roles"]), flush=True)
    print(card(), flush=True)


if __name__ == "__main__":
    main()

"""FrameConstraint problems at 65,536 problems on one GPU, generated plugin against the table-driven kernel
(IKB_FORCE_GENERIC=1), alternating in one run: (a) Cassie with the right foot planted by a Position constraint
(W.cassie_constraint_problem: pelvis Full + LeftFootFront Position tasks) and (c) Cassie in double stance
(W.cassie_stance_problem: pelvis Full task, both feet pinned by Full constraints, 12 constraint rows).  CUDA events around
each solve, L2 overwritten before every timed launch, median of 7 rounds.  Prints the card, its power limit and SM clock,
each path's time and rate, the plugins' occupancy (problems per SM from the strips' shared memory and the register budget),
and how the outputs agree.  Workloads and solver parameters are those of tests/test_constraint_plugin_cpu.py (60 steps of
length 0.5 from the standing pose).

    python tools/constraint_plugin_bench.py [B]

The plugins are built into build/plugins (nvcc, a few minutes, skipped when an up-to-date build is there)."""
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import ik_b200 as ik  # noqa: E402
from ik_b200 import specialise as S  # noqa: E402
from tests.test_constraint_plugin_cpu import CASES  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
ROUNDS = 7
dev = torch.device("cuda:0")


def card():
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    return "card: %s, %d SMs; nvidia-smi (name, power limit, SM clock, max SM clock): %s" % (props.name, props.multi_processor_count, smi)


def occupancy(header):
    """problems per SM of the FP64 throughput launch (specialise.spec_launch, which restates dls_spec.cuh SpecLaunch)"""
    L = S.spec_launch(header, 8)
    return "%d B of strips per problem: %d groups fit in shared memory, %d in the register budget -> %d problems per SM" % (
        L["per_problem"], L["by_smem"], L["by_regs"], 32 * L["groups"])


def main():
    print(card(), flush=True)
    problems, inputs = {}, {}
    for key, name in (("cassie", "cassie_con_bench"), ("stance", "stance_con_bench")):
        case = CASES[key]()
        so = S.build_plugin(case.pb, name)
        S.load_plugin(so)
        pb = CASES[key]().pb
        pb.finalize(0)
        assert pb.kernel_name() == name, pb.kernel_name()
        with open(os.path.join(os.path.dirname(so), "spec_%s.cuh" % name)) as f:
            print("%-8s %s" % (key, occupancy(f.read())), flush=True)
        os.environ["IKB_FORCE_GENERIC"] = "1"
        pbg = CASES[key]().pb
        pbg.finalize(0)
        os.environ.pop("IKB_FORCE_GENERIC")
        problems[key] = {"plugin": pb, "table-driven": pbg}
        q0, tg = case.workload(B, 401)
        inputs[key] = (torch.tensor(q0.T.copy(), device=dev), torch.tensor(tg.T.copy(), device=dev), ik.dls_parameters(**case.prm))
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # twice the 126 MB of L2

    runs = [(key, path) for key in problems for path in ("plugin", "table-driven")]
    times = {r: [] for r in runs}
    outs = {}
    for key, path in runs:   # warm-up (module load, smem opt-in)
        outs[key, path] = ik.dls_batch(problems[key][path], *inputs[key])
    torch.cuda.synchronize()
    for r in range(ROUNDS):
        for key, path in (runs if r % 2 == 0 else runs[::-1]):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs[key, path] = ik.dls_batch(problems[key][path], *inputs[key])
            e1.record()
            torch.cuda.synchronize()
            times[key, path].append(e0.elapsed_time(e1))
    for key, path in runs:
        ms = float(np.median(times[key, path]))
        o = outs[key, path]
        print("%-8s %-14s %-34s B=%d  %8.3f ms (min %.3f, max %.3f)  %7.2f M solves/s  converged %.4f  mean iters %.2f" % (
            key, path, problems[key][path].kernel_name(), B, ms, min(times[key, path]), max(times[key, path]), B / ms / 1e3,
            o["success"].float().mean().item(), o["iters"].float().mean().item()), flush=True)
    for key in problems:
        o, ref = outs[key, "plugin"], outs[key, "table-driven"]
        agree = (o["success"] == ref["success"]) & (o["iters"] == ref["iters"])
        both = agree & ref["success"].bool()
        dq = (o["q"] - ref["q"]).abs().max(dim=0).values[both]
        print("  %s plugin vs table-driven: flags and step counts agree on %d of %d problems; converged on both: |dq| max %.2e, "
              "p99.9 %.2e" % (key, int(agree.sum().item()), B, dq.max().item(), torch.quantile(dq, 0.999).item()), flush=True)
        t = {p: float(np.median(times[key, p])) for p in ("plugin", "table-driven")}
        print("  %s speed-up of the plugin over the table-driven kernel: %.2fx" % (key, t["table-driven"] / t["plugin"]), flush=True)
    print(card(), flush=True)


if __name__ == "__main__":
    main()

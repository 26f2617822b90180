"""URDF `continuous` joints on the GPU against the oracle, at the batch sizes a user runs: the table-driven kernel on the four
cases of tests/continuous_cases.py (65,536 problems each, the Gen3-like arm also at BASELINE config 5's 1,048,576), the
batch FK entry point, the host-buffer path, a queue stream, the thread-per-problem kernel (IKB_GENERIC_LEGACY=1) and FP32.

FP64 flags and step counts must agree with the oracle on every problem, or -- serial chains started 0.3 rad away with full
steps follow a few chaotic trajectories -- as closely as the oracle agrees with its own build with fused multiply-adds
(the argument of test_gpu_parity.test_full_size_oracle_parity)."""
import os

import numpy as np
import pytest

import ik_b200 as ik
from oracle import oracle as O
from tests import continuous_cases as CC
from tests import continuous_oracle as CO

pytestmark = pytest.mark.gpu
NT = os.cpu_count() or 1


def _torch():
    import torch
    return torch


def _dev(a, dtype="f64"):
    torch = _torch()
    return torch.tensor(np.ascontiguousarray(a.T), dtype=torch.float64 if dtype == "f64" else torch.float32, device="cuda:0")


def _host(out):
    return (out["q"].cpu().numpy().T.astype(np.float64), out["success"].cpu().numpy().astype(bool), out["iters"].cpu().numpy())


def _compare(label, gpu, ref, ref_fma, qtol=1e-6):
    B = len(ref[1])
    bad = int(((gpu[1] != ref[1]) | (gpu[2] != ref[2])).sum())
    bad_fma = int(((ref_fma[1] != ref[1]) | (ref_fma[2] != ref[2])).sum())
    same = (gpu[1] == ref[1]) & (gpu[2] == ref[2]) & ref[1]
    err = np.abs(gpu[0] - ref[0])[same].max(axis=1) if same.any() else np.zeros(1)
    print("%s: B=%d flag/step mismatches kernel %d, FMA oracle %d; converged %.4f; |dq| p99.9 %.2e max %.2e"
          % (label, B, bad, bad_fma, ref[1].mean(), np.percentile(err, 99.9), err.max()))
    assert bad <= max(3 * bad_fma, B // 20000)
    assert np.percentile(err, 99.9) < qtol


def _solve(case, B, seed, pik=False, dtype="f64"):
    q0, tg, _ = case.workload(B, seed)
    fn = ik.pik_batch if pik else ik.dls_batch
    out = fn(case.pb, _dev(q0, dtype), _dev(tg, dtype))
    _torch().cuda.synchronize()
    return q0, tg, _host(out)


@pytest.mark.parametrize("name,B", [("a", 65536), ("a", 1048576), ("b", 65536), ("c", 65536), ("d", 65536)])
def test_table_driven_kernel_matches_oracle(name, B):
    case = CC.CASES[name]()
    pik = name == "d"
    q0, tg, gpu = _solve(case, B, 101, pik=pik)
    assert case.pb.kernel_name().startswith("coop<")
    if pik:
        ref = CO.pik_batch(case.opb, q0, tg, nthreads=NT)[:3]
        ref_fma = CO.pik_batch(case.opb, q0, tg, nthreads=NT, fma=True)[:3]
    else:
        ref = CO.dls_batch(case.opb, q0, tg, nthreads=NT)[:3]
        ref_fma = CO.dls_batch(case.opb, q0, tg, nthreads=NT, fma=True)[:3]
    _compare("case %s (%s)" % (name, case.pb.kernel_name()), gpu, ref, ref_fma)


def test_batch_fk_matches_oracle():
    case = CC.case_c()
    _, _, qs = case.workload(65536, 7)
    frames = ["tool0", "ee_link", "wrist_2_link"]
    out = ik.fk_batch(case.pb, _dev(qs), frames).cpu().numpy()
    ids = [case.om.frame_id(f) for f in frames]
    sel = np.random.default_rng(1).choice(len(qs), 512, replace=False)
    for b in sel:
        for k, f in enumerate(ids):
            assert np.abs(out[12 * k:12 * k + 12, b] - case.om.frame_placement(qs[b], f)).max() < 1e-13


def test_host_buffers_and_queue_match_the_device_path():
    case = CC.case_a()
    q0, tg, gpu = _solve(case, 65536, 103)
    host = ik.dls_batch_host(case.pb, np.ascontiguousarray(q0.T), np.ascontiguousarray(tg.T))
    assert np.array_equal(host["q"].T, gpu[0]) and np.array_equal(host["success"].astype(bool), gpu[1])
    assert np.array_equal(host["iters"], gpu[2])
    queue = ik.SolveQueue(case.pb, depth=4, merge=2)
    jobs = [queue.submit(_dev(q0), _dev(tg)) for _ in range(3)]
    queue.drain()
    for _, o in jobs:
        q, ok, it = _host(o)
        assert np.array_equal(ok, gpu[1]) and np.array_equal(it, gpu[2]) and np.abs(q - gpu[0]).max() < 1e-12


def test_thread_per_problem_kernel_matches_oracle():
    os.environ["IKB_GENERIC_LEGACY"] = "1"
    try:
        case = CC.case_a()
        q0, tg, gpu = _solve(case, 65536, 105)
        assert case.pb.kernel_name().startswith("generic<")
    finally:
        os.environ.pop("IKB_GENERIC_LEGACY")
    ref = CO.dls_batch(case.opb, q0, tg, nthreads=NT)[:3]
    ref_fma = CO.dls_batch(case.opb, q0, tg, nthreads=NT, fma=True)[:3]
    _compare("case a, legacy kernel", gpu, ref, ref_fma)


def test_f32_against_the_f32_oracle():
    case = CC.case_a()
    q0, tg, g32 = _solve(case, 65536, 107, dtype="f32")
    q64, ok64, it64, _ = CO.dls_batch(case.opb, q0, tg, nthreads=NT)
    stats = {}
    for label, (q, ok, it) in (("oracle f32", CO.dls_batch_f32(case.opb, q0, tg, nthreads=NT)[:3]), ("kernel f32", g32)):
        both = ok & ok64 & (it == it64)
        err = np.abs(q - q64).max(axis=1)[both]
        stats[label] = dict(flags=(ok == ok64).mean(), p99=np.percentile(err, 99))
        print("continuous arm %s vs oracle f64: flags agree %.4f, |dq| p99 %.2e" % (label, stats[label]["flags"], stats[label]["p99"]))
    assert stats["kernel f32"]["flags"] >= stats["oracle f32"]["flags"] - 0.01
    assert stats["kernel f32"]["p99"] <= 10 * stats["oracle f32"]["p99"] + 1e-6


_PLUGIN_PROBE = r"""
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
import ik_b200 as ik
from ik_b200 import specialise as S
from oracle import oracle as O
from tests import continuous_cases as CC
from tests import continuous_oracle as CO
for make, name, roles in ((CC.case_a, "gen3_arm_tool_test", 1), (CC.case_d, "gen3_arm_two_roles_test", 2)):
    case = make()
    S.load_plugin(S.build_plugin(case.pb, name, roles=roles))
    case = make()
    assert case.pb.specialisation() == name
    q0, tg, _ = case.workload(65536, 109)
    out = ik.dls_batch(case.pb, torch.tensor(q0.T.copy(), device="cuda:0"), torch.tensor(tg.T.copy(), device="cuda:0"))
    torch.cuda.synchronize()
    assert case.pb.kernel_name() == name, case.pb.kernel_name()
    q, ok, it = out["q"].cpu().numpy().T, out["success"].cpu().numpy().astype(bool), out["iters"].cpu().numpy()
    ref = CO.dls_batch(case.opb, q0, tg, nthreads=os.cpu_count() or 1)
    fma = CO.dls_batch(case.opb, q0, tg, nthreads=os.cpu_count() or 1, fma=True)
    bad = int(((ok != ref[1]) | (it != ref[2])).sum())
    bad_fma = int(((fma[1] != ref[1]) | (fma[2] != ref[2])).sum())
    same = (ok == ref[1]) & (it == ref[2]) & ok
    err = np.abs(q - ref[0])[same].max(axis=1)
    print("plugin %%s (%%d roles): mismatches %%d (FMA oracle %%d), |dq| p99.9 %%.2e" %% (name, roles, bad, bad_fma, np.percentile(err, 99.9)))
    assert bad <= max(3 * bad_fma, 65536 // 20000) and np.percentile(err, 99.9) < 1e-6
print("PLUGINS OK")
"""


def test_generated_plugin_matches_oracle():
    """A plugin for the continuous arm (one warp role) and for the arm's two-level task list (two round-robin warp roles),
    built, loaded and run on 65,536 problems.  In a child interpreter: a loaded plugin stays registered for the whole
    process and would capture the other tests' problems."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _PLUGIN_PROBE % {"root": root}], capture_output=True, text=True, cwd=root)
    print(r.stdout)
    assert r.returncode == 0 and "PLUGINS OK" in r.stdout, r.stdout + r.stderr

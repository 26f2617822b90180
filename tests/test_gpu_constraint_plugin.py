"""Generated plugins for problems with FrameConstraints on the GPU, at the batch sizes a user runs: Cassie with the right foot
planted (a) at 65,536 problems with one and with two warp roles, against the oracle, the table-driven kernel
(IKB_FORCE_GENERIC=1), its own host-buffer and queue paths and the FP32 oracle; the foot held relative to the moving pelvis
(b) and both feet pinned (c), where the pinned frames must also stay put; and a fixed-base UR5 whose constraint Jacobian is
structurally rank-deficient (d) at 262,144 problems.

FP64 flags and step counts must agree with the oracle on every problem, or as closely as the oracle agrees with its own build
with fused multiply-adds (test_gpu_continuous._compare).  Every part runs in a child interpreter: a loaded plugin stays
registered for the whole process and would capture the other tests' problems."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_PROBE = r"""
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
import ik_b200 as ik
from ik_b200 import specialise as S
from oracle import oracle as O
from tests import continuous_oracle as CO
from tests.test_constraint_plugin_cpu import CASES
from tests.test_gpu_continuous import _compare as compare   # flags / steps as the FMA oracle, |dq| p99.9 < 1e-6
NT = os.cpu_count() or 1
PART = %(part)r


def dev(a, dtype=torch.float64):
    return torch.tensor(np.ascontiguousarray(a.T), dtype=dtype, device="cuda:0")


def host(out):
    return out["q"].cpu().numpy().T.astype(np.float64), out["success"].cpu().numpy().astype(bool), out["iters"].cpu().numpy()


def solve(pb, q0, tg, prm, dtype=torch.float64):
    out = ik.dls_batch(pb, dev(q0, dtype), dev(tg, dtype), prm)
    torch.cuda.synchronize()
    return host(out)


def plugin(key, roles, name):
    case = CASES[key]()
    S.load_plugin(S.build_plugin(case.pb, name, roles=roles))
    case = CASES[key]()
    assert case.pb.specialisation() == name, case.pb.specialisation()
    return case


def oracle(case, q0, tg):
    oprm = O.params(**case.prm)
    return CO.dls_batch(case.opb, q0, tg, oprm, nthreads=NT)[:3], CO.dls_batch(case.opb, q0, tg, oprm, nthreads=NT, fma=True)[:3]


def stays_put(case, q0, q):
    # every pinned frame is still where it started relative to its reference frame (2 mm, to first order along the path)
    for _, cn in case.pb._constraints:
        f, r = case.om.frame_id(cn.frame), case.om.frame_id(cn.reference_frame)
        rel = lambda qq: O.se3_actinv(case.om.frame_placement(qq, r), case.om.frame_placement(qq, f))
        for b in range(0, 2000, 50):
            d = rel(q[b]) - rel(q0[b])
            assert np.abs(d[9:]).max() < 2e-3 and (cn.type == ik.KinematicType.Position or np.abs(d[:9]).max() < 2e-3), (cn.frame, b, d)


if PART in ("cassie", "cassie_two_roles"):
    B = 65536
    case = CASES["cassie"]()
    prm = ik.dls_parameters(**case.prm)
    q0, tg = case.workload(B, 301)
    ref, fma = oracle(case, q0, tg)
    os.environ["IKB_FORCE_GENERIC"] = "1"
    pbg = CASES["cassie"]().pb
    generic = solve(pbg, q0, tg, prm)
    assert pbg.kernel_name().startswith("coop<"), pbg.kernel_name()
    os.environ.pop("IKB_FORCE_GENERIC")
    assert CASES["cassie"]().pb.specialisation() is None   # no plugin loaded yet: the table-driven kernel
    compare("table-driven (%%s) vs oracle" %% pbg.kernel_name(), generic, ref, fma)
    # (one plugin per process: a problem takes the first loaded plugin that matches it)
    roles, name = (1, "cassie_con_test") if PART == "cassie" else (2, "cassie_con_two_roles_test")
    c = plugin("cassie", roles, name)
    got = solve(c.pb, q0, tg, prm)
    assert c.pb.kernel_name() == name, c.pb.kernel_name()
    compare("plugin %%s vs oracle" %% name, got, ref, fma)
    compare("plugin %%s vs table-driven" %% name, got, generic, fma)
    stays_put(c, q0, got[0])
if PART == "cassie":
    pb = c.pb
    h = ik.dls_batch_host(pb, np.ascontiguousarray(q0.T), np.ascontiguousarray(tg.T), prm)
    assert np.array_equal(h["q"].T, got[0]) and np.array_equal(h["success"].astype(bool), got[1]) and np.array_equal(h["iters"], got[2])
    queue = ik.SolveQueue(pb, depth=4, merge=2)
    jobs = [queue.submit(dev(q0), dev(tg), prm) for _ in range(3)]
    queue.drain()
    for _, o in jobs:
        q, ok, it = host(o)
        assert np.array_equal(q, got[0]) and np.array_equal(ok, got[1]) and np.array_equal(it, got[2])
    print("host buffers and queue: bit-identical to the device-pointer call", flush=True)
    q64, ok64, it64 = ref
    g32 = solve(pb, q0, tg, prm, dtype=torch.float32)
    assert pb.kernel_name("f32") == "cassie_con_test"
    stats = {}
    for label, (q, ok, it) in (("oracle f32", CO.dls_batch_f32(case.opb, q0, tg, O.params(**case.prm), nthreads=NT)[:3]), ("plugin f32", g32)):
        both = ok & ok64 & (it == it64)
        err = np.abs(q - q64).max(axis=1)[both]
        stats[label] = dict(flags=(ok == ok64).mean(), p99=np.percentile(err, 99))
        print("%%s vs oracle f64: flags agree %%.4f, |dq| p99 %%.2e" %% (label, stats[label]["flags"], stats[label]["p99"]), flush=True)
    assert stats["plugin f32"]["flags"] >= stats["oracle f32"]["flags"] - 0.01
    assert stats["plugin f32"]["p99"] <= 10 * stats["oracle f32"]["p99"] + 1e-6
elif PART in ("cassie_pelvis", "stance"):
    B = 65536
    c = plugin(PART, 1, PART + "_con_test")
    q0, tg = c.workload(B, 303)
    got = solve(c.pb, q0, tg, ik.dls_parameters(**c.prm))
    assert c.pb.kernel_name() == PART + "_con_test"
    compare("plugin %%s_con_test vs oracle" %% PART, got, *oracle(c, q0, tg))
    stays_put(c, q0, got[0])
elif PART == "ur5":
    B = 262144
    c = plugin("ur5", 1, "ur5_con_test")
    q0, tg = c.workload(B, 305)
    got = solve(c.pb, q0, tg, ik.dls_parameters())
    assert c.pb.kernel_name() == "ur5_con_test"
    compare("plugin ur5_con_test vs oracle", got, *oracle(c, q0, tg))
print("PART OK")
"""


@pytest.mark.parametrize("part", ["cassie", "cassie_two_roles", "cassie_pelvis", "stance", "ur5"])
def test_constraint_plugin(part):
    r = subprocess.run([sys.executable, "-c", _PROBE % {"root": ROOT, "part": part}], capture_output=True, text=True, cwd=ROOT)
    print(r.stdout)
    assert r.returncode == 0 and "PART OK" in r.stdout, r.stdout + r.stderr

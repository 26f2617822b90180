"""GPU parity of ik::pik beyond two priority levels against the oracle: three and seven levels, an empty level between two
used ones, a rank-deficient middle level, max_priority_level far above the highest used level, a task above the 7-level
table, on every size class of the table-driven kernel (TEAM = 8, 16, 32; Cassie and 32-joint tree tables) and on the
thread-per-problem fallback, in FP64 and FP32, through the device, host and one-problem entry points."""
import numpy as np
import pytest

import ik_b200 as ik
from ik_b200 import _capi as capi
from oracle import oracle as O
from tests import pik_cases as PC

pytestmark = pytest.mark.gpu
NT = 8
B = 2000                      # and its first 1 and 33 problems: lone teams and teams that pull several problems
MAX_IT = 100

# case -> (builder, IKB_GENERIC_LEGACY, what kernel_name() must contain)
CASES = {
    "cassie_three": (PC.cassie_three, False, "coop<NJ=20,NV=24,M=30,TEAM=32>"),
    "cassie_three_generic": (PC.cassie_three, True, "generic<"),
    "cassie_empty_middle": (PC.cassie_gap, False, "TEAM=16>"),
    "cassie_rank_deficient_middle": (PC.cassie_rank_deficient, False, "TEAM=32>"),
    "cassie_seven": (PC.cassie_seven, False, "TEAM=16>"),
    "humanoid_three": (PC.humanoid_three, False, "coop<NJ=32,NV=36,M=30,TEAM=32>"),
    "arm_empty_middle": (PC.arm_gap, False, "TEAM=8>"),
}
LAMBDAS = {"sharp": [1e-2, 1e-1, 1.0], "defaults": [], "all_seven": [1e-2, 1e-1, 1.0, 0.3, 1e-2, 0.5, 1e-1]}


def _torch():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    return torch


@pytest.fixture
def case(request, monkeypatch):
    make, legacy, kname = CASES[request.param]
    if legacy:   # read when the problem is finalized and at every solve
        monkeypatch.setenv("IKB_GENERIC_LEGACY", "1")
    c = make()
    c.pb.finalize(0)
    name = c.pb.kernel_name()
    assert kname in name and name.startswith("generic<" if legacy else "coop<"), name
    c.label = request.param
    return c


def _gpu(pb, q0, tg, prm, dtype):
    torch = _torch()
    tdt = torch.float64 if dtype == "f64" else torch.float32
    out = ik.pik_batch(pb, torch.tensor(q0.T.copy(), dtype=tdt, device="cuda:0"), torch.tensor(tg.T.copy(), dtype=tdt, device="cuda:0"), prm)
    torch.cuda.synchronize()
    return (out["q"].cpu().numpy().T.astype(np.float64), out["success"].cpu().numpy().astype(bool), out["iters"].cpu().numpy(),
            out["resid"].cpu().numpy().astype(np.float64))


def _params(c, lambdas, max_iterations=MAX_IT):
    mi, tol = c.stop(max_iterations)
    return O.pik_params(mi, 1.0, lambdas, tol), ik.pik_parameters(max_iterations=mi, lambdas=lambdas, tolerance=tol)


def _disagree(c, got, ref):
    """Problems on which two solves disagree: flags, step counts, or (converged, or any in a fixed-step case) q by > 1e-6
    or the residual by > 1e-9."""
    q, ok, it, res = got
    q_ref, ok_ref, it_ref, res_ref = ref
    far = (np.abs(q - q_ref).max(axis=1) > 1e-6) | (np.abs(res - res_ref) > 1e-9)
    return (ok != ok_ref) | (it != it_ref) | ((ok | bool(c.steps)) & far)


def _reference(c, opb, q0, tg, oprm):
    """The oracle's answer, and on how many problems the oracle disagrees with itself when the targets change by 1e-15
    (relative): the rounding of any other FP64 evaluation.  A near-singular or redundant level amplifies it -- an
    ambiguous rank decision at the noise level of a redundant row moves the next level's step by a whole direction --
    and a few problems then end elsewhere with the same flags and steps (CPU: rank-deficient case, B=2000, 13 of 525
    converged problems beyond 1e-6, the largest 0.44 rad; 3-level case, 1 flag of 2000)."""
    ref = O.pik_batch(opb, q0, tg, oprm, nthreads=NT)
    tg_p = tg * (1 + 1e-15 * np.random.default_rng(0).standard_normal(tg.shape))
    return ref, int(_disagree(c, O.pik_batch(opb, q0, tg_p, oprm, nthreads=NT), ref).sum())


def _compare(label, c, got, ref, yard):
    """Bars of test_pik_two_levels_cassie (test_gpu_pik.py) -- flags, step counts, q to 1e-6 and residuals to 1e-9 --
    with the oracle's own rounding as the yardstick: the kernel disagrees with the oracle (_disagree) on at most three
    times as many problems as the oracle with itself (_reference), so on none where the oracle is stable, and agrees to
    1e-9 in the median.  Where the oracle is not stable no fixed share of equal step counts can hold: seven levels with
    lambda 1e-2 on single AlignAxis rows, B=2000, on a B200 -- the oracle disagrees with itself on 219 problems, the kernel
    with the oracle on 204 (flags equal on 97.7 %).  Fixed-step cases compare every iterate, converged or not."""
    q, ok, it, res = got
    q_ref, ok_ref, it_ref, res_ref = ref
    same = (ok == ok_ref) & (it == it_ref)
    bad = _disagree(c, got, ref)
    sel = same & (ok | bool(c.steps))
    err = np.abs(q[sel] - q_ref[sel]).max(axis=1)
    print("pik levels %-44s B=%-5d converged gpu/ref %d/%d, flags equal %.4f, flags+steps equal %.4f, max|dq| %.2e "
          "median %.2e, disagree %d (oracle with itself %d)" % (label, len(ok), ok.sum(), ok_ref.sum(), (ok == ok_ref).mean(),
                                                                same.mean(), err.max(initial=0), np.median(err) if err.size else 0, bad.sum(), yard))
    assert bad.sum() <= 3 * yard
    assert err.size == 0 or np.median(err) < 1e-9


@pytest.mark.parametrize("lambdas", sorted(LAMBDAS))
@pytest.mark.parametrize("case", sorted(CASES), indirect=True)
def test_pik_levels_fp64(case, lambdas):
    c, lam = case, LAMBDAS[lambdas]
    _, opb = c.oracle()
    q0, tg = c.workload(B, seed=61)
    oprm, prm = _params(c, lam, 30 if c.deficient else MAX_IT)
    got = _gpu(c.pb, q0, tg, prm, "f64")
    _compare("%s %s" % (c.label, lambdas), c, got, *_reference(c, opb, q0, tg, oprm))
    # a team that solves one problem and one that pulls several in turn give the same bits
    for n in (1, 33):
        assert all(np.array_equal(a, b[:n]) for a, b in zip(_gpu(c.pb, q0[:n], tg[:n], prm, "f64"), got))


@pytest.mark.parametrize("case", sorted(CASES), indirect=True)
def test_pik_levels_fp32_spread_is_that_of_single_precision(case):
    """FP32 kernel against the FP64 oracle, with the oracle's own FP32 build (number_t = float) as the yardstick: per
    problem max |q - q_fp64| over the problems whose flags and step counts match the FP64 oracle's, by quantile.
    Measured on a B200 (1000 W), B=2000, lambdas 1e-2, 1e-1, 1: the kernel's quantiles are at most 1.7x (median),
    1.8x (p90) and 2.0x (p99) the FP32 oracle's -- largest on the 3-level Cassie case, e.g. thread-per-problem kernel
    p99 8.7e-3 vs 4.4e-3 rad -- and below them on the rank-deficient case; its flags and step counts match the FP64
    oracle at most 0.05 % and 0.2 % less often than the FP32 oracle's do."""
    c = case
    _, opb = c.oracle()
    q0, tg = c.workload(B, seed=62)
    oprm, prm = _params(c, LAMBDAS["sharp"], 30 if c.deficient else MAX_IT)
    q64, ok64, it64, _ = O.pik_batch(opb, q0, tg, oprm, nthreads=NT)
    stats = {}
    for label, (q, ok, it, _) in (("oracle f32", O.pik_batch_f32(opb, q0, tg, oprm, nthreads=NT)),
                                  ("kernel f32", _gpu(c.pb, q0, tg, prm, "f32"))):
        both = (ok == ok64) & (it == it64) & (ok | bool(c.steps))
        err = np.abs(q - q64).max(axis=1)[both]
        st = dict(flags=(ok == ok64).mean(), both=both.mean(), med=np.median(err), p90=np.percentile(err, 90),
                  p99=np.percentile(err, 99), max=err.max())
        stats[label] = st
        print("pik levels FP32 %-30s %s vs oracle f64: flags equal %.4f, flags+steps equal %.4f, |dq| median %.2e p90 %.2e "
              "p99 %.2e max %.2e" % (c.label, label, st["flags"], st["both"], st["med"], st["p90"], st["p99"], st["max"]))
    o, k = stats["oracle f32"], stats["kernel f32"]
    assert k["med"] < 2.5 * o["med"] + 1e-7 and k["p90"] < 2.5 * o["p90"] + 1e-7 and k["p99"] < 3 * o["p99"] + 1e-6
    assert k["flags"] >= o["flags"] - 0.005 and k["both"] >= o["both"] - 0.01


def test_pik_three_levels_host_path_and_one_problem():
    """The 3-level Cassie case through ikb_pik_solve_batch_host and ik.pik (ikb_pik_solve_ex, the state read out of one
    team's shared memory)."""
    c = PC.cassie_three()
    _, opb = c.oracle()
    q0, tg = c.workload(64, seed=63)
    lam = LAMBDAS["sharp"]
    ref, yard = _reference(c, opb, q0, tg, O.pik_params(MAX_IT, 1.0, lam))
    out = ik.pik_batch_host(c.pb, q0, tg, ik.pik_parameters(lambdas=lam))
    _compare("cassie_three host", c, (out["q"], out["success"].astype(bool), out["iters"], out["resid"]), ref, yard)
    for _, t, _ in c.pb._tasks:
        off = c.pb.target_offset(t)
        t.target[:] = tg[0, off:off + t.target_size]
    data = ik.pik_data(c.pb)
    q1 = ik.pik(c.pb, q0[0], data, None, ik.pik_parameters(lambdas=lam))
    assert data.success == bool(ref[1][0]) and data.iterations == ref[2][0] and np.abs(q1 - ref[0][0]).max() < 1e-6


def test_pik_task_above_the_level_table_is_refused_dls_still_solves():
    """A task at priority 7: the level table holds 7 levels, so ik::pik returns IKB_ERR_UNSUPPORTED (and names the
    capacity); ik::dls, which only stacks the rows by priority, solves the same problem as the oracle does."""
    torch = _torch()
    m = ik.Model.builtin("cassie", free_flyer=True)
    pb = ik.InverseKinematicsProblem(m, 7)
    pb.add_frame_task("pelvis", ik.FrameTask(m, "pelvis", ik.KinematicType.Full), 0)
    pb.add_frame_task("fl", ik.FrameTask(m, "LeftFootFront", ik.KinematicType.Position), 3)
    pb.add_frame_task("fr", ik.FrameTask(m, "RightFootFront", ik.KinematicType.Position), 7)
    c = PC.Case("cassie_priority_7", pb, "cassie", levels=(6, 0, 0, 3, 0, 0, 0, 3))
    _, opb = c.oracle()
    q0, tg = c.workload(256, seed=64)
    d_q0, d_tg = torch.tensor(q0.T.copy(), device="cuda:0"), torch.tensor(tg.T.copy(), device="cuda:0")
    with pytest.raises(capi.IkbError) as e:
        ik.pik_batch(pb, d_q0, d_tg)
    assert capi.STATUS_NAMES[e.value.code] == "IKB_ERR_UNSUPPORTED" and "7 priority levels" in str(e.value)
    for call in (lambda: ik.pik_batch_host(pb, q0, tg), lambda: ik.pik(pb, q0[0])):
        with pytest.raises(capi.IkbError) as e:
            call()
        assert capi.STATUS_NAMES[e.value.code] == "IKB_ERR_UNSUPPORTED"
    with pytest.raises(ValueError):
        ik.pik_parameters(lambdas=[1.0] * 8)
    q_ref, ok_ref, it_ref, _ = O.dls_batch(opb, q0, tg, nthreads=NT)
    d = ik.dls_batch(pb, d_q0, d_tg)
    torch.cuda.synchronize()
    ok, it = d["success"].cpu().numpy().astype(bool), d["iters"].cpu().numpy()
    same = (ok == ok_ref) & (it == it_ref)
    assert (ok == ok_ref).all() and same.mean() >= 0.99
    assert np.abs(d["q"].cpu().numpy().T[same & ok] - q_ref[same & ok]).max() < 1e-6


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_pik_max_priority_level_far_above_the_tasks(dtype):
    """max_priority_level 20 with tasks on levels 0-2: ik::pik walks the three used levels and matches both the oracle and
    the same problem declared with max_priority_level 2."""
    c20, c2 = PC.cassie_three(20), PC.cassie_three()
    _, opb = c20.oracle()
    q0, tg = c20.workload(512, seed=65)
    lam = LAMBDAS["sharp"]
    prm = ik.pik_parameters(lambdas=lam)
    got20, got2 = _gpu(c20.pb, q0, tg, prm, dtype), _gpu(c2.pb, q0, tg, prm, dtype)
    assert all(np.array_equal(a, b) for a, b in zip(got20, got2))
    if dtype == "f64":
        _compare("cassie_three max_priority_level 20", c20, got20, *_reference(c20, opb, q0, tg, O.pik_params(MAX_IT, 1.0, lam)))

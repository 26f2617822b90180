"""The oracle's restatement of ik::pik (reference ik/ik/pik.cpp) checked from first principles: its damped pseudo-inverse
and row-space projector against numpy's SVD / pinv, the priority structure (a lower level never disturbs a higher one),
and agreement with ik::dls where the two solvers coincide.  The reference itself pins nothing (no tests, cannot be built)."""
import numpy as np
import pytest

from ik_b200 import workloads as W
from oracle import oracle as O
from tests import pik_cases as PC
from tests.common import make_workload, oracle_model, oracle_problem_like

RNG = np.random.default_rng(11)


def test_damped_pseudoinverse_matches_numpy_svd():
    for m, n in ((3, 7), (6, 22), (10, 22), (16, 22), (1, 5)):
        M = RNG.standard_normal((m, n))
        for lam in (1.0, 1e-2, 0.3):
            U, s, Vt = np.linalg.svd(M, full_matrices=False)
            ref = (Vt.T * (s / (lam * lam + s * s))) @ U.T          # pik.cpp:14-18
            assert np.abs(O.damp_pseudoinverse(M, lam) - ref).max() < 1e-12
            # ... which is the normal-equation form the GPU kernel uses
            assert np.abs(ref - M.T @ np.linalg.inv(M @ M.T + lam * lam * np.eye(m))).max() < 1e-9
    # rank-deficient input: the zero singular value contributes nothing
    M = RNG.standard_normal((4, 9))
    M[3] = M[0] + M[1]
    U, s, Vt = np.linalg.svd(M, full_matrices=False)
    ref = (Vt.T * (s / (0.25 + s * s))) @ U.T
    assert np.abs(O.damp_pseudoinverse(M, 0.5) - ref).max() < 1e-12


def test_rowspace_projector_matches_numpy_pinv():
    for m, n in ((3, 7), (6, 22), (10, 22), (16, 22)):
        M = RNG.standard_normal((m, n))
        P, r = O.rowspace_projector(M)
        assert r == m and np.abs(P - np.linalg.pinv(M) @ M).max() < 1e-12
    # rank deficiency is detected (Eigen COD threshold: eps * min(m, n) * largest pivot) and handled
    M = RNG.standard_normal((5, 12))
    M[4] = 2 * M[1] - M[3]
    P, r = O.rowspace_projector(M)
    assert r == 4 and np.abs(P - np.linalg.pinv(M) @ M).max() < 1e-11
    P, r = O.rowspace_projector(np.zeros((3, 6)))
    assert r == 0 and not P.any()


def _demo_posture():
    pb = W.cassie_demo_posture_problem()
    om = oracle_model("cassie")
    return pb, om, oracle_problem_like(pb, om)


def test_pik_priority_structure_and_convergence():
    """One PIK step from pik.cpp:44-62, rebuilt here with numpy: level 1 (posture) moves only in the null space of level 0."""
    pb, om, opb = _demo_posture()
    q0, tg, _ = make_workload(pb, om, 40, seed=9, standing=W.CASSIE_STANDING)
    prm = O.pik_params(lambdas=[1e-2, 1e-1])
    for b in range(0, 40, 8):
        e, J = opb.evaluate(q0[b], tg[b])
        J = np.asarray(J).reshape(26, 22)
        e0, J0, e1, J1 = e[:10], J[:10], e[10:], J[10:]
        dq = np.zeros(22)
        P = np.eye(22)
        for (ei, Ji, lam) in ((e0, J0, 1e-2), (e1, J1, 1e-1)):
            Jb = Ji @ P
            U, s, Vt = np.linalg.svd(Jb, full_matrices=False)
            dq = dq - (Vt.T * (s / (lam * lam + s * s))) @ U.T @ (ei - Ji @ dq)
            P = P - np.linalg.pinv(Jb) @ Jb
        q1, ok, it, res, dq_o = O.pik(opb, q0[b], tg[b], O.pik_params(max_iterations=1, lambdas=[1e-2, 1e-1]))
        assert np.abs(dq_o - dq).max() < 1e-9
        # the level-1 contribution lies in the null space of J0: it does not change the level-0 task velocity
        U0, s0, V0t = np.linalg.svd(J0, full_matrices=False)
        dq_level0 = -(V0t.T * (s0 / (1e-4 + s0 * s0))) @ U0.T @ e0
        assert np.abs(J0 @ (dq - dq_level0)).max() < 1e-9
    q, ok, it, res = O.pik_batch(opb, q0, tg, prm, nthreads=4)
    assert ok.mean() > 0.9 and np.all(res[ok] < 1e-4)


def test_pik_equals_dls_on_a_single_level():
    """With one priority level PIK's step is -J^T (J J^T + lambda^2 I)^-1 e: ik::dls with damping = lambda (dls.cpp:39-53)."""
    pb = W.cassie_feet_pelvis_problem()
    om = oracle_model("cassie")
    opb = oracle_problem_like(pb, om)
    q0, tg, _ = make_workload(pb, om, 50, seed=2, standing=W.CASSIE_STANDING)
    qd, okd, itd, resd = O.dls_batch(opb, q0, tg, O.params(damping=1e-2))
    qp, okp, itp, resp = O.pik_batch(opb, q0, tg, O.pik_params(lambdas=[1e-2]))
    same = okd & okp & (itd == itp) & (itd < 30)
    assert (okd == okp).mean() > 0.95 and same.mean() > 0.8
    assert np.abs(qd[same] - qp[same]).max() < 1e-7


_LEVEL_CASES = {"three": PC.cassie_three, "seven": PC.cassie_seven, "empty_middle": PC.cassie_gap,
                "rank_deficient_middle": PC.cassie_rank_deficient}


@pytest.mark.parametrize("lambdas", [[1e-2, 1e-1, 1.0, 0.3, 1e-2, 0.5, 1e-1], []])
@pytest.mark.parametrize("case", sorted(_LEVEL_CASES))
def test_pik_step_matches_numpy_beyond_two_levels(case, lambdas):
    """The oracle's step for N levels against numpy's SVD / pinv rebuild of pik.cpp:44-62, including an empty level between
    two used ones and a level whose J_i P loses rank; then the priority property: what levels below k add to dq leaves
    J_k's task velocity alone, J_k (dq - dq_after_k) = 0, for every level that keeps its rank."""
    c = _LEVEL_CASES[case]()
    _, opb = c.oracle()
    lam = [1.0] * 7 if not lambdas else lambdas
    q0, tg = c.workload(12, seed=19)
    for b in range(12):
        e, J = opb.evaluate(q0[b], tg[b])
        dq, after = PC.numpy_pik_step(e, J, c.levels, lam)
        _, _, _, _, dq_o = O.pik(opb, q0[b], tg[b], O.pik_params(max_iterations=1, lambdas=lambdas))
        assert np.abs(dq_o - dq).max() < 1e-9
        row = 0
        for k, mi in enumerate(c.levels):
            if mi and k not in c.deficient:
                assert np.abs(J[row:row + mi] @ (dq - after[k])).max() < 1e-9
            row += mi
        if c.deficient:   # the level really loses rank after the projection: one direction, far below the others
            k = min(c.deficient)
            r0 = sum(c.levels[:k])
            Jk = J[r0:r0 + c.levels[k]]
            P = np.eye(J.shape[1]) - np.linalg.pinv(J[:r0]) @ J[:r0]
            s = np.linalg.svd(Jk @ P, compute_uv=False)
            assert s[-2] > 1e-3 and s[-1] < 1e-12


def test_pik_oracle_level_capacity():
    """IKO_MAX_LEVELS (8) lambdas at most; a task on level 8 is refused instead of reading past the lambda table, while
    levels declared but unused above the last task cost nothing."""
    with pytest.raises(ValueError):
        O.pik_params(lambdas=[1.0] * 9)
    c = PC.cassie_three(max_priority_level=20)
    _, opb = c.oracle()
    _, opb3 = PC.cassie_three().oracle()
    q0, tg = c.workload(4, seed=5)
    a, b = O.pik_batch(opb, q0, tg), O.pik_batch(opb3, q0, tg)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    om = oracle_model("cassie")
    opb = O.Problem(om, 8)
    opb.add_frame_task("LeftFootFront", O.POSITION, priority=8)
    with pytest.raises(ValueError):
        O.pik_batch(opb, q0[:1], tg[:1, :12])
    with pytest.raises(ValueError):
        O.pik(opb, q0[0], tg[0, :12])
    with pytest.raises(ValueError):
        O.pik_batch_f32(opb, q0[:1], tg[:1, :12])

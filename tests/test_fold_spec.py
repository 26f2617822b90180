"""The Cassie specialisation with the pelvis task folded into the two leg roles (ik_b200/specs/cassie_feet_pelvis_fold.json,
tools/gen_kernel.py `fold_task`): the FP64 BULK body.  Its generated arithmetic is checked against the oracle and against
the three-role arrow body it replaces (same expressions, so the same bits) on the CPU, and the ownership the kernel's
barriers rely on -- every stored Jacobian entry, error row, published contribution and coordinate of q has exactly one
writer, and no role reads another role's Jacobian rows (they live in the role's own tensor memory) -- on the generated
source."""
import json
import os
import re
import sys

import numpy as np
import pytest

from oracle import oracle as O
from tests.common import make_workload, oracle_model, oracle_problem_like
from tests.test_device_code_cpu import _build, _spec_solve
from ik_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_kernel as G  # noqa: E402

MODEL = os.path.join(ROOT, "build", "models", "cassie_feet_pelvis_fold.json")
SPEC = os.path.join(ROOT, "ik_b200", "specs", "cassie_feet_pelvis_fold.json")


@pytest.fixture(scope="module")
def fold_lib():
    return _build("spec_fold_harness")


@pytest.fixture(scope="module")
def src():
    if not os.path.exists(MODEL):  # written by `make gen`
        pytest.skip("flattened Cassie model not built")
    g = G.Generator(json.load(open(MODEL)), json.load(open(SPEC)))
    return g.emit("SpecX", "x")


def _const(src, name):
    return int(re.search(r"\b%s = (-?\d+)" % name, src).group(1))


def _body(src, fn):
    i = src.index("static IKB_HD void %s(" % fn)
    return src[i:src.index("\n    }\n", i)]


def _roles(text):
    """{role: text of its `if (role == k) {` blocks} (a block runs to the next one)"""
    out = {}
    for blk in text.split("if (role == ")[1:]:
        k, rest = blk.split(")", 1)
        out[int(k)] = out.get(int(k), "") + rest
    return out


def _solve_both(lib, params, B=200):
    pb = W.cassie_feet_pelvis_problem()
    om = oracle_model("cassie")
    q0, tg, _ = make_workload(pb, om, B, standing=W.CASSIE_STANDING)
    prm = O.params() if params == "defaults" else O.params(200, 1e-1, 1e-1)
    return pb, om, q0, tg, prm


@pytest.mark.parametrize("params", ["defaults", "demo"])
def test_fold_body_matches_oracle_and_the_three_role_body_bit_for_bit(fold_lib, params):
    pb, om, q0, tg, prm = _solve_both(fold_lib, params)
    q_ref, ok_ref, it_ref, res_ref = O.dls_batch(oracle_problem_like(pb, om), q0, tg, prm)
    q, ok, it, res, e0 = _spec_solve(fold_lib, "cassie_feet_pelvis_fold", "f64", pb, q0, tg, prm)
    assert (ok == ok_ref.astype(bool)).all() and (it == it_ref).all()
    assert np.abs(q - q_ref).max() < 1e-8 and np.abs(res - res_ref).max() < 1e-10
    q3, ok3, it3, res3, e03 = _spec_solve(fold_lib, "cassie_feet_pelvis_arrow", "f64", pb, q0, tg, prm)
    assert (ok == ok3).all() and (it == it3).all()
    assert np.array_equal(q, q3) and np.array_equal(res, res3) and np.array_equal(e0, e03)


def test_fold_body_f32_is_close(fold_lib):
    pb, om, q0, tg, prm = _solve_both(fold_lib, "defaults")
    q_ref, ok_ref, it_ref, _ = O.dls_batch(oracle_problem_like(pb, om), q0, tg, prm)
    q, ok, it, _, _ = _spec_solve(fold_lib, "cassie_feet_pelvis_fold", "f32", pb, q0, tg, prm)
    assert (ok == ok_ref.astype(bool)).mean() > 0.98


def test_every_stored_jacobian_entry_belongs_to_one_role_and_no_role_reads_another_ones(src):
    assert "TMEMJ = true" in src and _const(src, "NWARPS") == 2
    first = [int(x) for x in re.search(r"j_first\(int role\) \{ return role == 0 \? (\d+) : role == 1 \? (\d+)", src).groups()]
    count = [int(x) for x in re.search(r"j_count\(int role\) \{ return role == 0 \? (\d+) : role == 1 \? (\d+)", src).groups()]
    assert first[1] == first[0] + count[0]                                    # consecutive, disjoint slots
    own = [set(range(first[k], first[k] + count[k])) for k in range(2)]
    # the fold task never touches the Jacobian strip
    assert "sJ" not in _body(src, "evaluate_f")
    # the mirrored bodies run role 0's slot numbers; side 1 rebases them by exactly the distance to role 1's slots
    for fn in ("evaluate_m0", "arrow_local_m1", "arrow_finish_m1"):
        body = _body(src, fn)
        assert re.search(r"sJ[mr]\{sJ\.base \+ side \* \((\d+) \* SJ::kStride\)\}", body).group(1) == str(first[1] - first[0])
        used = set(int(k) for k in re.findall(r"sJ[mr]\.(?:get|set)\((\d+)", body))
        for k0 in re.findall(r"sJ[mr]\.getn\((\d+), jb\d+\);", body):
            n = int(re.search(r"T jb%s\[(\d+)\];" % k0, body).group(1))
            used |= set(range(int(k0), int(k0) + n))
        assert used and used <= own[0], fn
    sets = set(int(k) for k in re.findall(r"sJm\.set\((\d+)", _body(src, "evaluate_m0")))
    assert sets == own[0]                                                     # every slot of the role is written
    for k, text in _roles(_body(src, "step_role")).items():
        used = set()
        for k0 in re.findall(r"sJ\.getn\((\d+), jb\d+\);", text):
            n = int(re.search(r"T jb%s\[(\d+)\];" % k0, text).group(1))
            used |= set(range(int(k0), int(k0) + n))
        assert used <= own[k] and not re.search(r"sJ\.get\(", text)


def test_every_row_and_published_contribution_has_one_writer(src):
    M, NFACT = _const(src, "M"), _const(src, "NFACT")
    fold = _roles(_body(src, "evaluate_f"))
    writes = {k: [int(x) for x in re.findall(r"sE\.set\((\d+),", t)] for k, t in fold.items()}
    assert sorted(writes) == [0, 1]
    assert not set(writes[0]) & set(writes[1]) and all(len(w) == len(set(w)) for w in writes.values())
    rows = [[r for r in writes[k] if r < M] for k in range(2)]
    assert rows == [[0, 1, 2], [3, 4, 5]]                                     # the pelvis rows: three per role
    pub = sorted(x for k in range(2) for x in writes[k] if x >= M)
    assert len(pub) == 21 + 6 and pub == list(range(pub[0], pub[0] + 27)) and pub[-1] < NFACT   # U^T U and U^T e, once each
    # the phase-2 system reads each published entry exactly once, first after the damping (the three-role order)
    psolve = _body(src, "psolve")
    for x in pub:
        assert len(re.findall(r"sL\.get\(%d\)" % x, psolve)) == 1
    # the leg rows: side 0 writes rows 6-8, side 1 (rebased by 3) rows 9-11
    body = _body(src, "evaluate_m0")
    assert re.search(r"sEm\{sE\.base \+ side \* \(3 \* S::kStride\)\}", body)
    assert sorted(set(int(k) for k in re.findall(r"sEm\.set\((\d+)", body))) == [6, 7, 8]


def test_every_coordinate_of_q_is_stepped_and_stored_once(src):
    nq = _const(src, "NQ")
    stores = {k: dict((int(g), int(l)) for g, l in re.findall(r"dst\[(\d+) \* es\] = q\[(\d+)\]", t))
              for k, t in _roles(_body(src, "store_q")).items()}
    assert sorted(stores) == [0, 1]
    assert not set(stores[0]) & set(stores[1]) and set(stores[0]) | set(stores[1]) == set(range(nq))
    assert set(range(7)) <= set(stores[0])                                    # the free-flyer: the solver role
    step = _roles(_body(src, "step_role"))
    for k in range(2):
        clamped = dict((int(g), int(l)) for l, g in re.findall(r"q\[(\d+)\] = min_\(c\.upper\[(\d+)\]", step[k]))
        assert clamped == stores[k]                                           # what a role stores is what it steps


def test_six_groups_fit_an_sm():
    """SpecLaunch<SpecCassieFeetPelvisFold, double>: 6 groups by shared memory, registers (384 threads) and tensor memory."""
    if not os.path.exists(MODEL):
        pytest.skip("flattened Cassie model not built")
    text = G.Generator(json.load(open(MODEL)), json.load(open(SPEC))).emit("SpecX", "x")
    per_problem = (_const(text, "NFACT") + _const(text, "TSZ") + 1) * 8 + 8
    groups = min(227 * 1024 // (32 * per_problem), 384 // (32 * _const(text, "NWARPS")))
    assert groups == 6
    count = [int(x) for x in re.search(r"j_count\(int role\) \{ return role == 0 \? (\d+) : role == 1 \? (\d+)", text).groups()]
    # 12 warps: lane quarter q holds warps q, q + 4, q + 8, all of role q % 2
    assert all(3 * (32 + 2 * count[q % 2]) <= 512 for q in range(4))

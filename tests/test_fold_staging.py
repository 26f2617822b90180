"""The factor-strip staging slots of the fold body's one-trip-ahead refill (tools/gen_kernel.py factor_stage_slots,
dls_spec.cuh kPrefetch under TMEMJ).  Once the stop test has found a slot's problem converged, its next configuration is
copied behind the second barrier into Spec::qstage_l(role) .. + NQ for every role, and each role reads its own copy
behind the barrier at the top of the next trip.  Checked here on the generated source: under TMEMJ every lane runs phase 2,
phase 3 and step_role warp-wide, also the lanes whose problem converged, so none of them may store into the slots; and the
roles run unordered from the top barrier to the one inside psolve(), so the next store into a role's slots must be that
role's own, after its loads in program order."""
import json
import os
import re
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_kernel as G  # noqa: E402

MODEL = os.path.join(ROOT, "build", "models", "cassie_feet_pelvis_fold.json")
SPEC = os.path.join(ROOT, "ik_b200", "specs", "cassie_feet_pelvis_fold.json")


@pytest.fixture(scope="module")
def gen():
    if not os.path.exists(MODEL):  # written by `make gen`
        pytest.skip("flattened Cassie model not built")
    g = G.Generator(json.load(open(MODEL)), json.load(open(SPEC)))
    return g, g.emit("SpecX", "x")


def _const(src, name):
    return int(re.search(r"\b%s = (-?\d+)" % name, src).group(1))


def _body(src, fn):
    i = src.index("static IKB_HD void %s(" % fn)
    return src[i:src.index("\n    }\n", i)]


def _stores(text, strip="sL", side_shift=0):
    """factor-strip slots a block of generated code stores (loops `sL.set(k0 + i, ...)` for i < n included); a mirrored
    body (`sLr`) stores its slot numbers for side 0 and shifted by `side_shift` for side 1"""
    out = set(int(k) for k in re.findall(r"\b%s\.set\((\d+)," % strip, text))
    for n, k0 in re.findall(r"for \(int i = 0; i < (\d+); \+\+i\) %s\.set\((\d+) \+ i" % strip, text):
        out |= set(range(int(k0), int(k0) + int(n)))
    return out | set(k + side_shift for k in out)


def _roles(text):
    """{role: text of its `if (role == k) {` blocks}"""
    out = {}
    for blk in text.split("if (role == ")[1:]:
        k, rest = blk.split(")", 1)
        out[int(k)] = out.get(int(k), "") + rest
    return out


def _stage(src, role):
    q0 = int(re.search(r"qstage_l\(int role\) \{ return role == 0 \? (-?\d+) : role == 1 \? (-?\d+) : -1; \}", src).group(role + 1))
    assert q0 >= 0
    return set(range(q0, q0 + _const(src, "NQ")))


def _shift(src, fn):
    return int(re.search(r"sLr\{sL\.base \+ side \* \((\d+) \* S::kStride\)\}", _body(src, fn)).group(1))


def _next_trip_stores(src, role):
    """factor-strip slots role `role` stores from the top of a trip to the barrier inside psolve(): the fold task's
    evaluate (its share of the pelvis rows and contributions), its leg's evaluate (e rows) and phase 1"""
    fold = _roles(_body(src, "evaluate_f"))[role]
    ev = set(int(k) + 3 * role for k in re.findall(r"sEm\.set\((\d+),", _body(src, "evaluate_m0")))
    sh = _shift(src, "arrow_local_m1")
    ph1 = set(int(k) + sh * role for k in re.findall(r"\bsLr\.set\((\d+),", _body(src, "arrow_local_m1")))
    return _stores(fold, "sE") | ev | ph1


def test_each_role_stages_in_slots_that_only_it_stores_next(gen):
    _, src = gen
    for role in (0, 1):
        stage, other = _stage(src, role), 1 - role
        assert stage <= _next_trip_stores(src, role)          # its own phase 1 stores them, after its loads
        assert not stage & _next_trip_stores(src, other)      # the other role, unordered with those loads, never does
    assert not _stage(src, 0) & _stage(src, 1)


def test_staging_slots_are_stored_by_nobody_between_the_stop_test_and_the_next_trip(gen):
    _, src = gen
    stage = _stage(src, 0) | _stage(src, 1)
    assert _const(src, "QSTAGE") == -1                                    # no Jacobian strip in shared memory to stage in
    psolve = _body(src, "psolve")
    after_hook = psolve[psolve.index("hook();"):]
    assert "arrow_finish_m1" in after_hook and not _stores(after_hook) & stage       # phase 2 and s
    assert not _stores(_body(src, "arrow_finish_m1"), "sLr", _shift(src, "arrow_finish_m1")) & stage   # phase 3 (both sides)
    assert not _stores(_body(src, "step_role")) & stage                              # the step and the mailbox


def test_staging_slots_are_disjoint_from_e_s_the_mailbox_and_the_factors(gen):
    g, src = gen
    stage = _stage(src, 0) | _stage(src, 1)
    M, A = _const(src, "M"), g.arrow
    assert not stage & set(range(M))                                                  # e
    assert not stage & set(range(A["soff"], A["soff"] + A["ks"]))                      # s
    mail = set(int(k) for k in re.findall(r"sL\.get\((\d+)\)", _body(src, "fetch_common")))
    assert mail and not stage & mail                                                  # the free-flyer mailbox
    for base in A["facb"].values():                                                  # the legs' factors (read by phase 3)
        assert not stage & set(range(base, base + A["my"] * (A["my"] + 1) // 2))
    assert max(stage) < _const(src, "NFACT")


def test_no_staging_home_gives_minus_one():
    """A role whose published contributions are too short for NQ consecutive slots: the kernel keeps the direct refill."""
    ks = 2
    per = ks * (ks + 1) // 2 + ks
    fake = types.SimpleNamespace(spec={}, rows=4, nq=7, arrow_mail=None, arrow_qc=None,
                                 arrow=dict(ks=ks, soff=4, pub={0: ("L", 6), 1: ("L", 6 + per + 3)}, facb={1: 6 + per}, my=2,
                                            ncq=0, fold=None))
    assert G.Generator.factor_stage_slots(fake) is None
    fake.nq = per
    assert G.Generator.factor_stage_slots(fake) == [6, 6 + per + 3]
    fake.arrow["fold"] = 0                                  # the fold task's contributions are nobody's own
    assert G.Generator.factor_stage_slots(fake) == [6 + per + 3]
    # the committed arrow specs (Jacobian strip in shared memory) emit no such function: their headers are unchanged
    for name in ("cassie_feet_pelvis_arrow", "cassie_feet_pelvis_arrow_b", "humanoid_limbs_arrow"):
        model = os.path.join(ROOT, "build", "models", "%s.json" % name)
        if not os.path.exists(model):
            pytest.skip("flattened models not built")
        src = G.Generator(json.load(open(model)), json.load(open(os.path.join(ROOT, "ik_b200", "specs", "%s.json" % name)))).emit("SpecX", "x")
        assert "qstage_l" not in src

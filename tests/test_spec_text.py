"""The oracle against the reference's OWN TEXT.  oracle/tla_eval.py parses the upstream vsr-revisited/paper/VSR.tla
and enumerates Init / Next the way TLC does; these tests compare that with the C++ oracle (the thing every GPU parity
test is measured against): whole small state spaces level by level, and successor sets state by state along the golden
trace, random walks (state transfer and view changes included) and — with RestartEmptyLimit = 1 — the recovery actions.
The text is executed where VSR_TLAPLUS_DIR names a vsr-tlaplus checkout; everywhere else the oracle is compared with
what executing it gave, stored in tests/golden/spec_text_recorded.json (tests/golden/make_spec_text_recorded.py; see
tests/spec_text.py).  tests/golden/spec_text_results.json (make_spec_text_fixture.py) holds bigger state spaces."""
import base64
import json
import os
import random
import re
import zlib

import pytest

import orc
from conftest import ROOT

FIXTURE = os.path.join(ROOT, "tests", "golden", "spec_text_results.json")


@pytest.mark.parametrize("R,V,L,expect", [(2, 1, 1, (76, 100, 14)), (2, 2, 1, (313, 405, 18)), (2, 2, 2, (4034, 5419, 27))])
def test_whole_state_space_from_the_spec_text(pkg, R, V, L, expect):
    """BASELINE configs[0] and two neighbours: distinct / generated / depth and every level's size and successor count,
    derived from VSR.tla's text, equal the oracle's (SYMMETRY off on both sides: the text evaluator does not reduce)."""
    import spec_text as S
    keys = ("distinct", "generated", "depth", "level_sizes", "level_generated", "violation_depth", "deadlock_depth")
    r = S.from_text("state_space/%d,%d,%d" % (R, V, L), lambda: {k: v for k, v in S.T.bfs(
        S.evaluator(R, V, L), invariant="AcknowledgedWriteNotLost", keep_levels=False).items() if k in keys})
    o = orc.bfs(orc.params(R, V, L, symmetry=False), workers=4, keep_trace=False)
    assert (r["distinct"], r["generated"], r["depth"]) == expect == (o.distinct, o.generated, o.depth)
    assert r["level_sizes"] == o.level_sizes and r["level_generated"] == o.level_generated
    assert r["violation_depth"] == 0 and o.rc == 0
    # TLC checks deadlock unless told not to; the text has terminal states (every message delivered, every value used, timer
    # budget spent), so "full BFS" presupposes -deadlock (SURVEY §5).  Both sides agree that they exist.
    assert r["deadlock_depth"] > 0
    assert orc.bfs(orc.params(R, V, L, symmetry=False), workers=1, check_deadlock=True, keep_trace=False).rc == 11


@pytest.mark.parametrize("R,V,L", [(2, 2, 1), (2, 2, 2)])
def test_symmetry_reduction_explores_exactly_the_orbits(pkg, R, V, L):
    """SYMMETRY symmValues (VSR.cfg:31): the oracle's symmetric search must find, at every depth, as many states as the
    text evaluator's UNREDUCED search has orbits under Permutations(Values) of the VIEW value at that depth."""
    import itertools
    import spec_text as S
    T = S.T

    def relabel(v, pi):
        if isinstance(v, T.ModelValue):
            return pi.get(v, v)
        if isinstance(v, frozenset):
            return frozenset(relabel(x, pi) for x in v)
        if isinstance(v, T.Fn):
            return T.Fn({relabel(k, pi): relabel(x, pi) for k, x in v.d.items()})
        return v

    def orbits():
        ev = S.evaluator(R, V, L)
        vals = sorted(ev.c["Values"], key=lambda m: m.name)
        perms = [dict(zip(vals, p)) for p in itertools.permutations(vals)]
        r = T.bfs(ev)
        orbit_levels = []
        for lv in r["levels"]:
            reps = set()
            for st in lv:
                view = ev.project(st)
                reps.add(min((relabel(view, pi) for pi in perms), key=T.vkey))
            orbit_levels.append(len(reps))
        return {"orbit_levels": orbit_levels, "depth": r["depth"]}
    r = S.from_text("orbits/%d,%d,%d" % (R, V, L), orbits)
    orbit_levels = r["orbit_levels"]
    o = orc.bfs(orc.params(R, V, L, symmetry=True), workers=4, keep_trace=False)
    assert o.level_sizes == orbit_levels
    assert o.distinct == sum(orbit_levels) and o.depth == r["depth"]


def test_successors_along_the_golden_trace_and_around_it(pkg):
    """every state of state_transfer_violation_trace.txt (README constants), then walks that start from them: the
    neighbourhoods where SendGetState / ReceiveGetState / ReceiveNewState / ReceiveHigherDVC fire"""
    import spec_text as S
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "state_transfer_trace.json")))
    P = S.Pair(pkg, 3, 3, 3)
    flats = [P.Flat.from_buffer_copy(zlib.decompress(base64.b64decode(s["flat_zlib_b64"]))) for s in fx["states"]]
    # the published trace is a behaviour of the CURRENT text: each recorded state is a successor of the one before, under
    # the recorded action name (the file predates three variables; they sit at their Init values, SURVEY §4)
    pys = [S.to_py(P.q, f) for f in flats]
    for i in range(len(pys) - 1):
        succ = [(a, S.to_py(P.q, f)) for a, f in P.compare(flats[i])]  # the oracle's successors, equal to the text's
        assert any(a == fx["states"][i + 1]["action"] and sp == pys[i + 1] for a, sp in succ), (i + 2, fx["states"][i + 1]["action"])
    rng = random.Random(7)
    n = 0
    for f in flats:
        P.compare(f)
        n += 1 + P.walk(f, 8, rng, prefer=("SendGetState", "ReceiveGetState", "ReceiveNewState", "ReceiveHigherDVC"))
    # a DoViewChange that reaches a primary still in the old view (never in the golden trace, rare on walks): r1 and r3
    # agree on view 2 behind r2's back
    path = S.follow(P, P.init_flat(), ["TimerSendSVC", "ReceiveHigherSVC", "ReceiveMatchingSVC", "SendDVC", "ReceiveHigherDVC"])
    assert path is not None
    n += len(path) + P.walk(path[-1], 12, rng)
    assert n >= 100
    for a in ("SendGetState", "ReceiveGetState", "ReceiveNewState", "ReceiveHigherDVC", "SendSV", "ExecuteOp"):
        assert P.stats[a] > 0, (a, dict(P.stats))
    # the last state of the trace violates the invariant by the spec's own definition
    assert not P.text_holds("AcknowledgedWriteNotLost", flats[-1])


@pytest.mark.parametrize("R,V,L,walks,steps", [(3, 2, 2, 6, 40), (3, 3, 3, 3, 40), (5, 2, 2, 2, 30)])
def test_successors_on_random_walks(pkg, R, V, L, walks, steps):
    import spec_text as S
    P = S.Pair(pkg, R, V, L)
    rng = random.Random(R * 100 + V * 10 + L)
    n = sum(P.walk(P.init_flat(), steps, rng) for _ in range(walks))
    assert n >= walks * steps // 2
    assert len([a for a in P.stats if P.stats[a]]) >= 9, dict(P.stats)


def test_recovery_actions_of_the_oracle_against_the_text(pkg):
    """RestartEmptyLimit = 1: RestartEmpty, ReceivesRecoveryMsg, ReceivesRecoveryResponseMsg, CompleteRecovery
    (VSR.tla:813-894) — the product refuses this constant, but the oracle restates the actions; here they meet the text"""
    import spec_text as S
    P = S.Pair(pkg, 3, 1, 1, restart=1)
    rng = random.Random(11)
    pref = ("RestartEmpty", "ReceivesRecoveryMsg", "ReceivesRecoveryResponseMsg", "CompleteRecovery")
    n = sum(P.walk(P.init_flat(), 40, rng, prefer=pref) for _ in range(8))
    assert n >= 100
    for a in pref:
        assert P.stats[a] > 0, (a, dict(P.stats))


def test_cfg2_counterexample_is_a_behaviour_of_the_spec_text(pkg):
    """The shipped VSR.cfg constants (R=3, 2 values, limit 2) violate AcknowledgedWriteNotLost at depth 28 — a finding of
    this repo, smaller than the model the spec's header calls the smallest known.  Independent of the oracle and the GPU:
    a behaviour of VSR.tla's text with exactly the action names of profiles/cfg2_counterexample exists and ends in a state
    that violates the spec's own definition of the invariant."""
    import spec_text as S
    acts = json.load(open(os.path.join(ROOT, "profiles", "cfg2_counterexample", "counterexample_actions.json")))["actions"]
    path = S.from_text("behaviour/cfg2/" + S.digest(["%d %s" % x for x in enumerate(acts)]),
                       lambda: S.behaviour(S.evaluator(3, 2, 2), acts[1:], "AcknowledgedWriteNotLost"))
    assert path is not None and len(path) == 28
    assert path[-2][1] and not path[-1][1]
    # the oracle finds the same behaviour
    assert S.behaviour(S.OracleEvaluator(pkg, 3, 2, 2), acts[1:], "AcknowledgedWriteNotLost") == path


def test_cfg3_counterexample_of_the_gpu_run_is_a_behaviour_of_the_spec_text(pkg):
    """README constants on 4 GPUs (profiles/cfg3_counterexample): violation at depth 24, the length of the published trace;
    a behaviour of the text with the GPU run's action names exists and ends with v1 acknowledged and every log empty"""
    import spec_text as S
    acts = json.load(open(os.path.join(ROOT, "profiles", "cfg3_counterexample", "counterexample_actions.json")))["actions"]
    path = S.from_text("behaviour/cfg3/" + S.digest(["%d %s" % x for x in enumerate(acts)]),
                       lambda: S.behaviour(S.evaluator(3, 3, 3), acts[1:], "AcknowledgedWriteNotLost"))
    assert path is not None and len(path) == 24
    assert all(ok for _, ok in path[:-1]) and not path[-1][1]
    assert S.behaviour(S.OracleEvaluator(pkg, 3, 3, 3), acts[1:], "AcknowledgedWriteNotLost") == path


@pytest.mark.parametrize("R,V,L,walks,steps", [(3, 2, 2, 5, 40), (3, 3, 3, 3, 40), (2, 3, 2, 3, 30)])
def test_product_host_next_against_the_text_directly(pkg, R, V, L, walks, steps):
    """No oracle in between: the PRODUCT's packed successor function (vsr_successors: canonical value labels, one successor
    standing for `mult` bindings under SYMMETRY) against the text, orbit by orbit.  Both sides are reduced to the smallest
    relabelling of the whole state (aux variables included) under Permutations(Values)."""
    import collections
    import itertools
    import spec_text as S
    T = S.T
    ev = S.evaluator(R, V, L)
    mc = pkg.ModelChecker.from_constants(R, V, L)  # SYMMETRY on
    vals = [T.ModelValue("v%d" % (i + 1)) for i in range(V)]  # the evaluator's Values
    perms = [dict(zip(vals, p)) for p in itertools.permutations(vals)]

    def relabel(v, pi):
        if isinstance(v, T.ModelValue):
            return pi.get(v, v)
        if isinstance(v, frozenset):
            return frozenset(relabel(x, pi) for x in v)
        if isinstance(v, T.Fn):
            return T.Fn({relabel(k, pi): relabel(x, pi) for k, x in v.d.items()})
        return v

    def orbit(st):
        f = T.Fn(dict(st))
        return min((relabel(f, pi) for pi in perms), key=T.vkey)
    rng = random.Random(R + 10 * V + 100 * L)
    compared = 0
    for _ in range(walks):
        state = mc.init_state()
        for _ in range(steps):
            py = T.parse_state_record(mc.to_tla(state))
            want = S.from_text("orbit_successors/%d,%d,%d/%s" % (R, V, L, S.state_key(py)),
                               lambda: S.successors_digest(collections.Counter((a, orbit(sp)) for a, sp in ev.successors(py))))
            got = collections.Counter()
            succ = mc.successors(state)
            for sb, act, mult in succ:
                got[(S.ACTIONS[act], orbit(T.parse_state_record(mc.to_tla(sb))))] += mult
            assert S.successors_digest(got) == want, {k: T.fmt(v) for k, v in py.items()}
            compared += 1
            if not succ:
                break
            state = rng.choice(succ)[0]
    assert compared >= walks * steps // 2


def test_two_clients_abort_in_the_text_as_the_loader_says(pkg):
    """ClientCount = 2 is refused by the loader with "TLC aborts on m.commit" (VSR.tla:421): executing the text confirms
    it — the first ReceivePrepareMsg evaluates the non-existent record field"""
    import spec_text as S

    def first_error():
        ev = S.T.load_vsr(S.SPEC, 3, 2, ["v1"], 1)
        frontier = ev.initial_states()
        try:
            for _ in range(4):
                frontier = [sp for st in frontier for _, sp in ev.successors(st)][:300]
        except S.T.EvalError as e:
            return str(e)
        return None
    assert re.search("has no field commit", S.from_text("two_clients_error", first_error) or "")
    with pytest.raises(pkg.VsrError, match="m.commit"):
        pkg.ModelChecker.from_cfg_text(pkg.cfg_text(3, ["v1"], 1).replace("ClientCount = 1", "ClientCount = 2"))


def test_oracle_equals_the_committed_spec_text_results():
    """runs everywhere (no reference needed): the numbers the text evaluator produced here, against the oracle"""
    fx = json.load(open(FIXTURE))
    for row in fx["state_spaces"]:
        R, V, L = row["R"], row["V"], row["L"]
        o = orc.bfs(orc.params(R, V, L, symmetry=False), workers=4, keep_trace=False, max_depth=row.get("max_depth", 0))
        n = len(row["level_sizes"])
        assert o.level_sizes[:n] == row["level_sizes"], (R, V, L)
        assert o.level_generated[:len(row["level_generated"])] == row["level_generated"], (R, V, L)
        if row["complete"]:
            assert (o.distinct, o.generated, o.depth) == (row["distinct"], row["generated"], row["depth"])

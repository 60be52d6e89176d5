"""The four ways to run the BFS on one GPU — ModelChecker.check (vsr_bfs), check(collect_levels=True), check_multi(1) and
dist.GpuEngine(world 1).run — drive the same level loop, vsr_bfs_sharded on a one-rank engine.  They must report the same
exploration, verdict and statistics for every way a search can end: complete, bounded by depth, at a violation (stopping
there or continuing past it), at a deadlock, and on a capacity overflow.  Their counterexamples have the same length and each
is a behaviour of Next from Init to the first violating (or a terminal) state.  Which of several equally short behaviours is
reported depends on the order the GPU's threads append states to a level, so two runs of the same path may differ there.
A one-rank checkpoint is the file at the given path, and a checkpoint written through one entry point continues through
another."""
import os

import pytest

import orc

pytestmark = pytest.mark.gpu

CAPS = dict(table_capacity=1 << 22, frontier_capacity=1 << 20)
INV2 = ("AcknowledgedWritesExistOnMajority",)


@pytest.fixture(scope="module")
def vdist(pkg):
    from vsr_tlaplus_b200 import dist
    return dist


def violated(pkg, mc, trace):
    mask = mc.invariant(trace[-1][1]) if trace else 0
    return [n for n, b in pkg.checker.INVARIANT_BITS.items() if mask & b]


def assert_counterexample(pkg, lit, trace, rc):
    """a behaviour of Next from Init, in literal states of `lit` (the model without SYMMETRY), that ends in the first state
    violating an invariant (rc 12) or in a state without successors (rc 11)"""
    assert trace[0] == ("Initial predicate", lit.init_state())
    for (_, a), (name, b) in zip(trace, trace[1:]):
        assert (b, name) in [(t, pkg.ACTION_NAMES[act]) for t, act, _ in lit.successors(a)]
    if rc == 12:
        assert lit.invariant(trace[-1][1]) != 0 and all(lit.invariant(st) == 0 for _, st in trace[:-1])
    else:
        assert lit.successors(trace[-1][1]) == []


def checker_outcome(res):
    return dict(rc=res.rc, generated=res.generated, distinct=res.distinct, queue=res.queue, depth=res.depth, complete=res.complete,
                level_sizes=res.level_sizes, level_generated=res.level_generated, violation_level=res.violation_level,
                violated_invariants=res.violated_invariants, h2_ties=res.h2_ties, fp_collisions=res.fp_collisions,
                kernel_launches=res.kernel_launches, trace=res.trace)


def four_paths(pkg, vdist, mc, deadlock=False, stop_on_violation=True, max_depth=0, caps=CAPS, lit=None):
    """outcome of each path, level_generated cut to the levels the search expanded; `lit` checks the counterexamples"""
    kw = dict(deadlock=deadlock, stop_on_violation=stop_on_violation, max_depth=max_depth, **caps)
    out = {"check": checker_outcome(mc.check(**kw)),
           "check(collect_levels)": checker_outcome(mc.check(collect_levels=True, **kw)),
           "check_multi(1)": checker_outcome(mc.check_multi(1, **kw))}
    eng = vdist.GpuEngine(mc, 0, 1, check_deadlock=deadlock, **caps)
    try:
        r = eng.run(max_depth=max_depth, stop_on_violation=stop_on_violation)
    finally:
        eng.close()
    trace = vdist.replay_trace(mc, r.trace_cands) if r.rc in (11, 12) or r.violation_level else []
    out["GpuEngine.run"] = dict(rc=r.rc, generated=r.generated, distinct=r.distinct, queue=r.queue, depth=r.depth, complete=r.complete,
                                level_sizes=r.level_sizes, level_generated=r.level_generated, violation_level=r.violation_level,
                                violated_invariants=violated(pkg, mc, trace), h2_ties=r.h2_ties, fp_collisions=r.fp_collisions,
                                kernel_launches=r.launches, trace=trace)
    expanded = len(r.level_generated)
    for o in out.values():
        o["level_generated"] = o["level_generated"][:expanded]
    first = out["check"]
    for name, o in out.items():
        for key in first:
            if key != "trace":
                assert o[key] == first[key], f"{name} and check() differ in {key}"
        assert len(o["trace"]) == len(first["trace"]), f"{name} and check() differ in the counterexample's length"
        if o["trace"]:
            assert_counterexample(pkg, lit, o["trace"], o["rc"])
    return first


def test_complete_small_space(pkg, vdist):
    o = four_paths(pkg, vdist, pkg.ModelChecker.from_constants(2, 1, 1))
    assert (o["rc"], o["complete"], o["generated"], o["distinct"], o["depth"]) == (0, True, 100, 76, 14)


def test_complete_space_without_symmetry(pkg, vdist):
    o = four_paths(pkg, vdist, pkg.ModelChecker.from_constants(3, 2, 1, symmetry=False), caps=dict(table_capacity=1 << 21, frontier_capacity=1 << 18))
    assert (o["rc"], o["complete"], o["distinct"], o["generated"], o["depth"]) == (0, True, 697364, 1831657, 30)  # pinned to the spec's text


@pytest.mark.parametrize("stop_on_violation", [True, False])
def test_violation_reports_the_first_violating_level(pkg, vdist, stop_on_violation):
    """whether the search stops at the violation or continues past it, the counterexample ends at the first violating depth"""
    mc = pkg.ModelChecker.from_constants(3, 2, 1, invariants=INV2)
    lit = pkg.ModelChecker.from_constants(3, 2, 1, symmetry=False, invariants=INV2)
    o = four_paths(pkg, vdist, mc, stop_on_violation=stop_on_violation, lit=lit)
    ref = orc.bfs(orc.params(3, 2, 1, invariant=2), workers=8, keep_trace=False, check_assumptions=False)
    assert o["rc"] == 12 == ref.rc and o["violation_level"] == ref.depth == len(o["trace"])
    assert o["violated_invariants"] == list(INV2)
    assert o["complete"] == (not stop_on_violation)


def test_bounded_depth(pkg, vdist):
    o = four_paths(pkg, vdist, pkg.ModelChecker.from_constants(3, 2, 2), max_depth=12)
    assert o["rc"] == 0 and o["depth"] == 12 and not o["complete"] and o["queue"] == o["level_sizes"][-1]


def test_deadlock(pkg, vdist):
    """VSR.tla has terminal states (DESIGN §5): with deadlock checking on the search stops at the first one, with a trace to it"""
    o = four_paths(pkg, vdist, pkg.ModelChecker.from_constants(2, 1, 1), deadlock=True, lit=pkg.ModelChecker.from_constants(2, 1, 1, symmetry=False))
    ref = orc.bfs(orc.params(2, 1, 1, symmetry=False), workers=1, check_deadlock=True, keep_trace=False)
    assert o["rc"] == 11 == ref.rc and o["depth"] == ref.depth and o["trace"]


def test_frontier_overflow(pkg, vdist):
    o = four_paths(pkg, vdist, pkg.ModelChecker.from_constants(3, 2, 2), max_depth=12, caps=dict(table_capacity=1 << 20, frontier_capacity=256))
    assert o["rc"] == 152 and not o["complete"]


def test_one_rank_checkpoint_is_the_plain_path_and_resumes_through_either_entry_point(pkg, vdist, tmp_path):
    mc = pkg.ModelChecker.from_constants(3, 2, 1, symmetry=False)
    caps = dict(table_capacity=1 << 21, frontier_capacity=1 << 18)
    whole = mc.check(stop_on_violation=False, **caps)
    a, b = str(tmp_path / "check.ckpt"), str(tmp_path / "engine.ckpt")
    assert mc.check(stop_on_violation=False, max_depth=17, checkpoint_path=a, checkpoint_seconds=1e9, **caps).depth == 17
    eng = vdist.GpuEngine(mc, 0, 1, **caps)
    try:
        assert eng.run(stop_on_violation=False, max_depth=17, checkpoint_path=b, checkpoint_seconds=1e9).depth == 17
        for p in (a, b):
            assert os.path.exists(p) and not os.path.exists(p + ".rank0")
        from_check = eng.run(stop_on_violation=False, recover_path=a)
    finally:
        eng.close()
    from_engine = mc.check(stop_on_violation=False, recover_path=b, **caps)
    for r in (from_check, from_engine):
        assert (r.rc, r.complete, r.generated, r.distinct, r.queue, r.depth) == (whole.rc, whole.complete, whole.generated, whole.distinct, whole.queue, whole.depth)
        assert r.level_sizes == whole.level_sizes and r.violation_level == whole.violation_level
        assert r.level_generated[:whole.depth - 1] == whole.level_generated[:whole.depth - 1]

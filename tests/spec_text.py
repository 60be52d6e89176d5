"""Helpers for tests/test_spec_text.py: the upstream VSR.tla executed by oracle/tla_eval.py, side by side with the
C++ oracle.  States travel between the two as text: the oracle prints a state (TLC value syntax), tla_eval parses it.

The spec text is not part of this repository.  Where VSR_TLAPLUS_DIR names a vsr-tlaplus checkout the tests execute it;
everywhere else they compare the oracle with what executing it gave, stored in tests/golden/spec_text_recorded.json
(written by tests/golden/make_spec_text_recorded.py).  Every such result goes through from_text()."""
import collections
import ctypes as C
import hashlib
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import tla_eval as T  # noqa: E402
import orc  # noqa: E402

_UPSTREAM = os.environ.get("VSR_TLAPLUS_DIR")
SPEC = os.path.join(_UPSTREAM, "vsr-revisited", "paper", "VSR.tla") if _UPSTREAM else None
LIVE = bool(SPEC and os.path.exists(SPEC))
RECORDED_PATH = os.path.join(ROOT, "tests", "golden", "spec_text_recorded.json")
RECORDED = {}
if not LIVE and os.path.exists(RECORDED_PATH):
    with open(RECORDED_PATH) as _f:
        RECORDED = json.load(_f)
ACTIONS = ["Initial predicate", "TimerSendSVC", "ReceiveHigherSVC", "ReceiveMatchingSVC", "SendDVC", "ReceiveHigherDVC",
           "ReceiveMatchingDVC", "SendSV", "ReceiveSV", "ReceiveClientRequest", "ReceivePrepareMsg", "ReceivePrepareOkMsg",
           "ExecuteOp", "SendGetState", "ReceiveGetState", "ReceiveNewState", "RestartEmpty", "ReceivesRecoveryMsg",
           "ReceivesRecoveryResponseMsg", "CompleteRecovery"]


def from_text(key, derive):
    """a result of executing the spec text: derive() it where the text is available (and remember it, so that
    make_spec_text_recorded.py can store it), else the stored one"""
    if LIVE:
        if key not in RECORDED:  # a state met again on a walk: the text gives the same answer
            RECORDED[key] = derive()
        return RECORDED[key]
    assert key in RECORDED, ("%s was not recorded from the spec text: rerun tests/golden/make_spec_text_recorded.py with the "
                             "vsr-tlaplus checkout (the walk or the oracle changed)" % key)
    return RECORDED[key]


def digest(items):
    """order-free 64-bit digest of a collection of strings"""
    return hashlib.sha256("\n".join(sorted(items)).encode()).hexdigest()[:16]


def state_key(st):
    """digest of a state (dict variable -> value), independent of how it was printed"""
    return digest([repr(T.vkey(T.Fn(dict(st))))])


def successors_digest(counter):
    """digest of a multiset of (action, state as T.Fn)"""
    return digest("%s %d %s" % (a, n, repr(T.vkey(s))) for (a, s), n in counter.items())


def evaluator(R, V, L, restart=0):
    """the spec text bound to the constants; None where the text is not available"""
    return T.load_vsr(SPEC, R, 1, ["v%d" % (i + 1) for i in range(V)], L, restart) if LIVE else None


def to_py(q, flat):
    return T.parse_state_record(orc.print_flat(q, flat))


class Pair:
    """one configuration: the text evaluator and the oracle (symmetry off: literal successors on both sides)"""

    def __init__(self, pkg, R, V, L, restart=0):
        self.Flat = pkg.checker.VsrFlatState
        self.ev = evaluator(R, V, L, restart)
        self.tag = "%d,%d,%d,%d" % (R, V, L, restart)
        self.q = orc.params(R, V, L, symmetry=False, restart=restart)
        self.q_awem = orc.params(R, V, L, symmetry=False, invariant=2, restart=restart)
        self.stats = collections.Counter()
        self.choose_retries = 0

    def init_flat(self):
        f = self.Flat()
        orc.lib().orc_init_flat(self.q, C.byref(f))
        return f

    def oracle_successors(self, flat, cap=512):
        out = (self.Flat * cap)()
        acts = (C.c_int * cap)()
        n = orc.lib().orc_successors_flat(self.q, C.byref(flat), out, acts, cap)
        assert 0 <= n <= cap, n
        return [(ACTIONS[acts[i]], out[i]) for i in range(n)]

    def compare(self, flat):
        """successors of one state from the text and from the oracle, as multisets of (action, whole next state);
        also the two safety invariants on the state itself.  Returns the oracle's successor flats."""
        st = to_py(self.q, flat)
        osucc = self.oracle_successors(flat)
        want = collections.Counter((a, T.Fn(to_py(self.q, f))) for a, f in osucc)
        text = from_text("successors/%s/%s" % (self.tag, state_key(st)), lambda: self._text_successors(st, want))
        if text["successors"] != successors_digest(want):
            raise AssertionError("successors differ from the text's\nstate: %s\n%s" % ({k: T.fmt(v) for k, v in st.items()}, text.get("diff", "")))
        for a, _ in osucc:
            self.stats[a] += 1
        assert text["AcknowledgedWriteNotLost"] == bool(orc.lib().orc_invariant_flat(self.q, C.byref(flat)))
        assert text["AcknowledgedWritesExistOnMajority"] == bool(orc.lib().orc_invariant_flat(self.q_awem, C.byref(flat)))
        return osucc

    def text_holds(self, name, flat):
        st = to_py(self.q, flat)
        return from_text("successors/%s/%s" % (self.tag, state_key(st)), lambda: self._text_successors(st, None))[name]

    def _text_successors(self, st, want):
        pick, got = 0, None
        while True:
            self.ev.choose_pick, self.ev.choose_log = pick, []
            got = collections.Counter((a, T.Fn(sp)) for a, sp in self.ev.successors(st))
            ambiguous = bool(self.ev.choose_log)
            if want is None or got == want or not ambiguous or pick >= 3:
                break
            pick += 1  # the result depended on which maximal DVC a CHOOSE took: try the others (TLC's order is not known here)
        self.ev.choose_pick = 0
        if pick and got == want:
            self.choose_retries += 1
        out = {"successors": successors_digest(got), "AcknowledgedWriteNotLost": bool(self.ev.holds("AcknowledgedWriteNotLost", st)),
               "AcknowledgedWritesExistOnMajority": bool(self.ev.holds("AcknowledgedWritesExistOnMajority", st))}
        if want is not None and got != want:
            out["diff"] = "only from the text: %s\nonly from the oracle: %s" % ([(a, T.fmt(s)) for (a, s) in (got - want)][:3],
                                                                                [(a, T.fmt(s)) for (a, s) in (want - got)][:3])
        return out

    def walk(self, flat, steps, rng, prefer=()):
        """compare along a random walk; `prefer` = actions taken whenever enabled (to reach rare neighbourhoods)"""
        n = 0
        for _ in range(steps):
            succ = self.compare(flat)
            n += 1
            if not succ:
                break
            pref = [f for a, f in succ if a in prefer]
            flat = rng.choice(pref) if pref and rng.random() < 0.7 else rng.choice(succ)[1]
        return n


def follow(P, flat, actions):
    """depth-first: a path from `flat` whose steps carry the given action names (every state on the way is compared);
    returns the flats of the path or None"""
    succ = P.compare(flat)
    if not actions:
        return [flat]
    for a, f in succ:
        if a == actions[0]:
            r = follow(P, f, actions[1:])
            if r:
                return [flat] + r
    return None


def find_behaviour(ev, actions, invariant):
    """depth-first search for a behaviour of the module whose i-th step is an `actions[i]` step and whose last state
    violates `invariant`; returns the list of states or None"""
    init = ev.initial_states()[0]
    dead = set()

    def rec(st, i, path):
        if i == len(actions):
            return path if not ev.holds(invariant, st) else None
        key = (i, T.Fn(st))
        if key in dead:
            return None
        for a, sp in ev.successors(st):
            if a == actions[i]:
                r = rec(sp, i + 1, path + [sp])
                if r:
                    return r
        dead.add(key)
        return None
    return rec(init, 0, [init])


class _OracleState(dict):
    __slots__ = ("flat",)


class OracleEvaluator:
    """the oracle behind the evaluator interface find_behaviour() uses (SYMMETRY off: literal successors)"""

    def __init__(self, pkg, R, V, L):
        self.P = Pair(pkg, R, V, L)

    def _state(self, flat):
        st = _OracleState(to_py(self.P.q, flat))
        st.flat = flat
        return st

    def initial_states(self):
        return [self._state(self.P.init_flat())]

    def successors(self, st):
        return [(a, self._state(f)) for a, f in self.P.oracle_successors(st.flat)]

    def holds(self, name, st):
        assert name == "AcknowledgedWriteNotLost"
        return bool(orc.lib().orc_invariant_flat(self.P.q, C.byref(st.flat)))


def behaviour(ev, actions, invariant):
    """find_behaviour() as JSON: the states' digests and the invariant's verdict on each"""
    path = find_behaviour(ev, actions, invariant)
    return None if path is None else [[state_key(st), bool(ev.holds(invariant, st))] for st in path]

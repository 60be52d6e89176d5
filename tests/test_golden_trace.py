"""The reference's only golden vector — state_transfer_violation_trace.txt, 24 states — against the oracle
(pins the oracle) and against the product's packed Next (pins the product to the same vector)."""
import base64
import ctypes as C
import json
import os
import re
import zlib

import pytest

import orc
from conftest import REF_TRACE

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = os.path.join(HERE, "golden", "state_transfer_trace.json")

# SURVEY §4 / Appendix A: the action of each of the 23 transitions
EXPECTED_ACTIONS = [
    "Initial predicate", "ReceiveClientRequest", "TimerSendSVC", "TimerSendSVC", "ReceivePrepareMsg", "ReceivePrepareOkMsg",
    "ExecuteOp", "ReceiveClientRequest", "ReceiveHigherSVC", "ReceiveMatchingSVC", "SendDVC", "TimerSendSVC", "SendDVC",
    "ReceiveMatchingDVC", "SendSV", "ReceiveClientRequest", "SendGetState", "ReceiveHigherSVC", "ReceiveMatchingSVC", "SendDVC",
    "SendDVC", "ReceiveMatchingDVC", "SendSV", "ReceiveSV"]


def load_fixture(pkg):
    Flat = pkg.checker.VsrFlatState
    with open(FIXTURE) as f:
        fx = json.load(f)
    assert fx["flat_state_bytes"] == C.sizeof(Flat), "VsrFlatState layout changed: regenerate tests/golden (make_trace_fixture.py)"
    states = [Flat.from_buffer_copy(zlib.decompress(base64.b64decode(s["flat_zlib_b64"]))) for s in fx["states"]]
    return fx, states


def test_fixture_shape(pkg):
    fx, states = load_fixture(pkg)
    assert len(states) == 24
    assert [s["action"] for s in fx["states"]] == EXPECTED_ACTIONS
    assert fx["constants"] == {"ReplicaCount": 3, "ClientCount": 1, "Values": 3, "StartViewOnTimerLimit": 3, "RestartEmptyLimit": 0}


def test_oracle_replays_golden_trace(pkg):
    """every consecutive pair is a step of the oracle's Next with the recorded action; the last state violates
    AcknowledgedWriteNotLost and no earlier one does"""
    fx, states = load_fixture(pkg)
    Flat = pkg.checker.VsrFlatState
    q = orc.params(3, 3, 3, symmetry=False)
    L = orc.lib()
    for i in range(23):
        cap = 128
        succ = (Flat * cap)()
        acts = (C.c_int * cap)()
        n = L.orc_successors_flat(q, C.byref(states[i]), succ, acts, cap)
        want = orc.digests_full_of(q, (Flat * 1)(states[i + 1]))[0]
        got = orc.digests_full_of(q, succ)[:n]
        assert any(g == want and pkg.ACTION_NAMES[acts[k]] == EXPECTED_ACTIONS[i + 1] for k, g in enumerate(got)), f"transition {i + 1}->{i + 2}"
    for i in range(23):
        assert L.orc_invariant_flat(q, C.byref(states[i])) == 1
    assert L.orc_invariant_flat(q, C.byref(states[23])) == 0
    for s in states:
        assert L.orc_check_assumptions_flat(q, C.byref(s)) == 0


def test_product_next_replays_golden_trace(pkg):
    """the packed, hand-lowered Next: pack each golden state, its successors (literal value names) contain the next
    golden state with the recorded action; invariant verdicts as in the file"""
    fx, states = load_fixture(pkg)
    mc = pkg.ModelChecker.from_cfg_text(pkg.cfg_text(3, ["v1", "v2", "v3"], 3, symmetry=False))
    packed = [mc.pack(s) for s in states]
    assert packed[0] == mc.init_state()
    for i in range(23):
        succ = mc.successors(packed[i])
        hits = [a for (t, a, m) in succ if t == packed[i + 1]]
        assert hits and pkg.ACTION_NAMES[hits[0]] == EXPECTED_ACTIONS[i + 1], f"transition {i + 1}->{i + 2}"
    assert [mc.invariant(p) for p in packed] == [0] * 23 + [1]
    # unpack(pack(x)) is the same TLA+ state
    q = orc.params(3, 3, 3, symmetry=False)
    Flat = pkg.checker.VsrFlatState
    for s, p in zip(states, packed):
        a = orc.digests_full_of(q, (Flat * 1)(s))[0]
        b = orc.digests_full_of(q, (Flat * 1)(mc.unpack(p)))[0]
        assert a == b


def test_product_symmetric_successors_cover_golden_trace(pkg):
    """with SYMMETRY on, the canonical successor set still contains (up to value permutation) each golden step"""
    fx, states = load_fixture(pkg)
    mc = pkg.ModelChecker.from_constants(3, 3, 3, symmetry=True)
    q = orc.params(3, 3, 3, symmetry=True)
    Flat = pkg.checker.VsrFlatState
    for i in range(23):
        p = mc.pack(states[i])  # canonicalises
        succ = mc.successors(p)
        want = orc.digests_full_of(q, (Flat * 1)(states[i + 1]))[0]
        got = orc.digests_full_of(q, (Flat * len(succ))(*[mc.unpack(t) for t, _, _ in succ]))
        assert want in got, f"transition {i + 1}->{i + 2}"


def test_product_printer_equals_oracle_printer(pkg):
    """TLC-format text of every golden state: two independent printers (product: csrc/vsr_host.cpp, oracle: tlc_text.cpp)"""
    fx, states = load_fixture(pkg)
    mc = pkg.ModelChecker.from_constants(3, 3, 3, symmetry=False)
    q = orc.params(3, 3, 3, symmetry=False)
    for s in states:
        assert mc.flat_to_tla(s) == orc.print_flat(q, s, True)


def test_oracle_printer_reproduces_reference_file_byte_for_byte(pkg):
    """parse -> print of the reference file gives the file back (17-variable form it was written in; location strings
    carried through): pins value syntax, variable order, record field order and the ordering of the message bag"""
    text = open(REF_TRACE, "rb").read()
    buf = C.create_string_buffer(1 << 20)
    n = orc.lib().orc_reprint_trace(text, 0, buf, len(buf))
    assert n > 0
    assert buf.raw[:n] == text


def test_fixture_is_current(pkg):
    """the committed fixture equals what the generating script makes from the reference file today"""
    fx, states = load_fixture(pkg)
    Flat = pkg.checker.VsrFlatState
    flats = (Flat * 64)()
    acts = (C.c_int * 64)()
    q = (C.c_int * 8)()
    n = orc.lib().orc_parse_trace(open(REF_TRACE, "rb").read(), q, flats, acts, 64)
    assert n == 24
    for i in range(n):
        assert bytes(flats[i]) == bytes(states[i])


def test_dump_trace_format_matches_reference_shape(pkg):
    """product `-dumpTrace tlc` text for the golden behaviour: same record skeleton as the reference file (the current
    spec has three more variables and other line numbers, so compare structure, not bytes; the locations the product reads
    from VSR.tla are checked in test_boundary.py::test_shipped_cfg_and_spec_load_unchanged)"""
    fx, states = load_fixture(pkg)
    mc = pkg.ModelChecker.from_cfg_text(pkg.cfg_text(3, ["v1", "v2", "v3"], 3, symmetry=False))
    trace = [(EXPECTED_ACTIONS[i], mc.pack(states[i])) for i in range(24)]
    text = mc.dump_trace_tlc(trace)
    ref = open(REF_TRACE).read()
    strip = lambda t: re.sub(r'location \|-> "[^"]*"', "location", t)
    drop = ("aux_restart |->", "rep_rec_number |->", "rep_rec_recv |->")
    ours = "\n".join(l for l in strip(text).split("\n") if not l.startswith(drop))
    assert ours == strip(ref)

#!/usr/bin/env python
"""Generates tests/golden/spec_text_results.json: what oracle/tla_eval.py derives from the TEXT of the reference's
vsr-revisited/paper/VSR.tla (read from the vsr-tlaplus checkout that VSR_TLAPLUS_DIR names).

  state_spaces   level sizes / successors generated per level / totals of breadth-first searches run by the text
                 evaluator (SYMMETRY off, VIEW on), complete for the small configurations, depth-bounded for bigger ones
  sweep          a longer successor-by-successor comparison of the C++ oracle with the text than the unit tests run:
                 states compared, mismatches (must be 0), per-action successor counts, CHOOSE picks that mattered
  cfg2_counterexample   the depth-28 AcknowledgedWriteNotLost violation of the shipped VSR.cfg constants re-found as a
                 behaviour of the text (action names of profiles/cfg2_counterexample)

tests/test_spec_text.py::test_oracle_equals_the_committed_spec_text_results checks the oracle against `state_spaces`
on every machine.

    VSR_TLAPLUS_DIR=<checkout> python tests/golden/make_spec_text_fixture.py                          # everything (about 20 minutes)
    VSR_TLAPLUS_DIR=<checkout> python tests/golden/make_spec_text_fixture.py --add-space R V L DEPTH  # one more state space (DEPTH 0 = complete)
"""
import base64
import json
import os
import random
import sys
import time
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _pkg  # noqa: E402
import spec_text as S  # noqa: E402


def space_row(R, V, L, depth):
    t = time.time()
    r = S.T.bfs(S.evaluator(R, V, L), invariant="AcknowledgedWriteNotLost", max_depth=depth, keep_levels=False)
    row = dict(R=R, V=V, L=L, max_depth=depth, complete=depth == 0, level_sizes=r["level_sizes"], level_generated=r["level_generated"],
               distinct=r["distinct"], generated=r["generated"], depth=r["depth"], violation_depth=r["violation_depth"],
               states_with_an_ambiguous_choose=r["ambiguous_choose"], seconds=round(time.time() - t, 1))
    if depth:  # the last level reached is not expanded by a depth-bounded run of the oracle: keep what both sides define
        row["level_generated"] = r["level_generated"][:len(r["level_sizes"]) - 1]
    return row


def main():
    assert S.LIVE, "set VSR_TLAPLUS_DIR to a vsr-tlaplus checkout"
    pkg = _pkg.load()
    if len(sys.argv) == 6 and sys.argv[1] == "--add-space":  # one more state space into the existing file (long runs)
        R, V, L, depth = map(int, sys.argv[2:6])
        row = space_row(R, V, L, depth)
        path = os.path.join(HERE, "spec_text_results.json")
        out = json.load(open(path))
        out["state_spaces"] = [x for x in out["state_spaces"] if (x["R"], x["V"], x["L"]) != (R, V, L)] + [row]
        json.dump(out, open(path, "w"), indent=1)
        print("added", R, V, L, row["distinct"], row["generated"], row["depth"], row["seconds"], "s")
        return
    out = {"source": "vsr-revisited/paper/VSR.tla (Vanlightly/vsr-tlaplus), executed by oracle/tla_eval.py", "state_spaces": []}
    for R, V, L, depth in [(2, 1, 1, 0), (2, 2, 1, 0), (2, 2, 2, 0), (3, 1, 1, 0), (2, 3, 2, 0), (2, 2, 3, 0), (3, 2, 1, 9), (3, 2, 2, 8), (3, 3, 3, 7), (5, 2, 2, 6)]:
        row = space_row(R, V, L, depth)
        out["state_spaces"].append(row)
        print(row["R"], row["V"], row["L"], row["distinct"], row["generated"], row["depth"], row["seconds"], "s", flush=True)

    sweep = {"configs": []}
    fx = json.load(open(os.path.join(HERE, "state_transfer_trace.json")))
    for R, V, L, restart, walks, steps in [(3, 2, 2, 0, 30, 45), (3, 3, 3, 0, 12, 45), (5, 2, 2, 0, 6, 30), (4, 2, 2, 0, 6, 30), (3, 2, 2, 1, 25, 45),
                                           (3, 1, 1, 2, 20, 45)]:
        P = S.Pair(pkg, R, V, L, restart=restart)
        rng = random.Random(1000 * R + 100 * V + 10 * L + restart)
        n = 0
        pref = ("RestartEmpty", "ReceivesRecoveryMsg", "ReceivesRecoveryResponseMsg", "CompleteRecovery") if restart else ()
        for _ in range(walks):
            n += P.walk(P.init_flat(), steps, rng, prefer=pref)
        if (R, V, L, restart) == (3, 3, 3, 0):
            for s in fx["states"]:
                f = P.Flat.from_buffer_copy(zlib.decompress(base64.b64decode(s["flat_zlib_b64"])))
                n += P.walk(f, 15, rng, prefer=("SendGetState", "ReceiveGetState", "ReceiveNewState", "ReceiveHigherDVC"))
        sweep["configs"].append(dict(R=R, V=V, L=L, RestartEmptyLimit=restart, states_compared=n, mismatches=0,
                                     successors_by_action=dict(P.stats), choose_picks_that_mattered=P.choose_retries))
        print("sweep", R, V, L, restart, n, dict(P.stats), P.choose_retries, flush=True)
    out["sweep"] = sweep

    acts = json.load(open(os.path.join(ROOT, "profiles", "cfg2_counterexample", "counterexample_actions.json")))["actions"]
    ev = S.evaluator(3, 2, 2)
    path = S.find_behaviour(ev, acts[1:], "AcknowledgedWriteNotLost")
    out["cfg2_counterexample"] = dict(constants=dict(ReplicaCount=3, Values=2, StartViewOnTimerLimit=2), actions=acts,
                                      found_as_behaviour_of_the_text=path is not None, states=len(path or []),
                                      last_state_violates_AcknowledgedWriteNotLost=bool(path) and not ev.holds("AcknowledgedWriteNotLost", path[-1]),
                                      acked_in_last_state=S.T.fmt(path[-1]["aux_client_acked"]) if path else None,
                                      logs_in_last_state=S.T.fmt(path[-1]["rep_log"]) if path else None)
    with open(os.path.join(HERE, "spec_text_results.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote spec_text_results.json")


if __name__ == "__main__":
    main()

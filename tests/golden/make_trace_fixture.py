#!/usr/bin/env python
"""Generates tests/golden/state_transfer_trace.json from the reference's only golden vector,
state_transfer_violation_trace.txt (24 states, TLC `dumpTrace tlc` text; stored unchanged beside this script).

The reference file is parsed with the oracle's TLC-value parser; each state is stored as the raw bytes
of a VsrFlatState (include/vsr_flat.h; zlib + base64, the struct is mostly zeros) next to its action
name.

    python tests/golden/make_trace_fixture.py
"""
import base64
import ctypes as C
import json
import os
import sys
import zlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import _pkg  # noqa: E402
import orc  # noqa: E402

SRC = os.path.join(HERE, "state_transfer_violation_trace.txt")


def main():
    pkg = _pkg.load()
    Flat = pkg.checker.VsrFlatState
    text = open(SRC, "rb").read()
    cap = 64
    flats = (Flat * cap)()
    acts = (C.c_int * cap)()
    q = (C.c_int * 8)()
    n = orc.lib().orc_parse_trace(text, q, flats, acts, cap)
    assert n == 24, n
    out = {
        "source": "state_transfer_violation_trace.txt (Vanlightly/vsr-tlaplus @ 7566e8af), parsed by oracle/tlc_text.cpp",
        "constants": {"ReplicaCount": q[0], "ClientCount": q[1], "Values": q[2], "StartViewOnTimerLimit": q[3], "RestartEmptyLimit": q[4]},
        "flat_state_bytes": C.sizeof(Flat),
        "states": [],
    }
    for i in range(n):
        raw = bytes(flats[i])
        out["states"].append({"position": i + 1, "action": pkg.ACTION_NAMES[acts[i]],
                              "flat_zlib_b64": base64.b64encode(zlib.compress(raw, 9)).decode()})
    with open(os.path.join(HERE, "state_transfer_trace.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", n, "states")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Generates tests/golden/spec_text_recorded.json: what oracle/tla_eval.py derives from the TEXT of the upstream
vsr-revisited/paper/VSR.tla for tests/test_spec_text.py — state-space summaries, per-state successor digests along the
tests' walks, the counterexample behaviours — so that those tests compare the oracle with the text on machines that do not
have the spec.  It runs tests/test_spec_text.py against the text and stores every result they took from it
(spec_text.from_text).

    python tests/golden/make_spec_text_recorded.py <vsr-tlaplus checkout>
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


def main():
    if len(sys.argv) != 2 or not os.path.exists(os.path.join(sys.argv[1], "vsr-revisited", "paper", "VSR.tla")):
        sys.exit(__doc__)
    os.environ["VSR_TLAPLUS_DIR"] = os.path.abspath(sys.argv[1])
    import pytest
    rc = pytest.main(["-q", "-p", "no:cacheprovider", os.path.join(ROOT, "tests", "test_spec_text.py")])
    if rc != 0:
        sys.exit("tests/test_spec_text.py failed against the spec text: nothing written")
    import spec_text
    assert spec_text.LIVE and spec_text.RECORDED
    with open(spec_text.RECORDED_PATH, "w") as f:
        json.dump(spec_text.RECORDED, f, indent=0, sort_keys=True)
        f.write("\n")
    print("wrote %s: %d results" % (spec_text.RECORDED_PATH, len(spec_text.RECORDED)))


if __name__ == "__main__":
    main()

"""The drop-in boundary (SURVEY §8b): TLC's cfg grammar, identity check of the .tla, exported C ABI, struct mirrors,
loud failure without a GPU."""
import ctypes as C
import os
import re
import subprocess

import pytest

from conftest import GOLDEN, REF_CFG, ROOT

HDR = os.path.join(ROOT, "include", "vsr_b200.h")


def test_library_exports_every_declared_symbol(pkg):
    lib = pkg.load_library()
    text = open(HDR).read()
    declared = set(re.findall(r"\b(vsr_[a-z0-9_]+)\s*\(", text))
    assert declared, "no declarations found"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/vsr_b200.h but not exported"
    assert declared == set(pkg.checker.EXPORTED_SYMBOLS)


def test_struct_mirrors_match_c_sizes(pkg, tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "vsr_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(VsrFlatState), sizeof(VsrMsg),'
                   ' sizeof(VsrModelInfo), sizeof(VsrRunOpts), sizeof(VsrStats), sizeof(VsrLevelInfo)); return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    ck = pkg.checker
    assert sizes == [C.sizeof(ck.VsrFlatState), C.sizeof(ck.VsrMsg), C.sizeof(ck.VsrModelInfo), C.sizeof(ck.VsrRunOpts),
                     C.sizeof(ck.VsrStats), C.sizeof(ck.VsrLevelInfo)]


def test_shipped_cfg_loads_unchanged(pkg):
    mc = pkg.ModelChecker.from_cfg(REF_CFG)
    i = mc.info
    assert (i.replica_count, i.client_count, i.value_count, i.start_view_on_timer_limit, i.restart_empty_limit) == (3, 1, 2, 2, 0)
    assert (i.symmetry, i.view, i.invariant, i.spec_verified) == (1, 1, 1, 0)  # no .tla given: nothing verified
    assert [bytes(i.value_names[k]).split(b"\0")[0] for k in range(2)] == [b"v1", b"v2"]
    assert i.state_bytes == 48


# The 20 VARIABLES of VSR.tla in declaration order and the 19 disjuncts of Next: what the loader checks a .tla against.
VARIABLES = ["replicas", "rep_status", "rep_log", "rep_view_number", "rep_op_number", "rep_commit_number", "rep_peer_op_number",
             "rep_client_table", "rep_last_normal_view", "rep_svc_recv", "rep_dvc_recv", "rep_sent_dvc", "rep_sent_sv",
             "rep_rec_number", "rep_rec_recv", "clients", "messages", "aux_svc", "aux_restart", "aux_client_acked"]


def stand_in_spec(pkg, module="VSR"):
    """A module with VSR.tla's outline (module name, VARIABLES, the action definitions, the disjuncts of Next, the
    definitions a cfg may name) and bodies of its own: not the spec the checker was lowered from.  Each action body is two
    lines, `    /\\ <action>_enabled` and `    /\\ UNCHANGED vars` (columns 5 to 21 of the second)."""
    lines = ["---- MODULE %s ----" % module, "EXTENDS Naturals", "VARIABLES " + ", ".join(VARIABLES), "",
             "vars == <<" + ", ".join(VARIABLES) + ">>", "", "Init == TRUE", ""]
    for a in pkg.ACTION_NAMES[1:]:
        lines += [a + " ==", "    /\\ %s_enabled" % a, "    /\\ UNCHANGED vars", ""]
    lines += ["Next =="] + ["    \\/ " + a for a in pkg.ACTION_NAMES[1:]] + [""]
    for d in ("view", "symmValues", "AcknowledgedWriteNotLost", "AcknowledgedWritesExistOnMajority", "NoLogDivergence", "TestInv"):
        lines.append(d + " == TRUE")
    return "\n".join(lines + ["===="]) + "\n"


def normalised_hash_of_refused(pkg, path):
    with pytest.raises(pkg.VsrError) as ei:
        pkg.ModelChecker.from_cfg(REF_CFG, str(path))
    assert ei.value.rc == 150 and "hand" in str(ei.value), str(ei.value)
    return re.search(r"normalised text hash ([0-9a-f]{16})", str(ei.value)).group(1)


def test_an_edited_spec_is_refused_and_comments_are_not_the_spec(pkg, tmp_path, monkeypatch):
    """Next and the invariants are hand-lowered, so a .tla whose text differs from VSR.tla must not load as "verified"
    even when it keeps the module name, the VARIABLES and the disjunct names; the text is compared after dropping
    comments, blank lines, trailing blanks and CR, and an edited definition body changes it."""
    text = stand_in_spec(pkg)
    p = tmp_path / "VSR.tla"
    p.write_text(text)
    h = normalised_hash_of_refused(pkg, p)
    p.write_text("\n".join(("\\* a comment line\n" + ln + "   \r") if i == 20 else ln + "\r" for i, ln in enumerate(text.split("\n")))
                 + "\n(* block\n (* nested *) comment *)\n\n")
    assert normalised_hash_of_refused(pkg, p) == h
    p.write_text(text.replace("AcknowledgedWriteNotLost == TRUE", "AcknowledgedWriteNotLost == TRUE \\/ FALSE"))
    assert normalised_hash_of_refused(pkg, p) != h
    # explicit override: loads, loudly, and is NOT reported as verified; the file's own hash and action locations are reported
    monkeypatch.setenv("VSR_B200_ALLOW_EDITED_SPEC", "1")
    p.write_text(text)
    mc = pkg.ModelChecker.from_cfg(REF_CFG, str(p))
    assert mc.info.spec_verified == 0
    fnv = 0xcbf29ce484222325
    for c in text.encode():
        fnv = ((fnv ^ c) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    assert mc.info.spec_hash == fnv
    lines = text.split("\n")
    for a, name in enumerate(pkg.ACTION_NAMES):
        want = "Unknown location" if a == 0 else "line %d, col 5 to line %d, col 21 of module VSR" % (
            lines.index(name + " ==") + 2, lines.index(name + " ==") + 3)
        assert mc.action_location(a) == want, name


@pytest.mark.parametrize("edit,frag", [
    (lambda t: t.replace("MODULE VSR", "MODULE VR_STATE_TRANSFER"), "MODULE VSR"),
    (lambda t: t.replace(", aux_client_acked", ""), "VARIABLES"),
    (lambda t: t.replace("    \\/ SendGetState\n", "    \\/ SendStateTransfer\n"), "disjunct"),
    (lambda t: t.replace("TestInv == TRUE\n", ""), "TestInv"),
])
def test_other_specs_are_refused_even_with_the_override(pkg, tmp_path, monkeypatch, edit, frag):
    """another module (the analysis specs are `MODULE VR_...`) or another outline is refused outright: the override only
    admits edited definition bodies"""
    p = tmp_path / "VSR.tla"
    p.write_text(edit(stand_in_spec(pkg)))
    normalised_hash_of_refused(pkg, p)
    monkeypatch.setenv("VSR_B200_ALLOW_EDITED_SPEC", "1")
    with pytest.raises(pkg.VsrError) as e:
        pkg.ModelChecker.from_cfg(REF_CFG, str(p))
    assert e.value.rc == 150 and frag in str(e.value), str(e.value)


def test_readme_constants_load(pkg, tmp_path):
    """README.md:13-18: the user edits only the constants"""
    cfg = open(REF_CFG).read().replace("Values = {v1, v2}", "Values = {v1, v2, v3}").replace("StartViewOnTimerLimit = 2", "StartViewOnTimerLimit = 3")
    p = tmp_path / "VSR.cfg"
    p.write_text(cfg)
    mc = pkg.ModelChecker.from_cfg(str(p))
    assert (mc.info.value_count, mc.info.start_view_on_timer_limit, mc.info.state_bytes) == (3, 3, 64)


@pytest.mark.parametrize("rel", ["analysis/03-state-transfer/VR_STATE_TRANSFER.cfg", "analysis/01-view-changes/VR_INC_RESEND.cfg"])
def test_analysis_cfgs_are_refused_loudly(pkg, rel):
    """the upstream analysis/ cfgs use SPECIFICATION / PROPERTY (liveness) — out of scope, must not be silently accepted"""
    with pytest.raises(pkg.VsrError) as e:
        pkg.ModelChecker.from_cfg(os.path.join(GOLDEN, os.path.basename(rel)))
    assert e.value.rc == 151


def test_cfg_grammar(pkg):
    base = pkg.cfg_text(3, ["v1", "v2"], 2)
    mc = pkg.ModelChecker.from_cfg_text(base)
    assert (mc.info.symmetry, mc.info.view, mc.info.invariant) == (1, 1, 1)
    # comments, commented-out keywords, inline comments after invariant names, no trailing newline (VSR.cfg:1,33-39)
    text = "\\* SPECIFICATION\n" + base.rstrip("\n") + "\n\\* PROPERTY\nAcknowledgedWritesExistOnMajority \\* less strict\n\\* NoLogDivergence"
    mc = pkg.ModelChecker.from_cfg_text(text)
    assert mc.info.invariant == 3
    # no SYMMETRY / VIEW lines
    mc = pkg.ModelChecker.from_cfg_text(pkg.cfg_text(3, ["a", "b"], 2, view=False, symmetry=False, invariants=["TestInv"]))
    assert (mc.info.symmetry, mc.info.view, mc.info.invariant) == (0, 0, 8)
    assert bytes(mc.info.value_names[1]).startswith(b"b")
    # a singleton Values has a trivial symmetry group
    assert pkg.ModelChecker.from_cfg_text(pkg.cfg_text(2, ["v1"], 1)).info.symmetry == 0


def test_specification_spec_is_init_next(pkg):
    """VSR.cfg's first line is a commented-out SPECIFICATION; `SPECIFICATION Spec` (VSR.tla:966: Init /\\ [][Next]_vars /\\
    WF_vars(Next)) in place of INIT/NEXT checks the same invariants over the same state graph, as in TLC"""
    base = pkg.cfg_text(3, ["v1", "v2"], 2)
    spec = base.replace("INIT Init\n", "").replace("NEXT Next\n", "SPECIFICATION Spec\n")
    assert "SPECIFICATION Spec" in spec and "INIT" not in spec
    a, b = pkg.ModelChecker.from_cfg_text(base), pkg.ModelChecker.from_cfg_text(spec)
    assert a.successors(a.init_state()) == b.successors(b.init_state())
    with pytest.raises(pkg.VsrError, match="Spec"):
        pkg.ModelChecker.from_cfg_text(spec.replace("SPECIFICATION Spec", "SPECIFICATION LivenessSpec"))


@pytest.mark.parametrize("mut,frag", [
    (lambda t: t.replace("INIT Init", "SPECIFICATION Spec\nINIT Init"), "SPECIFICATION"),
    (lambda t: t + "PROPERTY ViewChangeCompletes\n", "PROPERTY"),
    (lambda t: t + "CONSTRAINT Foo\n", "CONSTRAINT"),
    (lambda t: t.replace("ClientCount = 1", "ClientCount = 2"), "m.commit"),
    (lambda t: t.replace("RestartEmptyLimit = 0", "RestartEmptyLimit = 1"), "RestartEmptyLimit"),
    (lambda t: t.replace("    Nil = Nil\n", ""), "Nil"),
    (lambda t: t.replace("NEXT Next", "NEXT Foo"), "NEXT"),
    (lambda t: t.replace("AcknowledgedWriteNotLost", "NoSuchInvariant"), "NoSuchInvariant"),
    (lambda t: t.replace("ReplicaCount = 3", "ReplicaCount = 8"), "outside the packed encoding's range"),
    (lambda t: t.replace("    StartViewOnTimerLimit = 2\n", ""), "StartViewOnTimerLimit"),
])
def test_cfg_rejections_are_loud(pkg, mut, frag):
    with pytest.raises(pkg.VsrError) as e:
        pkg.ModelChecker.from_cfg_text(mut(pkg.cfg_text(3, ["v1", "v2"], 2)))
    assert e.value.rc == 151 and frag in str(e.value)


def test_no_gpu_means_loud_failure_not_fallback(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    mc = pkg.ModelChecker.from_constants(2, 1, 1)
    with pytest.raises(pkg.VsrError) as e:
        mc.check()
    assert e.value.rc == 153
    r = subprocess.run([os.path.join(ROOT, "vsr-tlaplus_b200", "vsrmc"), "-config", "/dev/null"], capture_output=True, text=True)
    assert r.returncode == 151


def test_init_has_the_hand_derivable_successors(pkg):
    """SURVEY §8c: Init has (R-1) + V successors, (R-1) + 1 distinct under symmetry"""
    for (R, V, L) in [(2, 1, 1), (3, 2, 2), (3, 3, 3), (5, 2, 2)]:
        mc = pkg.ModelChecker.from_constants(R, V, L, symmetry=True)
        succ = mc.successors(mc.init_state())
        assert sum(m for _, _, m in succ) == (R - 1) + V
        assert len({t for t, _, _ in succ}) == (R - 1) + 1
        mc = pkg.ModelChecker.from_constants(R, V, L, symmetry=False)
        assert len({t for t, _, _ in mc.successors(mc.init_state())}) == (R - 1) + V


def test_check_deadlock_keyword_of_the_cfg_is_honoured(pkg):
    """ADVICE round 1: CHECK_DEADLOCK FALSE in the cfg must switch deadlock checking off (TLC does), not be parsed and dropped."""
    base = pkg.cfg_text(2, ["v1"], 1)
    off = pkg.ModelChecker.from_cfg_text(base + "CHECK_DEADLOCK FALSE\n")
    on = pkg.ModelChecker.from_cfg_text(base + "CHECK_DEADLOCK TRUE\n")
    absent = pkg.ModelChecker.from_cfg_text(base)
    assert (off.info.check_deadlock, on.info.check_deadlock, absent.info.check_deadlock) == (0, 1, -1)
    assert off.run_opts().check_deadlock == 0 and on.run_opts().check_deadlock == 1 and absent.run_opts().check_deadlock == 0
    assert off.run_opts(deadlock=True).check_deadlock == 1  # an explicit argument wins, like TLC's command line over the cfg

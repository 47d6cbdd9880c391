"""Pins the oracle (oracle/tlc_oracle.py) against the only known-answer transcript the reference
holds for the hot path: README.md:267-321 (buggy pcal_intro) -- counts, trace, action locations --
and the verdict-only expectations (README.md:349-352, HourClock = 12 states)."""
import os
import tempfile

import pytest

from conftest import GOLDEN, ROOT, ref_results
from tla_rust_b200.front.spec import Model
from tla_rust_b200.front.pcal import translate_file
from tla_rust_b200.front.report import format_result
from oracle.tlc_oracle import Oracle
from test_frontend import README_BUGGY

README_TRACE = [
    dict(bob_account=10, money=(1, 10), alice_account=10, pc=("Transfer", "Transfer"), account_total=20),
    dict(bob_account=10, money=(1, 10), alice_account=10, pc=("A", "Transfer"), account_total=20),
    dict(bob_account=10, money=(1, 10), alice_account=10, pc=("A", "A"), account_total=20),
    dict(bob_account=10, money=(1, 10), alice_account=9, pc=("B", "A"), account_total=20),
    dict(bob_account=11, money=(1, 10), alice_account=9, pc=("C", "A"), account_total=20),
    dict(bob_account=11, money=(1, 10), alice_account=-1, pc=("C", "B"), account_total=20),
]
README_ACTIONS = [None, (35, 19, 40, 42), (35, 19, 40, 42), (42, 12, 45, 63), (47, 12, 50, 65), (42, 12, 45, 63)]


def _tuples(v):
    return tuple(_tuples(x) for x in v) if isinstance(v, list) else v


def test_readme_transcript_exact():
    """O1's report on the buggy pcal_intro (recorded from its source in tests/golden/reference/results.json) is the
    README's transcript: message, counts, the 6-state behaviour and its action locations; the report printer renders
    it as TLC does.  O1's sequential search is checked live on the repository's seats.tla, an assert failure as well:
    the same counts, message and behaviour length as the compiled model's sequential run on O2."""
    from tla_rust_b200.front.report import CheckResult
    rec = ref_results()["readme_buggy"]
    r = CheckResult()
    r.verdict, r.error_text = rec["verdict"], rec["error_text"]
    r.generated, r.distinct, r.queue, r.depth, r.init_states = (rec["generated"], rec["distinct"], rec["queue"],
                                                                rec["depth"], rec["init"])
    r.trace = [({k: _tuples(v) for k, v in st.items()}, _tuples(a)) for st, a in rec["trace"]]
    assert r.verdict == "assert"
    assert r.error_text == "Failure of assertion at line 16, column 4."
    assert (r.generated, r.distinct, r.queue, r.depth) == (9097, 6164, 999, 7)      # README.md:319-320
    assert [st for st, _ in r.trace] == README_TRACE                               # README.md:271-311
    assert [None if a is None else a[2] for _, a in r.trace] == README_ACTIONS      # README.md:278-306
    txt = format_result(r, rec["vars"], rec["module"])
    assert "State 6: <Action line 42, col 12 to line 45, col 63 of module pcal_intro>" in txt
    assert txt.rstrip().endswith("The depth of the complete state graph search is 7.")
    assert "9097 states generated, 6164 distinct states found, 999 states left on queue." in txt

    import shutil
    from oracle import cpu_engine
    from tla_rust_b200.checker import compile_model, encode_states
    d = tempfile.mkdtemp(prefix="tlag_t_")
    for f in ("seats.tla", "seats.cfg"):
        shutil.copy(os.path.join(ROOT, "tests", "specs", f), d)
    translate_file(os.path.join(d, "seats.tla"))
    m = Model(os.path.join(d, "seats.tla"))
    r = Oracle(m).run()
    init = m.initial_states()
    cm = compile_model(m, init)
    o2 = cpu_engine.run(cm, encode_states(cm, init), exact=True)
    assert r.verdict == "assert" and o2["verdict"] == 2
    assert r.error_text == cm.asserts[o2["detail"]][0] == "Failure of assertion at line 15, column 10."
    assert (r.generated, r.distinct, r.queue, r.depth) == (o2["generated"], o2["distinct"], o2["queue"], o2["depth"])
    assert len(r.trace) == o2["depth"] - 1 and r.trace[0][1] is None
    txt = format_result(r, m.vars, m.module_name)
    assert f"{r.generated} states generated, {r.distinct} distinct states found, {r.queue} states left on queue." in txt


def _fixture(name):
    from tla_rust_b200.compiled import load_compiled
    return load_compiled(os.path.join(GOLDEN, name + ".tlagz"))


def _o2(name):
    from oracle import cpu_engine
    cm, init, exp, info = _fixture(name)
    return exp, cpu_engine.run(cm, init, deadlock=info["deadlock"])


def _counts(r):
    return (r["verdict"], r["generated"], r["distinct"], r["depth"])


# The corpus models below are not part of this repository: their compiled form is (tests/golden/), with the result O1
# produced on their source (tests/golden/make_golden.py, tests/golden/make_reference_cases.py).  Each test checks what
# O1 recorded and the compiled model's run on ORACLE O2 against the numbers.
def test_bundled_specs_no_error():
    exp, o2 = _o2("pcal_intro")                           # README.md:349-352 "should produce no errors"
    r = exp["o1"]
    assert (r["verdict"], r["generated"], r["distinct"], r["depth"], r["init"]) == ("ok", 5850, 3800, 5, 400)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"], o2["init_states"]) == (0, 5850, 3800, 5, 400)
    exp, o2 = _o2("atomic_add")
    assert _counts(exp["o1"]) == ("ok", 7, 5, 4) and _counts(o2) == (0, 7, 5, 4)


def test_small_corpus_counts():
    exp, o2 = _o2("HourClock")
    assert (exp["o1"]["verdict"], exp["o1"]["distinct"]) == ("ok", 12) and o2["distinct"] == 12     # HourClock.tla:4-5
    exp, o2 = _o2("MCPaxos")
    assert _counts(exp["o1"]) == ("ok", 82, 25, 9) and _counts(o2) == (0, 82, 25, 9)
    r = ref_results()["o1"]["MCConsensus_nodeadlock"]
    assert not r["deadlock"] and (r["verdict"], r["distinct"], r["init"]) == ("ok", 4, 4)


def test_oracle_handles_raft_and_ssi_at_small_bounds():
    """BASELINE configs #4/#5 (raft.tla, serializableSnapshotIsolation.tla) through the front end and O1 at reduced
    bounds.  The reference holds no counts for them (parity unpinned at the TLC boundary, SURVEY §8c); these pin
    the oracle against itself: RECURSIVE operators, LAMBDA arguments, CHOOSE, bags as functions (raft.tla:117-135),
    @@ / :>, SelectSeq, CONSTRAINT semantics."""
    exp, o2 = _o2("MCssi")
    assert _counts(exp["o1"]) == ("ok", 945, 569, 9) and _counts(o2) == (0, 945, 569, 9)
    exp, o2 = _o2("MCraft")
    assert _counts(exp["o1"]) == ("ok", 6185, 694, 12) and _counts(o2) == (0, 6185, 694, 12)


# ---- the reference's SECOND known-answer transcript: AdvancedExamples/testout2 (TLC 1.57 on MCInnerSerial) ---------
def _testout2_numbers():
    t = ref_results()["testout2"]
    return t["init"], t["generated"], t["distinct"], t["queue"], t["diameter"]


def test_testout2_initial_states_match_the_front_end():
    """`Finished computing initial states: 4 distinct states generated.` (testout2:3): the initial states the front end
    computed for the compiled model"""
    import numpy as np
    cm, init, exp, info = _fixture("MCInnerSerial")
    assert len(np.unique(init.reshape(-1, cm.W), axis=0)) == exp["o2"]["levels"][0] == _testout2_numbers()[0] == 4


def test_testout2_final_counts_match_the_recorded_bytecode_run():
    """TLC: `6181 states generated, 195 distinct states found, 0 states left on queue.  The state graph has diameter
    5.` (22 h of CPU in 2001).  The AST oracle O1 cannot finish this model (a successor costs it minutes); the compiled
    model on the CPU bytecode engine O2 takes ~7 min on 8 cores, so its result is recorded in the fixture
    (tests/golden/make_golden.py) and re-run only with TLAG_SLOW=1."""
    import os
    from tla_rust_b200.compiled import load_compiled
    _init, gen, dist, queue, diam = _testout2_numbers()
    cm, init, exp, info = load_compiled(os.path.join(ROOT, "tests", "golden", "MCInnerSerial.tlagz"))
    o2 = exp["o2"]
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, gen, dist, diam) == (0, 6181, 195, 5)
    assert queue == 0 and sum(o2["levels"]) == dist and o2["levels"][0] == 4
    if os.environ.get("TLAG_SLOW"):
        from oracle import cpu_engine
        r = cpu_engine.run(cm, init, n_threads=os.cpu_count() or 1, deadlock=info["deadlock"])
        assert (r["generated"], r["distinct"], r["depth"], r["fp_xor"]) == (gen, dist, diam, o2["fp_xor"])


def test_readme_transcript_counts_from_the_bytecode_engine():
    """README.md:319-320 again, this time from the COMPILED model: the CPU bytecode engine in its sequential mode
    (one worker, FIFO order, stop at the first Assert failure) prints TLC's error-time numbers -- 9097 states
    generated, 6164 distinct, 999 left on queue, depth 7.  This pins the compiler's successor order and the
    initial-state order, not only the set of reachable states."""
    import os
    from tla_rust_b200.compiled import load_compiled
    from oracle import cpu_engine
    cm, init, exp, info = load_compiled(os.path.join(ROOT, "tests", "golden", "pcal_intro_readme_buggy.tlagz"))
    r = cpu_engine.run(cm, init, exact=True)
    assert (r["verdict"], r["generated"], r["distinct"], r["queue"], r["depth"]) == (2, 9097, 6164, 999, 7)
    assert cm.asserts[r["detail"]][0] == "Failure of assertion at line 16, column 4."

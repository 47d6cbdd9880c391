"""Dynamically-shaped values on the device (SURVEY §8a rows a4/a5: raft's message bag and history sets,
SSI's sequences / recursion): the bytecode lowering (sparse containers, partial functions, SubSeq, SelectSeq,
run-time \\X, UNION, tuple CHOOSE, unrolled RECURSIVE operators) against the AST oracle O1."""
import os

import pytest

from conftest import GOLDEN, ROOT, ref_case, ref_results
from tla_rust_b200.compiled import load_compiled
from tla_rust_b200.front.spec import Model
from tla_rust_b200.checker import compile_model, encode_states, decode_state
from tla_rust_b200.compile.types import TSparse, TPFun, TSeq
from oracle import cpu_engine
from oracle.tlc_oracle import Oracle

SPECS = os.path.join(ROOT, "tests", "specs")


def _o2(m, **kw):
    init = m.initial_states()
    cm = compile_model(m, init)
    return cm, cpu_engine.run(cm, encode_states(cm, init), deadlock=m.check_deadlock, **kw)


def _fixture_o2(name, **kw):
    """a compiled raft / SSI model (tests/golden/, tests/golden/reference/: raft.tla and serializableSnapshotIsolation.tla
    are not part of this repository) run on O2"""
    p = os.path.join(GOLDEN, name + ".tlagz")
    cm, init, exp, info = load_compiled(p) if os.path.exists(p) else ref_case(name)
    return cm, cpu_engine.run(cm, init, deadlock=info["deadlock"], **kw)


def test_containers_spec_matches_oracle():
    m = Model(os.path.join(SPECS, "Containers.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m, want_states=True, max_states=1 << 16)
    assert isinstance(cm.var_types["bag"], TSparse) and cm.var_types["bag"].vt is not None
    assert isinstance(cm.var_types["seen"], TSparse) and cm.var_types["seen"].vt is None
    assert isinstance(cm.var_types["pf"], TPFun) and isinstance(cm.var_types["q"], TSeq)
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == ("ok", 138101, 33884, 18)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 138101, 33884, 18)
    # the stored vectors decode to exactly the oracle's reachable set (canonical sparse encoding: one vector per value)
    seen = {tuple(sorted((k, repr(v)) for k, v in decode_state(cm, w).items())) for w in o2["states"][:o2["distinct"]]}
    assert len(seen) == o2["distinct"]


def test_containers_invariant_violation_depth_matches_oracle():
    import tempfile
    d = tempfile.mkdtemp(prefix="tlag_cont_")
    src = open(os.path.join(SPECS, "Containers.tla")).read()
    src = src.replace("BagOK    ==", "SeenShort == \\A s \\in seen : Len(s) <= 1\nBagOK    ==")
    open(os.path.join(d, "Containers.tla"), "w").write(src)
    open(os.path.join(d, "Containers.cfg"), "w").write(
        open(os.path.join(SPECS, "Containers.cfg")).read().replace("SeenOK", "SeenShort"))
    m = Model(os.path.join(d, "Containers.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert o1.verdict == "invariant" and o2["verdict"] == 1
    assert cm.invariants[o2["detail"]] == "SeenShort" == o1.invariant
    # invariants are evaluated when a state is expanded: the violating level may already have been expanded
    assert len(o1.trace) <= o2["depth"] <= len(o1.trace) + 1


def test_raft_small_bounds_on_bytecode_engine():
    """BASELINE config #4 at builder-chosen small bounds (the reference ships no cfg for raft.tla): O1 pins
    6185 / 694 / 12 (tests/test_oracle_golden.py); the compiled model must agree and TypeOK must hold (O1's run with
    TypeOK added to the invariants, recorded in tests/golden/reference/results.json)."""
    cm, o2 = _fixture_o2("MCraft")
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 6185, 694, 12)
    assert isinstance(cm.var_types["messages"], TSparse) and cm.var_types["messages"].cap == 3
    r = ref_results()["o1"]["MCraft_typeok"]
    assert (r["verdict"], r["distinct"]) == ("ok", 694)


def test_raft_three_servers_matches_oracle():
    cm, o2 = _fixture_o2("MCraft_s3")
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 93022, 7156, 14)


def test_raft_three_servers_larger_bounds_match_the_numbers_o1_produced():
    """3 servers, MaxTerm 3, MaxLogLen 2, MaxMessages 2, MaxClientRequests 2: O1 needs 175 s
    (run once: ok 1214920 / 91116 / 17); O2 takes 3 s."""
    cm, o2 = _fixture_o2("MCraft_s3_t3l2", n_threads=4)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 1214920, 91116, 17)


def test_raft_capacity_overflow_traps_instead_of_truncating():
    """A sparse container that is too small must stop the run with an evaluation error (verdict 4 / trap 2): MCraft.tla
    with the message bag's capacity bound MaxMessages + 1 cut to MaxMessages, compiled."""
    cm, o2 = _fixture_o2("MCraft_overflow")
    assert o2["verdict"] == 4


# ---- serializableSnapshotIsolation.tla (BASELINE config #5) on the bytecode engine -------------------------------
# Its invariants nest by-name definitions so deeply that inline expansion explodes; the compiler falls back to
# CALL/RET subroutines (one compiled copy per operator instance, static frames by call-graph level).
def test_ssi_compiles_with_subroutines_and_matches_oracle():
    import numpy as np
    from tla_rust_b200.compile.bytecode import OP
    cm, o2 = _fixture_o2("MCssi")
    ops = (cm.code & np.uint64(0xFF)).astype(int)
    assert int((ops == OP["CALL"]).sum()) > 50 and int((ops == OP["RET"]).sum()) > 10
    # O1 pins 945 / 569 / 9 for 2 transactions x 1 key with all eight invariants (tests/test_oracle_golden.py)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 945, 569, 9)


def test_ssi_two_keys_matches_the_numbers_o1_produced():
    """2 transactions x 2 keys: O1 needs 136 s (run once, numbers pinned here); O2 takes 2 s."""
    cm, o2 = _fixture_o2("MCssi_2x2", n_threads=4)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 50121, 29629, 13)


def test_ssi_three_transactions_matches_the_numbers_o1_produced():
    """3 transactions x 1 key: O1 needs 438 s (run once: ok 152554 / 90430 / 13); O2 takes 3 s."""
    cm, o2 = _fixture_o2("MCssi_3x1", n_threads=4)
    assert cm.frame_words <= 4096          # the CUDA engine's largest frame class
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 152554, 90430, 13)


def test_inline_budget_falls_back_to_subroutines(monkeypatch):
    """a budget Containers.tla exceeds when inlined (as SSI's invariants exceed the default one): the compiler falls back
    to subroutines, and the model still computes the same state space"""
    from tla_rust_b200.compile.lower import Lowering
    monkeypatch.setattr(Lowering, "CX_BUDGET", 2000)
    m = Model(os.path.join(SPECS, "Containers.tla"))
    init = m.initial_states()
    cm = compile_model(m, init)
    assert any("subroutines" in w for w in cm.warnings)
    o2 = cpu_engine.run(cm, encode_states(cm, init), deadlock=False)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 138101, 33884, 18)


def test_subroutine_mode_is_equivalent_on_models_that_also_inline():
    m = Model(os.path.join(SPECS, "Containers.tla"))
    init = m.initial_states()
    cm = compile_model(m, init, subroutines=True)
    o2 = cpu_engine.run(cm, encode_states(cm, init), deadlock=False)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 138101, 33884, 18)


def test_runtime_record_sets_and_domain_of_records():
    """[f : S, ...] with run-time components, membership in it, "f" \\in DOMAIN r on a tagged union
    (constructs of AdvancedExamples/InnerSerial.tla:5-30) -- tests/specs/RecSets.tla."""
    m = Model(os.path.join(SPECS, "RecSets.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == ("ok", 573, 169, 6)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 573, 169, 6)


def test_subsets_of_runtime_sets():
    """x' \\in SUBSET S, {R \\in SUBSET (S \\X S) : p}, \\E / \\A over it -- tests/specs/Subsets.tla."""
    m = Model(os.path.join(SPECS, "Subsets.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == ("ok", 124, 27, 4)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 124, 27, 4)


def test_pluscal_control_statements_end_to_end():
    """while / either / with / if-else / await / assert through pcal2tla, the compiler and O2 (tests/specs/loopy.tla)."""
    import shutil
    import tempfile
    from tla_rust_b200.front.pcal import translate_file
    d = tempfile.mkdtemp(prefix="tlag_loopy_")
    for f in ("loopy.tla", "loopy.cfg"):
        shutil.copy(os.path.join(SPECS, f), d)
    translate_file(os.path.join(d, "loopy.tla"))
    m = Model(os.path.join(d, "loopy.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == ("ok", 1222, 512, 11)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 1222, 512, 11)


@pytest.mark.parametrize("name,want", [("mac", ("ok", 26, 16, 7)), ("defn", ("deadlock", 17, 13, 5))])
def test_pluscal_macro_and_define_blocks(name, want):
    """macro (nested, token substitution) and define blocks of the PlusCal p-syntax (manual p.61), end to end."""
    import shutil
    import tempfile
    from tla_rust_b200.front.pcal import translate_file
    d = tempfile.mkdtemp(prefix="tlag_pc_")
    for ext in (".tla", ".cfg"):
        shutil.copy(os.path.join(SPECS, name + ext), d)
    translate_file(os.path.join(d, name + ".tla"))
    m = Model(os.path.join(d, name + ".tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == want
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == ({"ok": 0, "deadlock": 3}[want[0]],) + want[1:]


def test_subsets_of_a_runtime_set_over_a_two_word_universe():
    """Sub-mask enumeration with borrow across 32-bit words (universe 1..40) -- tests/specs/SubsetsWide.tla."""
    m = Model(os.path.join(SPECS, "SubsetsWide.tla"))
    o1 = Oracle(m).run()
    cm, o2 = _o2(m)
    assert cm.var_types["s"].size == 2
    assert (o1.verdict, o1.generated, o1.distinct, o1.depth) == ("ok", 2561, 243, 6)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, 2561, 243, 6)

"""Host logic + bytecode: compile -> ORACLE O2 (C bytecode engine on CPU) must equal ORACLE O1 (Python AST
evaluator); committed fixtures must load and reproduce their recorded counts on O2; C-ABI exports."""
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from tla_rust_b200.checker import encode_states, decode_state, pack_words, unpack_words
from tla_rust_b200.compiled import load_compiled
from tla_rust_b200.compile.types import TInt, TAtom, TRec, TSet, TFun, TTuple, TBool, Atoms, Codec
from tla_rust_b200.front.values import Fcn, ModelValue
from oracle import cpu_engine


def test_codec_roundtrip_and_ordinals():
    at = Atoms()
    cd = Codec(at)
    a1, a2 = ModelValue("a1"), ModelValue("a2")
    msg = TRec([{"type": TAtom(["1a"]), "bal": TInt(0, 1)},
                {"type": TAtom(["2b"]), "bal": TInt(0, 1), "acc": TAtom([a1, a2])}])
    assert msg.card() == 2 + 4
    vals = cd.enum(msg)
    assert [cd.ord_of(msg, v) for v in vals] == list(range(6))
    for v in vals:
        assert cd.unrep(msg, cd.rep(msg, v)) == v
    t = TFun([a1, a2], TSet(TTuple([TInt(0, 1), TBool()])))
    v = Fcn({a1: frozenset({(0, True)}), a2: frozenset()})
    assert cd.unrep(t, cd.rep(t, v)) == v


def test_fixtures_reproduce_on_cpu_engine(golden_names):
    assert "MCPaxos3" in golden_names and "pcal_intro" in golden_names
    for name in golden_names:
        cm, init, exp, info = load_compiled(os.path.join(GOLDEN, name + ".tlagz"))
        if exp["o2"]["distinct"] > 50000 or name == "MCInnerSerial":   # 195 states, but 7 minutes of CPU (TLAG_SLOW test)
            continue
        r = cpu_engine.run(cm, init, n_threads=2, deadlock=info["deadlock"])
        for k in ("verdict", "generated", "distinct", "depth", "fp_xor", "fp_sum", "levels"):
            assert r[k] == exp["o2"][k], (name, k)
        if "o1" in exp and exp["o1"]["verdict"] == "ok":
            assert (r["generated"], r["distinct"], r["depth"]) == (exp["o1"]["generated"], exp["o1"]["distinct"],
                                                                   exp["o1"]["depth"]), name
        # states decode back to TLA+ values
        st = decode_state(cm, init[0])
        assert set(st) == set(cm.vars)


def test_compile_matches_oracle_on_reference_models():
    """the corpus models compiled (tests/golden/) against the result O1 produced on their source"""
    for name, deadlock in (("MCPaxos", True), ("MCVoting", False), ("HourClock", True), ("AsynchInterface", True)):
        cm, iw, exp, info = load_compiled(os.path.join(GOLDEN, name + ".tlagz"))
        assert info["deadlock"] == deadlock
        for w in iw:
            assert (encode_states(cm, [decode_state(cm, w)])[0] == w).all()
        o2 = cpu_engine.run(cm, iw, deadlock=deadlock)
        o1 = exp["o1"]
        assert o1["verdict"] == "ok" and o2["verdict"] == 0
        assert (o1["generated"], o1["distinct"], o1["depth"]) == (o2["generated"], o2["distinct"], o2["depth"]), name


def test_pack_unpack_python_mirrors_c():
    cm, init, _, _ = load_compiled(os.path.join(GOLDEN, "pcal_intro.tlagz"))
    import ctypes as C
    L = cpu_engine.lib()
    lay = np.ascontiguousarray(cm.layout, dtype=np.int32)
    for w in init[:50]:
        frame = unpack_words(cm, w)
        st = np.zeros(cm.state_words_unpacked, dtype=np.int32)
        L.tlagcpu_unpack(lay.ctypes.data_as(C.c_void_p), lay.shape[0], np.ascontiguousarray(w).ctypes.data_as(C.c_void_p),
                         st.ctypes.data_as(C.c_void_p))
        assert st.tolist() == frame
        assert pack_words(cm, frame).tolist() == list(w)


def test_cabi_library_exports_every_declared_symbol():
    """The C-ABI library must load on a box without a GPU and export everything include/tlag.h declares."""
    import ctypes as C
    from tla_rust_b200 import engine
    if not os.path.exists(engine.LIB_PATH):
        engine.build_library()
    hdr = open(os.path.join(ROOT, "include", "tlag.h")).read()
    names = set(re.findall(r"\b(tlag_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 15
    L = C.CDLL(engine.LIB_PATH)
    for nme in names:
        assert hasattr(L, nme), nme
    assert set(engine.EXPORTS) <= names
    L.tlag_version.restype = C.c_char_p
    assert b"sm_100a" in L.tlag_version()


def test_engine_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from tla_rust_b200 import engine
    cm, init, _, _ = load_compiled(os.path.join(GOLDEN, "atomic_add.tlagz"))
    with pytest.raises(engine.EngineUnavailable):
        engine.Engine(cm)


def test_action_constraint_matches_the_ast_oracle():
    """ACTION-CONSTRAINT (cfg keyword, TLC/ConfigFileGrammar.tla:8-12): lowered as a conjunct of the in-model test after
    every completed successor; ORACLE O1 evaluates it on the AST (oracle/tlc_oracle.py: in_actions)."""
    from tla_rust_b200.front.spec import Model
    from tla_rust_b200.checker import compile_model, encode_states
    from oracle.tlc_oracle import Oracle
    spec = os.path.join(ROOT, "tests", "specs", "ActC.tla")
    m = Model(spec)
    assert [nm for nm, _, _ in m.action_constraints] == ["SmallStep"]
    o1 = Oracle(m).run()
    init = m.initial_states()
    cm = compile_model(m, init)
    o2 = cpu_engine.run(cm, encode_states(cm, init), deadlock=m.check_deadlock)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (0, o1.generated, o1.distinct, o1.depth)
    assert o1.distinct == 6 * 3                       # x stays in 0..5: the jumps to 6..8 are cut
    free = Oracle(Model(spec, cfg_text="INIT Init\nNEXT Next\nINVARIANT TypeOK\nCHECK_DEADLOCK FALSE\n")).run()
    assert free.distinct == 9 * 3 and free.generated > o1.generated

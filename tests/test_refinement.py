"""Refinement PROPERTYs (SURVEY §8f item 2): Init => Init2 and every transition satisfies [Next2]_v2.
Shipped cfgs that use it: Paxos/MCPaxos.cfg:12, MCVoting.cfg:9, HourClock/HourClock2.cfg:9."""
import os

import pytest

from conftest import GOLDEN, ROOT, ref_case, ref_results
from tla_rust_b200.compiled import load_compiled
from tla_rust_b200.front.spec import Model
from tla_rust_b200.checker import compile_model, encode_states, result_from_engine
from oracle import cpu_engine
from oracle.tlc_oracle import Oracle

SPEC = os.path.join(ROOT, "tests", "specs", "Clock3.tla")


def _model(prop):
    return Model(SPEC, cfg_text=f"SPECIFICATION Spec\nPROPERTY {prop}\n")


def test_good_property_holds_in_oracle_and_bytecode():
    m = _model("Good")
    r = Oracle(m).run()
    assert (r.verdict, r.distinct, r.generated) == ("ok", 3, 4)
    init = m.initial_states()
    cm = compile_model(m, init)
    o2 = cpu_engine.run(cm, encode_states(cm, init))
    assert (o2["verdict"], o2["distinct"], o2["generated"]) == (0, 3, 4)


def test_violated_action_property_is_reported():
    m = _model("Bad")
    r = Oracle(m).run()
    assert r.verdict == "property" and r.invariant == "Bad"
    init = m.initial_states()
    cm = compile_model(m, init)
    o2 = cpu_engine.run(cm, encode_states(cm, init))
    assert o2["verdict"] == 2
    res = result_from_engine(cm, dict(o2, queue_left=0))
    assert res.verdict == "property" and res.invariant == "Bad"


def test_initial_state_must_satisfy_the_property_init():
    m = _model("BadInit")
    assert m.check_refinement_init(m.initial_states()[0]) == "BadInit"
    assert Oracle(m).run().verdict == "property"


def test_shipped_refinement_cfgs_hold():
    """the compiled corpus models (tests/golden/) with the result O1 produced on their source"""
    res = ref_results()["o1"]
    for name, (cm, init, exp, info) in (("MCPaxos", load_compiled(os.path.join(GOLDEN, "MCPaxos.tlagz"))),
                                        ("HourClock2", ref_case("HourClock2"))):
        assert res[name]["refinements"] == 1 and info["deadlock"]
        o2 = cpu_engine.run(cm, init, deadlock=True)
        o1 = res[name]
        assert o1["verdict"] == "ok" and o2["verdict"] == 0
        assert (o1["generated"], o1["distinct"]) == (o2["generated"], o2["distinct"])

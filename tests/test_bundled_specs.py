"""Every bundled spec of the reference that has a .cfg (SURVEY §2a; north star: "bit-exact distinct-state count and
invariant verdict ... on every bundled spec"): ORACLE O1 (AST evaluator) against the compiled model run by
ORACLE O2 (C bytecode engine).  The reference holds no expected counts for these; the pinned numbers are O1's.
The models are the compiled corpus models of tests/golden/reference/ (tests/golden/make_reference_cases.py), with the
result O1 produced on their source recorded beside them.
Specs already covered by the committed GPU fixtures (MCPaxos, MCVoting, MCInnerFIFO, MCAlternatingBit, HourClock,
AsynchInterface) are in tests/test_compile_cpu.py / tests/test_gpu_parity.py."""
import os

import pytest

from conftest import ROOT, ref_case
from tla_rust_b200.front.spec import Model
from oracle import cpu_engine

V = {"ok": 0, "invariant": 1, "assert": 2, "deadlock": 3}

CASES = [
    # corpus path, (verdict, generated, distinct, depth)
    ("Paxos/MCConsensus.tla", ("deadlock", 7, 4, 1)),
    ("SpecifyingSystems/AsynchronousInterface/Channel.tla", ("ok", 30, 12, 2)),
    ("SpecifyingSystems/HourClock/HourClock2.tla", ("ok", 24, 12, 1)),
    ("SpecifyingSystems/Liveness/LiveHourClock.tla", ("ok", 24, 12, 1)),
    ("SpecifyingSystems/TLC/ABCorrectness.tla", ("ok", 36, 20, 3)),
    ("SpecifyingSystems/RealTime/MCRealTimeHourClock.tla", ("ok", 696, 216, 2)),          # [A]_v used as an action
    ("SpecifyingSystems/AdvancedExamples/MCInnerSequential.tla", ("ok", 24368, 3528, 9)),   # Seq capacity from sampling
    ("SpecifyingSystems/CachingMemory/MCInternalMemory.tla", ("ok", 21400, 4408, 10)),     # atom | record unions
    ("SpecifyingSystems/Liveness/MCLiveInternalMemory.tla", ("ok", 21400, 4408, 10)),
    ("SpecifyingSystems/CachingMemory/MCWriteThroughCache.tla", ("ok", 28170, 5196, 18)),  # recursive local function
]


def _check(name, want, n_threads=1):
    cm, init, exp, info = ref_case(name)
    o1 = exp["o1"]
    assert (o1["verdict"], o1["generated"], o1["distinct"], o1["depth"]) == want
    o2 = cpu_engine.run(cm, init, deadlock=info["deadlock"], n_threads=n_threads)
    assert (o2["verdict"], o2["generated"], o2["distinct"], o2["depth"]) == (V[want[0]],) + want[1:]
    assert (o2["fp_xor"], o2["fp_sum"], o2["levels"]) == (exp["o2"]["fp_xor"], exp["o2"]["fp_sum"], exp["o2"]["levels"])


@pytest.mark.parametrize("path,want", CASES, ids=[c[0].split("/")[-1][:-4] for c in CASES])
def test_bundled_spec_compiled_matches_oracle(path, want):
    _check(path.split("/")[-1][:-4], want)


@pytest.mark.parametrize("name", ["Assumes", "Logic"])
def test_assumption_only_modules(name):
    """No behaviour specification: TLC only evaluates the ASSUMEs (as for the corpus's PrintValues.tla and
    SimpleMath.tla); the repository's own assumption-only modules, tests/specs/."""
    m = Model(os.path.join(ROOT, "tests", "specs", name + ".tla"))
    assert all(v is True for _, v in m.check_assumes())
    assert m.next_node is None and not m.init_nodes


VARIATIONS = [
    # spec, (cfg text replacement ...), O1's counts -- other bounds than the shipped cfg, same specs
    ("FIFO/MCInnerFIFO.tla", (("qLen = 3", "qLen = 4"),), ("ok", 29100, 11640, 13)),
    ("TLC/MCAlternatingBit.tla", (("msgQLen = 2", "msgQLen = 3"),), ("ok", 2404, 372, 11)),
    ("TLC/MCAlternatingBit.tla", (("ackQLen = 2", "ackQLen = 3"),), ("ok", 2212, 344, 11)),
    ("CachingMemory/MCInternalMemory.tla", (("Adr = {a1, a2, a3}", "Adr = {a1, a2}"), ("Proc = {p1, p2}", "Proc = {p1, p2, p3}")),
     ("ok", 153916, 23544, 13)),
]
VARIATION_IDS = [c[0].split("/")[-1][:-4] + "-" + c[1][0][1].replace(" ", "") for c in VARIATIONS]


@pytest.mark.parametrize("path,subs,want", VARIATIONS, ids=VARIATION_IDS)
def test_bundled_spec_at_other_bounds(path, subs, want):
    _check(VARIATION_IDS[VARIATIONS.index((path, subs, want))], want, n_threads=2)

"""Regenerates tests/golden/reference/: the models of the tla-rust specification corpus (spacejam/tla-rust) that the CPU
tests check, in compiled form, with what the AST oracle O1 and the CPU bytecode engine O2 found on them.  The corpus
itself is not part of this repository; the tests run from these files.

    python tests/golden/make_reference_cases.py /path/to/tla-rust [--only name]

A case is either compiled from the corpus (with this repository's models/ where a case uses them) into <name>.tlagz,
run on O2 and, unless marked otherwise, on O1 (O1 and O2 must agree on the counts of a run without error), or only run
on O1.  results.json holds every O1 result, the facts of the source model a test checks (refinement PROPERTYs, size of
the SYMMETRY group), the numbers of the TLC transcript AdvancedExamples/testout2 and O1's whole report on pcal_intro.tla
with the labels A: and B: of README.md:232-236 (the run README.md:267-321 transcribes).
"""
from __future__ import annotations

import json
import os
import re
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tla_rust_b200.front.spec import Model  # noqa: E402
from tla_rust_b200.checker import compile_model, encode_states  # noqa: E402
from tla_rust_b200.compiled import save_compiled  # noqa: E402
from oracle.tlc_oracle import Oracle  # noqa: E402
from oracle import cpu_engine  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference")


def cases(ref):
    ex = ref + "/examples/"
    ss = ex + "SpecifyingSystems/"

    def cfg_sub(path, *subs):
        text = open(path).read()
        for a, b in subs:
            assert a in text, (path, a)
            text = text.replace(a, b)
        return text

    raft = ROOT + "/models/MCraft.tla"
    raft_s3 = open(ROOT + "/models/MCraft_s3.cfg").read()
    for k, v in (("MaxTerm", 3), ("MaxLogLen", 2), ("MaxClientRequests", 2)):
        raft_s3 = re.sub(rf"{k} = .*", f"{k} = {v}", raft_s3)
    # name: (tla path, Model kwargs, check deadlock (None: as the cfg says), run O1?, compile kwargs or None: O1 only)
    c = {
        # every bundled spec with a .cfg that no other fixture covers (tests/test_bundled_specs.py)
        "MCConsensus": (ex + "Paxos/MCConsensus.tla", {}, None, True, {}),
        "Channel": (ss + "AsynchronousInterface/Channel.tla", {}, None, True, {}),
        "HourClock2": (ss + "HourClock/HourClock2.tla", {}, None, True, {}),
        "LiveHourClock": (ss + "Liveness/LiveHourClock.tla", {}, None, True, {}),
        "ABCorrectness": (ss + "TLC/ABCorrectness.tla", {}, None, True, {}),
        "MCRealTimeHourClock": (ss + "RealTime/MCRealTimeHourClock.tla", {}, None, True, {}),
        "MCInnerSequential": (ss + "AdvancedExamples/MCInnerSequential.tla", {}, None, True, {}),
        "MCInternalMemory": (ss + "CachingMemory/MCInternalMemory.tla", {}, None, True, {}),
        "MCLiveInternalMemory": (ss + "Liveness/MCLiveInternalMemory.tla", {}, None, True, {}),
        "MCWriteThroughCache": (ss + "CachingMemory/MCWriteThroughCache.tla", {}, None, True, {"seq_cap": 2}),
        # ... and at other bounds than the shipped cfg
        "MCInnerFIFO-qLen=4": (ss + "FIFO/MCInnerFIFO.tla",
                               {"cfg_text": cfg_sub(ss + "FIFO/MCInnerFIFO.cfg", ("qLen = 3", "qLen = 4"))},
                               None, True, {"seq_cap": 6}),
        "MCAlternatingBit-msgQLen=3": (ss + "TLC/MCAlternatingBit.tla",
                                       {"cfg_text": cfg_sub(ss + "TLC/MCAlternatingBit.cfg", ("msgQLen = 2", "msgQLen = 3"))},
                                       None, True, {"seq_cap": 5}),
        "MCAlternatingBit-ackQLen=3": (ss + "TLC/MCAlternatingBit.tla",
                                       {"cfg_text": cfg_sub(ss + "TLC/MCAlternatingBit.cfg", ("ackQLen = 2", "ackQLen = 3"))},
                                       None, True, {"seq_cap": 5}),
        "MCInternalMemory-Adr={a1,a2}": (ss + "CachingMemory/MCInternalMemory.tla",
                                         {"cfg_text": cfg_sub(ss + "CachingMemory/MCInternalMemory.cfg",
                                                              ("Adr = {a1, a2, a3}", "Adr = {a1, a2}"),
                                                              ("Proc = {p1, p2}", "Proc = {p1, p2, p3}"))},
                                         None, True, {}),
        # Consensus has no next state: without deadlock checking its 4 initial states are the whole space
        "MCConsensus_nodeadlock": (ex + "Paxos/MCConsensus.tla", {}, False, True, None),
        # the shipped cfgs with a refinement PROPERTY (tests/test_refinement.py) and a SYMMETRY (tests/test_symmetry.py),
        # and MCVoting without its SYMMETRY
        "MCPaxos": (ex + "Paxos/MCPaxos.tla", {}, True, True, None),
        "MCVoting": (ex + "Paxos/MCVoting.tla", {}, False, True, None),
        "MCVoting_nosym": (ex + "Paxos/MCVoting.tla",
                           {"cfg_text": cfg_sub(ex + "Paxos/MCVoting.cfg", ("SYMMETRY MCSymmetry", ""))}, False, True, None),
        # raft.tla with TypeOK checked too (O1 only: TypeOK applies \\subseteq to the message bag), at MaxTerm 3 /
        # MaxLogLen 2 on 3 servers, and with a message bag one slot too small (the run must trap; tests/test_containers.py)
        "MCraft_typeok": (raft, {"extra_dirs": [ex],
                                 "cfg_text": cfg_sub(ROOT + "/models/MCraft.cfg", ("INVARIANT AtMostOneLeaderPerTerm",
                                                                                  "INVARIANT AtMostOneLeaderPerTerm TypeOK"))},
                          None, True, None),
        "MCraft_s3_t3l2": (raft, {"extra_dirs": [ex], "cfg_text": raft_s3}, None, False, {}),
        "MCraft_overflow": (raft, {"extra_dirs": [ex], "src_edit": ("<= MaxMessages + 1", "<= MaxMessages")}, None, False, {}),
    }
    return c


README_BUGGY = (("     alice_account := alice_account - money;", "     A: alice_account := alice_account - money;"),
                ("     bob_account := bob_account + money;", "     B: bob_account := bob_account + money;"))


def readme_run(ref):
    """O1 on the README's buggy pcal_intro: verdict, message, counts and the behaviour, as the report prints them"""
    import tempfile
    from tla_rust_b200.front.pcal import translate_file
    d = tempfile.mkdtemp(prefix="tlag_gold_")
    src = open(os.path.join(ref, "pcal_intro.tla")).read()
    for a, b in README_BUGGY:
        assert a in src
        src = src.replace(a, b)
    p = os.path.join(d, "pcal_intro.tla")
    open(p, "w").write(src)
    open(os.path.join(d, "pcal_intro.cfg"), "w").write("SPECIFICATION Spec\n")
    translate_file(p)
    m = Model(p)
    r = Oracle(m).run()
    return dict(r.summary(), error_text=r.error_text, vars=m.vars, module=m.module_name,
                trace=[[st, act] for st, act in r.trace])


def main():
    if len(sys.argv) < 2 or not os.path.isdir(sys.argv[1]):
        sys.exit(__doc__)
    ref = os.path.abspath(sys.argv[1])
    only = sys.argv[sys.argv.index("--only") + 1] if "--only" in sys.argv else None
    os.makedirs(OUT, exist_ok=True)
    rpath = os.path.join(OUT, "results.json")
    results = json.load(open(rpath)) if only and os.path.exists(rpath) else {"o1": {}}
    for name, (path, kw, deadlock, run_o1, ckw) in cases(ref).items():
        if only and name != only:
            continue
        t0 = time.time()
        kw = dict(kw)
        edit = kw.pop("src_edit", None)
        source = path.replace(ref, "<tla-rust>").replace(ROOT, "<repo>") + (" (edited: %s -> %s)" % edit if edit else "")
        if edit:
            import tempfile
            d = tempfile.mkdtemp(prefix="tlag_gold_")
            src = open(path).read()
            assert edit[0] in src
            open(os.path.join(d, os.path.basename(path)), "w").write(src.replace(*edit))
            cfg = path[:-4] + ".cfg"
            open(os.path.join(d, os.path.basename(cfg)), "w").write(open(cfg).read())
            path = os.path.join(d, os.path.basename(path))
        m = Model(path, **kw)
        if deadlock is not None:
            m.check_deadlock = deadlock
        m.check_assumes()
        init = m.initial_states()
        facts = {"source": source, "deadlock": m.check_deadlock, "refinements": len(m.refinements),
                 "symmetry_group": len(m.symmetry_group()) if m.cfg.symmetry else 0}
        o1 = dict(Oracle(m).run().summary()) if run_o1 else None
        if o1:
            results["o1"][name] = dict(o1, **facts)
        if ckw is not None:
            cm = compile_model(m, init, **ckw)
            iw = encode_states(cm, init)
            o2 = cpu_engine.run(cm, iw, n_threads=os.cpu_count() or 1, deadlock=m.check_deadlock, max_states=1 << 22)
            exp = {"o2": {k: o2[k] for k in ("verdict", "detail", "generated", "distinct", "depth", "init_states",
                                             "fp_xor", "fp_sum", "levels", "state_idx")}}
            if o1:
                exp["o1"] = o1
                if o1["verdict"] == "ok":
                    assert (o1["generated"], o1["distinct"], o1["depth"]) == (o2["generated"], o2["distinct"], o2["depth"]), \
                        (name, o1, exp["o2"])
            save_compiled(os.path.join(OUT, name + ".tlagz"), cm, iw, exp,
                          dict(facts, code_len=int(len(cm.code)), W=cm.W))
            print(f"{name}: W={cm.W} code={len(cm.code)} "
                  f"o2={ {k: o2[k] for k in ('verdict', 'generated', 'distinct', 'depth')} } o1={o1} ({time.time() - t0:.1f}s)",
                  flush=True)
        else:
            print(f"{name}: o1={o1} ({time.time() - t0:.1f}s)", flush=True)
    if not only:
        txt = open(ref + "/examples/SpecifyingSystems/AdvancedExamples/testout2").read()
        m1 = re.search(r"Finished computing initial states: (\d+) distinct states generated", txt)
        m2 = re.search(r"^(\d+) states generated, (\d+) distinct states found, (\d+) states left on queue\.\s*$", txt, re.M)
        m3 = re.search(r"The state graph has diameter (\d+)\.", txt)
        results["readme_buggy"] = readme_run(ref)
        results["testout2"] = {"init": int(m1.group(1)), "generated": int(m2.group(1)), "distinct": int(m2.group(2)),
                               "queue": int(m2.group(3)), "diameter": int(m3.group(1))}
    with open(rpath, "w") as f:
        json.dump(results, f, indent=1, sort_keys=True)
        f.write("\n")

if __name__ == "__main__":
    main()

"""Front end: parser over every module of the repository, cfg grammar, PlusCal translation layout, ASSUMEs."""
import glob
import os
import shutil
import tempfile

import pytest

from conftest import GOLDEN, ROOT
from tla_rust_b200.front.parser import parse_module_text, parse_expr_text, read_text
from tla_rust_b200.front.spec import parse_cfg, Model
from tla_rust_b200.front.pcal import translate_text
from tla_rust_b200.front.values import ModelValue, fmt


# the constructs of the Standard/ modules of the specification corpus that few specs use: user-defined infix and
# prefix operators (a (+) b == ..., -. a == ...) and an instance's infix operator applied qualified (a R!+ b)
OPERATOR_MODULE = r"""---------------------------- MODULE Ops ----------------------------
EXTENDS Naturals
-. a == 0 - a
a (+) b == a + b
R == INSTANCE Naturals
x == 1 R!+ 2
y == x (+) 3
=============================================================================
"""


def test_parse_whole_corpus():
    # every module of the repository (models/, the demo and test specs), and the operator forms above
    files = glob.glob(os.path.join(ROOT, "models", "**", "*.tla"), recursive=True) + \
        glob.glob(os.path.join(ROOT, "tests", "specs", "*.tla"))
    assert len(files) >= 19
    for f in files:
        parse_module_text(read_text(f))
    m = parse_module_text(OPERATOR_MODULE)
    assert m is not None


def test_junction_lists_and_precedence():
    e = parse_expr_text("/\\ a = 1\n/\\ \\/ b\n   \\/ c\n/\\ d")
    assert e.k == "and" and len(e.a[0]) == 3 and e.a[0][1].k == "or"
    e = parse_expr_text("a + b * c - d")
    # TLA+ table: `-` (11-11) binds tighter than `+` (10-10), `*` (13-13) tighter than both
    assert e.a[0] == "+" and e.a[2].a[0] == "-" and e.a[2].a[1].a[0] == "*"
    e = parse_expr_text("[f EXCEPT ![a].b = @ + 1, ![c] = 2]")
    assert e.k == "except" and len(e.a[1]) == 2
    e = parse_expr_text("{x \\in S : x > 1} \\cup {f[x] : x \\in S}")
    assert e.a[1].k == "setfilter" and e.a[2].k == "setmap"
    e = parse_expr_text("Inv!2 /\\ V!ShowsSafeAt(Q, b, v) /\\ Thm!:")
    assert [x.k for x in e.a[0][0].a[0]] + [e.a[0][1].k] == ["sel", "sel", "sel"] or e.k == "and"


def test_cfg_grammar():
    # TLC/ConfigFileGrammar.tla:8-33 + MCPaxos.cfg:9 module-scoped override + comments
    c = parse_cfg("""SPECIFICATION Spec \\* c1
    CONSTANTS a1=a1 Acceptor <- MCAcceptor N = 3 S = {x, "s", 2} (* c2 *)
      Ballot <-[Voting] MCBallot
    INVARIANT Inv1 Inv2
    PROPERTY P SYMMETRY Sym CONSTRAINT C ACTION-CONSTRAINT AC""")
    assert c.specification == "Spec" and c.invariants == ["Inv1", "Inv2"]
    assert ("a1", ModelValue("a1")) in c.const_assign and ("N", 3) in c.const_assign
    assert ("S", frozenset({ModelValue("x"), "s", 2})) in c.const_assign
    assert ("Ballot", "Voting", "MCBallot") in c.const_subst and ("Acceptor", None, "MCAcceptor") in c.const_subst
    assert c.symmetry == "Sym" and c.constraints == ["C"] and c.action_constraints == ["AC"] and c.properties == ["P"]


README_BUGGY = (("     alice_account := alice_account - money;", "     A: alice_account := alice_account - money;"),
                ("     bob_account := bob_account + money;", "     B: bob_account := bob_account + money;"))


def test_pcal_layout_matches_readme_locations():
    """The README trace names Transfer(self) as 'line 35, col 19 to line 40, col 42' etc (README.md:278-306): the
    compiled buggy pcal_intro (tests/golden/pcal_intro_readme_buggy.tlagz, translated when it was made) holds exactly
    those action locations and the assert message TLC prints.  The translator, run now on the repository's PlusCal
    specs, must put every action where the compiled fixtures of those specs recorded it, and each location must span
    the action's definition: it starts at `Name(self) ==` and ends at the last column of its last line."""
    from tla_rust_b200.compiled import load_compiled
    from tla_rust_b200.checker import compile_model
    cm, _, _, _ = load_compiled(os.path.join(GOLDEN, "pcal_intro_readme_buggy.tlagz"))
    locs = {a[0]: a[1] for a in cm.actions}
    assert (locs["Transfer"], locs["A"], locs["B"]) == ((35, 19, 40, 42), (42, 12, 45, 63), (47, 12, 50, 65))
    assert {a[0] for a in cm.asserts} == {"Failure of assertion at line 16, column 4."}
    for name in ("race", "lock"):
        out, had = translate_text(open(os.path.join(ROOT, "models", "demo", name + ".tla")).read())
        assert had
        lines = out.split("\n")
        d = tempfile.mkdtemp(prefix="tlag_layout_")
        open(os.path.join(d, name + ".tla"), "w").write(out)
        shutil.copy(os.path.join(ROOT, "models", "demo", name + ".cfg"), d)
        m = Model(os.path.join(d, name + ".tla"))
        got = compile_model(m, m.initial_states()).actions
        want, _, _, _ = load_compiled(os.path.join(GOLDEN, "demo_" + name + ".tlagz"))
        assert [(a[0], tuple(a[1])) for a in got] == [(a[0], tuple(a[1])) for a in want.actions]
        for act, (l, c, el, ec) in ((a[0], a[1]) for a in got if a[0] != "Next"):
            assert lines[l - 1].startswith(act + "(self) == ") and len(lines[l - 1]) > c
            assert len(lines[el - 1]) == ec


def test_assumes_and_printvalues():
    import io
    m = Model(os.path.join(ROOT, "tests", "specs", "Logic.tla"))
    res = m.check_assumes()
    assert len(res) == 5 and all(v is True for _, v in res)
    m = Model(os.path.join(ROOT, "tests", "specs", "Assumes.tla"))
    m.ev.out = io.StringIO()
    res = m.check_assumes()
    assert len(res) == 4 and all(v is True for _, v in res)
    assert m.ev.print_out[0] == '<<"two plus two: ", 4>>'

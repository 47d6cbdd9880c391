"""Boundary B0: the reference's Makefile flow (`make` -> `pcal2tla *tla` ; `tlc *tla`, Makefile:1-7) driven
by this repo's bin/ wrappers, on builder-authored PlusCal specs of the same shape (models/demo)."""
import os
import shutil
import subprocess
import sys
import tempfile

import pytest

from conftest import ROOT


def _run_make(target="all"):
    d = tempfile.mkdtemp(prefix="tlag_cli_")
    for f in os.listdir(os.path.join(ROOT, "models", "demo")):
        shutil.copy(os.path.join(ROOT, "models", "demo", f), d)
    env = dict(os.environ)
    env["PATH"] = os.path.join(ROOT, "bin") + os.pathsep + os.path.dirname(sys.executable) + os.pathsep + env["PATH"]
    p = subprocess.run(["make", target], cwd=d, env=env, capture_output=True, text=True, timeout=300)
    return d, p


def test_pcal2tla_in_place_translation_cfg_and_backup():
    d, p = _run_make("transpile")
    assert p.returncode == 0, p.stderr
    txt = open(os.path.join(d, "race.tla")).read()
    assert "\\* BEGIN TRANSLATION" in txt and "\\* END TRANSLATION" in txt and "Spec == Init /\\ [][Next]_vars" in txt
    assert os.path.exists(os.path.join(d, "race.old")) and os.path.exists(os.path.join(d, "lock.old"))
    # idempotent: translating again replaces the block instead of appending a second one
    _ = subprocess.run([sys.executable, os.path.join(ROOT, "bin", "pcal2tla"), os.path.join(d, "race.tla")], check=True,
                       capture_output=True)
    assert open(os.path.join(d, "race.tla")).read().count("BEGIN TRANSLATION") == 1


def test_tlc_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    d, p = _run_make("all")
    assert p.returncode != 0                       # make stops: no CPU fallback exists
    assert "CUDA" in (p.stdout + p.stderr)


@pytest.mark.gpu
def test_make_flow_on_gpu_reports_like_tlc():
    d, p = _run_make("all")
    out = p.stdout
    assert p.returncode != 0                       # race.tla violates its invariant -> make stops (Makefile:6-7)
    # lock.tla (checked first: glob order) passes
    assert "Model checking completed. No error has been found." in out
    assert "45 states generated, 26 distinct states found, 0 states left on queue." in out
    assert "The depth of the complete state graph search is 8." in out
    # race.tla: TLC-format counterexample (README.md:267-321 layout)
    assert "Error: Invariant Correct is violated." in out
    assert "State 1: <Initial predicate>" in out and "/\\ counter = 0" in out
    assert "State 5: <Action line" in out and "of module race>" in out
    assert '/\\ pc = <<"Done", "Done">>' in out and "/\\ counter = 1" in out


class _CpuShimEngine:
    """Stand-in for tla_rust_b200.engine.Engine backed by the CPU bytecode oracle: lets the CPU suite drive the
    whole `tlc` control flow (compile, report formatting, capacity retry).  Test infrastructure only."""

    def __init__(self, cm, deadlock=True, device=0, native=False, exact=False):
        self.cm, self.deadlock, self.r, self.exact = cm, deadlock, None, exact

    def seed(self, iw):
        self.iw = iw

    def result(self):
        import numpy as np
        if self.r is None:
            return {"distinct": int(len(np.unique(self.iw, axis=0))), "depth": 1}
        return self.r

    def step(self):
        from oracle import cpu_engine
        r = cpu_engine.run(self.cm, self.iw, deadlock=self.deadlock, want_states=True, max_states=1 << 17, exact=self.exact)
        self.states = r.pop("states")
        r.update(queue_left=r.get("queue", 0), device_seconds=r["seconds"])
        self.r = r
        return {"verdict": r["verdict"], "expanded": 0}

    def run(self):
        self.step()
        return self.r

    def trace(self, idx):
        import numpy as np
        return self.states[idx:idx + 1], np.array([-1])       # (the shim keeps no parent links: one-state "trace")

    def launches(self):
        return 0

    def close(self):
        pass


def test_tlc_flow_and_capacity_retry_on_cpu_shim(monkeypatch):
    import io
    import tla_rust_b200.engine as eng
    from tla_rust_b200.cli import check_file
    from tla_rust_b200.compile import types as T
    monkeypatch.setattr(eng, "Engine", _CpuShimEngine)
    spec = os.path.join(ROOT, "tests", "specs", "Containers.tla")
    # default sparse capacity too small for `seen` (two elements are reachable): one doubling 1 -> 2, then success
    monkeypatch.setattr(T, "SPARSE_CAP", 1)
    out = io.StringIO()
    rc = check_file(spec, out=out, verbose=False)
    text = out.getvalue()
    assert rc == 0, text
    assert text.count("Note: a default container capacity was exceeded") == 1
    assert "Model checking completed. No error has been found." in text
    assert "138101 states generated, 33884 distinct states found, 0 states left on queue." in text
    assert T.SPARSE_CAP == 1                      # restored


def test_demo_specs_through_tlc_flow_on_cpu_shim(monkeypatch):
    """The specs of the GPU make-flow test (models/demo), compiled by the current compiler and checked through
    check_file with the CPU shim: lock.tla passes, race.tla violates its invariant."""
    import io
    import tla_rust_b200.engine as eng
    from tla_rust_b200.cli import check_file
    from tla_rust_b200.front.pcal import translate_file
    monkeypatch.setattr(eng, "Engine", _CpuShimEngine)
    d = tempfile.mkdtemp(prefix="tlag_demo_")
    for f in ("lock.tla", "lock.cfg", "race.tla", "race.cfg"):
        shutil.copy(os.path.join(ROOT, "models", "demo", f), d)
    translate_file(os.path.join(d, "lock.tla"))
    translate_file(os.path.join(d, "race.tla"))
    out = io.StringIO()
    assert check_file(os.path.join(d, "lock.tla"), out=out, verbose=False) == 0
    assert "Model checking completed. No error has been found." in out.getvalue()
    assert "45 states generated, 26 distinct states found, 0 states left on queue." in out.getvalue()
    out = io.StringIO()
    assert check_file(os.path.join(d, "race.tla"), out=out, verbose=False) == 12
    assert "Invariant Correct is violated" in out.getvalue()
    # ./states/ (reference .gitignore:2): the report of every run, and the behaviour leading to an error
    assert "No error has been found" in open(os.path.join(d, "states", "lock.out")).read()
    assert not os.path.exists(os.path.join(d, "states", "lock.trace"))
    tr = open(os.path.join(d, "states", "race.trace")).read()
    assert tr.startswith("State 1:") and "/\\ counter" in tr


def test_config1_as_written_reference_makefile_and_specs(monkeypatch, capfd):
    """BASELINE config #1 as the reference runs it: a Makefile of the reference's shape (models/demo/Makefile:
    `pcal2tla *tla` then `tlc *tla`) over two passing PlusCal specs, one with its own .cfg (lock.tla) and one whose .cfg
    the translator writes (mac.tla: pcal_intro.tla and atomic_add.tla play these parts in the reference), copied to a
    scratch directory (pcal2tla rewrites in place) with this repo's bin/ on PATH.  `make transpile` runs as real
    processes (the translator is host code); `tlc *tla` then runs in-process with the CPU shim standing in for the GPU
    engine (the demo specs run on the device in test_make_flow_on_gpu_reports_like_tlc)."""
    import glob
    import tla_rust_b200.engine as eng
    from tla_rust_b200.cli import tlc_main
    d = tempfile.mkdtemp(prefix="tlag_ref_")
    for f in ("Makefile", "lock.tla", "lock.cfg"):
        shutil.copy(os.path.join(ROOT, "models", "demo", f), d)
    shutil.copy(os.path.join(ROOT, "tests", "specs", "mac.tla"), d)
    env = dict(os.environ)
    env["PATH"] = os.path.join(ROOT, "bin") + os.pathsep + os.path.dirname(sys.executable) + os.pathsep + env["PATH"]
    p = subprocess.run(["make", "transpile"], cwd=d, env=env, capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert os.path.exists(os.path.join(d, "mac.cfg")) and os.path.exists(os.path.join(d, "lock.old"))
    assert "BEGIN TRANSLATION" in open(os.path.join(d, "mac.tla")).read()
    # what `make test` would run: tlc *tla (glob order), stopping at the first failing module
    monkeypatch.setattr(eng, "Engine", _CpuShimEngine)
    monkeypatch.chdir(d)
    rc = tlc_main(sorted(glob.glob("*tla")))
    sys.stdout.flush()
    out = capfd.readouterr().out
    assert rc == 0, out
    assert out.count("Model checking completed. No error has been found.") == 2
    assert "45 states generated, 26 distinct states found, 0 states left on queue." in out         # lock
    assert "26 states generated, 16 distinct states found, 0 states left on queue." in out         # mac


def test_constraint_on_initial_states_and_view_warning(monkeypatch, capfd):
    """Initial states outside the CONSTRAINT are generated and counted, not explored (as TLC and ORACLE O1 do); a cfg
    VIEW is reported as not applied instead of being dropped silently."""
    import tla_rust_b200.engine as eng
    from tla_rust_b200.cli import check_file
    from tla_rust_b200.front.spec import Model
    from oracle.tlc_oracle import Oracle
    spec = os.path.join(ROOT, "tests", "specs", "Cinit.tla")
    m = Model(spec)
    o1 = Oracle(m).run()
    monkeypatch.setattr(eng, "Engine", _CpuShimEngine)
    rc = check_file(spec, verbose=False, engine="interp")
    sys.stdout.flush()
    out = capfd.readouterr().out
    assert rc == 0, out
    assert "VIEW x is not applied" in out
    assert f"{o1.generated} states generated, {o1.distinct} distinct states found, 0 states left on queue." in out


def test_error_is_replayed_sequentially_for_tlc_exact_counts(monkeypatch, capfd):
    """TLC's single worker stops at the failed assert (README.md:267-321: 9097 generated / 6164 distinct / 999 on queue
    for the buggy pcal_intro).  `tlc` finds the error with the parallel search (whole-level counts: 1729 generated /
    661 distinct on tests/specs/seats.tla, an oversold pool of seats), then replays the model as ONE sequential worker
    (TLAG_F_EXACT on the device; ORACLE O2's sequential mode behind the CPU shim here) and reports that run: the counts
    of the AST oracle's sequential search, which stops where TLC does."""
    import tla_rust_b200.engine as eng
    from tla_rust_b200.cli import check_file
    from tla_rust_b200.front.pcal import translate_file
    from tla_rust_b200.front.spec import Model
    from oracle.tlc_oracle import Oracle
    d = tempfile.mkdtemp(prefix="tlag_readme_")
    for f in ("seats.tla", "seats.cfg"):
        shutil.copy(os.path.join(ROOT, "tests", "specs", f), d)
    p = os.path.join(d, "seats.tla")
    translate_file(p)
    o1 = Oracle(Model(p)).run()
    assert o1.verdict == "assert" and (o1.generated, o1.distinct, o1.queue, o1.depth) == (1271, 582, 166, 6)
    monkeypatch.setattr(eng, "Engine", _CpuShimEngine)
    rc = check_file(p, verbose=False, engine="interp")
    sys.stdout.flush()
    out = capfd.readouterr().out
    assert rc == 12
    assert "Failure of assertion at line 15, column 10." in out
    assert "1271 states generated, 582 distinct states found, 166 states left on queue." in out
    assert "The depth of the complete state graph search is 6." in out

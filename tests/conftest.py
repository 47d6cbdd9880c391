import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# the corpus models the CPU tests check, compiled (tests/golden/make_reference_cases.py)
REF_GOLDEN = os.path.join(GOLDEN, "reference")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def ref_results():
    """what ORACLE O1 found on corpus models, the facts of their source a test checks, the TLC transcript numbers"""
    import json
    with open(os.path.join(REF_GOLDEN, "results.json")) as f:
        return json.load(f)


def ref_case(name):
    """-> (CompiledModel, init_words, expected, info) of a compiled corpus model (tests/golden/reference/)"""
    from tla_rust_b200.compiled import load_compiled
    return load_compiled(os.path.join(REF_GOLDEN, name + ".tlagz"))


@pytest.fixture(scope="session")
def golden_names():
    return sorted(f[:-6] for f in os.listdir(GOLDEN) if f.endswith(".tlagz"))

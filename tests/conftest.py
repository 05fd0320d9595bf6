import json
import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
sys.path.insert(0, os.path.join(REPO, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_cases():
    with open(os.path.join(GOLDEN, "cases.json")) as fh:
        return {c["name"]: c for c in json.load(fh)["cases"]}


def load_trace(name):
    """Rows of tests/golden/traces/<name>.tsv as dicts + header comments."""
    rows, meta = [], {"counters": []}
    with open(os.path.join(GOLDEN, "traces", name + ".tsv")) as fh:
        cols = None
        for line in fh:
            line = line.rstrip("\n")
            if line.startswith("# counter "):
                meta["counters"].append(line[len("# counter "):])
            elif line.startswith("#"):
                if "init_lnL=" in line:
                    meta["init_lnL"] = float(line.split("init_lnL=")[1])
                if line.startswith("# last_tree="):
                    meta["last_tree"] = line[len("# last_tree="):]
            elif cols is None:
                cols = line.split("\t")
            else:
                rows.append(dict(zip(cols, line.split("\t"))))
    return rows, meta


@pytest.fixture
def fake_backend(monkeypatch):
    """Route the product's host logic to the oracle-backed FakeEngine (CPU tests only)."""
    from cybayes_b200 import likelihood
    from fake_engine import FakeEngine
    likelihood.reset_engines()
    likelihood._plan_cache.clear()
    monkeypatch.setattr(likelihood, "_engine_factory", FakeEngine)
    FakeEngine.instances.clear()
    yield FakeEngine
    likelihood.reset_engines()


@pytest.fixture
def gpu_backend():
    from cybayes_b200 import likelihood
    likelihood.reset_engines()
    likelihood._plan_cache.clear()
    yield likelihood
    likelihood.reset_engines()


def run_reference_script(script_name, argv, monkeypatch, capsys):
    """Run one of the reference's unmodified, byte-compiled driver scripts (oracle/_ref/<name>.code, built by
    oracle/build_ref.sh from a CyBayes checkout; the project does not vendor the reference's code) on top of
    cybayes_b200/compat; returns its stdout."""
    import runpy
    path = os.path.join(REPO, "oracle", "_ref", script_name + ".code")
    if not os.path.exists(path):
        pytest.skip("no reference driver available (oracle/build_ref.sh)")
    monkeypatch.syspath_prepend(os.path.join(REPO, "cybayes_b200", "compat"))
    names = ("config", "utils", "mcmc_gamma", "ML_gamma", "mcmc", "ML")
    for m in names:
        monkeypatch.delitem(sys.modules, m, raising=False)
    monkeypatch.setattr(sys, "argv", [script_name + ".py"] + list(argv))
    try:
        runpy.run_path(path, run_name="__main__")
    finally:
        for m in names:
            sys.modules.pop(m, None)
    return capsys.readouterr().out


def check_nongamma_trace(out, name, rel):
    rows, meta = load_trace(name)
    gens = [l.split("\t") for l in out.splitlines() if len(l.split("\t")) == 6 and l.split("\t")[0].isdigit()]
    assert len(gens) == len(rows)
    for f, g in zip(gens, rows):
        assert (f[4], f[5], f[3]) == (g["param"], g["move"], g["TL"]), (f, g)
        for col, idx in (("state_lnL", 1), ("proposed_ll", 2)):
            want = float(g[col])
            assert abs(float(f[idx]) - want) <= rel * abs(want), (f, g)

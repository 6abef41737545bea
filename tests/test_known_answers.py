"""Known answers of the reference (benchmarks/test_list.csv, the 32 FlatZinc rows) through the
committed golden TNF fixtures.  CPU part: the oracle's root fixpoint is pinned, and the oracle finds the
reference's optimum on the instances it finishes in seconds.  GPU part: the CUDA engine reproduces
the same optimum, bit-exact root fixpoints and dive subproblems on every fixture.  (That the fixtures
are what the front-end makes of the FlatZinc sources is checked by regenerating them with
tests/golden/make_golden.py from a reference checkout.)
"""
import hashlib

import numpy as np
import pytest

from tests import golden_io

ALL = golden_io.names()
WITH_ANSWER = [n for n in ALL if golden_io.load(n)[1]["expected"] is not None]
SLOW_ON_CPU = {"triangular9", "pat12", "pat13"}


def test_fixture_inventory():
    assert len(WITH_ANSWER) == 32 and len(ALL) == 37


def sha_of(r):
    h = hashlib.sha256()
    h.update(b"F" if r["failed"] else b"-")
    if not r["failed"]:
        h.update(r["lb"].tobytes())
        h.update(r["ub"].tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("name", ALL)
def test_oracle_root_fixpoint_is_pinned(name):
    from oracle import oracle_py as orc
    pb, info = golden_io.load(name)
    assert sha_of(orc.fixpoint(pb)) == info["root_sha"]


@pytest.mark.parametrize("name", [n for n in WITH_ANSWER if n not in SLOW_ON_CPU])
def test_oracle_finds_the_reference_optimum(name):
    from oracle import oracle_py as orc
    pb, info = golden_io.load(name)
    r = orc.solve(pb, depth=4, timeout_ms=60000)
    assert r["has_solution"] and r["exhaustive"]
    assert golden_io.user_objective(info, r["lb"], r["ub"]) == info["expected"]


# ---- GPU ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", ALL)
def test_gpu_root_fixpoint_bit_exact(name):
    from oracle import oracle_py as orc
    from turbo_b200 import engine
    pb, info = golden_io.load(name)
    o = orc.fixpoint(pb)
    with engine.Solver(pb) as s:
        g = s.propagate()
    assert g["failed"] == o["failed"]
    assert np.array_equal(g["lb"], o["lb"]) and np.array_equal(g["ub"], o["ub"])
    assert sha_of(dict(failed=g["failed"], lb=g["lb"], ub=g["ub"])) == info["root_sha"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["accap_a3", "trains15", "pat1", "sudoku_opt4", "bug2", "pennies5"])
def test_gpu_dive_subproblems_bit_exact(name):
    from oracle import oracle_py as orc
    from turbo_b200 import engine
    pb, _ = golden_io.load(name)
    depth = 5
    with engine.Solver(pb) as s:
        g = s.dive_batch(0, 1 << depth, depth)
    for idx in range(1 << depth):
        o = orc.dive(pb, idx, depth)
        assert g["remaining_depth"][idx] == o["remaining_depth"] and g["leaf_kind"][idx] == o["leaf_kind"], idx
        if o["leaf_kind"] != 1:
            assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"]), idx


@pytest.mark.gpu
@pytest.mark.parametrize("name", WITH_ANSWER)
def test_gpu_finds_the_reference_optimum(name):
    """test_turbo.sh protocol (reference test_turbo.sh:34-67): the objective must equal the expected
    one unless the run timed out."""
    from turbo_b200 import engine
    from turbo_b200.model import Model
    pb, info = golden_io.load(name)
    with engine.Solver(pb, timeout_ms=60000) as s:
        g = s.solve()
    assert g["has_solution"]
    if g["exhaustive"]:
        assert golden_io.user_objective(info, g["lb"], g["ub"]) == info["expected"]
    # every reported solution is re-checked (TNF level here: the .fzn sources do not travel)
    from tests.test_oracle_ops import REL
    for p in pb.props:
        assert REL[int(p["op"])](int(g["lb"][p["x"]]), int(g["lb"][p["y"]]), int(g["lb"][p["z"]]))

"""GPU parity tests: the CUDA engine (through the C ABI) against the CPU oracle, bit for bit.

Everything here needs a B200.
"""
import numpy as np
import pytest

from tests import tnf_gen
from turbo_b200 import abi

pytestmark = pytest.mark.gpu

KINDS = [abi.MEM_TCN_SHARED, abi.MEM_STORE_SHARED, abi.MEM_GLOBAL]


@pytest.fixture(scope="module")
def eng():
    from turbo_b200 import engine
    assert engine.device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    return engine


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle_py
    return oracle_py


def assert_same_store(g, o, what):
    assert g["failed"] == o["failed"], what
    if not o["failed"]:
        bad = np.nonzero((g["lb"] != o["lb"]) | (g["ub"] != o["ub"]))[0]
        assert len(bad) == 0, (what, bad[:5], g["lb"][bad[:5]], o["lb"][bad[:5]], g["ub"][bad[:5]], o["ub"][bad[:5]])


@pytest.mark.parametrize("fp", [abi.FP_AC1, abi.FP_WAC1])
@pytest.mark.parametrize("kind", KINDS)
def test_root_fixpoint_bit_exact(eng, orc, kind, fp):
    for seed, (nv, npr) in enumerate([(8, 5), (33, 64), (100, 300), (1000, 3000), (5000, 20000), (20000, 6000)]):
        pb = tnf_gen.planted(nv, npr, seed)
        if kind == abi.MEM_TCN_SHARED and pb.nvars * 8 + pb.nprops * 8 > 200_000:
            continue
        o = orc.fixpoint(pb)
        with eng.Solver(pb, mem_kind=kind, fixpoint=fp) as s:
            assert s.config()["mem_kind"] == kind
            g = s.propagate()
        assert_same_store(g, o, (kind, fp, nv, npr))
        assert g["stats"]["num_deductions"] > 0


@pytest.mark.parametrize("kind", KINDS)
def test_failed_and_unsat_stores(eng, orc, kind):
    # no planted solution: many of these fail at the root; the failure flag must agree
    nfailed = 0
    for seed in range(30):
        pb = tnf_gen.random_net(20, 40, 500 + seed, lo=-5, hi=5)
        o = orc.fixpoint(pb)
        with eng.Solver(pb, mem_kind=kind) as s:
            g = s.propagate()
        assert_same_store(g, o, (kind, seed))
        nfailed += o["failed"]
    assert nfailed > 0


def test_batch_of_perturbed_stores(eng, orc):
    pb = tnf_gen.planted(400, 1200, 3)
    rng = np.random.default_rng(0)
    B = 64
    lb = np.tile(pb.lb, (B, 1))
    ub = np.tile(pb.ub, (B, 1))
    for b in range(B):          # random extra narrowing, sometimes inconsistent
        vs = rng.integers(3, pb.nvars, size=8)
        for v in vs:
            m = int(rng.integers(pb.lb[v], pb.ub[v] + 1))
            if rng.random() < 0.5:
                lb[b, v] = m
            else:
                ub[b, v] = m
    with eng.Solver(pb) as s:
        g = s.propagate_batch(lb, ub)
    for b in range(B):
        o = orc.fixpoint(pb, lb[b], ub[b])
        assert_same_store(dict(lb=g["lb"][b], ub=g["ub"][b], failed=bool(g["failed"][b])), o, b)


def test_infinite_and_extreme_bounds(eng, orc):
    NI, PI = abi.NEG_INF, abi.POS_INF
    big = 2 ** 31 - 2
    lb = [0, 1, 2, NI, NI, 5, big, -big, NI, 0]
    ub = [0, 1, 2, PI, 10, PI, big, -big, PI, 1]
    props = [(abi.OP_ADD, 3, 4, 5), (abi.OP_ADD, 8, 6, 6), (abi.OP_ADD, 8, 7, 7), (abi.OP_LEQ, 1, 3, 4),
             (abi.OP_LEQ, 9, 5, 4), (abi.OP_MUL, 8, 6, 2), (abi.OP_MAX, 3, 4, 5), (abi.OP_EQ, 0, 4, 5)]
    for k in range(1, len(props) + 1):
        pb = abi.Problem(lb, ub, np.array(props[:k], np.int32))
        o = orc.fixpoint(pb)
        for kind in KINDS:
            with eng.Solver(pb, mem_kind=kind) as s:
                g = s.propagate()
            assert_same_store(g, o, (k, kind))


@pytest.mark.parametrize("kind", KINDS)
def test_every_dive_subproblem_bit_exact(eng, orc, kind):
    for seed, depth in [(11, 4), (12, 6), (13, 5)]:
        strat = [(abi.VAR_INPUT_ORDER, abi.VAL_SPLIT, list(range(3, 40))), (abi.VAR_FIRST_FAIL, abi.VAL_MIN, [])]
        pb = tnf_gen.planted(120, 200, seed, strategies=strat, objective=True)
        with eng.Solver(pb, mem_kind=kind) as s:
            g = s.dive_batch(0, 1 << depth, depth)
        for idx in range(1 << depth):
            o = orc.dive(pb, idx, depth)
            assert g["remaining_depth"][idx] == o["remaining_depth"], (seed, idx)
            assert g["leaf_kind"][idx] == o["leaf_kind"], (seed, idx)
            if o["leaf_kind"] != 1:
                assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"]), (seed, idx)


@pytest.mark.parametrize("var_order", range(5))
@pytest.mark.parametrize("val_order", range(4))
def test_dive_all_orders(eng, orc, var_order, val_order):
    strat = [(var_order, val_order, list(range(3, 30))), (abi.VAR_FIRST_FAIL, abi.VAL_MIN, [])]
    pb = tnf_gen.planted(60, 90, 21, strategies=strat)
    depth = 5
    with eng.Solver(pb) as s:
        g = s.dive_batch(0, 1 << depth, depth)
    for idx in range(1 << depth):
        o = orc.dive(pb, idx, depth)
        assert g["remaining_depth"][idx] == o["remaining_depth"] and g["leaf_kind"][idx] == o["leaf_kind"]
        if o["leaf_kind"] != 1:
            assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"])


@pytest.mark.parametrize("kind", KINDS)
def test_solve_status_and_optimum(eng, orc, kind):
    nsat = 0
    for seed in range(30):
        pb = tnf_gen.search_instance(seed) if seed < 14 else tnf_gen.random_net(16, 9, 5000 + seed, lo=-4, hi=4)
        o = orc.solve(pb, depth=0)
        nsat += o["has_solution"]
        with eng.Solver(pb, mem_kind=kind, subproblems_power=4) as s:
            g = s.solve()
        assert g["exhaustive"] and o["exhaustive"]
        assert g["has_solution"] == o["has_solution"], seed
        assert g["objective"] == o["objective"], seed
        if g["has_solution"]:
            from tests.test_oracle_ops import REL
            for p in pb.props:
                assert REL[int(p["op"])](int(g["lb"][p["x"]]), int(g["lb"][p["y"]]), int(g["lb"][p["z"]]))
    assert nsat >= 14


def test_single_block_node_counts_match_oracle(eng, orc):
    """With one block the subproblems are visited in index order exactly like the oracle, so the
    whole trace (nodes, failures, solutions, skipped/solved subproblems, depth) is comparable."""
    for seed in range(12):
        pb = tnf_gen.search_instance(seed) if seed < 8 else tnf_gen.random_net(18, 10, 4000 + seed, lo=-4, hi=4)
        for depth in (0, 3):
            o = orc.solve(pb, depth=depth)
            with eng.Solver(pb, or_blocks=1, subproblems_power=depth, fixpoint=abi.FP_AC1) as s:
                g = s.solve()
            for key in ("nodes", "fails", "solutions", "eps_solved_subproblems", "eps_skipped_subproblems", "depth_max"):
                assert g["stats"][key] == o["stats"][key], (seed, depth, key, g["stats"][key], o["stats"][key])
            assert g["objective"] == o["objective"]


def test_satisfaction(eng, orc):
    pb = tnf_gen.planted(60, 80, 5, objective=False)
    with eng.Solver(pb, subproblems_power=3) as s:
        g = s.solve()
    assert g["has_solution"] and not g["exhaustive"]
    from tests.test_oracle_ops import REL
    for p in pb.props:
        assert REL[int(p["op"])](int(g["lb"][p["x"]]), int(g["lb"][p["y"]]), int(g["lb"][p["z"]]))


def test_cutnodes_and_stop(eng):
    pb = tnf_gen.planted(300, 500, 9, objective=True, slack=200)
    with eng.Solver(pb, cutnodes=50) as s:
        g = s.solve()
    assert not g["exhaustive"]
    assert g["stats"]["nodes"] <= 50 * g["stats"]["num_blocks"] + g["stats"]["num_blocks"]
    with eng.Solver(pb, timeout_ms=200) as s:
        g = s.solve()
    assert g["stats"]["timers_ns"][abi.TIMER_OVERALL] < 5e9


# ---- STORE_CLUSTER: the store striped over a thread-block cluster's distributed shared memory ---------

@pytest.mark.parametrize("csize", [2, 4, 8])
@pytest.mark.parametrize("fp", [abi.FP_AC1, abi.FP_WAC1])
def test_cluster_fixpoint_bit_exact(eng, orc, csize, fp):
    for seed, (nv, npr) in enumerate([(8, 5), (100, 300), (5000, 20000), (40000, 120000)]):
        pb = tnf_gen.planted(nv, npr, 70 + seed)
        o = orc.fixpoint(pb)
        with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=csize, fixpoint=fp) as s:
            cfg = s.config()
            assert cfg["mem_kind"] == abi.MEM_STORE_CLUSTER and cfg["cluster_size"] == csize
            g = s.propagate()
        assert_same_store(g, o, (csize, fp, nv, npr))


def test_cluster_is_chosen_when_the_store_exceeds_one_sm(eng, orc):
    pb = tnf_gen.planted(60000, 90000, 5)          # 480 KB store: does not fit 227 KB
    o = orc.fixpoint(pb)
    with eng.Solver(pb) as s:
        cfg = s.config()
        assert cfg["mem_kind"] == abi.MEM_STORE_CLUSTER and cfg["cluster_size"] == 4
        g = s.propagate()
    assert_same_store(g, o, "auto cluster")


def test_cluster_failed_stores_and_batch(eng, orc):
    for seed in range(10):
        pb = tnf_gen.random_net(20, 40, 500 + seed, lo=-5, hi=5)
        o = orc.fixpoint(pb)
        with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
            g = s.propagate()
        assert_same_store(g, o, seed)


def test_cluster_dive_and_solve(eng, orc):
    strat = [(abi.VAR_INPUT_ORDER, abi.VAL_SPLIT, list(range(3, 40))), (abi.VAR_FIRST_FAIL, abi.VAL_MIN, [])]
    pb = tnf_gen.planted(120, 200, 11, strategies=strat, objective=True)
    depth = 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=4) as s:
        g = s.dive_batch(0, 1 << depth, depth)
    for idx in range(1 << depth):
        o = orc.dive(pb, idx, depth)
        assert g["remaining_depth"][idx] == o["remaining_depth"] and g["leaf_kind"][idx] == o["leaf_kind"], idx
        if o["leaf_kind"] != 1:
            assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"]), idx
    for seed in range(8):
        pb = tnf_gen.search_instance(seed)
        o = orc.solve(pb, depth=0)
        with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2, subproblems_power=4) as s:
            g = s.solve()
        assert g["exhaustive"] and g["has_solution"] == o["has_solution"] and g["objective"] == o["objective"], seed
        with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2, or_blocks=1, subproblems_power=3, fixpoint=abi.FP_AC1) as s:
            g = s.solve()
        o = orc.solve(pb, depth=3)
        for key in ("nodes", "fails", "solutions", "eps_solved_subproblems", "eps_skipped_subproblems", "depth_max"):
            assert g["stats"][key] == o["stats"][key], (seed, key)


# ---- the layout pass specialises the device table on the root domains -------------------------------------

def test_propagate_rejects_a_store_outside_the_root(eng):
    pb = tnf_gen.planted(50, 80, 1)
    lb, ub = pb.lb.copy(), pb.ub.copy()
    v = int(np.argmax(pb.ub - pb.lb))
    ub[v] += 1
    with eng.Solver(pb) as s:
        with pytest.raises(eng.TurboError) as e:
            s.propagate(lb, ub)
        assert "root store" in str(e.value)
        s.propagate(pb.lb, pb.ub)           # the solver is still usable


@pytest.mark.parametrize("kind", KINDS)
def test_caller_store_with_an_empty_folded_constant(eng, orc, kind):
    """Variable 1 is the constant 1 and the `x` of a LEQ: the device table folds it away (class leq_t) and
    never loads it, yet a caller store in which it is empty must fail like the oracle's deduce does; an
    empty variable no propagator mentions must not."""
    lb = [0, 1, 2, 0, 0, 7]
    ub = [0, 1, 2, 9, 9, 7]
    props = np.array([(abi.OP_LEQ, 1, 3, 4), (abi.OP_ADD, 4, 3, 2)], np.int32)
    pb = abi.Problem(lb, ub, props)
    for bad, want_failed in ((1, True), (5, False)):
        l, u = pb.lb.copy(), pb.ub.copy()
        u[bad] = l[bad] - 1
        o = orc.fixpoint(pb, l, u)
        assert o["failed"] == want_failed
        with eng.Solver(pb, mem_kind=kind) as s:
            g = s.propagate(l, u)
        assert_same_store(g, o, (kind, bad))


@pytest.mark.parametrize("fp", [abi.FP_AC1, abi.FP_WAC1])
@pytest.mark.parametrize("kind", KINDS)
def test_exact_and_extended_arithmetic_classes_together(eng, orc, kind, fp):
    """Some variables get infinite or 2^30-sized bounds (extended-integer classes), the others stay small
    (32-bit classes); constants of every size; one network."""
    for seed in range(6):
        pb = tnf_gen.planted(300, 900, 900 + seed, spread=2000, slack=500,
                             mix={abi.OP_ADD: 0.4, abi.OP_LEQ: 0.2, abi.OP_EQ: 0.15, abi.OP_MIN: 0.05, abi.OP_MAX: 0.05,
                                  abi.OP_MUL: 0.05, abi.OP_TDIV: 0.05, abi.OP_TMOD: 0.05})
        rng = np.random.default_rng(seed)
        lb, ub = pb.lb.astype(np.int64), pb.ub.astype(np.int64)
        res = {int(p["x"]) for p in pb.props if int(p["op"]) in (abi.OP_EQ, abi.OP_LEQ)}
        for v in rng.choice(np.arange(3, pb.nvars), size=60, replace=False):
            if int(v) in res:
                continue
            how = rng.integers(0, 4)
            if how == 0:
                lb[v] = abi.NEG_INF
            elif how == 1:
                ub[v] = abi.POS_INF
            elif how == 2:
                lb[v], ub[v] = -(2 ** 30), 2 ** 30
            else:
                lb[v], ub[v] = abi.NEG_INF, abi.POS_INF
        big = abi.Problem(lb, ub, pb.props)
        classes = {k for k, n in eng.layout_describe(big)["classes"].items() if n}
        assert {"add_s", "add_g"} <= classes
        o = orc.fixpoint(big)
        with eng.Solver(big, mem_kind=kind, fixpoint=fp) as s:
            g = s.propagate()
        assert_same_store(g, o, (kind, fp, seed))

"""tb_solve_batch: K roots of one network (narrowings of the solver's root) searched in one launch, each as if it were
the root of its own tb_solve. The oracle is oracle_py.solve on a problem with root r's domains."""
import numpy as np
import pytest

from tests import golden_io, tnf_gen
from tools.batch_solve import make_roots, root_problem, valid
from turbo_b200 import abi

pytestmark = pytest.mark.gpu

CONFIGS = [dict(), dict(or_blocks=1, subproblems_power=0)]


@pytest.fixture(scope="module")
def eng():
    from turbo_b200 import engine
    assert engine.device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    return engine


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle_py
    return oracle_py


def network(name):
    if name == "planted_sat":
        return tnf_gen.planted(60, 80, 5, objective=False)
    if name == "planted_opt":
        return tnf_gen.search_instance(3)
    if name == "random_opt":
        return tnf_gen.random_net(16, 9, 5011, lo=-4, hi=4)
    return golden_io.load(name)[0]


def oracle_answers(orc, pb, lb, ub):
    return [orc.solve(root_problem(pb, lb[r], ub[r]), depth=0) for r in range(lb.shape[0])]


def check_against(pb, lb, ub, g, want, what):
    for r, o in enumerate(want):
        assert bool(g["has_solution"][r]) == o["has_solution"], (what, r)
        assert bool(g["exhaustive"][r]) == o["exhaustive"], (what, r)
        obj = o["objective"] if o["objective"] is not None else abi.POS_INF
        assert int(g["objective"][r]) == obj, (what, r, int(g["objective"][r]), obj)
        if o["has_solution"]:
            assert valid(pb, lb[r], ub[r], g["lb"][r], g["ub"][r]), (what, r)


@pytest.mark.parametrize("name", ["pat2", "pat10", "pat1", "sudoku_opt2", "sudoku_opt3", "pennies5", "reified_in",
                                  "planted_sat", "planted_opt", "random_opt"])
def test_every_root_equals_the_oracle(eng, orc, name):
    """Batches of 1, 7 and a few hundred roots (some empty at the root, some failing after propagation), in the default
    grid and with a single block, which must carry nothing from one root to the next."""
    pb = network(name)
    k = 64 if name in ("pat1", "pennies5") else 240
    lb, ub = make_roots(pb, k, seed=11)
    want = oracle_answers(orc, pb, lb, ub)
    assert any(o["has_solution"] for o in want)
    assert any(not o["has_solution"] for o in want) or name == "reified_in"
    for opts in CONFIGS:
        with eng.Solver(pb, **opts) as s:
            for n in (1, 7, k):
                g = s.solve_batch(lb[:n], ub[:n])
                check_against(pb, lb[:n], ub[:n], g, want[:n], (name, opts, n))
                assert g["stats"]["eps_num_subproblems"] == n << g["stats"]["subproblems_power"]


@pytest.mark.parametrize("opts", CONFIGS)
def test_no_incumbent_leaks_between_roots(eng, orc, opts):
    """Root B is root A's box with the objective at least A's optimum + k: it must report its own optimum, which an
    incumbent carried over from A would prune away."""
    for name in ("pat2", "planted_opt"):
        pb = network(name)
        a = orc.solve(pb)["objective"]
        lbs, ubs = [pb.lb.copy()], [pb.ub.copy()]
        for k in (1, 2, 3):
            lb, ub = pb.lb.copy(), pb.ub.copy()
            lb[pb.obj_var] = min(a + k, ub[pb.obj_var])
            lbs.append(lb)
            ubs.append(ub)
        lb, ub = np.stack(lbs), np.stack(ubs)
        want = oracle_answers(orc, pb, lb, ub)
        assert sum(o["has_solution"] for o in want[1:]) >= 1, name
        with eng.Solver(pb, **opts) as s:
            check_against(pb, lb, ub, s.solve_batch(lb, ub), want, (name, opts))
            # B first, then A: the order of the roots does not matter either
            check_against(pb, lb[::-1], ub[::-1], s.solve_batch(lb[::-1], ub[::-1]), want[::-1], (name, opts, "reversed"))


@pytest.mark.parametrize("opts", CONFIGS)
def test_satisfaction_stops_per_root(eng, orc, opts):
    pb = tnf_gen.planted(60, 80, 5, objective=False)
    lb, ub = make_roots(pb, 120, seed=3, nfix=4, empty_frac=0.2)
    # and roots around the planted solution with most variables fixed: searches that end on their solution
    near_lb, near_ub = make_roots(pb, 40, seed=4, around=pb.planted.astype(np.int64), free=3, empty_frac=0)
    lb, ub = np.vstack([lb, near_lb]), np.vstack([ub, near_ub])
    want = oracle_answers(orc, pb, lb, ub)
    nsat = sum(o["has_solution"] for o in want)
    assert 0 < nsat < len(want)
    with eng.Solver(pb, **opts) as s:
        g = s.solve_batch(lb, ub)
    for r, o in enumerate(want):
        assert bool(g["has_solution"][r]) == o["has_solution"], r
        if o["has_solution"]:
            assert not g["exhaustive"][r] and valid(pb, lb[r], ub[r], g["lb"][r], g["ub"][r]), r
        else:
            assert g["exhaustive"][r], r
        assert g["objective"][r] == abi.POS_INF


@pytest.mark.parametrize("opts", CONFIGS)
def test_a_solved_satisfaction_root_is_never_exhaustive(eng, orc, opts):
    """The first solution stops a satisfaction root with exhaustive = 0, as tb_solve and the oracle report it, even when
    that solution is the last node of the root's search: (a) a root fixed to a solution (propagation alone solves it),
    (b) a root whose only solution is on the last branch (x + y = 1, y <= x over 0..1: the root fixpoint prunes
    nothing, x = 0 fails, x = 1, y = 0 is the rightmost leaf)."""
    last = abi.Problem([0, 1, 2, 0, 0, 1], [0, 1, 2, 1, 1, 1], np.array([(abi.OP_ADD, 5, 3, 4), (abi.OP_LEQ, 1, 4, 3)], np.int32))
    planted = tnf_gen.planted(60, 80, 5, objective=False)
    for pb, extra in ((last, [([0, 1, 2, 1, 0, 1], [0, 1, 2, 1, 0, 1]), ([0, 1, 2, 0, 0, 1], [0, 1, 2, 0, 1, 1])]),
                      (planted, [(planted.planted, planted.planted)])):
        lb = np.vstack([pb.lb] + [np.asarray(l, np.int32) for l, _ in extra])
        ub = np.vstack([pb.ub] + [np.asarray(u, np.int32) for _, u in extra])
        want = oracle_answers(orc, pb, lb, ub)
        assert any(o["has_solution"] for o in want)
        with eng.Solver(pb, **opts) as s:
            g = s.solve_batch(lb, ub)
            for r in range(len(want)):          # each root alone too: with one root the search is the same as tb_solve's
                check_against(pb, lb[r:r + 1], ub[r:r + 1], s.solve_batch(lb[r:r + 1], ub[r:r + 1]), want[r:r + 1], (opts, r, "alone"))
        check_against(pb, lb, ub, g, want, opts)
        for r, o in enumerate(want):
            if o["has_solution"]:
                assert not g["exhaustive"][r], r


def test_copies_of_the_root_equal_solve_and_leave_solve_as_it_was(eng):
    for pb in (tnf_gen.search_instance(4), tnf_gen.planted(60, 80, 5, objective=False)):
        with eng.Solver(pb, subproblems_power=4) as s:
            before = s.solve()
            g = s.solve_batch(np.tile(pb.lb, (9, 1)), np.tile(pb.ub, (9, 1)))
            after = s.solve()
        assert before["has_solution"]
        for key in ("has_solution", "exhaustive", "objective"):
            assert before[key] == after[key], key
        assert g["has_solution"].all() and (g["exhaustive"] == before["exhaustive"]).all()
        if pb.obj_var >= 0:
            assert (g["objective"] == before["objective"]).all()
            for r in range(9):
                assert int(g["lb"][r][pb.obj_var]) == before["objective"]


def test_exhaustiveness_is_per_root_under_a_budget(eng, orc, monkeypatch):
    """Easy roots of accap_a3 next to its full root, which does not finish in a second: the easy ones are exhaustive
    with the oracle's optimum, the full one is not, and its store, if any, is a solution. The full root keeps blocks
    busy while the others wait: its subproblems are split at the tail inside the batch."""
    monkeypatch.setenv("TB_SPLIT_MIN_NODES", "256")
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    with eng.Solver(pb, timeout_ms=1000) as s:
        sol = s.solve()
    assert sol["has_solution"]
    lb, ub = make_roots(pb, 48, seed=5, around=sol["lb"].astype(np.int64), free=12)
    lb, ub = np.vstack([lb, pb.lb]), np.vstack([ub, pb.ub])
    want = oracle_answers(orc, pb, lb[:-1], ub[:-1])
    assert all(o["exhaustive"] for o in want)
    with eng.Solver(pb, timeout_ms=1000) as s:
        g = s.solve_batch(lb, ub)
    check_against(pb, lb[:-1], ub[:-1], {k: v[:-1] if k != "stats" else v for k, v in g.items()}, want, "easy roots")
    assert not g["exhaustive"][-1]
    if g["has_solution"][-1]:
        assert valid(pb, pb.lb, pb.ub, g["lb"][-1], g["ub"][-1])
        assert g["objective"][-1] == g["lb"][-1][pb.obj_var]
    assert g["stats"]["eps_split_subproblems"] > 0


@pytest.mark.parametrize("opts", CONFIGS)
def test_cut_blocks_leave_their_roots_unproven(eng, orc, opts):
    """With cutnodes a block stops; no root it was searching may report exhaustive, and every root that does report
    exhaustive has the oracle's answer."""
    pb = tnf_gen.search_instance(5)
    lb, ub = make_roots(pb, 40, seed=7, nfix=1, empty_frac=0)
    want = oracle_answers(orc, pb, lb, ub)
    with eng.Solver(pb, cutnodes=30, **opts) as s:
        g = s.solve_batch(lb, ub)
    for r, o in enumerate(want):
        if g["exhaustive"][r]:
            assert bool(g["has_solution"][r]) == o["has_solution"] and o["exhaustive"], r
            assert int(g["objective"][r]) == (o["objective"] if o["objective"] is not None else abi.POS_INF), r
    if opts:
        # one block takes the roots in order: what it proved is a prefix, and the root it was cut on is not in it
        assert not g["exhaustive"].all() and g["stats"]["nodes"] <= 30
        first_open = int(np.argmin(g["exhaustive"]))
        assert g["exhaustive"][:first_open].all() and not g["exhaustive"][first_open:].any()


def test_rejections(eng):
    pb = tnf_gen.search_instance(2)
    with eng.Solver(pb) as s:
        wide_lb, wide_ub = pb.lb.copy(), pb.ub.copy()
        wide_ub[5] += 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_batch(wide_lb[None], wide_ub[None])
        assert e.value.status == 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_batch(np.zeros((0, pb.nvars), np.int32), np.zeros((0, pb.nvars), np.int32))
        assert e.value.status == 1
        s.stream_solutions(4)
        with pytest.raises(eng.TurboError) as e:
            s.solve_batch(pb.lb[None], pb.ub[None])
        assert e.value.status == 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
        with pytest.raises(eng.TurboError) as e:
            s.solve_batch(pb.lb[None], pb.ub[None])
        assert e.value.status == 4
    a, b = eng.Solver(pb), eng.Solver(pb)
    try:
        eng.link_peers([a, b])
        with pytest.raises(eng.TurboError) as e:
            a.solve_batch(pb.lb[None], pb.ub[None])
        assert e.value.status == 4
    finally:
        a.close()
        b.close()

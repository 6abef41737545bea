"""tb_solve_groups: roots of one network gathered in groups, each group solved over the union of its roots' boxes with
one incumbent and one stop word for all of them. A group's oracle answer is the reduction of its roots' answers: any
solution, the minimum objective, exhaustive when every root is."""
import itertools

import numpy as np
import pytest

from tests import golden_io, tnf_gen
from tools.batch_solve import make_roots, referenced, root_problem, valid
from tools.group_solve import cubes, hole_boxes, with_disequality
from turbo_b200 import abi

CONFIGS = [dict(), dict(or_blocks=1, subproblems_power=0)]
NETWORKS = ["pat2", "pat10", "pat1", "sudoku_opt2", "sudoku_opt3", "pennies5", "reified_in", "planted_sat",
            "planted_opt", "random_opt"]


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


def reduce_answers(want, groups, ngroups):
    out = []
    for g in range(ngroups):
        mine = [want[r] for r in range(len(want)) if groups[r] == g]
        objs = [o["objective"] for o in mine if o["has_solution"] and o["objective"] is not None]
        out.append(dict(has_solution=any(o["has_solution"] for o in mine), exhaustive=all(o["exhaustive"] for o in mine),
                        objective=min(objs) if objs else abi.POS_INF))
    return out


def check_groups(pb, lb, ub, groups, g, want, what):
    for k, o in enumerate(want):
        assert bool(g["has_solution"][k]) == o["has_solution"], (what, k)
        assert bool(g["exhaustive"][k]) == o["exhaustive"], (what, k)
        assert int(g["objective"][k]) == o["objective"], (what, k, int(g["objective"][k]), o["objective"])
        if o["has_solution"]:
            members = np.nonzero(groups == k)[0]
            assert any(valid(pb, lb[r], ub[r], g["lb"][k], g["ub"][k]) for r in members), (what, k)
            if pb.obj_var >= 0:
                assert int(g["lb"][k][pb.obj_var]) == o["objective"], (what, k)


def scattered_groups(k, ngroups, seed):
    """Every group gets at least one root, and the roots of a group are spread over the batch."""
    return (np.random.default_rng(seed).permutation(k) % ngroups).astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NETWORKS)
def test_every_group_equals_the_reduced_oracle(eng, orc, name):
    pb = network(name)
    k = 64 if name in ("pat1", "pennies5") else 240
    lb, ub = make_roots(pb, k, seed=11)
    want = oracle_answers(orc, pb, lb, ub)
    for ngroups in (1, 5, k // 3):
        groups = scattered_groups(k, ngroups, seed=ngroups)
        red = reduce_answers(want, groups, ngroups)
        for opts in CONFIGS:
            with eng.Solver(pb, **opts) as s:
                g = s.solve_groups(lb, ub, groups)
            assert len(g["has_solution"]) == ngroups
            check_groups(pb, lb, ub, groups, g, red, (name, opts, ngroups))


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_identity_groups_equal_the_batch(eng, opts):
    for name in ("pat2", "planted_sat", "planted_opt", "random_opt"):
        pb = network(name)
        lb, ub = make_roots(pb, 120, seed=2)
        with eng.Solver(pb, **opts) as s:
            b = s.solve_batch(lb, ub)
            g = s.solve_groups(lb, ub, np.arange(lb.shape[0]))
        for key in ("has_solution", "exhaustive", "objective"):
            assert np.array_equal(b[key], g[key]), (name, opts, key)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_cubes_in_one_group_equal_solve(eng, orc, opts):
    """Cube-and-conquer: the root split into an exact partition, all cubes in one group, answers as the whole root."""
    for name in ("pat2", "sudoku_opt3", "planted_opt", "random_opt", "planted_sat"):
        pb = network(name)
        o = orc.solve(pb)
        for k in (8, 64):
            lb, ub = cubes(pb, k)
            assert lb.shape[0] > 1
            with eng.Solver(pb, **opts) as s:
                whole = s.solve()
                g = s.solve_groups(lb, ub, np.zeros(lb.shape[0], np.int32))
            assert bool(g["has_solution"][0]) == whole["has_solution"] == o["has_solution"], (name, k)
            assert bool(g["exhaustive"][0]) == whole["exhaustive"] == o["exhaustive"], (name, k)
            if pb.obj_var >= 0:
                assert int(g["objective"][0]) == whole["objective"] == o["objective"], (name, k)
            if o["has_solution"]:
                assert valid(pb, pb.lb, pb.ub, g["lb"][0], g["ub"][0]), (name, k)


def test_cubes_partition_the_root():
    """Every point of the root lies in exactly one cube (small boxes, enumerated)."""
    for seed in range(4):
        rng = np.random.default_rng(seed)
        n = 5
        lb = rng.integers(-3, 2, size=n)
        ub = lb + rng.integers(0, 4, size=n)
        lb[0] = ub[0] = 0
        props = np.array([(abi.OP_ADD, 1, 2, 3), (abi.OP_LEQ, 0, 3, 4)], np.int32)
        pb = abi.Problem(lb, ub, props, [(abi.VAR_INPUT_ORDER, abi.VAL_MIN, [4, 2])], obj_var=1)
        for k in (1, 2, 7, 16, 1000):
            clb, cub = cubes(pb, k)
            assert clb.shape[0] >= min(k, 1) and (clb <= cub).all()
            assert (clb >= pb.lb).all() and (cub <= pb.ub).all()
            for pt in itertools.product(*[range(int(a), int(b) + 1) for a, b in zip(pb.lb, pb.ub)]):
                pt = np.array(pt)
                assert ((clb <= pt) & (pt <= cub)).all(axis=1).sum() == 1, (seed, k, pt)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_a_hole_equals_the_disequality(eng, orc, opts):
    """{x <= v-1} u {x >= v+1} as one group equals the network with x != v added as TNF propagators; v is x's value
    in an optimal solution, so that the hole matters, and the returned store avoids it."""
    for name in ("planted_opt", "random_opt", "pat2"):
        pb = network(name)
        o = orc.solve(pb)
        assert o["has_solution"]
        xs = [v for v in range(pb.nvars) if pb.lb[v] < o["lb"][v] < pb.ub[v]][:3]
        assert xs, name
        for x in xs:
            v = int(o["lb"][x])
            lb, ub = hole_boxes(pb, x, v)
            want = orc.solve(with_disequality(pb, x, v))
            with eng.Solver(pb, **opts) as s:
                g = s.solve_groups(lb, ub, [0, 0])
            assert bool(g["has_solution"][0]) == want["has_solution"], (name, x)
            assert bool(g["exhaustive"][0]) == want["exhaustive"], (name, x)
            if want["has_solution"]:
                assert int(g["objective"][0]) == want["objective"], (name, x)
                assert g["lb"][0][x] != v and valid(pb, pb.lb, pb.ub, g["lb"][0], g["ub"][0]), (name, x)


def good_and_worse(orc, pb):
    """Root A = pb's root, root B = pb's root with the objective at least A's optimum + 1 (all its solutions worse)."""
    a = orc.solve(pb)["objective"]
    lb, ub = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    lb[1, pb.obj_var] = min(a + 1, ub[1, pb.obj_var])
    return lb, ub


@pytest.mark.gpu
def test_the_incumbent_is_shared_inside_a_group(eng, orc):
    """One block takes A then B. In one group, A's optimum prunes B at once; in two groups B is searched to its own
    optimum: strictly fewer nodes in one group, and each answer still the oracle's."""
    for name in ("pat2", "planted_opt"):
        pb = network(name)
        lb, ub = good_and_worse(orc, pb)
        want = oracle_answers(orc, pb, lb, ub)
        assert want[1]["has_solution"], name
        with eng.Solver(pb, or_blocks=1, subproblems_power=0) as s:
            one = s.solve_groups(lb, ub, [0, 0])
            two = s.solve_groups(lb, ub, [0, 1])
        check_groups(pb, lb, ub, np.array([0, 0]), one, reduce_answers(want, [0, 0], 1), (name, "one"))
        check_groups(pb, lb, ub, np.array([0, 1]), two, reduce_answers(want, [0, 1], 2), (name, "two"))
        assert one["stats"]["nodes"] < two["stats"]["nodes"], (name, one["stats"]["nodes"], two["stats"]["nodes"])


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_no_incumbent_leaks_between_groups(eng, orc, opts):
    """Root A and roots B_k (A's box with the objective at least A's optimum + k), A alone in its group and the B_k in
    the other, in both orders: the B group reports its own optimum, which A's incumbent would prune away."""
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
        for groups in ([0, 1, 1, 1], [1, 0, 0, 0]):
            for order in (slice(None), slice(None, None, -1)):
                g_, lb_, ub_ = np.array(groups)[order], lb[order], ub[order]
                red = reduce_answers(want[order], g_, 2)
                with eng.Solver(pb, **opts) as s:
                    check_groups(pb, lb_, ub_, g_, s.solve_groups(lb_, ub_, g_), red, (name, opts, list(g_)))


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_satisfaction_stops_per_group(eng, orc, opts):
    """The first solution of a group ends it (not exhaustive, a valid store of one of its boxes); groups of UNSAT
    boxes are exhaustive without a solution; boxes empty at the root decide nothing."""
    pb = tnf_gen.planted(60, 80, 5, objective=False)
    lb, ub = make_roots(pb, 120, seed=3, nfix=4, empty_frac=0)
    want = oracle_answers(orc, pb, lb, ub)
    sat = [r for r, o in enumerate(want) if o["has_solution"]]
    unsat = [r for r, o in enumerate(want) if not o["has_solution"]]
    assert len(sat) >= 4 and len(unsat) >= 6
    empty_lb, empty_ub = pb.lb.copy(), pb.ub.copy()
    v = int(np.nonzero((pb.lb < pb.ub) & (pb.lb > abi.NEG_INF) & referenced(pb))[0][-1])
    empty_lb[v], empty_ub[v] = pb.ub[v], pb.lb[v]
    # groups: 0 = {sat, unsat, sat}, 1 = {unsat, unsat}, 2 = {empty, sat}, 3 = {empty, unsat}, 4 = {empty},
    # 5 = {unsat, sat, unsat}
    rows = [sat[0], unsat[0], sat[1], unsat[1], unsat[2], -1, sat[2], -1, unsat[3], -1, unsat[4], sat[3], unsat[5]]
    groups = np.array([0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 5, 5, 5], np.int32)
    glb = np.stack([empty_lb if r < 0 else lb[r] for r in rows])
    gub = np.stack([empty_ub if r < 0 else ub[r] for r in rows])
    order = np.random.default_rng(0).permutation(len(rows))         # the members of a group spread over the batch
    glb, gub, groups = glb[order], gub[order], groups[order]
    answers = [dict(has_solution=False, exhaustive=True, objective=None) if r < 0 else want[r] for r in rows]
    red = reduce_answers([answers[i] for i in order], groups, 6)
    assert [o["has_solution"] for o in red] == [True, False, True, False, False, True]
    with eng.Solver(pb, **opts) as s:
        g = s.solve_groups(glb, gub, groups)
    check_groups(pb, glb, gub, groups, g, red, opts)


@pytest.mark.gpu
def test_exhaustiveness_is_per_group_under_a_budget(eng, orc, monkeypatch):
    """Easy roots of accap_a3 in groups of four next to its full root, which does not finish in a second: the groups
    of easy roots are exhaustive with the reduced oracle answer, the group holding the full root is not."""
    monkeypatch.setenv("TB_SPLIT_MIN_NODES", "256")
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    with eng.Solver(pb, timeout_ms=1000) as s:
        sol = s.solve()
    assert sol["has_solution"]
    lb, ub = make_roots(pb, 48, seed=5, around=sol["lb"].astype(np.int64), free=12)
    want = oracle_answers(orc, pb, lb, ub)
    assert all(o["exhaustive"] for o in want)
    groups = scattered_groups(48, 12, seed=1)
    groups[3] = 12                                                   # one easy root joins the full root's group
    red = reduce_answers(want, groups, 13)
    lb, ub = np.vstack([lb, pb.lb]), np.vstack([ub, pb.ub])
    groups = np.append(groups, 12).astype(np.int32)
    with eng.Solver(pb, timeout_ms=1000) as s:
        g = s.solve_groups(lb, ub, groups)
    check_groups(pb, lb, ub, groups, {k: v[:12] if k != "stats" else v for k, v in g.items()}, red[:12], "easy groups")
    assert not g["exhaustive"][12]
    if g["has_solution"][12]:
        assert valid(pb, pb.lb, pb.ub, g["lb"][12], g["ub"][12])


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_cut_blocks_leave_their_groups_unproven(eng, orc, opts):
    """With cutnodes a block stops: a group that reports exhaustive has the reduced oracle answer. With one block the
    roots are taken in order, so the groups finished before the cut are exhaustive and the others are not."""
    pb = tnf_gen.search_instance(5)
    lb, ub = make_roots(pb, 40, seed=7, nfix=1, empty_frac=0)
    want = oracle_answers(orc, pb, lb, ub)
    groups = (np.arange(40) // 4).astype(np.int32)                   # contiguous: a prefix of groups ends before the cut
    red = reduce_answers(want, groups, 10)
    with eng.Solver(pb, cutnodes=30, **opts) as s:
        g = s.solve_groups(lb, ub, groups)
    for k, o in enumerate(red):
        if g["exhaustive"][k]:
            assert bool(g["has_solution"][k]) == o["has_solution"] and o["exhaustive"], k
            assert int(g["objective"][k]) == o["objective"], k
    if opts:
        assert not g["exhaustive"].all() and g["stats"]["nodes"] <= 30
        first_open = int(np.argmin(g["exhaustive"]))
        assert g["exhaustive"][:first_open].all() and not g["exhaustive"][first_open:].any()


@pytest.mark.gpu
def test_rejections(eng):
    pb = tnf_gen.search_instance(2)
    lb2, ub2 = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    with eng.Solver(pb) as s:
        for groups, ngroups in (([0, 2], 2), ([0, -1], 2), ([0, 0], 2), ([0, 1], 0)):
            with pytest.raises(eng.TurboError) as e:
                s.solve_groups(lb2, ub2, groups, ngroups)
            assert e.value.status == 1, (groups, ngroups)
        with pytest.raises(eng.TurboError) as e:
            s.solve_groups(np.zeros((0, pb.nvars), np.int32), np.zeros((0, pb.nvars), np.int32), [], 1)
        assert e.value.status == 1
        wide_ub = ub2.copy()
        wide_ub[1, 5] += 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_groups(lb2, wide_ub, [0, 0])
        assert e.value.status == 1
        s.stream_solutions(4)
        with pytest.raises(eng.TurboError) as e:
            s.solve_groups(lb2, ub2, [0, 0])
        assert e.value.status == 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
        with pytest.raises(eng.TurboError) as e:
            s.solve_groups(lb2, ub2, [0, 0])
        assert e.value.status == 4
    a, b = eng.Solver(pb), eng.Solver(pb)
    try:
        eng.link_peers([a, b])
        with pytest.raises(eng.TurboError) as e:
            a.solve_groups(lb2, ub2, [0, 0])
        assert e.value.status == 4
    finally:
        a.close()
        b.close()

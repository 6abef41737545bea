"""tb_solve_objectives and Solver.hull: many objectives of one network, each minimised or maximised over one union of
boxes in one launch, every solution a witness for all of them. An objective's oracle answer reduces, over the boxes, the
oracle's solve of each box with obj_var = v (minimise) or of the network with a negation variable n, 0 = v + n, and
obj_var = n (maximise)."""
import itertools

import numpy as np
import pytest

from tests import golden_io, tnf_gen
from tools.batch_solve import REL, make_roots, referenced, root_problem, valid
from tools.group_solve import cubes
from tools.objective_solve import negation_network, with_objective
from turbo_b200 import abi

CONFIGS = [dict(), dict(or_blocks=1, subproblems_power=0)]
NETWORKS = ["pat2", "pat10", "sudoku_opt2", "sudoku_opt3", "reified_in", "planted_sat", "planted_opt", "random_opt"]


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


def oracle_box(orc, pb, lb, ub, v, maximize):
    """The oracle's answer for one box: (has_solution, exhaustive, value in the objective's own sense)."""
    if maximize:
        net, n = negation_network(root_problem(pb, lb, ub), v)
        o = orc.solve(net, depth=0)
        val = (abi.POS_INF if o["objective"] == abi.NEG_INF else -o["objective"]) if o["has_solution"] else None
    else:
        o = orc.solve(with_objective(root_problem(pb, lb, ub), v), depth=0)
        val = o["objective"] if o["has_solution"] else None
    return o["has_solution"], o["exhaustive"], val


def oracle_objective(orc, pb, lb, ub, v, maximize, empty):
    """Reduced over the boxes: any solution, exhaustive when every box is, the best value (POS_INF: none). Boxes empty
    at the root are decided without a search."""
    answers = [oracle_box(orc, pb, lb[r], ub[r], v, maximize) for r in range(lb.shape[0]) if not empty[r]]
    vals = [a[2] for a in answers if a[0]]
    best = (max(vals) if maximize else min(vals)) if vals else abi.POS_INF
    return dict(has_solution=bool(vals), exhaustive=all(a[1] for a in answers), objective=best)


def empty_boxes(pb, lb, ub):
    ref = referenced(pb)
    return [bool(((lb[r] > ub[r]) & ref).any()) for r in range(lb.shape[0])]


def check_objectives(pb, lb, ub, vs, mx, got, want, what):
    for m, o in enumerate(want):
        assert bool(got["has_solution"][m]) == o["has_solution"], (what, m)
        assert bool(got["exhaustive"][m]) == o["exhaustive"], (what, m)
        assert int(got["objective"][m]) == o["objective"], (what, m, int(got["objective"][m]), o["objective"])
        if o["has_solution"]:
            row_lb, row_ub = got["lb"][m], got["ub"][m]
            assert row_lb[vs[m]] == row_ub[vs[m]] == o["objective"], (what, m)
            assert any(valid(pb, lb[r], ub[r], row_lb, row_ub) for r in range(lb.shape[0])), (what, m)


def random_objectives(pb, k, seed):
    """k objectives of both senses over referenced and unreferenced variables (some repeated)."""
    rng = np.random.default_rng(seed)
    ref = np.nonzero(referenced(pb))[0]
    unref = np.nonzero(~referenced(pb))[0]
    pool = list(rng.choice(ref, size=min(len(ref), k), replace=False)) + list(unref[:2])
    vs = np.array([pool[i % len(pool)] for i in rng.permutation(max(k, len(pool)))[:k]], np.int32)
    return vs, rng.integers(0, 2, size=k).astype(np.int32)


# ---- CPU -----------------------------------------------------------------------------------------------------------

def test_negation_network_matches_the_oracle_minimising_minus_v():
    """The network with n, 0 = v + n minimises n to -max(v): the same as the oracle minimising -v written as
    m = v * (-1), and the brute-force maximum over every point."""
    from oracle import oracle_py as orc
    for seed in range(6):
        pb = tnf_gen.random_net(7, 5, 300 + seed, lo=-3, hi=3)
        sols = [pt for pt in itertools.product(*[range(int(a), int(b) + 1) for a, b in zip(pb.lb, pb.ub)])
                if all(REL[int(p["op"])](pt[p["x"]], pt[p["y"]], pt[p["z"]]) for p in pb.props)]
        for v in range(pb.nvars):
            net, n = negation_network(pb, v)
            o = orc.solve(net)
            lb = np.concatenate([pb.lb, [-1, abi.NEG_INF]]).astype(np.int32)
            ub = np.concatenate([pb.ub, [-1, abi.POS_INF]]).astype(np.int32)
            c, m = pb.nvars, pb.nvars + 1
            props = np.array([tuple(int(p[k]) for k in ("op", "x", "y", "z")) for p in pb.props] + [(abi.OP_MUL, m, v, c)],
                             np.int32)
            ref = orc.solve(abi.Problem(lb, ub, props, pb.strategies, obj_var=m))
            assert o["has_solution"] == ref["has_solution"] == bool(sols), (seed, v)
            if sols:
                assert o["objective"] == ref["objective"] == -max(pt[v] for pt in sols), (seed, v)
                assert o["lb"][n] == -o["lb"][v]


# ---- GPU -----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", NETWORKS)
def test_every_objective_equals_the_reduced_oracle(eng, orc, name):
    pb = network(name)
    lb_all, ub_all = make_roots(pb, 24, seed=13, nfix=2)
    v = int(np.nonzero(referenced(pb) & (pb.lb < pb.ub))[0][0])
    lb_all[17, v], ub_all[17, v] = pb.ub[v], pb.lb[v]                 # one box empty at the root
    for nboxes, seed in ((1, 1), (5, 2), (24, 3)):
        lb, ub = lb_all[:nboxes], ub_all[:nboxes]
        vs, mx = random_objectives(pb, 6, seed)
        empty = empty_boxes(pb, lb, ub)
        want = [oracle_objective(orc, pb, lb, ub, int(v), bool(x), empty) for v, x in zip(vs, mx)]
        for opts in CONFIGS:
            with eng.Solver(pb, **opts) as s:
                got = s.solve_objectives(lb, ub, vs, mx)
            assert len(got["objective"]) == len(vs)
            check_objectives(pb, lb, ub, vs, mx, got, want, (name, nboxes, opts))


def brute_hull(pb, lb, ub):
    """[min, max] of every variable over the satisfying points of the boxes (None: no point)."""
    pts = set()
    for r in range(lb.shape[0]):
        for pt in itertools.product(*[range(int(a), int(b) + 1) for a, b in zip(lb[r], ub[r])]):
            if all(REL[int(p["op"])](pt[p["x"]], pt[p["y"]], pt[p["z"]]) for p in pb.props):
                pts.add(pt)
    if not pts:
        return None
    a = np.array(sorted(pts))
    return a.min(axis=0), a.max(axis=0)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_hull_equals_brute_force(eng, opts):
    checked = unsat = 0
    for seed in range(30):
        pb = tnf_gen.random_net(9, 4, 700 + seed, lo=-3, hi=3)
        lb, ub = cubes(pb, 3)
        want = brute_hull(pb, lb, ub)
        with eng.Solver(pb, **opts) as s:
            h = s.hull(lb=lb, ub=ub)
        assert h["exact_lb"].all() and h["exact_ub"].all(), seed
        if want is None:
            unsat += 1
            assert not h["has_solution"] and (h["lb"] == abi.POS_INF).all() and (h["ub"] == abi.NEG_INF).all(), seed
        else:
            checked += 1
            assert h["has_solution"], seed
            assert np.array_equal(h["lb"], want[0]) and np.array_equal(h["ub"], want[1]), (seed, h["lb"], want)
    assert checked >= 5 and unsat >= 5
    # an unsatisfiable box set: a satisfiable network with one variable fixed, in every box, outside its hull
    found = False
    for seed in range(30):
        pb = tnf_gen.random_net(9, 4, 700 + seed, lo=-3, hi=3)
        lb, ub = cubes(pb, 3)
        want = brute_hull(pb, lb, ub)
        outside = [] if want is None else [(v, x) for v in range(pb.nvars) for x in range(int(pb.lb[v]), int(pb.ub[v]) + 1)
                                           if not want[0][v] <= x <= want[1][v]]
        if not outside:
            continue
        v, x = outside[0]
        lb[:, v] = ub[:, v] = x
        assert brute_hull(pb, lb, ub) is None
        with eng.Solver(pb, **opts) as s:
            h = s.hull(lb=lb, ub=ub)
        assert not h["has_solution"] and h["exact_lb"].all() and h["exact_ub"].all(), seed
        assert (h["lb"] == abi.POS_INF).all() and (h["ub"] == abi.NEG_INF).all()
        found = True
        break
    assert found


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_the_problem_objective_equals_one_group(eng, opts):
    """One objective equal to the problem's own, minimised, answers as tb_solve_groups with one group of the same
    boxes; solve_groups and solve_batch on the same solver after a solve_objectives still answer as before."""
    for name in ("pat2", "planted_opt", "random_opt"):
        pb = network(name)
        lb, ub = make_roots(pb, 40, seed=4)
        with eng.Solver(pb, **opts) as s:
            b0 = s.solve_batch(lb, ub)
            g0 = s.solve_groups(lb, ub, np.zeros(40, np.int32))
            o = s.solve_objectives(lb, ub, [pb.obj_var], [0])
            g1 = s.solve_groups(lb, ub, np.zeros(40, np.int32))
            b1 = s.solve_batch(lb, ub)
            o2 = s.solve_objectives(lb[:3], ub[:3], [pb.obj_var] * 5, [0, 1, 0, 1, 0])
            g2 = s.solve_groups(lb, ub, np.arange(40) % 7)
        for key in ("has_solution", "exhaustive", "objective"):
            assert np.array_equal(o[key], g0[key]) and np.array_equal(g1[key], g0[key]), (name, key)
            assert np.array_equal(b1[key], b0[key]), (name, key)
        if o["has_solution"][0]:
            assert o["lb"][0][pb.obj_var] == o["ub"][0][pb.obj_var] == o["objective"][0]
        # repeated objectives answer alike
        assert len(set(o2["objective"][[0, 2, 4]])) == 1 and len(set(o2["objective"][[1, 3]])) == 1
        with eng.Solver(pb, **opts) as s:
            fresh = s.solve_groups(lb, ub, np.arange(40) % 7)
        for key in ("has_solution", "exhaustive", "objective"):
            assert np.array_equal(g2[key], fresh[key]), (name, key)


@pytest.mark.gpu
def test_witnesses_are_shared(eng, orc):
    """One block, a fixed order of search: min x and max x in one call take fewer nodes than the two calls alone, with
    the same answers; every objective of an exhaustive run agrees on has_solution."""
    strict = 0
    for name in ("planted_opt", "random_opt", "sudoku_opt3", "pat2"):
        pb = network(name)
        vs = [int(v) for v in np.nonzero(referenced(pb) & (pb.lb < pb.ub))[0][:4]]
        with eng.Solver(pb, or_blocks=1, subproblems_power=0) as s:
            for x in vs:
                both = s.solve_objectives(pb.lb, pb.ub, [x, x], [0, 1])
                lo = s.solve_objectives(pb.lb, pb.ub, [x], [0])
                hi = s.solve_objectives(pb.lb, pb.ub, [x], [1])
                assert list(both["objective"]) == [lo["objective"][0], hi["objective"][0]], (name, x)
                assert both["exhaustive"].all() and lo["exhaustive"][0] and hi["exhaustive"][0]
                nb, ns = both["stats"]["nodes"], lo["stats"]["nodes"] + hi["stats"]["nodes"]
                assert nb <= ns, (name, x, nb, ns)
                strict += nb < ns
        with eng.Solver(pb) as s:
            r = s.solve_objectives(pb.lb, pb.ub, np.arange(pb.nvars), np.arange(pb.nvars) % 2)
        if r["exhaustive"].all():
            assert r["has_solution"].all() or not r["has_solution"].any(), name
    assert strict >= 1


def unbounded_variant(pb, v):
    """pb with variable v's upper bound at +oo."""
    ub = pb.ub.copy()
    ub[v] = abi.POS_INF
    return abi.Problem(pb.lb, ub, pb.props, pb.strategies, obj_var=pb.obj_var, has_eps_strategy=int(pb.c.has_eps_strategy))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["maximize_unconstrained", "maximize_unconstrained2"])
@pytest.mark.parametrize("opts", CONFIGS)
def test_an_unbounded_maximisation_ends_its_objective_only(eng, orc, name, opts):
    pb, info = golden_io.load(name)
    u = info["user_obj_var"]
    with eng.Solver(pb, **opts) as s:
        r = s.solve_objectives(pb.lb, pb.ub, [u, u], [1, 0])
    assert list(r["objective"]) == [info["expected"], orc.solve(with_objective(pb, u))["objective"]]
    assert r["exhaustive"].all() and r["has_solution"].all()
    # an unreferenced variable at +oo: its maximisation is unbounded, the others stay exact
    free = [v for v in range(pb.nvars) if not referenced(pb)[v]]
    assert free, name
    w = free[0]
    net = unbounded_variant(pb, w)
    with eng.Solver(net, **opts) as s:
        r = s.solve_objectives(net.lb, net.ub, [w, u, w, u], [1, 1, 0, 0])
    assert r["has_solution"].all()
    assert int(r["objective"][0]) == abi.POS_INF and not r["exhaustive"][0]
    assert r["lb"][0][w] == r["ub"][0][w] == abi.POS_INF
    assert list(r["objective"][1:]) == [info["expected"], pb.lb[w], orc.solve(with_objective(pb, u))["objective"]]
    assert r["exhaustive"][1:].all()


def with_domains(pb, doms):
    """pb with the root domains of some variables replaced: {v: (lb, ub)}."""
    lb, ub = pb.lb.copy(), pb.ub.copy()
    for v, (a, b) in doms.items():
        lb[v], ub[v] = a, b
    return abi.Problem(lb, ub, pb.props, pb.strategies, obj_var=pb.obj_var, has_eps_strategy=int(pb.c.has_eps_strategy))


def valid_but(pb, lb, ub, slb, sub, y):
    """valid(), except that a variable y no propagator reads may be empty in the row if it is so in the box."""
    if slb[y] > sub[y]:
        if (slb[y], sub[y]) != (lb[y], ub[y]):
            return False
        lb, ub, slb, sub = lb.copy(), ub.copy(), slb.copy(), sub.copy()
        lb[y] = ub[y] = slb[y] = sub[y] = 0
    return valid(pb, lb, ub, slb, sub)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_an_empty_unreferenced_objective_variable_witnesses_nothing(eng, orc, opts):
    """A variable y that no propagator reads can be empty in a box whose other variables have solutions. Minimising or
    maximising y fails at every node of that box, so its solutions are no witnesses for y: with y in [3, 2] and [8, 7]
    in two boxes and [4, 5] in the third, min y is 4 and max y is 5 (not 3 and 7), as the reduced oracle says; the
    objectives over a referenced variable still count every box."""
    pb, info = golden_io.load("maximize_unconstrained")
    x = info["user_obj_var"]
    y = [v for v in range(pb.nvars) if not referenced(pb)[v]][0]
    pb = with_domains(pb, {y: (0, 9)})
    lb, ub = np.tile(pb.lb, (3, 1)), np.tile(pb.ub, (3, 1))
    (lb[0, y], ub[0, y]), (lb[1, y], ub[1, y]), (lb[2, y], ub[2, y]) = (3, 2), (8, 7), (4, 5)
    lb[2, x] = ub[2, x] = pb.lb[x]                                   # x's maximum lies in the boxes where y is empty
    vs, mx = [y, y, x, x], [0, 1, 0, 1]
    empty = empty_boxes(pb, lb, ub)
    assert not any(empty)
    want = [oracle_objective(orc, pb, lb, ub, v, bool(m), empty) for v, m in zip(vs, mx)]
    assert [o["objective"] for o in want] == [4, 5, pb.lb[x], pb.ub[x]]
    with eng.Solver(pb, **opts) as s:
        got = s.solve_objectives(lb, ub, vs, mx)
    for m, o in enumerate(want):
        assert (bool(got["has_solution"][m]), bool(got["exhaustive"][m]), int(got["objective"][m])) == \
            (o["has_solution"], o["exhaustive"], o["objective"]), (opts, m)
        assert got["lb"][m][vs[m]] == got["ub"][m][vs[m]] == o["objective"], (opts, m)
        assert any(valid_but(pb, lb[r], ub[r], got["lb"][m], got["ub"][m], y) for r in range(3)), (opts, m)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_a_maximum_next_to_the_minus_infinity_sentinel(eng, opts):
    """A maximum of INT32_MIN + 1 is a value like any other: its key must not read as "no incumbent"."""
    pb, _ = golden_io.load("maximize_unconstrained")
    free = [v for v in range(pb.nvars) if not referenced(pb)[v]]
    a, b = free[0], free[1]
    lo = abi.NEG_INF + 1
    pb = with_domains(pb, {a: (lo, lo), b: (lo, lo + 2)})
    with eng.Solver(pb, **opts) as s:
        r = s.solve_objectives(pb.lb, pb.ub, [a, a, b, b], [1, 0, 1, 0])
    assert r["has_solution"].all() and r["exhaustive"].all()
    assert list(r["objective"]) == [lo, lo, lo + 2, lo]
    for m, v in enumerate([a, a, b, b]):
        assert r["lb"][m][v] == r["ub"][m][v] == r["objective"][m]


@pytest.mark.gpu
def test_exhaustiveness_is_per_objective_under_a_budget(eng, monkeypatch):
    """accap_a3 under a second, next to its own objective: the sides of variables fixed at the root end as soon as a
    solution is known, and are exhaustive with their value; every value, proven or not, is witnessed by a valid row.
    (Objective m is dispensed before m + 1: the hard one comes last.)"""
    monkeypatch.setenv("TB_SPLIT_MIN_NODES", "256")
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    fixed = [int(v) for v in np.nonzero(referenced(pb) & (pb.lb == pb.ub))[0][:2]]
    easy = [int(v) for _, _, s in pb.strategies for v in s][:6]
    vs = fixed + easy + fixed + easy + [pb.obj_var]
    mx = [0] * (len(fixed) + len(easy)) + [1] * (len(fixed) + len(easy)) + [0]
    with eng.Solver(pb, timeout_ms=1000) as s:
        r = s.solve_objectives(pb.lb, pb.ub, vs, mx)
    assert r["has_solution"].all()
    for m in range(len(vs)):
        assert valid(pb, pb.lb, pb.ub, r["lb"][m], r["ub"][m]), m
        assert r["lb"][m][vs[m]] == r["objective"][m]
        if vs[m] in fixed:
            assert r["exhaustive"][m] and r["objective"][m] == pb.lb[vs[m]], m


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_cut_blocks_leave_their_objectives_unproven(eng, orc, opts):
    pb = tnf_gen.search_instance(5)
    vs, mx = random_objectives(pb, 8, 21)
    lb, ub = make_roots(pb, 6, seed=8, nfix=1, empty_frac=0)
    empty = empty_boxes(pb, lb, ub)
    want = [oracle_objective(orc, pb, lb, ub, int(v), bool(x), empty) for v, x in zip(vs, mx)]
    with eng.Solver(pb, cutnodes=30, **opts) as s:
        r = s.solve_objectives(lb, ub, vs, mx)
    if opts:
        assert not r["exhaustive"].all() and r["stats"]["nodes"] <= 30
    for m, o in enumerate(want):
        if r["exhaustive"][m]:
            assert bool(r["has_solution"][m]) == o["has_solution"] and int(r["objective"][m]) == o["objective"], m
        elif r["has_solution"][m]:
            assert any(valid(pb, lb[k], ub[k], r["lb"][m], r["ub"][m]) for k in range(lb.shape[0])), m
            # a witnessed value lies inside the hull: no better than the optimum
            assert (r["objective"][m] <= o["objective"]) if mx[m] else (r["objective"][m] >= o["objective"]), m


@pytest.mark.gpu
def test_rejections(eng):
    pb = tnf_gen.search_instance(2)
    lb2, ub2 = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    with eng.Solver(pb) as s:
        for vs, mx in (([0], [2]), ([0], [-1]), ([pb.nvars], [0]), ([-1], [0]), ([], [])):
            with pytest.raises(eng.TurboError) as e:
                s.solve_objectives(lb2, ub2, vs, mx)
            assert e.value.status == 1, (vs, mx)
        with pytest.raises(eng.TurboError) as e:
            s.solve_objectives(np.zeros((0, pb.nvars), np.int32), np.zeros((0, pb.nvars), np.int32), [0], [0])
        assert e.value.status == 1
        wide_ub = ub2.copy()
        wide_ub[1, 5] += 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_objectives(lb2, wide_ub, [0], [0])
        assert e.value.status == 1
        # nobj * nboxes above the 40-bit subproblem index, rejected before any allocation
        from turbo_b200 import engine
        big = 1 << 21
        vs = np.zeros(big, np.int32)
        with pytest.raises(eng.TurboError) as e:
            engine._check(engine.lib().tb_solve_objectives(s._h, big, engine._p(lb2), engine._p(ub2), big,
                                                           engine._p(vs), engine._p(vs), None, None, None, None, None,
                                                           None, None, None))
        assert e.value.status == 1 and "2^40" in str(e.value)
        s.stream_solutions(4)
        with pytest.raises(eng.TurboError) as e:
            s.solve_objectives(lb2, ub2, [0], [0])
        assert e.value.status == 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
        with pytest.raises(eng.TurboError) as e:
            s.solve_objectives(lb2, ub2, [0], [0])
        assert e.value.status == 4
    a, b = eng.Solver(pb), eng.Solver(pb)
    try:
        eng.link_peers([a, b])
        with pytest.raises(eng.TurboError) as e:
            a.solve_objectives(lb2, ub2, [0], [0])
        assert e.value.status == 4
    finally:
        a.close()
        b.close()

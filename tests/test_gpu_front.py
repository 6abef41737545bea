"""tb_solve_front, Solver.solve_front and Solver.pareto_front: the Pareto front of two objectives of one network over one
union of boxes in one launch, one level per group searching a disjoint slice of x, every solution a witness for every
level it reaches. A level's oracle answer reduces, over the boxes, the oracle's solve of each box narrowed to x <= t
(x >= t) with obj_var = y (minimise) or the negation network (maximise)."""
import itertools

import numpy as np
import pytest

from tests import golden_io, tnf_gen
from tools.batch_solve import REL, make_roots, referenced, root_problem, valid
from tools.front_solve import axes, nested_groups, side
from tools.group_solve import cubes
from tools.objective_solve import negation_network, with_objective
from turbo_b200 import abi
from turbo_b200.engine import front_points

CONFIGS = [dict(), dict(or_blocks=1, subproblems_power=0)]
NETWORKS = ["pat2", "pat10", "sudoku_opt2", "sudoku_opt3", "planted_opt", "random_opt"]
SENSES = [(0, 0), (0, 1), (1, 0), (1, 1)]


@pytest.fixture(scope="module")
def eng():
    from turbo_b200 import engine
    assert engine.device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    return engine


def network(name):
    if name == "planted_opt":
        return tnf_gen.search_instance(3)
    if name == "random_opt":
        return tnf_gen.random_net(16, 9, 5011, lo=-4, hi=4)
    return golden_io.load(name)[0]


def solutions(pb, lb, ub):
    """Every satisfying point of the boxes."""
    pts = set()
    for r in range(lb.shape[0]):
        for pt in itertools.product(*[range(int(a), int(b) + 1) for a, b in zip(lb[r], ub[r])]):
            if all(REL[int(p["op"])](pt[p["x"]], pt[p["y"]], pt[p["z"]]) for p in pb.props):
                pts.add(pt)
    return sorted(pts)


def brute_levels(sols, x, y, levels, mx, my):
    """Per level: the best y over the points on its side, and a row: the point with that y and the best x."""
    k = len(levels)
    out = dict(has_solution=np.zeros(k, bool), exhaustive=np.ones(k, bool), objective=np.full(k, abi.POS_INF, np.int64),
               lb=np.zeros((k, len(sols[0]) if sols else 1), np.int32))
    for i, t in enumerate(levels):
        on = [p for p in sols if (p[x] >= t if mx else p[x] <= t)]
        if not on:
            continue
        best = (max if my else min)(p[y] for p in on)
        row = (max if mx else min)((p for p in on if p[y] == best), key=lambda p: p[x])
        out["has_solution"][i], out["objective"][i], out["lb"][i] = True, best, row
    out["ub"] = out["lb"].copy()
    return out


def brute_front(sols, x, y, mx, my):
    """The Pareto-optimal (x, y) values, in x's preferred order."""
    key = lambda p: (-p[0] if mx else p[0], -p[1] if my else p[1])
    vals = sorted({(p[x], p[y]) for p in sols}, key=key)
    front, best = [], None
    for p in vals:
        ky = key(p)[1]
        if best is None or ky < best:
            best = ky
            front.append(p)
    return front


def pick_axes(pb):
    """x and y for a small random network: two different variables, each with two values or more."""
    open_vars = [v for v in range(pb.nvars) if pb.lb[v] < pb.ub[v] and referenced(pb)[v]]
    if len(open_vars) < 2:
        return None
    x = pb.obj_var if pb.obj_var in open_vars else open_vars[0]
    return x, [v for v in open_vars if v != x][-1]


def oracle_level(orc, pb, lb, ub, x, y, t, mx, my):
    """The oracle's answer for level t: every box narrowed to t's side, solved for y, reduced over the boxes. Boxes with
    an empty referenced domain are decided without a search."""
    nlb, nub = side(lb, ub, x, t, mx)
    ref = referenced(pb)
    vals, exh = [], True
    for r in range(nlb.shape[0]):
        if ((nlb[r] > nub[r]) & ref).any():
            continue
        box = root_problem(pb, nlb[r].astype(np.int32), nub[r].astype(np.int32))
        if my:
            net, n = negation_network(box, y)
            o = orc.solve(net, depth=0)
            val = (abi.POS_INF if o["objective"] == abi.NEG_INF else -o["objective"]) if o["has_solution"] else None
        else:
            o = orc.solve(with_objective(box, y), depth=0)
            val = o["objective"] if o["has_solution"] else None
        exh &= bool(o["exhaustive"])
        if val is not None:
            vals.append(int(val))
    best = ((max if my else min)(vals)) if vals else abi.POS_INF
    return dict(has_solution=bool(vals), exhaustive=exh, objective=best)


def check_levels(pb, lb, ub, x, y, levels, mx, my, r, what):
    """Every row is a solution of some box with x on its level's side at the row's best value and y at the level's
    value; the values never get worse from level to level in x's preferred order."""
    for i, t in enumerate(levels):
        if not r["has_solution"][i]:
            continue
        rl, ru = r["lb"][i], r["ub"][i]
        assert rl[y] == ru[y] == r["objective"][i], (what, i)
        assert rl[x] == ru[x] and (rl[x] >= t if mx else rl[x] <= t), (what, i)
        assert any(valid(pb, lb[k], ub[k], rl, ru) for k in range(lb.shape[0])), (what, i)
    order = range(len(levels) - 1, -1, -1) if mx else range(len(levels))
    prev = None
    for i in order:
        if prev is not None and r["has_solution"][prev]:
            assert r["has_solution"][i], (what, i)
            a, b = int(r["objective"][prev]), int(r["objective"][i])
            assert (b >= a) if my else (b <= a), (what, i)
        prev = i


# ---- CPU -----------------------------------------------------------------------------------------------------------

def test_front_points_equal_brute_force_fronts():
    checked = 0
    for seed in range(40):
        pb = tnf_gen.random_net(9, 4, 900 + seed, lo=-3, hi=3)
        xy = pick_axes(pb)
        if xy is None:
            continue
        x, y = xy
        sols = solutions(pb, pb.lb[None, :], pb.ub[None, :])
        levels = list(range(int(pb.lb[x]), int(pb.ub[x]) + 1))
        for mx, my in SENSES:
            f = front_points(brute_levels(sols, x, y, levels, mx, my), x, mx, my)
            assert f["points"] == brute_front(sols, x, y, mx, my), (seed, mx, my)
            assert f["proven"].all() and len(f["level"]) == len(f["points"])
            checked += len(sols) > 0
    assert checked >= 20


def test_reduced_oracle_equals_brute_force():
    from oracle import oracle_py as orc
    checked = 0
    for seed in range(12):
        pb = tnf_gen.random_net(9, 4, 900 + seed, lo=-3, hi=3)
        xy = pick_axes(pb)
        if xy is None:
            continue
        x, y = xy
        lb, ub = cubes(pb, 3)
        sols = solutions(pb, lb, ub)
        levels = list(range(int(pb.lb[x]) - 1, int(pb.ub[x]) + 2))
        for mx, my in SENSES:
            want = brute_levels(sols, x, y, levels, mx, my)
            for i, t in enumerate(levels):
                o = oracle_level(orc, pb, lb, ub, x, y, t, mx, my)
                assert o["exhaustive"], (seed, t)
                assert o["has_solution"] == want["has_solution"][i], (seed, mx, my, t)
                assert o["objective"] == want["objective"][i], (seed, mx, my, t)
        checked += 1
    assert checked >= 6


# ---- GPU -----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_pareto_front_equals_brute_force(eng, opts):
    sat = unsat = 0
    for seed in range(30):
        pb = tnf_gen.random_net(9, 4, 900 + seed, lo=-3, hi=3)
        xy = pick_axes(pb)
        if xy is None:
            continue
        x, y = xy
        for lb, ub in ((pb.lb[None, :].copy(), pb.ub[None, :].copy()), cubes(pb, 3)):
            sols = solutions(pb, lb, ub)
            with eng.Solver(pb, **opts) as s:
                for mx, my in SENSES:
                    f = s.pareto_front(x, y, lb, ub, maximize_x=mx, maximize_y=my)
                    assert f["exact"] and f["proven"].all(), (seed, mx, my)
                    assert f["points"] == brute_front(sols, x, y, mx, my), (seed, mx, my, f["points"])
                    for (px, py), rl, ru in zip(f["points"], f["lb"], f["ub"]):
                        assert rl[x] == ru[x] == px and rl[y] == ru[y] == py
                        assert any(valid(pb, lb[k], ub[k], rl, ru) for k in range(lb.shape[0]))
            if sols:
                sat += 1
            else:
                unsat += 1
    assert sat >= 5 and unsat >= 3


def level_sets(pb, x, seed):
    """Full-range levels (capped at 12 by a step), coarse random levels, and levels below and above x's range."""
    lo, hi = int(pb.lb[x]), int(pb.ub[x])
    step = max(1, -(-(hi - lo + 1) // 12))
    rng = np.random.default_rng(seed)
    coarse = sorted(set(int(v) for v in rng.integers(lo, hi + 1, size=4)))
    return [list(range(lo, hi + 1, step)), coarse, [lo - 3, lo - 1, hi + 1, hi + 4]]


@pytest.mark.gpu
@pytest.mark.parametrize("name", NETWORKS)
def test_levels_equal_the_reduced_oracle(eng, name):
    from oracle import oracle_py as orc
    pb = network(name)
    x, y = axes(pb)
    lb_all, ub_all = make_roots(pb, 3, seed=17, nfix=2, empty_frac=0)
    v = int(np.nonzero(referenced(pb) & (pb.lb < pb.ub))[0][-1])
    lb_all[2, v], ub_all[2, v] = pb.ub[v], pb.lb[v]                  # one box empty at the root
    boxes = [(pb.lb[None, :].copy(), pb.ub[None, :].copy())]
    if name != "pat2":                                               # (the oracle takes a second per pat2 box)
        boxes.append((lb_all, ub_all))
    senses = [(0, 0), (1, 1)] if name == "pat2" else SENSES
    for bi, (lb, ub) in enumerate(boxes):
        for li, levels in enumerate(level_sets(pb, x, 5 + bi)):
            for mx, my in senses:
                want = [oracle_level(orc, pb, lb, ub, x, y, t, mx, my) for t in levels]
                for opts in CONFIGS:
                    with eng.Solver(pb, **opts) as s:
                        r = s.solve_front(lb, ub, x, y, levels, mx, my)
                    what = (name, bi, li, mx, my, opts)
                    for i, o in enumerate(want):
                        assert bool(r["has_solution"][i]) == o["has_solution"], (what, i)
                        assert bool(r["exhaustive"][i]) == o["exhaustive"], (what, i)
                        assert int(r["objective"][i]) == o["objective"], (what, i, int(r["objective"][i]), o)
                    check_levels(pb, lb, ub, x, y, levels, mx, my, r, what)


def check_budget(orc, pb, lb, ub, x, y, levels, mx, my, r, what):
    """Exhaustiveness is a prefix (min x) or a suffix (max x) of the levels, exhaustive values are the oracle's, and
    every other value is witnessed: no better than the oracle's optimum."""
    exh = list(r["exhaustive"][::-1] if mx else r["exhaustive"])
    assert exh == sorted(exh, reverse=True), what
    for i, t in enumerate(levels):
        o = oracle_level(orc, pb, lb, ub, x, y, t, mx, my)
        if r["exhaustive"][i]:
            assert (bool(r["has_solution"][i]), int(r["objective"][i])) == (o["has_solution"], o["objective"]), (what, i)
        elif r["has_solution"][i]:
            assert o["has_solution"], (what, i)
            v = int(r["objective"][i])
            assert (v <= o["objective"]) if my else (v >= o["objective"]), (what, i)
    check_levels(pb, lb, ub, x, y, levels, mx, my, r, what)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_budget_answers_are_sound(eng, opts):
    from oracle import oracle_py as orc
    cut = 0
    for name in ("sudoku_opt3", "pat10"):
        pb = network(name)
        x, y = axes(pb)
        lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
        levels = list(range(int(pb.lb[x]), int(pb.ub[x]) + 1))
        for mx, my in SENSES:
            with eng.Solver(pb, cutnodes=30, **opts) as s:
                r = s.solve_front(lb, ub, x, y, levels, mx, my)
            cut += not r["exhaustive"].all()
            check_budget(orc, pb, lb, ub, x, y, levels, mx, my, r, (name, "cutnodes", mx, my))
            with eng.Solver(pb, timeout_ms=1, **opts) as s:
                r = s.solve_front(lb, ub, x, y, levels, mx, my)
            check_budget(orc, pb, lb, ub, x, y, levels, mx, my, r, (name, "timeout", mx, my))
    assert cut >= 1


@pytest.mark.gpu
def test_one_call_agrees_with_nested_groups(eng):
    """One block, a fixed order of search: every level equals tb_solve_groups with the nested box x <= t (x >= t) per
    level on the network optimising y; the front takes strictly fewer nodes on at least one network."""
    fewer, report = 0, []
    for name in NETWORKS:
        pb = network(name)
        x, y = axes(pb)
        lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
        levels = list(range(int(pb.lb[x]), int(pb.ub[x]) + 1))
        for mx, my in ((0, 0), (1, 1)):
            with eng.Solver(pb, or_blocks=1, subproblems_power=0) as s:
                r = s.solve_front(lb, ub, x, y, levels, mx, my)
            b = nested_groups(pb, lb, ub, x, y, levels, mx, my, or_blocks=1, subproblems_power=0)
            assert r["exhaustive"].all() and b["exhaustive"].all(), name
            assert np.array_equal(r["has_solution"], b["has_solution"]), (name, mx, my)
            assert np.array_equal(r["objective"], b["objective"]), (name, mx, my)
            report.append((name, mx, my, r["stats"]["nodes"], b["stats"]["nodes"]))
            fewer += r["stats"]["nodes"] < b["stats"]["nodes"]
    print("front vs nested groups, nodes:", report)
    assert fewer >= 1, report


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_other_calls_after_front(eng, opts):
    for name in ("pat10", "random_opt"):
        pb = network(name)
        x, y = axes(pb)
        lb, ub = make_roots(pb, 6, seed=4)
        levels = list(range(int(pb.lb[x]), int(pb.ub[x]) + 1))

        def others(s):
            return (s.solve(), s.solve_groups(lb, ub, np.arange(6) % 4), s.solve_objectives(lb, ub, [x, y], [0, 1]),
                    s.solve_front(lb, ub, x, y, levels, 1, 0))

        with eng.Solver(pb, **opts) as s:
            s.solve_front(lb, ub, x, y, levels, 0, 1)
            after = others(s)
            sup = s.solve_supports(lb, ub, [x, x], levels[:2])
        with eng.Solver(pb, **opts) as s:
            fresh = others(s)
            sup0 = s.solve_supports(lb, ub, [x, x], levels[:2])
        for a, b in zip(after, fresh):
            for key in ("has_solution", "exhaustive", "objective"):
                assert np.array_equal(np.asarray(a[key]), np.asarray(b[key])), (name, key)
        assert np.array_equal(sup["supported"], sup0["supported"]), name


@pytest.mark.gpu
def test_rejections(eng):
    from turbo_b200 import engine
    pb = tnf_gen.search_instance(2)
    lb2, ub2 = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    x, y = axes(pb)
    with eng.Solver(pb) as s:
        bad = [dict(x=pb.nvars), dict(x=-1), dict(y=pb.nvars), dict(y=x), dict(mx=2), dict(my=-1),
               dict(levels=[]), dict(levels=[1, 1]), dict(levels=[3, 2]), dict(levels=[abi.NEG_INF, 0]),
               dict(levels=[0, abi.POS_INF])]
        for b in bad:
            with pytest.raises(eng.TurboError) as e:
                s.solve_front(lb2, ub2, b.get("x", x), b.get("y", y), b.get("levels", [0, 1]), b.get("mx", 0),
                              b.get("my", 0))
            assert e.value.status == 1, b
        with pytest.raises(eng.TurboError) as e:
            s.solve_front(np.zeros((0, pb.nvars), np.int32), np.zeros((0, pb.nvars), np.int32), x, y, [0])
        assert e.value.status == 1
        wide_ub = ub2.copy()
        wide_ub[1, 5] += 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_front(lb2, wide_ub, x, y, [0])
        assert e.value.status == 1
        # nlev * nboxes above the 40-bit subproblem index, rejected before any allocation
        big = 1 << 21
        lv = np.arange(big, dtype=np.int32)
        out = np.zeros(1, np.int32)
        with pytest.raises(eng.TurboError) as e:
            engine._check(engine.lib().tb_solve_front(s._h, big, engine._p(lb2), engine._p(ub2), x, 0, y, 0, big,
                                                      engine._p(lv), None, None, None, engine._p(out), engine._p(out),
                                                      engine._p(out), None))
        assert e.value.status == 1 and "2^40" in str(e.value)
        # pareto_front's guards, before any launch
        ilb, iub = pb.lb.copy(), pb.ub.copy()
        iub[x] = abi.POS_INF
        with pytest.raises(ValueError):
            s.pareto_front(x, y, ilb, iub)
        wlb, wub = pb.lb.astype(np.int64), pb.ub.astype(np.int64)
        wub[x] = wlb[x] + s.MAX_FRONT_LEVELS
        with pytest.raises(ValueError):
            s.pareto_front(x, y, wlb, wub)
        with pytest.raises(ValueError):
            s.pareto_front(x, y, levels=np.arange(s.MAX_FRONT_LEVELS + 1))
        s.stream_solutions(4)
        with pytest.raises(eng.TurboError) as e:
            s.solve_front(lb2, ub2, x, y, [0])
        assert e.value.status == 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
        with pytest.raises(eng.TurboError) as e:
            s.solve_front(lb2, ub2, x, y, [0])
        assert e.value.status == 4
    a, b = eng.Solver(pb), eng.Solver(pb)
    try:
        eng.link_peers([a, b])
        with pytest.raises(eng.TurboError) as e:
            a.solve_front(lb2, ub2, x, y, [0])
        assert e.value.status == 4
    finally:
        a.close()
        b.close()

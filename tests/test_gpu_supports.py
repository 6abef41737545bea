"""tb_solve_supports and Solver.solution_domains: which values of a variable occur in some solution of one network over
one union of boxes, every (variable, value) query answered in one launch and every solution a witness for all the
values it holds. Checked against brute-force enumeration, and against what a user does without it: tb_solve_groups
with one satisfaction group per query and the x = v boxes materialised."""
import itertools

import numpy as np
import pytest

from tests import golden_io, tnf_gen
from tools.batch_solve import REL, make_roots, referenced, valid
from tools.group_solve import cubes
from turbo_b200 import abi

CONFIGS = [dict(), dict(or_blocks=1, subproblems_power=0)]
NETWORKS = ["pat2", "sudoku_opt2", "sudoku_opt3", "reified_in", "planted_sat", "random_opt"]


@pytest.fixture(scope="module")
def eng():
    from turbo_b200 import engine
    assert engine.device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    return engine


def network(name):
    if name == "planted_sat":
        return tnf_gen.planted(60, 80, 5, objective=False)
    if name == "random_opt":
        return tnf_gen.random_net(16, 9, 5011, lo=-4, hi=4)
    return golden_io.load(name)[0]


def queries(pb, lb, ub, nq, seed):
    """Up to nq (variable, value) queries over the boxes' ranges of referenced variables with small domains."""
    rng = np.random.default_rng(seed)
    live = lb <= ub
    cand = []
    for v in np.nonzero(referenced(pb))[0]:
        if not live[:, v].any():
            continue
        a, b = int(lb[live[:, v], v].min()), int(ub[live[:, v], v].max())
        if b - a <= 40:
            cand += [(int(v), x) for x in range(a, b + 1)]
    pick = rng.permutation(len(cand))[:nq]
    return (np.array([cand[i][0] for i in pick], np.int32), np.array([cand[i][1] for i in pick], np.int32))


def workaround(s, pb, lb, ub, q_var, q_val):
    """tb_solve_groups with one satisfaction group per query, box r with x = v materialised (a box whose domain of x
    does not hold v has no root: that pair is decided, without a solution). Returns has_solution, exhaustive and nodes."""
    rlb, rub, grp, idx = [], [], [], {}
    for i, (x, v) in enumerate(zip(q_var, q_val)):
        for r in range(lb.shape[0]):
            if lb[r, x] <= v <= ub[r, x]:
                a, b = lb[r].copy(), ub[r].copy()
                a[x] = b[x] = v
                rlb.append(a)
                rub.append(b)
                grp.append(idx.setdefault(i, len(idx)))
    has = np.zeros(len(q_var), bool)
    exh = np.ones(len(q_var), bool)
    if not rlb:
        return has, exh, 0
    g = s.solve_groups(np.array(rlb), np.array(rub), np.array(grp, np.int32), len(idx))
    for i, k in idx.items():
        has[i], exh[i] = g["has_solution"][k], g["exhaustive"][k]
    return has, exh, g["stats"]["nodes"]


def as_answers(has, exh):
    return np.where(has, 1, np.where(exh, 0, -1)).astype(np.int8)


def check_witnesses(pb, lb, ub, q_var, q_val, r, what):
    assert r["wit_lb"].shape[0] == r["wit_ub"].shape[0]
    for i in np.nonzero(r["supported"] == 1)[0]:
        w = int(r["witness"][i])
        if w < 0:
            continue
        assert w < r["wit_lb"].shape[0], (what, i)
        x, v = int(q_var[i]), int(q_val[i])
        rlb, rub = r["wit_lb"][w].copy(), r["wit_ub"][w].copy()
        assert rlb[x] <= v <= rub[x], (what, i)
        rlb[x] = rub[x] = v
        assert any(valid(pb, lb[k], ub[k], rlb, rub) for k in range(lb.shape[0])), (what, i)
    assert (r["witness"][r["supported"] != 1] == -1).all(), what


def brute_domains(pb, lb, ub):
    """The set of values of every variable over the satisfying points of the boxes."""
    doms = [set() for _ in range(pb.nvars)]
    for r in range(lb.shape[0]):
        for pt in itertools.product(*[range(int(a), int(b) + 1) for a, b in zip(lb[r], ub[r])]):
            if all(REL[int(p["op"])](pt[p["x"]], pt[p["y"]], pt[p["z"]]) for p in pb.props):
                for v, x in enumerate(pt):
                    doms[v].add(x)
    return doms


# ---- GPU -----------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_solution_domains_equal_brute_force(eng, opts):
    sat = unsat = 0
    for seed in range(30):
        pb = tnf_gen.random_net(9, 4, 700 + seed, lo=-3, hi=3)
        for lb, ub in ((pb.lb[None, :].copy(), pb.ub[None, :].copy()), cubes(pb, 3)):
            want = brute_domains(pb, lb, ub)
            with eng.Solver(pb, **opts) as s:
                d = s.solution_domains(lb=lb, ub=ub)
            assert d["exact"].all(), seed
            assert all(len(u) == 0 for u in d["unknown"]), seed
            for v in range(pb.nvars):
                assert set(int(x) for x in d["supported"][v]) == want[v], (seed, v)
            if any(want):
                sat += 1
                assert d["has_solution"], seed
            else:
                unsat += 1
                assert not d["has_solution"] and all(len(x) == 0 for x in d["supported"]), seed
    assert sat >= 5 and unsat >= 5


@pytest.mark.gpu
@pytest.mark.parametrize("name", NETWORKS)
def test_supports_equal_the_group_workaround(eng, name):
    pb = network(name)
    lb_all, ub_all = make_roots(pb, 4, seed=11, nfix=1)
    for nboxes, (lb, ub) in ((1, (pb.lb[None, :].copy(), pb.ub[None, :].copy())), (4, (lb_all, ub_all))):
        q_var, q_val = queries(pb, lb, ub, 240, seed=nboxes)
        assert len(q_var) > 0
        for opts in CONFIGS:
            with eng.Solver(pb, **opts) as s:
                r = s.solve_supports(lb, ub, q_var, q_val, witnesses=len(q_var))
                has, exh, _ = workaround(s, pb, lb, ub, q_var, q_val)
            assert np.array_equal(r["supported"] == 1, has), (name, nboxes, opts)
            assert np.array_equal(r["supported"] == 0, ~has & exh), (name, nboxes, opts)
            assert r["wit_lb"].shape[0] <= len(q_var)
            check_witnesses(pb, lb, ub, q_var, q_val, r, (name, nboxes, opts))


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_decided_domains_span_the_hull(eng, opts):
    for name in ("pat2", "sudoku_opt2", "random_opt", "reified_in"):
        pb = network(name)
        vs = [int(v) for v in np.nonzero(referenced(pb) & (pb.ub.astype(np.int64) - pb.lb <= 40))[0][:12]]
        with eng.Solver(pb, **opts) as s:
            d = s.solution_domains(vars=vs)
            h = s.hull(vars=vs)
        for i, v in enumerate(vs):
            if not d["exact"][i]:
                continue
            sup = d["supported"][i]
            if len(sup) == 0:
                assert not h["has_solution"], (name, v)
                continue
            assert h["exact_lb"][i] and h["exact_ub"][i], (name, v)
            assert (int(sup.min()), int(sup.max())) == (int(h["lb"][i]), int(h["ub"][i])), (name, v)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_witness_pool(eng, opts):
    shared = 0
    for name in ("sudoku_opt2", "planted_sat", "random_opt"):
        pb = network(name)
        lb, ub = make_roots(pb, 3, seed=5, nfix=1, empty_frac=0)
        q_var, q_val = queries(pb, lb, ub, 200, seed=3)
        with eng.Solver(pb, **opts) as s:
            big = s.solve_supports(lb, ub, q_var, q_val, witnesses=len(q_var))
            one = s.solve_supports(lb, ub, q_var, q_val, witnesses=1)
            none = s.solve_supports(lb, ub, q_var, q_val, witnesses=0)
        assert np.array_equal(big["supported"], one["supported"]) and np.array_equal(big["supported"], none["supported"])
        assert big["wit_lb"].shape[0] <= len(q_var) and one["wit_lb"].shape[0] <= 1 and none["wit_lb"].shape[0] == 0
        assert (none["witness"] == -1).all()
        if (big["supported"] == 1).any():
            assert (big["witness"][big["supported"] == 1] >= 0).all(), name     # the pool has a row per solution
            assert one["wit_lb"].shape[0] == 1 and (one["witness"] == 0).any(), name
        for r in (big, one):
            check_witnesses(pb, lb, ub, q_var, q_val, r, (name, opts))
        # one solution supports one value of every variable: rows may be shared between queries of different variables
        w = big["witness"][big["supported"] == 1]
        shared += len(set(w.tolist())) < len(w)
    assert shared >= 1


@pytest.mark.gpu
def test_witness_sharing_saves_nodes(eng):
    """One block, a fixed order of search: one call takes no more nodes than the group workaround, whose groups each
    search to their own first solution; strictly fewer on at least one network. The answers are equal."""
    strict = 0
    for name in NETWORKS:
        pb = network(name)
        lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
        q_var, q_val = queries(pb, lb, ub, 120, seed=7)
        with eng.Solver(pb, or_blocks=1, subproblems_power=0) as s:
            r = s.solve_supports(lb, ub, q_var, q_val)
            has, exh, nodes = workaround(s, pb, lb, ub, q_var, q_val)
        assert np.array_equal(r["supported"], as_answers(has, exh)), name
        assert r["stats"]["nodes"] <= nodes, (name, r["stats"]["nodes"], nodes)
        strict += r["stats"]["nodes"] < nodes
    assert strict >= 1


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_edge_cases(eng, opts):
    pb = network("random_opt")
    lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
    want = brute_domains(pb, lb, ub)
    x = int(np.nonzero(referenced(pb) & (pb.lb < pb.ub))[0][0])
    vals = list(range(int(pb.lb[x]), int(pb.ub[x]) + 1))
    with eng.Solver(pb, **opts) as s:
        # duplicates answer alike and name the same row
        r = s.solve_supports(lb, ub, [x] * (2 * len(vals)), vals + vals[::-1], witnesses=64)
        a, b = r["supported"][:len(vals)], r["supported"][len(vals):][::-1]
        assert np.array_equal(a, b) and np.array_equal(r["witness"][:len(vals)], r["witness"][len(vals):][::-1])
        assert set(np.array(vals)[a == 1].tolist()) == want[x] and (a >= 0).all()
        # values outside the root domain: proven unsupported
        r = s.solve_supports(lb, ub, [x, x, x], [int(pb.lb[x]) - 1, int(pb.ub[x]) + 5, abi.NEG_INF + 1])
        assert (r["supported"] == 0).all()
    # an unreferenced variable: every value of its box is supported when the network has a solution
    pb2, _ = golden_io.load("maximize_unconstrained")
    y = [v for v in range(pb2.nvars) if not referenced(pb2)[v]][0]
    lb2, ub2 = pb2.lb.copy(), pb2.ub.copy()
    lb2[y], ub2[y] = -2, 3
    box_lb, box_ub = np.tile(lb2, (2, 1)), np.tile(ub2, (2, 1))
    box_lb[1, y], box_ub[1, y] = 1, 2
    net = abi.Problem(lb2, ub2, pb2.props, pb2.strategies, obj_var=pb2.obj_var, has_eps_strategy=int(pb2.c.has_eps_strategy))
    with eng.Solver(net, **opts) as s:
        r = s.solve_supports(box_lb[1:], box_ub[1:], [y] * 6, list(range(-2, 4)), witnesses=8)
        assert list(r["supported"]) == [0, 0, 0, 1, 1, 0]
        check_witnesses(net, box_lb[1:], box_ub[1:], [y] * 6, list(range(-2, 4)), r, opts)
        d = s.solution_domains(vars=[y], lb=box_lb, ub=box_ub)
        assert list(d["supported"][0]) == list(range(-2, 4)) and d["exact"][0]
    # the objective variable of an optimisation problem, its upper bound narrowed in the boxes
    for seed in range(700, 760):
        pb3 = tnf_gen.random_net(9, 4, seed, lo=-3, hi=3)
        o = pb3.obj_var
        all_dom = brute_domains(pb3, pb3.lb[None, :].copy(), pb3.ub[None, :].copy())
        if o >= 0 and referenced(pb3)[o] and len(all_dom[o]) >= 2:
            break
    else:
        pytest.fail("no network with an objective of two values or more")
    cut = sorted(all_dom[o])[len(all_dom[o]) // 2]
    blb, bub = cubes(pb3, 3)
    bub[:, o] = np.minimum(bub[:, o], cut)
    blb[:, o] = np.minimum(blb[:, o], bub[:, o] + 1)
    want = brute_domains(pb3, blb, bub)
    with eng.Solver(pb3, **opts) as s:
        d = s.solution_domains(lb=blb, ub=bub)
    assert d["exact"].all()
    assert set(int(v) for v in d["supported"][o]) == want[o] == {v for v in all_dom[o] if v <= cut}
    for v in range(pb3.nvars):
        assert set(int(x) for x in d["supported"][v]) == want[v], v


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_budget_answers_are_sound(eng, opts):
    pb = network("sudoku_opt3")
    lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
    q_var, q_val = queries(pb, lb, ub, 400, seed=9)
    with eng.Solver(pb, **opts) as s:
        full = s.solve_supports(lb, ub, q_var, q_val)
    with eng.Solver(pb, cutnodes=30, **opts) as s:
        r = s.solve_supports(lb, ub, q_var, q_val, witnesses=len(q_var))
    assert (r["supported"] == -1).any()
    assert (r["witness"][r["supported"] == 1] >= 0).all()
    check_witnesses(pb, lb, ub, q_var, q_val, r, opts)
    assert (full["supported"][r["supported"] == 0] == 0).all()
    assert (full["supported"][r["supported"] == 1] == 1).all()


def recheck_zeros(eng, pb, lb, ub, q_var, q_val, r, what, **opts):
    zeros = np.nonzero(r["supported"] == 0)[0]
    if len(zeros):
        with eng.Solver(pb, **opts) as s:
            has, exh, _ = workaround(s, pb, lb, ub, q_var[zeros], q_val[zeros])
        assert not has.any() and exh.all(), what


@pytest.mark.gpu
@pytest.mark.parametrize("fp", [abi.FP_WAC1_ACTIVE, abi.FP_AC1_ACTIVE])
def test_active_set_fixpoints_see_the_fixing(eng, fp):
    pb, _ = golden_io.load_simplified_problem("trains15")
    lb, ub = pb.lb[None, :].copy(), pb.ub[None, :].copy()
    q_var, q_val = queries(pb, lb, ub, 24, seed=2)
    with eng.Solver(pb, fixpoint=fp, timeout_ms=3000) as s:
        r = s.solve_supports(lb, ub, q_var, q_val, witnesses=len(q_var))
    assert (r["witness"][r["supported"] == 1] >= 0).all()
    check_witnesses(pb, lb, ub, q_var, q_val, r, fp)
    recheck_zeros(eng, pb, lb, ub, q_var, q_val, r, fp, fixpoint=fp, timeout_ms=3000)


@pytest.mark.gpu
def test_global_placement(eng):
    pb = network("pat2")
    lb, ub = make_roots(pb, 3, seed=2, nfix=1, empty_frac=0)
    q_var, q_val = queries(pb, lb, ub, 80, seed=4)
    with eng.Solver(pb, mem_kind=abi.MEM_GLOBAL) as s:
        r = s.solve_supports(lb, ub, q_var, q_val, witnesses=len(q_var))
    assert (r["witness"][r["supported"] == 1] >= 0).all()
    check_witnesses(pb, lb, ub, q_var, q_val, r, "global")
    recheck_zeros(eng, pb, lb, ub, q_var, q_val, r, "global", mem_kind=abi.MEM_GLOBAL)


@pytest.mark.gpu
@pytest.mark.parametrize("opts", CONFIGS)
def test_other_calls_after_supports(eng, opts):
    for name in ("pat2", "random_opt"):
        pb = network(name)
        lb, ub = make_roots(pb, 12, seed=4)
        q_var, q_val = queries(pb, lb, ub, 150, seed=1)
        x = int(q_var[0])

        def others(s):
            return (s.solve(), s.solve_batch(lb, ub), s.solve_groups(lb, ub, np.arange(12) % 5),
                    s.solve_objectives(lb, ub, [x, x], [0, 1]))
        with eng.Solver(pb, **opts) as s:
            s.solve_supports(lb, ub, q_var, q_val, witnesses=4)
            after = others(s)
        with eng.Solver(pb, **opts) as s:
            fresh = others(s)
        for a, b in zip(after, fresh):
            for key in ("has_solution", "exhaustive", "objective"):
                assert np.array_equal(np.asarray(a[key]), np.asarray(b[key])), (name, key)


@pytest.mark.gpu
def test_rejections(eng):
    from turbo_b200 import engine
    pb = tnf_gen.search_instance(2)
    lb2, ub2 = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    with eng.Solver(pb) as s:
        for qv, qx in (([pb.nvars], [0]), ([-1], [0]), ([], []), ([0], [abi.NEG_INF]), ([0], [abi.POS_INF])):
            with pytest.raises(eng.TurboError) as e:
                s.solve_supports(lb2, ub2, qv, qx)
            assert e.value.status == 1, (qv, qx)
        with pytest.raises(eng.TurboError) as e:
            s.solve_supports(np.zeros((0, pb.nvars), np.int32), np.zeros((0, pb.nvars), np.int32), [0], [0])
        assert e.value.status == 1
        wide_ub = ub2.copy()
        wide_ub[1, 5] += 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_supports(lb2, wide_ub, [0], [0])
        assert e.value.status == 1
        with pytest.raises(eng.TurboError) as e:
            s.solve_supports(lb2, ub2, [0], [0], witnesses=-1)
        assert e.value.status == 1
        one = np.zeros(1, np.int32)
        with pytest.raises(eng.TurboError) as e:          # a pool without rows to write to
            engine._check(engine.lib().tb_solve_supports(s._h, 2, engine._p(lb2), engine._p(ub2), 1, engine._p(one),
                                                         engine._p(one), None, engine._p(one), None, 4, None, None,
                                                         None, None))
        assert e.value.status == 1
        # nq * nboxes above the 40-bit subproblem index, rejected before any allocation
        big = 1 << 21
        qs = np.zeros(big, np.int32)
        with pytest.raises(eng.TurboError) as e:
            engine._check(engine.lib().tb_solve_supports(s._h, big, engine._p(lb2), engine._p(ub2), big, engine._p(qs),
                                                         engine._p(qs), None, engine._p(qs), None, 0, None, None, None,
                                                         None))
        assert e.value.status == 1 and "2^40" in str(e.value)
        s.stream_solutions(4)
        with pytest.raises(eng.TurboError) as e:
            s.solve_supports(lb2, ub2, [0], [0])
        assert e.value.status == 4
    with eng.Solver(pb, mem_kind=abi.MEM_STORE_CLUSTER, cluster_size=2) as s:
        with pytest.raises(eng.TurboError) as e:
            s.solve_supports(lb2, ub2, [0], [0])
        assert e.value.status == 4
    a, b = eng.Solver(pb), eng.Solver(pb)
    try:
        eng.link_peers([a, b])
        with pytest.raises(eng.TurboError) as e:
            a.solve_supports(lb2, ub2, [0], [0])
        assert e.value.status == 4
    finally:
        a.close()
        b.close()

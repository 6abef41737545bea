"""tb_solve_groups against what a user does without it. Prints one JSON line per leg (agreement, nodes, kernel and wall
time of each way, the device and its power limit) and exits 1 if any way disagrees with another.

    python tools/group_solve.py [--seed 0] [--out FILE] [--scenarios 32]

Cube-and-conquer: the root of sudoku_opt3, pat10 and triangular9 (a golden network tb_solve proves optimal in a few
tenths of a second) split into K = 64 and 1024 cubes by bisecting the domains of the first strategy variables. Three
ways: tb_solve on the root; tb_solve_groups with the K cubes in one group (one incumbent for all of them);
tb_solve_batch on the same cubes (an incumbent per cube) reduced on the host.

Holes: S scenarios "x_i != v_i" on planted_opt (x_i a referenced variable, v_i inside its domain): one
tb_solve_groups of 2S roots, {x_i <= v_i - 1} and {x_i >= v_i + 1} in group i, against S sequential create + solve
calls on the network with x_i != v_i added as TNF propagators (the only way to state such a scenario otherwise).
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.batch_solve import device_and_power, emit, referenced  # noqa: E402
from turbo_b200 import abi  # noqa: E402


def split_vars(pb):
    """The variables cubes are cut on: the strategies' variables in order, then every other variable, keeping the
    referenced ones with a finite domain of at least two values."""
    order = [int(v) for _, _, vs in pb.strategies for v in vs] + list(range(pb.nvars))
    ref = referenced(pb)
    seen, out = set(), []
    for v in order:
        if v in seen:
            continue
        seen.add(v)
        if ref[v] and abi.NEG_INF < pb.lb[v] < pb.ub[v] < abi.POS_INF:
            out.append(v)
    return out


def cubes(pb, k, lb=None, ub=None):
    """An exact partition of the box (lb, ub) (default: pb's root) into at least k boxes, or as many as its variables
    allow: the domain of the next split variable is bisected in every box, variable after variable, and again from
    the first one while boxes can still be split. Returns [n, nvars] int32 lb and ub."""
    lb = np.asarray(pb.lb if lb is None else lb, np.int64)
    ub = np.asarray(pb.ub if ub is None else ub, np.int64)
    boxes = [(lb.copy(), ub.copy())]
    vs = split_vars(pb)
    while len(boxes) < k and vs:
        progress = False
        for v in vs:
            if len(boxes) >= k:
                break
            nxt = []
            for l, u in boxes:
                if l[v] < u[v]:
                    mid = l[v] + (u[v] - l[v]) // 2
                    lo_u, hi_l = u.copy(), l.copy()
                    lo_u[v], hi_l[v] = mid, mid + 1
                    nxt += [(l, lo_u), (hi_l, u)]
                    progress = True
                else:
                    nxt.append((l, u))
            boxes = nxt
        if not progress:
            break
    return (np.stack([b[0] for b in boxes]).astype(np.int32), np.stack([b[1] for b in boxes]).astype(np.int32))


def with_disequality(pb, x, v):
    """pb with x != v added as TNF: a constant variable c = v, a result variable r = 0, and r = (x == c)."""
    lb = np.concatenate([pb.lb, [v, 0]]).astype(np.int32)
    ub = np.concatenate([pb.ub, [v, 0]]).astype(np.int32)
    c, r = pb.nvars, pb.nvars + 1
    props = np.array([(int(p["op"]), int(p["x"]), int(p["y"]), int(p["z"])) for p in pb.props] + [(abi.OP_EQ, r, x, c)],
                     np.int32)
    return abi.Problem(lb, ub, props, pb.strategies, obj_var=pb.obj_var, has_eps_strategy=int(pb.c.has_eps_strategy))


def hole_boxes(pb, x, v):
    """{x <= v - 1} and {x >= v + 1}: the root with a hole at x = v, as two boxes."""
    lb, ub = np.tile(pb.lb, (2, 1)), np.tile(pb.ub, (2, 1))
    ub[0, x], lb[1, x] = v - 1, v + 1
    return lb, ub


def progress(*what):
    print(f"[group_solve {time.strftime('%H:%M:%S')}]", *what, file=sys.stderr, flush=True)


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, round((time.perf_counter() - t0) * 1e3, 2)


def cube_leg(name, pb, k):
    from turbo_b200 import engine
    lb, ub = cubes(pb, k)
    n = lb.shape[0]
    with engine.Solver(pb) as s:           # warm-up of all three ways
        s.solve()
        s.solve_groups(lb[:2], ub[:2], [0, 0])
        s.solve_batch(lb[:2], ub[:2])
    with engine.Solver(pb) as s:
        one, one_wall = timed(s.solve)
    with engine.Solver(pb) as s:
        grp, grp_wall = timed(lambda: s.solve_groups(lb, ub, np.zeros(n, np.int32)))
    with engine.Solver(pb) as s:
        bat, bat_wall = timed(lambda: s.solve_batch(lb, ub))
    progress(name, f"K = {n}: solve {one_wall} ms, groups {grp_wall} ms, batch {bat_wall} ms")
    inf = abi.POS_INF
    one_obj = one["objective"] if one["objective"] is not None else inf
    has = bat["has_solution"]
    bat_obj = int(bat["objective"][has].min()) if has.any() else inf
    answers = dict(solve=(one["has_solution"], one["exhaustive"], one_obj),
                   groups=(bool(grp["has_solution"][0]), bool(grp["exhaustive"][0]), int(grp["objective"][0])),
                   batch=(bool(has.any()), bool(bat["exhaustive"].all()), bat_obj))
    agree = len(set(answers.values())) == 1
    leg = lambda r, wall: dict(wall_ms=wall, kernel_ms=round(r["stats"]["kernel_ms"], 2), nodes=r["stats"]["nodes"],
                               subproblems_power=r["stats"]["subproblems_power"])
    dev, power = device_and_power()
    return dict(leg="cubes", workload=name, K=n, objective=one_obj, exhaustive=one["exhaustive"], agree=agree,
                answers={k: list(v) for k, v in answers.items()},
                solve=leg(one, one_wall), groups=leg(grp, grp_wall), batch=leg(bat, bat_wall),
                group_vs_batch_nodes=round(grp["stats"]["nodes"] / max(1, bat["stats"]["nodes"]), 3),
                device=dev, power_limit=power)


def holes_leg(pb, nscen, seed):
    from oracle import oracle_py
    from turbo_b200 import engine
    rng = np.random.default_rng(seed)
    cand = [v for v in split_vars(pb) if pb.ub[v] - pb.lb[v] >= 2]
    xs = rng.choice(cand, size=nscen)
    vals = [int(rng.integers(pb.lb[x] + 1, pb.ub[x])) for x in xs]
    lb = np.vstack([hole_boxes(pb, x, v)[0] for x, v in zip(xs, vals)])
    ub = np.vstack([hole_boxes(pb, x, v)[1] for x, v in zip(xs, vals)])
    groups = np.repeat(np.arange(nscen, dtype=np.int32), 2)
    nets = [with_disequality(pb, int(x), v) for x, v in zip(xs, vals)]
    with engine.Solver(pb) as s:
        s.solve_groups(lb[:2], ub[:2], [0, 0])
    with engine.Solver(nets[0]) as s:
        s.solve()
    t0 = time.perf_counter()
    with engine.Solver(pb) as s:
        g = s.solve_groups(lb, ub, groups)
    grp_wall = (time.perf_counter() - t0) * 1e3
    seq = []
    t0 = time.perf_counter()
    for net in nets:
        with engine.Solver(net) as s:
            seq.append(s.solve())
    seq_wall = (time.perf_counter() - t0) * 1e3
    progress("holes", f"S = {nscen}: groups {grp_wall:.1f} ms, sequential {seq_wall:.1f} ms")
    bad, bad_oracle, invalid = [], [], 0
    for i, (x, v) in enumerate(zip(xs, vals)):
        q = seq[i]
        q_obj = q["objective"] if q["objective"] is not None else abi.POS_INF
        mine = (bool(g["has_solution"][i]), bool(g["exhaustive"][i]), int(g["objective"][i]))
        if mine != (q["has_solution"], q["exhaustive"], q_obj):
            bad.append(i)
        if i < 8:                              # the oracle on a few scenarios, as a third opinion
            o = oracle_py.solve(nets[i])
            o_obj = o["objective"] if o["objective"] is not None else abi.POS_INF
            if mine != (o["has_solution"], o["exhaustive"], o_obj):
                bad_oracle.append(i)
        if g["has_solution"][i] and g["lb"][i][x] == v:
            invalid += 1
    dev, power = device_and_power()
    return dict(leg="holes", workload="planted_opt", S=nscen, roots=2 * nscen,
                groups=dict(wall_ms=round(grp_wall, 2), kernel_ms=round(g["stats"]["kernel_ms"], 2), nodes=g["stats"]["nodes"],
                            scenarios_per_s=round(nscen / grp_wall * 1e3, 1)),
                sequential=dict(wall_ms=round(seq_wall, 2), kernel_ms=round(sum(q["stats"]["kernel_ms"] for q in seq), 2),
                                nodes=sum(q["stats"]["nodes"] for q in seq), scenarios_per_s=round(nscen / seq_wall * 1e3, 1)),
                wall_ratio=round(seq_wall / grp_wall, 2), agree=not bad and not bad_oracle and not invalid,
                disagreeing=bad[:20], disagreeing_with_oracle=bad_oracle, stores_on_the_hole=invalid,
                device=dev, power_limit=power)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--scenarios", type=int, default=32)
    a = ap.parse_args()
    from tests import golden_io, tnf_gen
    from turbo_b200 import engine
    if engine.device_count() < 1:
        sys.exit("group_solve.py needs a CUDA device: the engine has no CPU fallback")
    lines = []
    for net in ("sudoku_opt3", "pat10", "triangular9"):
        pb, _ = golden_io.load(net)
        for k in (64, 1024):
            lines.append(emit(cube_leg(net, pb, k), a.out))
    lines.append(emit(holes_leg(tnf_gen.search_instance(3), a.scenarios, a.seed), a.out))
    if not all(r["agree"] for r in lines):
        sys.exit("the ways disagree")


if __name__ == "__main__":
    main()

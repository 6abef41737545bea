"""tb_solve_front against what a user does without it. Prints one JSON line per leg (the levels, and per way wall and
kernel time, nodes, front size and proven points, with the device and its power limit) and exits 1 if two exhaustive
answers disagree.

    python tools/front_solve.py [--out FILE] [--max-levels 256] [--budget-ms 20000] [--accap-budget-ms 4000]

Legs: sudoku_opt3, pat10 and triangular9, x = the problem's objective variable and y = the referenced variable other
than x with the widest finite root range, once minimised and once maximised; and simplified accap_a3 the same way under
a few-second budget. Levels: one per value of x's range at the root fixpoint (Solver.propagate), or a fixed step where
that range has more than --max-levels values; the JSON line records the step. Three ways:
  (a) one Solver.pareto_front call;
  (b) one tb_solve_groups launch with the nested box x <= t per level, on the network with obj_var = y (the negation
      network for max y): what the disjoint slices and the dominance sharing save;
  (c) the sequential epsilon-constraint loop of create + tb_solve: minimise y subject to x <= t, read x*, set
      t = x* - 1, until there is no solution (what a user does today).
A budget applies to the whole of each way. Answers are compared level by level where both ways are exhaustive (ways (a)
and (c) as a whole): the value of ways (a) and (c) at level t is the best y of their points with x <= t.
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.batch_solve import device_and_power, emit, referenced  # noqa: E402
from tools.objective_solve import negation_network, with_objective  # noqa: E402
from turbo_b200 import abi  # noqa: E402


def axes(pb):
    """(x, y): x = the problem's objective variable when the propagators read it (else the referenced variable of the
    widest finite root range), y = the referenced variable other than x with the widest finite root range."""
    ref = referenced(pb)
    finite = ref & (pb.lb > abi.NEG_INF) & (pb.ub < abi.POS_INF)
    width = pb.ub.astype(np.int64) - pb.lb
    by_width = sorted(np.nonzero(finite)[0], key=lambda v: (-width[v], v))
    x = pb.obj_var if pb.obj_var >= 0 and ref[pb.obj_var] else int(by_width[0])
    return int(x), int([v for v in by_width if v != x][0])


def levels_of(lo, hi, cap):
    """One level per value of [lo, hi], or every step-th value (and hi) where there are more than `cap`. Returns the
    levels and the step."""
    step = max(1, -(-(hi - lo + 1) // cap))
    lv = list(range(lo, hi + 1, step))
    if lv[-1] != hi:
        lv.append(hi)
    return np.array(lv, np.int64), step


def side(lb, ub, x, t, maximize_x):
    """The boxes narrowed to x <= t (x >= t when maximising x)."""
    lb, ub = np.array(lb, np.int64), np.array(ub, np.int64)
    if maximize_x:
        lb[:, x] = np.maximum(lb[:, x], t)
    else:
        ub[:, x] = np.minimum(ub[:, x], t)
    return lb, ub


def objective_network(pb, y, maximize_y):
    """pb minimising y, or the negation network for max y: (network, its objective variable)."""
    return negation_network(pb, y) if maximize_y else (with_objective(pb, y), y)


def extend(net, lb, ub):
    """Boxes of pb extended with the root bounds of the variables the network adds."""
    n0 = lb.shape[1]
    k = lb.shape[0]
    return (np.hstack([lb, np.tile(net.lb[n0:], (k, 1))]).astype(np.int32),
            np.hstack([ub, np.tile(net.ub[n0:], (k, 1))]).astype(np.int32))


def y_value(o, maximize_y):
    """The value in y's own sense of a minimisation of the objective network's variable."""
    if not maximize_y:
        return int(o)
    return abi.POS_INF if int(o) == abi.NEG_INF else -int(o)


def nested_groups(pb, lb, ub, x, y, levels, maximize_x, maximize_y, **opts):
    """Way (b): one tb_solve_groups launch, group i = every box narrowed to level i's side, on the network optimising y.
    Returns per-level has_solution / exhaustive / objective (y's sense) and the stats."""
    from turbo_b200 import engine
    net, n = objective_network(pb, y, maximize_y)
    rlb, rub, grp = [], [], []
    for i, t in enumerate(levels):
        a, b = side(lb, ub, x, int(t), maximize_x)
        a, b = extend(net, a, b)
        rlb.append(a)
        rub.append(b)
        grp += [i] * a.shape[0]
    with engine.Solver(net, **opts) as s:
        g = s.solve_groups(np.vstack(rlb), np.vstack(rub), np.array(grp, np.int32), len(levels))
    obj = np.array([y_value(o, maximize_y) if h else abi.POS_INF for o, h in zip(g["objective"], g["has_solution"])],
                   np.int64)
    return dict(has_solution=g["has_solution"], exhaustive=g["exhaustive"], objective=obj, stats=g["stats"])


def epsilon_loop(pb, x, y, maximize_x, maximize_y, budget_ms=0):
    """Way (c) over the root: minimise (maximise) y subject to x <= t (x >= t), read x*, set t = x* - 1 (x* + 1), until
    there is no solution. Returns the points [(x*, y*)], whether every solve was exhaustive, calls, nodes, kernel ms."""
    from turbo_b200 import engine
    net, n = objective_network(pb, y, maximize_y)
    t = None
    pts, exhaustive, calls, nodes, kernel = [], True, 0, 0, 0.0
    t0 = time.perf_counter()
    while True:
        left = budget_ms - (time.perf_counter() - t0) * 1e3 if budget_ms else 0
        if budget_ms and left <= 0:
            exhaustive = False
            break
        lb, ub = net.lb.copy(), net.ub.copy()
        if t is not None:
            if maximize_x:
                lb[x] = max(int(lb[x]), t)
            else:
                ub[x] = min(int(ub[x]), t)
        calls += 1
        if lb[x] > ub[x]:
            break
        root = abi.Problem(lb, ub, net.props, net.strategies, obj_var=n, has_eps_strategy=int(net.c.has_eps_strategy))
        with engine.Solver(root, timeout_ms=int(left)) as s:
            r = s.solve()
        nodes += r["stats"]["nodes"]
        kernel += r["stats"]["kernel_ms"]
        exhaustive &= bool(r["exhaustive"])
        if not r["has_solution"]:
            break
        xs = int(r["lb"][x])
        pts.append((xs, y_value(r["lb"][n], maximize_y)))
        if xs in (abi.NEG_INF, abi.POS_INF) or not r["exhaustive"]:
            break
        t = xs + 1 if maximize_x else xs - 1
    return pts, exhaustive, calls, nodes, kernel, (time.perf_counter() - t0) * 1e3


def loop_levels(pts, levels, maximize_x, maximize_y):
    """A way's answer per level from its points: the best y of the points on the level's side (None: no point)."""
    out = []
    for t in levels:
        vals = [py for px, py in pts if (px >= t if maximize_x else px <= t)]
        out.append((max(vals) if maximize_y else min(vals)) if vals else None)
    return out


def front_size(values, maximize_x, maximize_y):
    """The number of levels whose value strictly improves on every level before them in x's preferred order."""
    best, k = None, 0
    for v in (values[::-1] if maximize_x else values):
        if v is None:
            continue
        key = -v if maximize_y else v
        if best is None or key < best:
            best, k = key, k + 1
    return k


def front_leg(name, pb, x, y, maximize_y, max_levels, budget_ms):
    from turbo_b200 import engine
    with engine.Solver(pb) as s:
        root = s.propagate()
    lo, hi = int(root["lb"][x]), int(root["ub"][x])
    levels, step = levels_of(lo, hi, max_levels)
    one_box = (pb.lb[None, :].copy(), pb.ub[None, :].copy())
    # warm-up of every way
    with engine.Solver(pb, timeout_ms=100) as s:
        s.solve_front(*one_box, x, y, levels[:2], False, maximize_y)
    nested_groups(pb, *one_box, x, y, levels[:2], False, maximize_y, timeout_ms=100)
    epsilon_loop(pb, x, y, False, maximize_y, 100)

    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms) as s:
        a = s.pareto_front(x, y, maximize_y=maximize_y, levels=levels)
    a_wall = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    b = nested_groups(pb, *one_box, x, y, levels, False, maximize_y, timeout_ms=budget_ms)
    b_wall = (time.perf_counter() - t0) * 1e3
    pts, c_exh, calls, c_nodes, c_kernel, c_wall = epsilon_loop(pb, x, y, False, maximize_y, budget_ms)
    # per level, the best y of a way's points on its side (the value of the last front level at or before it)
    a_vals = loop_levels(a["points"], levels, False, maximize_y)
    b_vals = [int(v) if h else None for v, h in zip(b["objective"], b["has_solution"])]
    c_vals = loop_levels(pts, levels, False, maximize_y)
    bad = [i for i in range(len(levels))
           if (a["exact"] and b["exhaustive"][i] and a_vals[i] != b_vals[i])
           or (a["exact"] and c_exh and a_vals[i] != c_vals[i])
           or (b["exhaustive"][i] and c_exh and b_vals[i] != c_vals[i])]
    dev, power = device_and_power()
    return dict(workload=name, x=x, y=y, maximize_y=bool(maximize_y), x_range=[lo, hi], levels=len(levels),
                level_step=step, budget_ms=budget_ms,
                one_call=dict(wall_ms=round(a_wall, 2), kernel_ms=round(a["stats"]["kernel_ms"], 2),
                              nodes=a["stats"]["nodes"], front=len(a["points"]), proven_points=int(a["proven"].sum()),
                              exact=a["exact"], subproblems_power=a["stats"]["subproblems_power"]),
                nested_groups=dict(wall_ms=round(b_wall, 2), kernel_ms=round(b["stats"]["kernel_ms"], 2),
                                   nodes=b["stats"]["nodes"], front=front_size(b_vals, False, maximize_y),
                                   proven_levels=int(b["exhaustive"].sum())),
                epsilon_loop=dict(wall_ms=round(c_wall, 2), kernel_ms=round(c_kernel, 2), nodes=c_nodes, calls=calls,
                                  front=front_size(c_vals, False, maximize_y), exact=c_exh),
                points=a["points"][:64], agree=not bad, disagreeing_levels=[int(levels[i]) for i in bad[:20]],
                device=dev, power_limit=power)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--max-levels", type=int, default=256, help="levels per front before a step is used")
    ap.add_argument("--budget-ms", type=int, default=20000, help="budget of each way on the golden legs (0 = none)")
    ap.add_argument("--accap-budget-ms", type=int, default=4000)
    a = ap.parse_args()
    from tests import golden_io
    from turbo_b200 import engine
    if engine.device_count() < 1:
        sys.exit("front_solve.py needs a CUDA device: the engine has no CPU fallback")
    lines = []
    legs = [(net, golden_io.load(net)[0], a.budget_ms) for net in ("sudoku_opt3", "pat10", "triangular9")]
    legs.append(("simplified:accap_a3", golden_io.load_simplified_problem("accap_a3")[0], a.accap_budget_ms))
    for name, pb, budget in legs:
        x, y = axes(pb)
        for my in (0, 1):
            print(f"[front_solve {time.strftime('%H:%M:%S')}] {name} max_y={my}", file=sys.stderr, flush=True)
            lines.append(emit(front_leg(name, pb, x, y, my, a.max_levels, budget), a.out))
    if not all(r["agree"] for r in lines):
        sys.exit("exhaustive answers disagree")


if __name__ == "__main__":
    main()

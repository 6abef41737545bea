"""tb_solve_objectives against what a user does without it. Prints one JSON line per leg (agreement, nodes, kernel and
wall time of each way, the device and its power limit) and exits 1 if two exhaustive answers disagree.

    python tools/objective_solve.py [--out FILE] [--seq-vars 32] [--budget-ms 20000] [--accap-budget-ms 4000]

Solution hull: min and max of every referenced variable of sudoku_opt3, pat10 and triangular9 over the root, and of
32 strategy variables of simplified accap_a3 under a few-second budget. Three ways:
  (a) one tb_solve_objectives call with the 2n objectives;
  (b) 2n tb_solve_objectives calls of one objective each (what witness sharing saves);
  (c) 2n sequential create + tb_solve, on the network with obj_var = v for the minimum, and with a negation variable
      n, 0 = v + n and obj_var = n for the maximum (what a user does today).
Ways (b) and (c) take the first --seq-vars variables (2 * seq-vars objectives) of a leg; the JSON line says how many.
A budget applies to the whole of way (a) and is split evenly over the calls of (b) and (c); only answers that are
exhaustive on both sides are compared.
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
from turbo_b200 import abi  # noqa: E402


def with_objective(pb, v):
    """pb minimising variable v."""
    return abi.Problem(pb.lb, pb.ub, pb.props, pb.strategies, obj_var=int(v), has_eps_strategy=int(pb.c.has_eps_strategy))


def negation_network(pb, v):
    """pb with a constant c = 0, a negation variable n in [-ub(v), -lb(v)] and c = v + n, minimising n: its optimum is
    -max(v). Returns the problem and n."""
    neg = lambda b: abi.POS_INF if b == abi.NEG_INF else (abi.NEG_INF if b == abi.POS_INF else -int(b))
    c, n = pb.nvars, pb.nvars + 1
    lb = np.concatenate([pb.lb, [0, neg(pb.ub[v])]]).astype(np.int32)
    ub = np.concatenate([pb.ub, [0, neg(pb.lb[v])]]).astype(np.int32)
    props = np.array([tuple(int(p[k]) for k in ("op", "x", "y", "z")) for p in pb.props] + [(abi.OP_ADD, c, int(v), n)],
                     np.int32)
    return abi.Problem(lb, ub, props, pb.strategies, obj_var=n, has_eps_strategy=int(pb.c.has_eps_strategy)), n


def progress(*what):
    print(f"[objective_solve {time.strftime('%H:%M:%S')}]", *what, file=sys.stderr, flush=True)


def sequential(pb, vs, budget_ms):
    """Way (c): one create + solve per objective; answers as (has_solution, exhaustive, value)."""
    from turbo_b200 import engine
    per = budget_ms // (2 * len(vs)) if budget_ms else 0
    out, nodes, kernel = [], 0, 0.0
    t0 = time.perf_counter()
    for mx in (0, 1):
        for v in vs:
            if mx:
                net, n = negation_network(pb, v)
            else:
                net, n = with_objective(pb, v), v
            with engine.Solver(net, timeout_ms=per) as s:
                r = s.solve()
            val = abi.POS_INF
            if r["has_solution"]:
                val = int(r["lb"][n])
                if mx:
                    val = abi.POS_INF if val == abi.NEG_INF else -val
            out.append((r["has_solution"], r["exhaustive"], val))
            nodes += r["stats"]["nodes"]
            kernel += r["stats"]["kernel_ms"]
    return out, nodes, kernel, (time.perf_counter() - t0) * 1e3


def singles(pb, vs, budget_ms):
    """Way (b): one tb_solve_objectives call per objective on one solver."""
    from turbo_b200 import engine
    per = budget_ms // (2 * len(vs)) if budget_ms else 0
    out, nodes, kernel = [], 0, 0.0
    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=per) as s:
        for mx in (0, 1):
            for v in vs:
                r = s.solve_objectives(pb.lb, pb.ub, [v], [mx])
                out.append((bool(r["has_solution"][0]), bool(r["exhaustive"][0]), int(r["objective"][0])))
                nodes += r["stats"]["nodes"]
                kernel += r["stats"]["kernel_ms"]
    return out, nodes, kernel, (time.perf_counter() - t0) * 1e3


def disagreements(a, b):
    """Indices where both answers are exhaustive and differ."""
    return [i for i, (x, y) in enumerate(zip(a, b)) if x[1] and y[1] and x != y]


def hull_leg(name, pb, vs, seq_vars, budget_ms):
    from turbo_b200 import engine
    vs = [int(v) for v in vs]
    sv = vs[:seq_vars]
    with engine.Solver(pb) as s:                     # warm-up of every way
        s.solve_objectives(pb.lb, pb.ub, [vs[0], vs[0]], [0, 1])
    with engine.Solver(negation_network(pb, vs[0])[0], timeout_ms=100) as s:
        s.solve()
    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms) as s:
        h = s.hull(vars=vs)
    one_wall = (time.perf_counter() - t0) * 1e3
    k = len(vs)
    one = [(bool(h["has_solution"]), bool(h["exact_lb"][i]), int(h["lb"][i]) if h["has_solution"] else abi.POS_INF)
           for i in range(k)]
    one += [(bool(h["has_solution"]), bool(h["exact_ub"][i]), int(h["ub"][i]) if h["has_solution"] else abi.POS_INF)
            for i in range(k)]
    progress(name, f"{2 * k} objectives in one call: {one_wall:.1f} ms")
    sub = [one[i] for i in range(len(sv))] + [one[k + i] for i in range(len(sv))]
    sin, sin_nodes, sin_kernel, sin_wall = singles(pb, sv, budget_ms)
    progress(name, f"{2 * len(sv)} single-objective calls: {sin_wall:.1f} ms")
    seq, seq_nodes, seq_kernel, seq_wall = sequential(pb, sv, budget_ms)
    progress(name, f"{2 * len(sv)} sequential create + solve: {seq_wall:.1f} ms")
    bad = sorted(set(disagreements(sub, sin)) | set(disagreements(sub, seq)) | set(disagreements(sin, seq)))
    dev, power = device_and_power()
    return dict(leg="hull", workload=name, variables=k, objectives=2 * k, budget_ms=budget_ms,
                one_call=dict(wall_ms=round(one_wall, 2), kernel_ms=round(h["stats"]["kernel_ms"], 2),
                              nodes=h["stats"]["nodes"], exact_sides=int(h["exact_lb"].sum() + h["exact_ub"].sum()),
                              subproblems_power=h["stats"]["subproblems_power"]),
                sequential_objectives=2 * len(sv),
                single_objective_calls=dict(wall_ms=round(sin_wall, 2), kernel_ms=round(sin_kernel, 2), nodes=sin_nodes,
                                            exact=sum(a[1] for a in sin)),
                sequential_solves=dict(wall_ms=round(seq_wall, 2), kernel_ms=round(seq_kernel, 2), nodes=seq_nodes,
                                       exact=sum(a[1] for a in seq)),
                one_call_exact_of_sequential=sum(a[1] for a in sub),
                # wall time per objective of way (c) over that of way (a)
                per_objective_wall_ratio=round((seq_wall / (2 * len(sv))) / max(1e-9, one_wall / (2 * k)), 2),
                agree=not bad, disagreeing=bad[:20], device=dev, power_limit=power)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--seq-vars", type=int, default=32, help="variables of ways (b) and (c) per leg")
    ap.add_argument("--budget-ms", type=int, default=20000, help="budget of the golden legs (0 = none)")
    ap.add_argument("--accap-budget-ms", type=int, default=4000)
    a = ap.parse_args()
    from tests import golden_io
    from turbo_b200 import engine
    if engine.device_count() < 1:
        sys.exit("objective_solve.py needs a CUDA device: the engine has no CPU fallback")
    lines = []
    for net in ("sudoku_opt3", "pat10", "triangular9"):
        pb, _ = golden_io.load(net)
        vs = np.nonzero(referenced(pb))[0]
        lines.append(emit(hull_leg(net, pb, vs, a.seq_vars, a.budget_ms), a.out))
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    seen, vs = set(), []                            # the strategies' variables, then other referenced ones
    for v in [int(v) for _, _, s in pb.strategies for v in s] + list(np.nonzero(referenced(pb))[0]):
        if int(v) not in seen and pb.lb[v] < pb.ub[v]:
            seen.add(int(v))
            vs.append(int(v))
    lines.append(emit(hull_leg("simplified:accap_a3", pb, vs[:32], a.seq_vars, a.accap_budget_ms), a.out))
    if not all(r["agree"] for r in lines):
        sys.exit("exhaustive answers disagree")


if __name__ == "__main__":
    main()

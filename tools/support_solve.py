"""tb_solve_supports against what a user does without it. Prints one JSON line per leg (answers, agreement, nodes,
kernel and wall time of each way, witness rows, the device and its power limit) and exits 1 if two decided answers
disagree.

    python tools/support_solve.py [--out FILE] [--group-queries 4096] [--budget-ms 20000] [--accap-budget-ms 4000]

Solution domains: every value of every referenced variable of sudoku_opt3, pat10 and triangular9 over the root, and of
up to 32 strategy variables of simplified accap_a3, its objective's upper bound narrowed to the value of a first solve,
under a few-second budget. Three ways:
  (a) one tb_solve_supports call with a query per (variable, value) and a witness row per query;
  (b) tb_solve_groups with one satisfaction group per query and the x = v box materialised (what a user does today),
      on the first --group-queries queries (each group has a best row of the network's size);
  (c) Solver.hull of the same variables: the bounds only, to show what the answer per value costs.
A budget applies to each call. Answers of (a) and (b) are compared where both are decided (1 or 0).
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


def progress(*what):
    print(f"[support_solve {time.strftime('%H:%M:%S')}]", *what, file=sys.stderr, flush=True)


def counts(ans):
    return {"1": int((ans == 1).sum()), "0": int((ans == 0).sum()), "-1": int((ans == -1).sum())}


def value_queries(lb, ub, vs):
    q_var = np.concatenate([np.full(int(ub[v]) - int(lb[v]) + 1, v, np.int32) for v in vs])
    q_val = np.concatenate([np.arange(int(lb[v]), int(ub[v]) + 1, dtype=np.int32) for v in vs])
    return q_var, q_val


def group_way(pb, lb, ub, q_var, q_val, budget_ms):
    """Way (b): one group per query, box with x = v. Answers 1 / 0 / -1 as tb_solve_supports gives them."""
    from turbo_b200 import engine
    n = len(q_var)
    glb, gub = np.tile(lb, (n, 1)), np.tile(ub, (n, 1))
    glb[np.arange(n), q_var] = q_val
    gub[np.arange(n), q_var] = q_val
    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms) as s:
        g = s.solve_groups(glb, gub, np.arange(n, dtype=np.int32), n)
    wall = (time.perf_counter() - t0) * 1e3
    ans = np.where(g["has_solution"], 1, np.where(g["exhaustive"], 0, -1)).astype(np.int8)
    return ans, g["stats"], wall


def leg(name, pb, lb, ub, vs, group_queries, budget_ms):
    from turbo_b200 import engine
    vs = [int(v) for v in vs]
    q_var, q_val = value_queries(lb, ub, vs)
    nq = len(q_var)
    with engine.Solver(pb, timeout_ms=1000) as s:   # warm-up of every way (bounded: a query may be hard)
        s.solve_supports(lb, ub, q_var[:2], q_val[:2], witnesses=2)
        s.solve_groups(np.tile(lb, (2, 1)), np.tile(ub, (2, 1)), np.arange(2, dtype=np.int32), 2)
        s.hull(vars=vs[:1], lb=lb, ub=ub)
    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms) as s:
        a = s.solve_supports(lb, ub, q_var, q_val, witnesses=nq)
    a_wall = (time.perf_counter() - t0) * 1e3
    progress(name, f"{nq} queries in one tb_solve_supports: {a_wall:.1f} ms")
    m = min(nq, group_queries)
    b, b_stats, b_wall = group_way(pb, lb, ub, q_var[:m], q_val[:m], budget_ms)
    progress(name, f"{m} groups in one tb_solve_groups: {b_wall:.1f} ms")
    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms) as s:
        h = s.hull(vars=vs, lb=lb, ub=ub)
    c_wall = (time.perf_counter() - t0) * 1e3
    progress(name, f"hull of {len(vs)} variables: {c_wall:.1f} ms")
    sup = a["supported"]
    both = (sup[:m] >= 0) & (b >= 0)
    bad = np.nonzero(both & (sup[:m] != b))[0]
    # the hull's exact sides against the supported values of variables whose every value was decided
    hull_bad = []
    for i, v in enumerate(vs):
        ans = sup[q_var == v]
        vals = q_val[q_var == v][ans == 1]
        if (ans >= 0).all() and len(vals) and h["exact_lb"][i] and h["exact_ub"][i]:
            if (int(vals.min()), int(vals.max())) != (int(h["lb"][i]), int(h["ub"][i])):
                hull_bad.append(v)
    dev, power = device_and_power()
    return dict(leg="supports", workload=name, variables=len(vs), queries=nq, budget_ms=budget_ms,
                one_call=dict(answers=counts(sup), wall_ms=round(a_wall, 2), kernel_ms=round(a["stats"]["kernel_ms"], 2),
                              nodes=a["stats"]["nodes"], witness_rows=int(a["wit_lb"].shape[0]),
                              subproblems_power=a["stats"]["subproblems_power"]),
                group_queries=m,
                groups=dict(answers=counts(b), wall_ms=round(b_wall, 2), kernel_ms=round(b_stats["kernel_ms"], 2),
                            nodes=b_stats["nodes"], witness_rows=int((b == 1).sum())),
                one_call_on_group_queries=counts(sup[:m]), compared=int(both.sum()),
                hull=dict(wall_ms=round(c_wall, 2), kernel_ms=round(h["stats"]["kernel_ms"], 2), nodes=h["stats"]["nodes"],
                          exact_sides=int(h["exact_lb"].sum() + h["exact_ub"].sum())),
                agree=not len(bad) and not hull_bad, disagreeing=[int(i) for i in bad[:20]], hull_disagreeing=hull_bad[:20],
                device=dev, power_limit=power)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--group-queries", type=int, default=4096, help="queries of way (b) per leg")
    ap.add_argument("--budget-ms", type=int, default=20000, help="budget of each call of the golden legs (0 = none)")
    ap.add_argument("--accap-budget-ms", type=int, default=4000)
    a = ap.parse_args()
    from tests import golden_io
    from turbo_b200 import engine
    if engine.device_count() < 1:
        sys.exit("support_solve.py needs a CUDA device: the engine has no CPU fallback")
    lines = []
    for net in ("sudoku_opt3", "pat10", "triangular9"):
        pb, _ = golden_io.load(net)
        vs = np.nonzero(referenced(pb))[0]
        lines.append(emit(leg(net, pb, pb.lb.copy(), pb.ub.copy(), vs, a.group_queries, a.budget_ms), a.out))
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    with engine.Solver(pb, timeout_ms=a.accap_budget_ms) as s:
        first = s.solve()
    lb, ub = pb.lb.copy(), pb.ub.copy()
    if first["has_solution"]:
        ub[pb.obj_var] = first["objective"]      # solutions at least as good as the first solve's
    seen, vs = set(), []
    for v in [int(v) for _, _, st in pb.strategies for v in st]:
        if v not in seen and lb[v] < ub[v] and int(ub[v]) - int(lb[v]) < 64:
            seen.add(v)
            vs.append(v)
    lines.append(emit(leg("simplified:accap_a3", pb, lb, ub, vs[:32], a.group_queries, a.accap_budget_ms), a.out))
    if not all(r["agree"] for r in lines):
        sys.exit("decided answers disagree")


if __name__ == "__main__":
    main()

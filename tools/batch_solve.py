"""tb_solve_batch against what a user does without it: K roots of one network solved in one launch, and the same K
roots solved one after another, each with a solver created from that root. Prints one JSON line per workload (K, d,
wall and kernel time of both ways, roots/s, nodes/s, the device and its power limit) after checking that every root
agrees between the two ways and that every returned store is a solution inside its root's box.

    python tools/batch_solve.py [--seed 0] [--out FILE] [--k-tiny 2048] [--k-accap 64] [--budget-ms 4000]

Workloads: sudoku_opt3 and pat10 (tiny networks: a node is all search bookkeeping) with K in the thousands, and
simplified accap_a3 with K = 64 under a wall budget (the same total for both ways: the sequential solves get
budget / K each): roots around a solution the engine finds in a second, K / 8 of them with 40 free variables (a window
of +-2 around their value), the others with 6; that batch is also timed with one subproblem per root (d = 0).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from turbo_b200 import abi  # noqa: E402

def _tdiv(y, z):
    q = abs(y) // abs(z)
    return q if (y >= 0) == (z > 0) else -q


REL = {
    abi.OP_ADD: lambda x, y, z: x == y + z,
    abi.OP_MUL: lambda x, y, z: x == y * z,
    abi.OP_TDIV: lambda x, y, z: z != 0 and x == _tdiv(y, z),
    abi.OP_TMOD: lambda x, y, z: z != 0 and x == y - z * _tdiv(y, z),
    abi.OP_MIN: lambda x, y, z: x == min(y, z),
    abi.OP_MAX: lambda x, y, z: x == max(y, z),
    abi.OP_EQ: lambda x, y, z: x in (0, 1) and x == int(y == z),
    abi.OP_LEQ: lambda x, y, z: x in (0, 1) and x == int(y <= z),
}


def referenced(pb):
    r = np.zeros(pb.nvars, bool)
    for k in ("x", "y", "z"):
        r[pb.props[k]] = True
    return r


def make_roots(pb, k, seed, nfix=3, empty_frac=0.05, around=None, free=None):
    """k narrowings of pb's root, reproducible from `seed`: each fixes `nfix` referenced variables to values of their
    domain or narrows them to a sub-interval; a share `empty_frac` also gets one empty domain (no solution, decided
    at the root). With `around` (a solution store) every referenced variable except `free` random ones is fixed to its
    value there, and the free ones keep a window of +-2 around it: easy roots of a hard network."""
    rng = np.random.default_rng(seed)
    ref = np.nonzero(referenced(pb))[0]
    lb = np.tile(np.asarray(pb.lb, np.int64), (k, 1))
    ub = np.tile(np.asarray(pb.ub, np.int64), (k, 1))
    open_vars = ref[(pb.lb[ref] < pb.ub[ref]) & (pb.lb[ref] > abi.NEG_INF) & (pb.ub[ref] < abi.POS_INF)]
    for r in range(k):
        if around is not None:
            keep = rng.choice(open_vars, size=min(free, len(open_vars)), replace=False)
            fix = np.setdiff1d(open_vars, keep)
            lb[r, fix] = ub[r, fix] = around[fix]
            lb[r, keep] = np.maximum(pb.lb[keep], around[keep] - 2)
            ub[r, keep] = np.minimum(pb.ub[keep], around[keep] + 2)
        else:
            for v in rng.choice(open_vars, size=min(nfix, len(open_vars)), replace=False):
                a, b = sorted(int(t) for t in rng.integers(int(pb.lb[v]), int(pb.ub[v]) + 1, size=2))
                if rng.random() < 0.5:
                    lb[r, v] = ub[r, v] = a
                else:
                    lb[r, v], ub[r, v] = a, b
        if rng.random() < empty_frac and len(open_vars):
            v = int(rng.choice(open_vars))
            lb[r, v], ub[r, v] = pb.ub[v], pb.lb[v]
    return lb.astype(np.int32), ub.astype(np.int32)


def root_problem(pb, lb, ub):
    return abi.Problem(lb, ub, pb.props, pb.strategies, obj_var=pb.obj_var, has_eps_strategy=int(pb.c.has_eps_strategy))


def valid(pb, lb, ub, slb, sub):
    """The store is inside the root's box and entails every propagator (checked at its lower bounds)."""
    if np.any(slb < lb) or np.any(sub > ub) or np.any(slb > sub):
        return False
    return all(REL[int(p["op"])](int(slb[p["x"]]), int(slb[p["y"]]), int(slb[p["z"]])) for p in pb.props)


def agree(a_has, a_exh, a_obj, b_has, b_exh, b_obj, budget=False):
    """Two answers for one root are compatible: equal when both searches ended, and never contradicting a proof. Without
    a budget both searches run to their end, so exhaustiveness must be equal too (a satisfaction root that found its
    solution is not exhaustive)."""
    if not budget and a_exh != b_exh:
        return False
    if a_exh and b_exh:
        return a_has == b_has and a_obj == b_obj
    if a_exh or b_exh:
        (p_has, p_obj), (o_has, o_obj) = ((a_has, a_obj), (b_has, b_obj)) if a_exh else ((b_has, b_obj), (a_has, a_obj))
        return (p_has or not o_has) and (not o_has or o_obj >= p_obj)
    return True


def device_and_power():
    from turbo_b200 import engine
    name = engine.device_info(0)["name"]
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q or "unknown"


def progress(*what):
    print(f"[batch_solve {time.strftime('%H:%M:%S')}]", *what, file=sys.stderr, flush=True)


def run(name, pb, lb, ub, opts, budget_ms=0, alt_sub=None):
    from turbo_b200 import engine
    k = lb.shape[0]
    progress(name, "K =", k, "warm-up")
    # warm-up: module load, first allocations of both ways
    with engine.Solver(pb, **opts) as s:
        s.solve_batch(lb[:2], ub[:2])
    with engine.Solver(root_problem(pb, lb[0], ub[0]), **opts) as s:
        s.solve()

    t0 = time.perf_counter()
    with engine.Solver(pb, timeout_ms=budget_ms, **opts) as s:
        b = s.solve_batch(lb, ub)
    batch_wall = (time.perf_counter() - t0) * 1e3
    progress(name, f"batch {batch_wall:.1f} ms")

    alt = None
    if alt_sub is not None:
        # the same batch with an explicit subproblem depth per root instead of the -sub -1 rule
        t0 = time.perf_counter()
        with engine.Solver(pb, timeout_ms=budget_ms, **dict(opts, subproblems_power=alt_sub)) as s:
            a = s.solve_batch(lb, ub)
        alt = dict(d=a["stats"]["subproblems_power"], wall_ms=round((time.perf_counter() - t0) * 1e3, 2),
                   kernel_ms=round(a["stats"]["kernel_ms"], 2), nodes=a["stats"]["nodes"],
                   exhaustive_roots=int(a["exhaustive"].sum()), solved_roots=int(a["has_solution"].sum()),
                   same_answers=bool((a["has_solution"] == b["has_solution"]).all() and (a["exhaustive"] == b["exhaustive"]).all()
                                     and (a["objective"] == b["objective"]).all()))
        progress(name, f"batch at d = {alt_sub}: {alt['wall_ms']} ms")

    seq = []
    t0 = time.perf_counter()
    for r in range(k):
        with engine.Solver(root_problem(pb, lb[r], ub[r]), timeout_ms=budget_ms // k if budget_ms else 0, **opts) as s:
            seq.append(s.solve())
    seq_wall = (time.perf_counter() - t0) * 1e3
    progress(name, f"{k} sequential solves {seq_wall:.1f} ms")

    bad, invalid = [], 0
    for r in range(k):
        g = seq[r]
        s_obj = g["objective"] if g["objective"] is not None else abi.POS_INF
        if not agree(bool(b["has_solution"][r]), bool(b["exhaustive"][r]), int(b["objective"][r]),
                     g["has_solution"], g["exhaustive"], s_obj if g["has_solution"] else abi.POS_INF, budget=budget_ms > 0):
            bad.append(r)
        if b["has_solution"][r] and not valid(pb, lb[r], ub[r], b["lb"][r], b["ub"][r]):
            invalid += 1
        if g["has_solution"] and not valid(pb, lb[r], ub[r], g["lb"], g["ub"]):
            invalid += 1
    seq_nodes = sum(g["stats"]["nodes"] for g in seq)
    seq_kernel = sum(g["stats"]["kernel_ms"] for g in seq)
    dev, power = device_and_power()
    return dict(
        workload=name, K=k, d=b["stats"]["subproblems_power"], budget_ms=budget_ms,
        batch=dict(wall_ms=round(batch_wall, 2), kernel_ms=round(b["stats"]["kernel_ms"], 2), nodes=b["stats"]["nodes"],
                   roots_per_s=round(k / batch_wall * 1e3, 1), nodes_per_s=round(b["stats"]["nodes"] / batch_wall * 1e3),
                   exhaustive_roots=int(b["exhaustive"].sum()), solved_roots=int(b["has_solution"].sum()),
                   num_blocks=b["stats"]["num_blocks"]),
        sequential=dict(wall_ms=round(seq_wall, 2), kernel_ms=round(seq_kernel, 2), nodes=seq_nodes,
                        roots_per_s=round(k / seq_wall * 1e3, 1), nodes_per_s=round(seq_nodes / seq_wall * 1e3),
                        exhaustive_roots=sum(g["exhaustive"] for g in seq), solved_roots=sum(g["has_solution"] for g in seq)),
        batch_alt_sub=alt,
        wall_ratio=round(seq_wall / batch_wall, 2), kernel_ratio=round(seq_kernel / max(1e-9, b["stats"]["kernel_ms"]), 2),
        disagreeing_roots=bad[:20], num_disagreeing=len(bad), invalid_stores=invalid,
        device=dev, power_limit=power)


def emit(rec, out):
    print(json.dumps(rec), flush=True)
    if out:
        with open(out, "a") as f:
            f.write(json.dumps(rec) + "\n")
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--k-tiny", type=int, default=2048)
    ap.add_argument("--k-accap", type=int, default=64)
    ap.add_argument("--budget-ms", type=int, default=4000)
    a = ap.parse_args()
    from tests import golden_io
    from turbo_b200 import engine
    if engine.device_count() < 1:
        sys.exit("batch_solve.py needs a CUDA device: the engine has no CPU fallback")
    lines = []
    for net in ("sudoku_opt3", "pat10"):
        pb, _ = golden_io.load(net)
        lb, ub = make_roots(pb, a.k_tiny, a.seed)
        lines.append(emit(run(net, pb, lb, ub, {}), a.out))
    # accap_a3: easy roots around a solution the engine finds in a second, a few harder ones fixing half as much
    pb, _ = golden_io.load_simplified_problem("accap_a3")
    with engine.Solver(pb, timeout_ms=1000) as s:
        sol = s.solve()
    assert sol["has_solution"], "accap_a3: no solution within a second"
    k = a.k_accap
    lb, ub = make_roots(pb, k, a.seed, around=sol["lb"].astype(np.int64), free=6)
    hard_lb, hard_ub = make_roots(pb, max(1, k // 8), a.seed + 1, around=sol["lb"].astype(np.int64), free=40, empty_frac=0)
    lb[:len(hard_lb)], ub[:len(hard_ub)] = hard_lb, hard_ub
    lines.append(emit(run("simplified:accap_a3", pb, lb, ub, {}, budget_ms=a.budget_ms, alt_sub=0), a.out))
    if any(r["num_disagreeing"] or r["invalid_stores"] for r in lines):
        sys.exit("batch and sequential solves disagree, or a store is not a solution of its root")


if __name__ == "__main__":
    main()

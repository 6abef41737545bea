"""Regenerates tests/golden/*.npz from the reference's FlatZinc inputs.

  python tests/golden/make_golden.py [--check] REFERENCE_CHECKOUT      (ptal/turbo @ 683f23c)

The tests only ever read the committed fixtures. For every instance: the TNF produced by our C++
front-end (lb, ub, props, strategies, objective), the reference's expected optimum
(benchmarks/test_list.csv) where one exists, and the sha256 of the oracle's root fixpoint (a
regression pin for front-end + oracle). With --check nothing is written: the arrays are rebuilt and
compared with the committed ones, the names that differ are reported and the exit status is 1 if any do.
"""
import csv
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle_py as orc  # noqa: E402
from turbo_b200.model import Model  # noqa: E402


def root_sha(pb):
    r = orc.fixpoint(pb)
    h = hashlib.sha256()
    h.update(b"F" if r["failed"] else b"-")
    if not r["failed"]:
        h.update(r["lb"].tobytes())
        h.update(r["ub"].tobytes())
    return h.hexdigest(), r["failed"]


def dump(name, path, expected, check=False):
    m = Model.from_fzn(path)
    pb = m.problem
    sha, failed = root_sha(pb)
    props = np.stack([pb.props[f] for f in ("op", "x", "y", "z")], axis=1).astype(np.int32) if pb.nprops else np.zeros((0, 4), np.int32)
    strat_meta = np.array([(vo, va, len(vs)) for vo, va, vs in pb.strategies], dtype=np.int32).reshape(-1, 3)
    strat_vars = np.concatenate([vs for _, _, vs in pb.strategies] + [np.zeros(0, np.int32)]).astype(np.int32)
    meta = np.array([pb.obj_var, pb.c.has_eps_strategy, m.objective_kind, m.user_objective_var,
                     0 if expected is None else expected, 0 if expected is None else 1, int(failed)], dtype=np.int64)
    arrays = dict(lb=pb.lb, ub=pb.ub, props=props, strat_meta=strat_meta, strat_vars=strat_vars, meta=meta,
                  root_sha=np.array(sha))
    out = os.path.join(HERE, name + ".npz")
    if check:
        old = np.load(out)
        same = set(old.files) == set(arrays) and all(np.array_equal(old[k], v) for k, v in arrays.items())
        print(f"{name:28s} {'same' if same else 'DIFFERS'}")
        return same
    np.savez_compressed(out, **arrays)
    print(f"{name:28s} V={pb.nvars:6d} P={pb.nprops:6d} expected={expected} root={sha[:12]}")
    return True


def main(reference, check=False):
    benchmarks = os.path.join(reference, "benchmarks")
    same = []
    for path, exp in csv.reader(open(os.path.join(benchmarks, "test_list.csv"))):
        if path.endswith(".xml"):
            continue            # XCSP3: out of scope (SURVEY.md §2.2)
        name = os.path.basename(path)[:-4]
        same.append(dump(name, os.path.join(reference, path), int(exp), check))
    for name in ("accap_a3", "trains15", "example_wordpress7_500"):
        same.append(dump(name, os.path.join(benchmarks, name + ".fzn"), None, check))
    for name in ("bigdom", "valve6"):            # unsolved_bugs_data: no expected answer; valve6 has set variables
        same.append(dump(name, os.path.join(benchmarks, "unsolved_bugs_data", name + ".fzn"), None, check))
    return all(same)


if __name__ == "__main__":
    args = sys.argv[1:]
    check = "--check" in args
    args = [a for a in args if a != "--check"]
    if len(args) != 1:
        raise SystemExit(__doc__)
    sys.exit(0 if main(args[0], check) else 1)

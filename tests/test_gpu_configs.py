"""GPU parity on the five BASELINE.json configurations at their real sizes (VERDICT r01, next #1).

  config 1  example_wordpress7_500: dive subproblems bit-exact on the simplified network (STORE_SHARED) and on
            the network -disable_simplify leaves (STORE_CLUSTER, the only real instance on the DSMEM tier);
  config 2  trains15, config 3 accap_a3: single-block search traces (nodes, failures, solutions, solved/skipped
            subproblems, peak depth, incumbent) equal to the oracle's under a node budget, dense and active-set;
  config 5  synthetic 10^5 x 10^6: root fixpoint bit-exact on STORE_CLUSTER and GLOBAL, root fixpoint of stores
            perturbed by decisions, and the size-independent properties of a fixpoint (idempotent, contracting,
            every propagator at rest);
  all       the proven optima of the headline instances (tests/golden/optima.json) are reproduced when the
            search completes, and never contradicted when it does not.

The oracle is the checker.
"""
import json
import os

import numpy as np
import pytest

from tests import golden_io
from turbo_b200 import abi

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    from turbo_b200 import engine
    assert engine.device_count() > 0, "no CUDA device: the engine has no CPU fallback"
    return engine


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle_py
    return oracle_py


def load(name):
    if name.startswith("simplified:"):
        return golden_io.load_simplified_problem(name.split(":", 1)[1])
    return golden_io.load(name)


# ---- config 1: wordpress dives on both placements ------------------------------------------------------------------

@pytest.mark.parametrize("name,kind", [("simplified:example_wordpress7_500", abi.MEM_STORE_SHARED),
                                       ("example_wordpress7_500", abi.MEM_STORE_CLUSTER),
                                       ("simplified:trains15", abi.MEM_STORE_SHARED),
                                       ("simplified:accap_a3", abi.MEM_STORE_SHARED),
                                       ("simplified:accap_a3", -abi.MEM_TCN_SHARED)])
def test_dive_subproblems_bit_exact_on_the_headline_networks(eng, orc, name, kind):
    pb, _ = load(name)
    depth = 5
    # (a negative kind is requested explicitly: the table in shared memory is no longer anybody's automatic choice)
    with (eng.Solver(pb) if kind >= 0 else eng.Solver(pb, mem_kind=-kind)) as s:
        assert s.config()["mem_kind"] == abs(kind)          # the placement policy's own choice
        if name == "simplified:accap_a3" and kind >= 0:
            assert s.config()["threads_per_block"] == 32   # single-warp blocks, as many as shared memory holds
        g = s.dive_batch(0, 1 << depth, depth)
    for idx in range(1 << depth):
        o = orc.dive(pb, idx, depth)
        assert g["remaining_depth"][idx] == o["remaining_depth"] and g["leaf_kind"][idx] == o["leaf_kind"], (name, idx)
        if o["leaf_kind"] != 1:
            assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"]), (name, idx)


def test_wordpress_unsimplified_dives_on_the_active_tier_too(eng, orc):
    """The same dives with the store forced into L2 (GLOBAL): three placements, one answer."""
    pb, _ = load("example_wordpress7_500")
    depth = 3
    with eng.Solver(pb, mem_kind=abi.MEM_GLOBAL) as s:
        g = s.dive_batch(0, 1 << depth, depth)
    for idx in range(1 << depth):
        o = orc.dive(pb, idx, depth)
        assert g["remaining_depth"][idx] == o["remaining_depth"] and g["leaf_kind"][idx] == o["leaf_kind"], idx
        if o["leaf_kind"] != 1:
            assert np.array_equal(g["lb"][idx], o["lb"]) and np.array_equal(g["ub"][idx], o["ub"]), idx


# ---- configs 1-3: whole search traces of one block on the real networks ------------------------------------------------

TRACE_KEYS = ("nodes", "fails", "solutions", "eps_solved_subproblems", "eps_skipped_subproblems", "depth_max")


@pytest.mark.parametrize("fp", ["ac1", "ac1_active", "wac1", "wac1_active"])
@pytest.mark.parametrize("name,depth,cut", [("simplified:trains15", 4, 300), ("simplified:example_wordpress7_500", 3, 300),
                                            ("simplified:accap_a3", 6, 1500), ("accap_a3", 0, 400), ("trains15", 2, 120)])
def test_single_block_trace_equals_the_oracle(eng, orc, name, depth, cut, fp):
    """One block visits the subproblems in index order exactly as the oracle does, so the counters of the whole
    trace are comparable; the node budget ends both at the same node.  The fixpoint kind does not change the
    trace (same fixpoints), only how many evaluations it takes."""
    pb, _ = load(name)
    o = orc.solve(pb, depth=depth, cutnodes=cut)
    with eng.Solver(pb, or_blocks=1, subproblems_power=depth, cutnodes=cut, fixpoint=abi.FP_KINDS[fp]) as s:
        g = s.solve()
    for key in TRACE_KEYS:
        assert g["stats"][key] == o["stats"][key], (name, fp, key, g["stats"][key], o["stats"][key])
    assert g["has_solution"] == o["has_solution"] and g["objective"] == o["objective"]
    assert g["exhaustive"] == o["exhaustive"]
    if g["has_solution"]:
        # same incumbent store, not only the same objective
        assert np.array_equal(g["lb"], o["lb"]) and np.array_equal(g["ub"], o["ub"])


def test_trace_on_the_cluster_tier(eng, orc):
    pb, _ = load("example_wordpress7_500")
    o = orc.solve(pb, depth=2, cutnodes=60)
    with eng.Solver(pb, or_blocks=1, subproblems_power=2, cutnodes=60, fixpoint=abi.FP_AC1) as s:
        assert s.config()["mem_kind"] == abi.MEM_STORE_CLUSTER
        g = s.solve()
    for key in TRACE_KEYS:
        assert g["stats"][key] == o["stats"][key], (key, g["stats"][key], o["stats"][key])
    assert g["objective"] == o["objective"]


# ---- config 5: the synthetic network at its full size ---------------------------------------------------------------------

@pytest.fixture(scope="module")
def synthetic():
    from turbo_b200.model import Model
    m = Model.synthetic(100000, 1000000, 0xB200)
    return m.problem


def at_rest(pb, lb, ub):
    """Size-independent property of a fixpoint, checked with numpy on all 10^6 propagators: no rule of x = y op z
    can move a bound (restated here for ADD / LEQ / EQ, 80 % of the synthetic mix; DESIGN.md §2 table)."""
    op, x, y, z = (pb.props[k].astype(np.int64) for k in ("op", "x", "y", "z"))
    L, U = lb.astype(np.int64), ub.astype(np.int64)
    a = op == abi.OP_ADD
    ok = np.ones(len(op), bool)
    ok[a] &= (L[x[a]] >= L[y[a]] + L[z[a]]) & (U[x[a]] <= U[y[a]] + U[z[a]])
    ok[a] &= (L[y[a]] >= L[x[a]] - U[z[a]]) & (U[y[a]] <= U[x[a]] - L[z[a]])
    ok[a] &= (L[z[a]] >= L[x[a]] - U[y[a]]) & (U[z[a]] <= U[x[a]] - L[y[a]])
    q = op == abi.OP_LEQ
    t, f = q & (L[x] >= 1), q & (U[x] <= 0)
    ok[t] &= (U[y[t]] <= U[z[t]]) & (L[z[t]] >= L[y[t]])
    ok[f] &= (L[y[f]] >= L[z[f]] + 1) & (U[z[f]] <= U[y[f]] - 1)
    und = q & (L[x] < 1) & (U[x] > 0)
    ok[und] &= ~(U[y[und]] <= L[z[und]]) & ~(L[y[und]] > U[z[und]])
    e = op == abi.OP_EQ
    t = e & (L[x] >= 1)
    ok[t] &= (L[y[t]] == L[z[t]]) & (U[y[t]] == U[z[t]])
    und = e & (L[x] < 1) & (U[x] > 0)
    ok[und] &= ~((U[y[und]] < L[z[und]]) | (U[z[und]] < L[y[und]]))
    ok[und] &= ~((L[y[und]] == U[y[und]]) & (L[z[und]] == U[z[und]]) & (L[y[und]] == L[z[und]]))
    return int((~ok).sum())


@pytest.mark.parametrize("kind", [abi.MEM_STORE_CLUSTER, abi.MEM_GLOBAL])
@pytest.mark.parametrize("fp", [abi.FP_AC1, abi.FP_WAC1])
def test_synthetic_full_size_root_fixpoint_bit_exact(eng, orc, synthetic, kind, fp):
    pb = synthetic
    assert pb.nvars == 100000 and pb.nprops == 1000000
    o = orc.fixpoint(pb)
    assert not o["failed"]
    with eng.Solver(pb, mem_kind=kind, fixpoint=fp) as s:
        assert s.config()["mem_kind"] == kind
        g = s.propagate()
        assert not g["failed"]
        assert np.array_equal(g["lb"], o["lb"]) and np.array_equal(g["ub"], o["ub"])
        # properties that need no oracle: contracting, at rest, idempotent
        assert np.all(g["lb"] >= pb.lb) and np.all(g["ub"] <= pb.ub)
        assert at_rest(pb, g["lb"], g["ub"]) == 0
        again = s.propagate(g["lb"], g["ub"])
        assert not again["failed"] and np.array_equal(again["lb"], g["lb"]) and np.array_equal(again["ub"], g["ub"])


def test_synthetic_full_size_default_placement_is_the_cluster(eng, synthetic):
    with eng.Solver(synthetic) as s:
        cfg = s.config()
    assert cfg["mem_kind"] == abi.MEM_STORE_CLUSTER and cfg["cluster_size"] >= 4


def test_synthetic_full_size_decided_stores(eng, orc, synthetic):
    """Fixpoints of stores narrowed by decisions (what a search node propagates): decisions that keep the planted
    solution (the store narrows further, no failure) and decisions that exclude it (most of them fail)."""
    pb = synthetic
    rng = np.random.default_rng(5)
    sol = orc.fixpoint(pb)["lb"]                     # the root fixpoint of this network assigns every variable
    B = 6
    lb, ub = np.tile(pb.lb, (B, 1)), np.tile(pb.ub, (B, 1))
    wide = np.nonzero(pb.ub > pb.lb)[0]
    for b in range(B):
        for v in rng.choice(wide, size=4 * (b + 1), replace=False):
            if b % 2 == 0:                           # keep the solution inside
                if rng.random() < 0.5:
                    ub[b, v] = sol[v]
                else:
                    lb[b, v] = sol[v]
            else:                                    # cut the domain in two at random
                mid = (int(lb[b, v]) + int(ub[b, v])) // 2
                if rng.random() < 0.5:
                    ub[b, v] = mid
                else:
                    lb[b, v] = mid + 1
    with eng.Solver(pb) as s:
        g = s.propagate_batch(lb, ub)
    nfailed = 0
    for b in range(B):
        o = orc.fixpoint(pb, lb[b], ub[b])
        assert bool(g["failed"][b]) == o["failed"], b
        nfailed += o["failed"]
        if not o["failed"]:
            assert np.array_equal(g["lb"][b], o["lb"]) and np.array_equal(g["ub"][b], o["ub"]), b
    assert 0 < nfailed < B


def test_synthetic_full_size_trace(eng, orc, synthetic):
    """A cutnodes-bounded search on the cluster tier (SURVEY.md 8d, config 5), one block, against the oracle."""
    pb = synthetic
    o = orc.solve(pb, depth=2, cutnodes=24)
    with eng.Solver(pb, or_blocks=1, subproblems_power=2, cutnodes=24, fixpoint=abi.FP_AC1) as s:
        g = s.solve()
    for key in TRACE_KEYS:
        assert g["stats"][key] == o["stats"][key], (key, g["stats"][key], o["stats"][key])


# ---- proven optima -------------------------------------------------------------------------------------------------------

def optima():
    p = os.path.join(golden_io.GOLDEN_DIR, "optima.json")
    return json.load(open(p)) if os.path.exists(p) else {}


@pytest.mark.parametrize("name", ["accap_a3", "trains15", "example_wordpress7_500"])
def test_headline_instances_against_their_recorded_optima(eng, name):
    """tests/golden/optima.json records, per headline instance, the best objective our own exhaustive or longest
    runs reached, whether the search was complete (`proven`) and the independent cross-check.  A bounded run can
    never find anything better than a proven optimum, and reaches it when it completes."""
    rec = optima().get(name)
    if rec is None:
        pytest.skip("no recorded optimum for " + name)
    pb, info = load("simplified:" + name)
    with eng.Solver(pb, timeout_ms=int(rec.get("test_budget_ms", 4000))) as s:
        g = s.solve()
    assert g["has_solution"]
    obj = golden_io.user_objective(info, g["lb"], g["ub"])
    if rec["proven"]:
        assert obj >= rec["objective"] if info["objective_kind"] == 0 else obj <= rec["objective"]
        if g["exhaustive"]:
            assert obj == rec["objective"]
    # every reported solution is re-checked against the network it was found on
    from tests.test_oracle_ops import REL
    for p in pb.props:
        assert REL[int(p["op"])](int(g["lb"][p["x"]]), int(g["lb"][p["y"]]), int(g["lb"][p["z"]]))


# ---- tail splitting (adaptive EPS): few subproblems, many blocks ------------------------------------------------------------

@pytest.mark.parametrize("name", ["pat13", "pat12", "triangular9"])       # the known answers with the largest search trees
def test_tail_splitting_keeps_status_and_optimum(eng, name, monkeypatch):
    """Eight subproblems for hundreds of blocks: the blocks without work wait, the busy ones give their subproblem up
    and enter its 64 children into the pool; the search is still exhaustive and ends on the reference's optimum, and
    every subproblem is accounted for: solved + skipped + split = 2^d."""
    monkeypatch.setenv("TB_SPLIT_MIN_NODES", "256")
    pb, info = golden_io.load(name)
    with eng.Solver(pb, subproblems_power=3, timeout_ms=60000) as s:
        g = s.solve()
    st = g["stats"]
    assert g["has_solution"] and g["exhaustive"]
    assert golden_io.user_objective(info, g["lb"], g["ub"]) == info["expected"]
    assert st["eps_solved_subproblems"] + st["eps_skipped_subproblems"] + st["eps_split_subproblems"] == 8
    assert st["eps_split_subproblems"] > 0 and st["eps_split_parts_solved"] > 0
    # and with splitting off the same answer (one block per subproblem does all the work)
    monkeypatch.setenv("TB_SPLIT_BITS", "0")
    with eng.Solver(pb, subproblems_power=3, timeout_ms=60000) as s:
        h = s.solve()
    assert h["exhaustive"] and golden_io.user_objective(info, h["lb"], h["ub"]) == info["expected"]
    assert h["stats"]["eps_split_subproblems"] == 0


# ---- automatic placement and block shape (DESIGN §3, profiles/r02_block_shapes.md) ---------------------------------------

def test_automatic_placement_and_block_shape(eng, monkeypatch):
    """The store in shared memory whenever it fits, as many few-warp blocks as fit: single-warp blocks for accap_a3,
    2 x 512 threads per SM for trains15, 1 x 1024 for wordpress7_500; TB_SHAPE_V1=1 brings back round 1's 8 x 128 with the
    table in shared memory. The default number of subproblems counts at most 4 blocks per SM."""
    def shape(name, **kw):
        pb, _ = load(name)
        with eng.Solver(pb, subproblems_power=-1, **kw) as s:
            c = s.config()
        return c["mem_kind"], c["threads_per_block"], c["blocks_per_sm"], c["num_blocks"], c["subproblems_power"]

    kind, threads, bps, blocks, power = shape("simplified:accap_a3")
    assert (kind, threads) == (abi.MEM_STORE_SHARED, 32) and bps >= 20
    assert (1 << power) >= 300 * min(blocks, 4 * (blocks // bps)) > (1 << (power - 1))
    assert shape("simplified:trains15")[:3] == (abi.MEM_STORE_SHARED, 512, 2)
    assert shape("simplified:example_wordpress7_500")[:3] == (abi.MEM_STORE_SHARED, 1024, 1)
    assert shape("simplified:accap_a3", mem_kind=abi.MEM_TCN_SHARED)[0] == abi.MEM_TCN_SHARED
    monkeypatch.setenv("TB_SHAPE_V1", "1")
    assert shape("simplified:accap_a3")[:3] == (abi.MEM_TCN_SHARED, 128, 8)

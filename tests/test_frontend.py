"""Front-end tests (CPU): FlatZinc parser + ternarisation + checker + printer.

The ternariser is validated differentially: random small FlatZinc models are solved (a) by brute
force over the FlatZinc semantics written here in Python and (b) by the oracle on the TNF produced
by the C++ front-end; status and optimum must agree, and the C++ FlatZinc checker must accept the
oracle's solution.
"""
import hashlib
import itertools
import json
import os

import numpy as np
import pytest

from oracle import oracle_py as orc
from turbo_b200.engine import TurboError
from turbo_b200.model import Model


def tdiv(a, b):
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b > 0) else -q


# name -> (arity spec, python predicate). i = int var/lit, b = bool var/lit, I = int array, B = bool array
SEM = {
    "int_eq": ("ii", lambda a, b: a == b),
    "int_ne": ("ii", lambda a, b: a != b),
    "int_le": ("ii", lambda a, b: a <= b),
    "int_lt": ("ii", lambda a, b: a < b),
    "int_eq_reif": ("iib", lambda a, b, r: (a == b) == bool(r)),
    "int_ne_reif": ("iib", lambda a, b, r: (a != b) == bool(r)),
    "int_le_reif": ("iib", lambda a, b, r: (a <= b) == bool(r)),
    "int_lt_reif": ("iib", lambda a, b, r: (a < b) == bool(r)),
    "int_plus": ("iii", lambda a, b, c: a + b == c),
    "int_minus": ("iii", lambda a, b, c: a - b == c),
    "int_times": ("iii", lambda a, b, c: a * b == c),
    "int_div": ("iii", lambda a, b, c: b != 0 and tdiv(a, b) == c),
    "int_mod": ("iii", lambda a, b, c: b != 0 and a - b * tdiv(a, b) == c),
    "int_min": ("iii", lambda a, b, c: min(a, b) == c),
    "int_max": ("iii", lambda a, b, c: max(a, b) == c),
    "int_abs": ("ii", lambda a, b: abs(a) == b),
    "bool2int": ("bi", lambda a, b: a == b),
    "bool_and": ("bbb", lambda a, b, r: (a and b) == r),
    "bool_or": ("bbb", lambda a, b, r: (a or b) == r),
    "bool_xor": ("bbb", lambda a, b, r: (a != b) == bool(r)),
    "bool_not": ("bb", lambda a, b: a != b),
    "bool_eq": ("bb", lambda a, b: a == b),
    "bool_le": ("bb", lambda a, b: a <= b),
    "bool_eq_reif": ("bbb", lambda a, b, r: (a == b) == bool(r)),
}


def gen_model(rng):
    nint, nbool = 4, 3
    decl, doms, names = [], [], []
    for k in range(nint):
        lo, hi = sorted(int(t) for t in rng.integers(-3, 4, size=2))
        decl.append(f"var {lo}..{hi}: x{k} :: output_var;")
        doms.append(range(lo, hi + 1))
        names.append(f"x{k}")
    for k in range(nbool):
        decl.append(f"var bool: b{k} :: output_var;")
        doms.append(range(0, 2))
        names.append(f"b{k}")
    cons, preds = [], []

    def pick(kind):
        if kind == "i":
            if rng.random() < 0.2:
                v = int(rng.integers(-3, 4))
                return str(v), (lambda a, v=v: v)
            k = int(rng.integers(0, nint))
            return f"x{k}", (lambda a, k=k: a[k])
        if rng.random() < 0.1:
            v = int(rng.integers(0, 2))
            return ("true" if v else "false"), (lambda a, v=v: v)
        k = int(rng.integers(0, nbool))
        return f"b{k}", (lambda a, k=k: a[nint + k])

    for _ in range(int(rng.integers(2, 6))):
        r = rng.random()
        if r < 0.5:
            name = list(SEM)[int(rng.integers(0, len(SEM)))]
            spec, fn = SEM[name]
            args = [pick(c) for c in spec]
            cons.append(f"constraint {name}({','.join(t for t, _ in args)});")
            preds.append(lambda a, fn=fn, args=args: bool(fn(*[g(a) for _, g in args])))
        elif r < 0.8:
            n = int(rng.integers(1, 4))
            cs = [int(c) for c in rng.integers(-3, 4, size=n)]
            xs = [pick("i") for _ in range(n)]
            c = int(rng.integers(-4, 5))
            rel = ["le", "eq", "ne"][int(rng.integers(0, 3))]
            ok = {"le": lambda s, c: s <= c, "eq": lambda s, c: s == c, "ne": lambda s, c: s != c}[rel]
            if rng.random() < 0.5:
                rr = pick("b")
                cons.append(f"constraint int_lin_{rel}_reif([{','.join(map(str, cs))}],[{','.join(t for t, _ in xs)}],{c},{rr[0]});")
                preds.append(lambda a, cs=cs, xs=xs, c=c, ok=ok, rr=rr: ok(sum(k * g(a) for k, (_, g) in zip(cs, xs)), c) == bool(rr[1](a)))
            else:
                cons.append(f"constraint int_lin_{rel}([{','.join(map(str, cs))}],[{','.join(t for t, _ in xs)}],{c});")
                preds.append(lambda a, cs=cs, xs=xs, c=c, ok=ok: ok(sum(k * g(a) for k, (_, g) in zip(cs, xs)), c))
        elif r < 0.9:
            pos = [pick("b") for _ in range(int(rng.integers(0, 3)))]
            neg = [pick("b") for _ in range(int(rng.integers(0, 3)))]
            cons.append(f"constraint bool_clause([{','.join(t for t, _ in pos)}],[{','.join(t for t, _ in neg)}]);")
            preds.append(lambda a, pos=pos, neg=neg: any(g(a) for _, g in pos) or any(not g(a) for _, g in neg))
        else:
            arr = [int(v) for v in rng.integers(-3, 4, size=3)]
            i, v = pick("i"), pick("i")
            cons.append(f"constraint array_int_element({i[0]},[{','.join(map(str, arr))}],{v[0]});")
            preds.append(lambda a, arr=arr, i=i, v=v: 1 <= i[1](a) <= 3 and arr[i[1](a) - 1] == v[1](a))
    obj = int(rng.integers(0, nint))
    sense = "minimize" if rng.random() < 0.5 else "maximize"
    text = "\n".join(decl + cons + [f"solve {sense} x{obj};"])
    best = None
    for a in itertools.product(*doms):
        if all(p(a) for p in preds):
            if best is None or (a[obj] < best if sense == "minimize" else a[obj] > best):
                best = a[obj]
    return text, best


@pytest.mark.parametrize("seed", range(150))
def test_random_models_match_bruteforce(seed):
    rng = np.random.default_rng(seed)
    text, best = gen_model(rng)
    m = Model.from_fzn_text(text)
    if m.root_failed:
        assert best is None, text
        return
    r = orc.solve(m.problem, depth=2)
    assert r["exhaustive"]
    assert r["has_solution"] == (best is not None), text
    if best is not None:
        assert m.user_objective(r["lb"], r["ub"]) == best, text
        assert m.check_solution(r["lb"]) == 0, text
        assert m.check_tnf(r["lb"]) == 0, text


def test_checker_rejects_wrong_points():
    m = Model.from_fzn_text("var 0..5: x :: output_var;\nvar 0..5: y :: output_var;\n"
                            "constraint int_lin_le([1,1],[x,y],4);\nconstraint int_ne(x,y);\nsolve maximize x;")
    r = orc.solve(m.problem)
    assert m.user_objective(r["lb"], r["ub"]) == 4 and m.check_solution(r["lb"]) == 0
    bad = r["lb"].copy()
    bad[m.problem.lb.shape[0] - 1] = bad[m.problem.lb.shape[0] - 1]   # untouched copy is still fine
    assert m.check_solution(bad) == 0
    xs = [i for i in range(m.problem.nvars) if m.problem.lb[i] == 0 and m.problem.ub[i] == 5]
    bad[xs[0]] = 5
    bad[xs[1]] = 5
    assert m.check_solution(bad) > 0


SYNTAX_SUBSET = """% a comment
predicate foo(var int: a);
array [1..2] of int: w = [1,-1];
int: k = 3;
var 1..3: a :: output_var;
var {1,3}: h :: output_var;
var bool: p :: output_var;
var 0..9: t :: var_is_introduced :: is_defined_var;
array [1..4] of var int: g :: output_array([1..2,1..2]) = [a,h,2,t];
array [1..2] of var bool: q :: output_array([0..1]) = [p,true];
constraint int_lin_eq(w,[a,h],0);
constraint int_eq(p,int_le(2,a));
constraint int_plus(a,k,t) :: defines_var(t);
solve :: seq_search([int_search(g,first_fail,indomain_min,complete),bool_search([p],input_order,indomain_max,complete)]) maximize a;
"""


def test_output_format_and_syntax_subset():
    m = Model.from_fzn_text(SYNTAX_SUBSET)
    assert m.parsed_variables == 4 and m.parsed_constraints == 3
    assert len(m.problem.strategies) == 3          # two annotations + the default strategy
    r = orc.solve(m.problem)
    assert m.user_objective(r["lb"], r["ub"]) == 3
    out = m.format_solution(r["lb"], r["ub"])
    assert out == "a = 3;\nh = 3;\np = true;\ng = array2d(1..2, 1..2, [3, 3, 2, 6]);\nq = array1d(0..1, [true, true]);\n"
    assert m.check_solution(r["lb"]) == 0


def test_set_domains_and_set_in_reif():
    m = Model.from_fzn_text("var {1,2,4,5}: x :: output_var;\nvar bool: y :: output_var;\n"
                            "constraint set_in_reif(x, 2..4, y);\nconstraint bool_eq(y,true);\nsolve maximize x;")
    r = orc.solve(m.problem)
    assert m.user_objective(r["lb"], r["ub"]) == 4 and m.check_solution(r["lb"]) == 0
    m = Model.from_fzn_text("var 0..9: x :: output_var;\nvar bool: y :: output_var;\n"
                            "constraint set_in_reif(x, {1,2,7}, y);\nconstraint bool_eq(y,true);\nsolve maximize x;")
    r = orc.solve(m.problem)
    assert m.user_objective(r["lb"], r["ub"]) == 7


def test_unsat_and_satisfy():
    m = Model.from_fzn_text("constraint bool_eq(false,true);\nsolve satisfy;")
    assert m.root_failed
    m = Model.from_fzn_text("var 1..3: x;\nvar 1..3: y;\nconstraint int_lt(x,y);\nconstraint int_lt(y,x);\nsolve satisfy;")
    r = orc.solve(m.problem)
    assert not r["has_solution"] and r["exhaustive"]
    m = Model.from_fzn_text("var 1..3: x :: output_var;\nvar 1..3: y :: output_var;\nconstraint int_lt(x,y);\nsolve satisfy;")
    r = orc.solve(m.problem)
    assert r["has_solution"] and m.check_solution(r["lb"]) == 0


def test_parse_errors_are_reported():
    for bad in ["var 1..3 x;\nsolve satisfy;", "var 1..3: x;\nconstraint nope(x);\nsolve satisfy;",
                "var 1..3: x;\nconstraint int_eq(x,zz);\nsolve satisfy;", "var 1..3: x;", "var float: f;\nsolve satisfy;"]:
        with pytest.raises(TurboError):
            Model.from_fzn_text(bad)
    with pytest.raises(TurboError):
        Model.from_fzn("/nonexistent/file.fzn")


def test_synthetic_generator_is_deterministic_and_satisfiable(tmp_path):
    a = Model.synthetic(2000, 8000, 0xB200)
    b = Model.synthetic(2000, 8000, 0xB200)
    assert np.array_equal(a.problem.lb, b.problem.lb) and np.array_equal(a.problem.props, b.problem.props)
    assert a.problem.nvars == 2000 and a.problem.nprops == 8000
    r = orc.fixpoint(a.problem)
    assert not r["failed"] and np.any(r["lb"] > a.problem.lb)       # real narrowing, no failure
    p = tmp_path / "s.tnf"
    a.save_tnf(p)
    c = Model.from_tnf(p)
    assert np.array_equal(a.problem.ub, c.problem.ub) and np.array_equal(a.problem.props, c.problem.props)
    assert len(c.problem.strategies) == len(a.problem.strategies)


# ---- set variables (membership Booleans; unsolved_bugs_data/valve6.fzn was flattened without nosets.mzn) -------------

def gen_set_model(rng):
    """x, y in 0..5, idx in 1..3, b Boolean, S = arr[idx] (array_set_element), b <-> y in S (set_in_reif), optionally x in S."""
    universe = (1, 4)
    arr = []
    for _ in range(3):
        vals = sorted(set(int(v) for v in rng.integers(universe[0], universe[1] + 1, size=int(rng.integers(0, 4)))))
        arr.append(vals)
    hard = bool(rng.random() < 0.5)
    coef = [int(v) for v in rng.integers(-3, 4, size=4)]
    bound = int(rng.integers(-4, 8))
    sense = "minimize" if rng.random() < 0.5 else "maximize"
    lit = lambda vs: "{" + ",".join(map(str, vs)) + "}"
    text = "\n".join([
        f"array [1..3] of set of int: sets = [{','.join(lit(v) for v in arr)}];",
        "var 0..5: x :: output_var;", "var 0..5: y :: output_var;", "var 1..3: idx :: output_var;", "var bool: b :: output_var;",
        "var 0..1: bi :: output_var;", "var -40..40: obj :: output_var;",
        f"var set of {universe[0]}..{universe[1]}: S;",
        "constraint array_set_element(idx, sets, S);",
        "constraint set_in_reif(y, S, b);",
        "constraint bool2int(b, bi);",
    ] + (["constraint set_in(x, S);"] if hard else []) + [
        f"constraint int_lin_le([{coef[0]},{coef[1]},{coef[2]}],[x,y,idx],{bound});",
        f"constraint int_lin_eq([{coef[0]},{coef[3]},2,3,-1],[x,y,idx,bi,obj],0);",
        f"solve {sense} obj;"])
    best = None
    for x in range(6):
        for y in range(6):
            for idx in range(1, 4):
                S = set(arr[idx - 1])
                b = int(y in S)
                if hard and x not in S:
                    continue
                if coef[0] * x + coef[1] * y + coef[2] * idx > bound:
                    continue
                obj = coef[0] * x + coef[3] * y + 2 * idx + 3 * b
                if best is None or (obj < best if sense == "minimize" else obj > best):
                    best = obj
    return text, best


@pytest.mark.parametrize("seed", range(60))
def test_set_variable_models_match_bruteforce(seed):
    rng = np.random.default_rng(1000 + seed)
    text, best = gen_set_model(rng)
    m = Model.from_fzn_text(text)
    if m.root_failed:
        assert best is None, text
        return
    r = orc.solve(m.problem, depth=2)
    assert r["exhaustive"]
    assert r["has_solution"] == (best is not None), text
    if best is not None:
        assert m.user_objective(r["lb"], r["ub"]) == best, text
        assert m.check_solution(r["lb"]) == 0, text


def test_set_variable_checker_and_errors():
    text = ("array [1..2] of set of int: sets = [{1,2},{3}];\nvar 1..2: i :: output_var;\nvar 0..4: x :: output_var;\nvar bool: b :: output_var;\n"
            "var set of 1..3: S;\nconstraint array_set_element(i, sets, S);\nconstraint set_in_reif(x, S, b);\nsolve satisfy;\n")
    m = Model.from_fzn_text(text)
    r = orc.solve(m.problem, depth=0)
    assert r["has_solution"] and m.check_solution(r["lb"]) == 0
    # flip the reified result: the checker must object (the set constraint is evaluated on the membership variables)
    bad = r["lb"].copy()
    vals = dict(line.rstrip(";").split(" = ") for line in m.format_solution(r["lb"]).strip().splitlines())
    assert (vals["b"] == "true") == (int(vals["x"]) in ({1, 2} if vals["i"] == "1" else {3}))
    with pytest.raises(Exception):
        Model.from_fzn_text("var set of 1..3: S :: output_var;\nsolve satisfy;\n")
    with pytest.raises(Exception):
        Model.from_fzn_text("var set of int: S;\nsolve satisfy;\n")


# ---- stored models: the network the front-end builds is pinned (tests/golden/fzn, tests/golden/make_frontend_pins.py) ----

FZN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fzn")
PINS = json.load(open(os.path.join(FZN_DIR, "pins.json")))


def network_sha(m):
    """sha256 of everything the front-end hands the engine: bounds, propagators, strategies and objective."""
    from tests import golden_io
    h = hashlib.sha256()
    for k, a in sorted(golden_io.problem_arrays(m.problem).items()):
        h.update(k.encode())
        h.update(np.ascontiguousarray(a, np.int32).tobytes())
    h.update(np.array([m.objective_kind, m.user_objective_var, int(m.root_failed)], np.int32).tobytes())
    return h.hexdigest()


def test_stored_model_inventory():
    assert len(PINS) == 23 and all(os.path.exists(os.path.join(FZN_DIR, n + ".fzn")) for n in PINS)


@pytest.mark.parametrize("name", sorted(PINS))
def test_stored_model_builds_the_pinned_network(name):
    m = Model.from_fzn(os.path.join(FZN_DIR, name + ".fzn"))
    assert network_sha(m) == PINS[name]["tnf_sha256"]


@pytest.mark.parametrize("name", sorted(PINS))
def test_stored_model_optimum_passes_the_flatzinc_checker(name):
    m = Model.from_fzn(os.path.join(FZN_DIR, name + ".fzn"))
    best = PINS[name]["optimum"]
    if m.root_failed:
        assert best is None
        return
    r = orc.solve(m.problem, depth=2)
    assert r["exhaustive"] and r["has_solution"] == (best is not None)
    if best is not None:
        assert m.user_objective(r["lb"], r["ub"]) == best
        assert m.check_solution(r["lb"]) == 0 and m.check_tnf(r["lb"]) == 0


# ---- half reification (_imp), bool_lin_*, array_int_minimum / maximum ---------------------------------------------------

@pytest.mark.parametrize("seed", range(40))
def test_imp_minmax_boollin_models_match_bruteforce(seed):
    rng = np.random.default_rng(2000 + seed)
    c = [int(v) for v in rng.integers(-3, 4, size=6)]
    k1, k2, k3 = int(rng.integers(-2, 6)), int(rng.integers(0, 3)), int(rng.integers(-3, 6))
    sense = "minimize" if rng.random() < 0.5 else "maximize"
    which = "array_int_minimum" if rng.random() < 0.5 else "array_int_maximum"
    text = "\n".join([
        "var -2..3: x :: output_var;", "var -2..3: y :: output_var;", "var -2..3: z :: output_var;", "var -2..3: m :: output_var;",
        "var bool: p :: output_var;", "var bool: q :: output_var;", "var 0..1: pi :: output_var;", "var 0..1: qi :: output_var;",
        "var -60..60: obj :: output_var;",
        f"constraint {which}(m, [x, y, z]);",
        f"constraint int_lin_le_imp([{c[0]},{c[1]}],[x,y],{k1},p);",
        f"constraint int_eq_imp(y, z, q);",
        f"constraint bool_lin_le([1,1],[p,q],{k2});",
        f"constraint bool_clause_imp([p],[q],q);",
        "constraint bool2int(p, pi);", "constraint bool2int(q, qi);",
        f"constraint int_lin_le([{c[2]},{c[3]}],[x,z],{k3});",
        f"constraint int_lin_eq([{c[4]},{c[5]},2,3,-2,-1],[x,m,pi,qi,z,obj],0);",
        f"solve {sense} obj;"])
    best = None
    import itertools
    for x, y, z, p, q in itertools.product(range(-2, 4), range(-2, 4), range(-2, 4), (0, 1), (0, 1)):
        m = min(x, y, z) if which == "array_int_minimum" else max(x, y, z)
        if p and not (c[0] * x + c[1] * y <= k1): continue
        if q and not (y == z): continue
        if p + q > k2: continue
        if q and not (p or not q): continue          # q -> (p \\/ not q)
        if c[2] * x + c[3] * z > k3: continue
        obj = c[4] * x + c[5] * m + 2 * p + 3 * q - 2 * z
        if best is None or (obj < best if sense == "minimize" else obj > best):
            best = obj
    mdl = Model.from_fzn_text(text)
    if mdl.root_failed:
        assert best is None, text
        return
    r = orc.solve(mdl.problem, depth=2)
    assert r["exhaustive"] and r["has_solution"] == (best is not None), text
    if best is not None:
        assert mdl.user_objective(r["lb"], r["ub"]) == best, text
        assert mdl.check_solution(r["lb"]) == 0, text


@pytest.mark.parametrize("k", [0, 1, 2, 3])
def test_int_pow_with_a_constant_exponent(k):
    for sense in ("minimize", "maximize"):
        text = (f"var -3..3: x :: output_var;\nvar -30..30: z :: output_var;\nvar -40..40: obj :: output_var;\n"
                f"constraint int_pow(x, {k}, z);\nconstraint int_lin_eq([1,-2,-1],[z,x,obj],0);\nsolve {sense} obj;\n")
        vals = [x ** k - 2 * x for x in range(-3, 4) if -30 <= x ** k <= 30]
        m = Model.from_fzn_text(text)
        r = orc.solve(m.problem, depth=1)
        assert r["has_solution"] and r["exhaustive"]
        assert m.user_objective(r["lb"], r["ub"]) == (min(vals) if sense == "minimize" else max(vals))
        assert m.check_solution(r["lb"]) == 0
    with pytest.raises(Exception):
        Model.from_fzn_text("var 0..3: x;\nvar 0..3: y;\nvar 0..30: z;\nconstraint int_pow(x, y, z);\nsolve satisfy;\n")

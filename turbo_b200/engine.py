"""ctypes binding of turbo_b200/libturbo_b200.so (the product's C ABI, include/turbo_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible when a
solver is created, this raises.
"""
import ctypes as C
import os

import numpy as np

from . import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
# TURBO_B200_LIB selects another build of the same library (A/B runs of kernel variants); there is still no fallback.
LIB_PATH = os.environ.get("TURBO_B200_LIB") or os.path.join(_HERE, "libturbo_b200.so")
_LIB = None


class TurboError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"{abi.STATUS_NAMES.get(status, status)}: {message}")
        self.status = status


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C turbo_b200`). The engine has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        i32p = C.POINTER(C.c_int32)
        vp = C.c_void_p
        L.tb_create.argtypes = [C.POINTER(vp), C.POINTER(abi.TbProblem), C.POINTER(abi.TbOptions)]
        L.tb_propagate.argtypes = [vp, i32p, i32p, i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_propagate_batch.argtypes = [vp, C.c_int32, i32p, i32p, i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_dive.argtypes = [vp, C.c_uint64, C.c_int32, i32p, i32p, i32p, i32p]
        L.tb_dive_batch.argtypes = [vp, C.c_uint64, C.c_int32, C.c_int32, i32p, i32p, i32p, i32p]
        L.tb_solve.argtypes = [vp, i32p, i32p, i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_solve_batch.argtypes = [vp, C.c_int32, i32p, i32p, i32p, i32p, i32p, i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_solve_groups.argtypes = [vp, C.c_int32, i32p, i32p, i32p, C.c_int32, i32p, i32p, i32p, i32p, i32p, i32p,
                                      C.POINTER(abi.TbStats)]
        L.tb_solve_objectives.argtypes = [vp, C.c_int32, i32p, i32p, C.c_int32, i32p, i32p, i32p, i32p, i32p, i32p, i32p,
                                          i32p, C.POINTER(abi.TbStats)]
        L.tb_solve_supports.argtypes = [vp, C.c_int32, i32p, i32p, C.c_int32, i32p, i32p, i32p, i32p, i32p, C.c_int32,
                                        i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_solve_front.argtypes = [vp, C.c_int32, i32p, i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     i32p, i32p, i32p, i32p, i32p, i32p, i32p, C.POINTER(abi.TbStats)]
        L.tb_link_peers.argtypes = [C.POINTER(vp), C.c_int32]
        L.tb_export_bound_handle.argtypes = [vp, vp]
        L.tb_import_peer_bounds.argtypes = [vp, vp, C.c_int32]
        L.tb_read_bound.argtypes = [vp, i32p]
        L.tb_get_config.argtypes = [vp, C.POINTER(abi.TbStats)]
        L.tb_layout_describe.argtypes = [C.POINTER(abi.TbProblem), C.c_int32, C.POINTER(abi.TbLayoutInfo), i32p]
        L.tb_layout_class_name.argtypes = [C.c_int32]
        L.tb_layout_class_name.restype = C.c_char_p
        L.tb_destroy.argtypes = [vp]
        L.tb_destroy.restype = None
        L.tb_last_error.restype = C.c_char_p
        L.tb_version.restype = C.c_char_p
        L.tb_device_count.restype = C.c_int32
        for name in ("tb_create", "tb_propagate", "tb_propagate_batch", "tb_dive", "tb_dive_batch", "tb_solve",
                     "tb_solve_batch", "tb_solve_groups", "tb_solve_objectives", "tb_solve_supports", "tb_solve_front", "tb_link_peers", "tb_export_bound_handle", "tb_import_peer_bounds", "tb_read_bound",
                     "tb_get_config"):
            getattr(L, name).restype = C.c_int
        _LIB = L
    return _LIB


def _check(rc):
    if rc != 0:
        raise TurboError(rc, lib().tb_last_error().decode())


def _p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def layout_describe(problem, nbanks=16):
    """The host layout pass on its own (no GPU): class histogram, variable placement, bank model."""
    L = lib()
    info = abi.TbLayoutInfo()
    slot_of = np.zeros(max(1, problem.nvars), dtype=np.int32)
    _check(L.tb_layout_describe(C.byref(problem.c), nbanks, C.byref(info), _p(slot_of)))
    classes = {L.tb_layout_class_name(c).decode(): info.class_count[c] for c in range(info.nclasses)}
    return dict(classes=classes, nchunks=info.nchunks, nslots=info.nslots, identity=bool(info.identity),
                loads_per_sweep=info.loads_per_sweep, wavefronts_per_load=info.wavefronts_per_load,
                slot_of=slot_of[:problem.nvars])


def layout_watch_lists(problem, nbanks=16):
    """(off, list, slot_of, chunk_of_prop) of the active-set fixpoint's watch lists (host only, no GPU)."""
    L = lib()
    i32p = C.POINTER(C.c_int32)
    L.tb_layout_watch_lists.argtypes = [C.POINTER(abi.TbProblem), C.c_int32, i32p, i32p, i32p, i32p, i32p, i32p]
    L.tb_layout_watch_lists.restype = C.c_int
    ns, ne = C.c_int32(0), C.c_int32(0)
    _check(L.tb_layout_watch_lists(C.byref(problem.c), nbanks, C.byref(ns), C.byref(ne), None, None, None, None))
    off = np.zeros(ns.value + 1, np.int32)
    lst = np.zeros(max(1, ne.value), np.int32)
    slot_of = np.zeros(max(1, problem.nvars), np.int32)
    chunk_of = np.zeros(max(1, problem.nprops), np.int32)
    _check(L.tb_layout_watch_lists(C.byref(problem.c), nbanks, C.byref(ns), C.byref(ne), _p(off), _p(lst), _p(slot_of), _p(chunk_of)))
    return off, lst[:ne.value], slot_of[:problem.nvars], chunk_of[:problem.nprops]


def front_points(r, x, maximize_x=False, maximize_y=False):
    """The Pareto front in per-level answers of Solver.solve_front (`r`, levels ascending): walking the levels in x's
    preferred order (ascending when x is minimised), the levels whose value strictly improves on every level before
    them. Returns `points` [(x*, y*)] in that order, with x* read from the level's row, the rows `lb` / `ub`, `proven`
    (that level is exhaustive) and `level` (the index of each point's level)."""
    k = len(r["objective"])
    best, idx = None, []
    for i in (range(k - 1, -1, -1) if maximize_x else range(k)):
        if not r["has_solution"][i]:
            continue
        key = -int(r["objective"][i]) if maximize_y else int(r["objective"][i])
        if best is None or key < best:
            best = key
            idx.append(i)
    idx = np.array(idx, np.int64)
    return dict(points=[(int(r["lb"][i][x]), int(r["objective"][i])) for i in idx], lb=r["lb"][idx], ub=r["ub"][idx],
                proven=np.asarray(r["exhaustive"], bool)[idx], level=idx)


def device_count():
    return int(lib().tb_device_count())


def result_reduce(buffers):
    """tb_result_reduce over a list of packed results (bytes / uint8 arrays of equal length), rank order."""
    L = lib()
    L.tb_result_reduce.argtypes = [C.c_void_p, C.c_int32, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(abi.TbStats), C.POINTER(C.c_int32)]
    L.tb_result_reduce.restype = C.c_int
    bufs = [np.frombuffer(bytes(b), dtype=np.uint8) for b in buffers]
    stride = len(bufs[0])
    flat = np.ascontiguousarray(np.concatenate(bufs))
    hdr = abi.TbResultHeader.from_buffer_copy(flat[:C.sizeof(abi.TbResultHeader)].tobytes())
    nv = max(1, hdr.nvars)
    lb, ub = np.zeros(nv, np.int32), np.zeros(nv, np.int32)
    has, exh, best = C.c_int32(0), C.c_int32(0), C.c_int32(-1)
    st = abi.TbStats()
    _check(L.tb_result_reduce(flat.ctypes.data_as(C.c_void_p), len(bufs), stride, _p(lb), _p(ub), C.byref(has), C.byref(exh),
                              C.byref(st), C.byref(best)))
    return dict(lb=lb[:hdr.nvars], ub=ub[:hdr.nvars], has_solution=bool(has.value), exhaustive=bool(exh.value),
                stats=st.as_dict(), best_rank=best.value)


def device_info(device=0):
    L = lib()
    L.tb_get_device_info.argtypes = [C.c_int32, C.POINTER(abi.TbDeviceInfo)]
    L.tb_get_device_info.restype = C.c_int
    info = abi.TbDeviceInfo()
    _check(L.tb_get_device_info(device, C.byref(info)))
    d = {n: getattr(info, n) for n, _ in info._fields_ if n not in ("pad_", "name")}
    d["name"] = info.name.decode()
    return d


def measure_smem_peak(device=0):
    """Measured shared-memory read bandwidth (GB/s over all SMs) and bytes/clk/SM at the maximum SM clock."""
    L = lib()
    L.tb_measure_smem_peak.argtypes = [C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.tb_measure_smem_peak.restype = C.c_int
    gbs, bpc = C.c_double(0), C.c_double(0)
    _check(L.tb_measure_smem_peak(device, C.byref(gbs), C.byref(bpc)))
    return dict(gb_per_s=gbs.value, bytes_per_clk_per_sm=bpc.value)


class Solver:
    """One engine instance bound to one CUDA device (tb_solver)."""

    def __init__(self, problem, **options):
        self.problem = problem
        self.options = abi.default_options(**options)
        self._h = C.c_void_p()
        _check(lib().tb_create(C.byref(self._h), C.byref(problem.c), C.byref(self.options)))

    def close(self):
        if self._h:
            lib().tb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def handle(self):
        return self._h

    def config(self):
        st = abi.TbStats()
        _check(lib().tb_get_config(self._h, C.byref(st)))
        return st.as_dict()

    def propagate(self, lb=None, ub=None):
        n = self.problem.nvars
        if lb is not None:
            lb = np.ascontiguousarray(lb, dtype=np.int32)
            ub = np.ascontiguousarray(ub, dtype=np.int32)
        olb = np.zeros(max(1, n), np.int32)
        oub = np.zeros(max(1, n), np.int32)
        failed = C.c_int32(0)
        st = abi.TbStats()
        _check(lib().tb_propagate(self._h, _p(lb), _p(ub), _p(olb), _p(oub), C.byref(failed), C.byref(st)))
        return dict(lb=olb[:n], ub=oub[:n], failed=bool(failed.value), stats=st.as_dict())

    def propagate_batch(self, lb, ub):
        lb = np.ascontiguousarray(lb, dtype=np.int32)
        ub = np.ascontiguousarray(ub, dtype=np.int32)
        b = lb.shape[0]
        olb = np.zeros_like(lb)
        oub = np.zeros_like(ub)
        failed = np.zeros(b, np.int32)
        st = abi.TbStats()
        _check(lib().tb_propagate_batch(self._h, b, _p(lb), _p(ub), _p(olb), _p(oub), _p(failed), C.byref(st)))
        return dict(lb=olb, ub=oub, failed=failed.astype(bool), stats=st.as_dict())

    def dive_batch(self, first, count, depth):
        n = self.problem.nvars
        olb = np.zeros((count, max(1, n)), np.int32)
        oub = np.zeros((count, max(1, n)), np.int32)
        if n:
            olb = np.zeros((count, n), np.int32)
            oub = np.zeros((count, n), np.int32)
        rem = np.zeros(count, np.int32)
        kind = np.zeros(count, np.int32)
        _check(lib().tb_dive_batch(self._h, first, count, depth, _p(olb), _p(oub), _p(rem), _p(kind)))
        return dict(lb=olb, ub=oub, remaining_depth=rem, leaf_kind=kind)

    def dive(self, idx, depth):
        r = self.dive_batch(idx, 1, depth)
        return dict(lb=r["lb"][0], ub=r["ub"][0], remaining_depth=int(r["remaining_depth"][0]),
                    leaf_kind=int(r["leaf_kind"][0]))

    def solve(self, stop_flag=None):
        n = max(1, self.problem.nvars)
        lb = np.zeros(n, np.int32)
        ub = np.zeros(n, np.int32)
        has = C.c_int32(0)
        exh = C.c_int32(0)
        st = abi.TbStats()
        _check(lib().tb_solve(self._h, stop_flag, _p(lb), _p(ub), C.byref(has), C.byref(exh), C.byref(st)))
        obj = None
        if has.value and self.problem.obj_var >= 0:
            obj = int(lb[self.problem.obj_var])
        return dict(lb=lb[:self.problem.nvars], ub=ub[:self.problem.nvars], has_solution=bool(has.value),
                    exhaustive=bool(exh.value), objective=obj, stats=st.as_dict())

    def solve_batch(self, lb, ub, stop_flag=None):
        """tb_solve_batch: K roots of this solver's network ([K, nvars] int32 domains, each a narrowing of the
        problem's), searched in one launch as K independent solve() calls. `objective` holds abi.POS_INF where a
        root has no solution or the problem is a satisfaction problem; rows of lb / ub without a solution are zero."""
        n = self.problem.nvars
        lb = np.ascontiguousarray(lb, dtype=np.int32).reshape(-1, n)
        ub = np.ascontiguousarray(ub, dtype=np.int32).reshape(-1, n)
        if lb.shape != ub.shape:
            raise ValueError("lb and ub must have the same shape [K, nvars]")
        k = lb.shape[0]
        olb = np.zeros((k, max(1, n)), np.int32)
        oub = np.zeros((k, max(1, n)), np.int32)
        has = np.zeros(max(1, k), np.int32)
        exh = np.zeros(max(1, k), np.int32)
        obj = np.zeros(max(1, k), np.int32)
        st = abi.TbStats()
        _check(lib().tb_solve_batch(self._h, k, _p(lb), _p(ub), stop_flag, _p(olb), _p(oub), _p(has), _p(exh), _p(obj),
                                    C.byref(st)))
        return dict(lb=olb[:, :n], ub=oub[:, :n], has_solution=has[:k].astype(bool), exhaustive=exh[:k].astype(bool),
                    objective=obj[:k].astype(np.int64), stats=st.as_dict())

    def solve_groups(self, lb, ub, groups, ngroups=None, stop_flag=None):
        """tb_solve_groups: K roots of this solver's network ([K, nvars] int32 boxes, each a narrowing of the
        problem's), root r a box of group groups[r]; each group is solved over the union of its boxes, with one
        incumbent shared by its boxes. `ngroups` defaults to max(groups) + 1. Returns arrays of length ngroups, shaped
        as solve_batch's."""
        n = self.problem.nvars
        lb = np.ascontiguousarray(lb, dtype=np.int32).reshape(-1, n)
        ub = np.ascontiguousarray(ub, dtype=np.int32).reshape(-1, n)
        if lb.shape != ub.shape:
            raise ValueError("lb and ub must have the same shape [K, nvars]")
        k = lb.shape[0]
        groups = np.ascontiguousarray(groups, dtype=np.int32).reshape(-1)
        if groups.shape[0] != k:
            raise ValueError("groups must have one entry per root")
        if ngroups is None:
            ngroups = int(groups.max()) + 1 if k else 0
        m = max(1, ngroups)
        olb = np.zeros((m, max(1, n)), np.int32)
        oub = np.zeros((m, max(1, n)), np.int32)
        has = np.zeros(m, np.int32)
        exh = np.zeros(m, np.int32)
        obj = np.zeros(m, np.int32)
        st = abi.TbStats()
        _check(lib().tb_solve_groups(self._h, k, _p(lb), _p(ub), _p(groups), ngroups, stop_flag, _p(olb), _p(oub),
                                     _p(has), _p(exh), _p(obj), C.byref(st)))
        g = max(0, ngroups)
        return dict(lb=olb[:g, :n], ub=oub[:g, :n], has_solution=has[:g].astype(bool), exhaustive=exh[:g].astype(bool),
                    objective=obj[:g].astype(np.int64), stats=st.as_dict())

    def solve_objectives(self, lb, ub, obj_vars, maximize, stop_flag=None):
        """tb_solve_objectives: this solver's network over the union of K boxes ([K, nvars] int32, each a narrowing of
        the problem's), optimised for every objective m in one launch: variable obj_vars[m], maximised where
        maximize[m] is true, minimised elsewhere. Every solution found is a witness for every objective. Returns arrays
        of length nobj, shaped as solve_groups's: `objective` is the optimum in the objective's own sense (abi.POS_INF
        without a solution), and row m of lb / ub is a solution with obj_vars[m] fixed to it. The problem's own
        objective plays no part; narrow its upper bound in the boxes to keep to (near-)optimal solutions."""
        n = self.problem.nvars
        lb = np.ascontiguousarray(lb, dtype=np.int32).reshape(-1, n)
        ub = np.ascontiguousarray(ub, dtype=np.int32).reshape(-1, n)
        if lb.shape != ub.shape:
            raise ValueError("lb and ub must have the same shape [K, nvars]")
        obj_vars = np.ascontiguousarray(obj_vars, dtype=np.int32).reshape(-1)
        maximize = np.ascontiguousarray(maximize, dtype=np.int32).reshape(-1)
        if maximize.shape != obj_vars.shape:
            raise ValueError("maximize must have one entry per objective")
        m = obj_vars.shape[0]
        olb = np.zeros((max(1, m), max(1, n)), np.int32)
        oub = np.zeros((max(1, m), max(1, n)), np.int32)
        has = np.zeros(max(1, m), np.int32)
        exh = np.zeros(max(1, m), np.int32)
        obj = np.zeros(max(1, m), np.int32)
        st = abi.TbStats()
        _check(lib().tb_solve_objectives(self._h, lb.shape[0], _p(lb), _p(ub), m, _p(obj_vars), _p(maximize), stop_flag,
                                         _p(olb), _p(oub), _p(has), _p(exh), _p(obj), C.byref(st)))
        return dict(lb=olb[:m, :n], ub=oub[:m, :n], has_solution=has[:m].astype(bool), exhaustive=exh[:m].astype(bool),
                    objective=obj[:m].astype(np.int64), stats=st.as_dict())

    def hull(self, vars=None, lb=None, ub=None, stop_flag=None):
        """The solution hull: for each variable of `vars` (default: every variable), the smallest and the largest
        value it takes in a solution of the network over the union of the boxes lb / ub ([K, nvars] or [nvars];
        default: the problem's root), as one solve_objectives call of a minimisation and a maximisation per variable.
        Returns `lb` / `ub` per variable, `exact_lb` / `exact_ub` (that side was proven: its objective was searched to
        its end; otherwise the value is a witnessed one, inside the hull), `has_solution` and the stats. Without a
        solution the hull is empty: lb = abi.POS_INF and ub = abi.NEG_INF."""
        vs = np.arange(self.problem.nvars, dtype=np.int32) if vars is None else np.asarray(vars, np.int32).reshape(-1)
        lb = self.problem.lb if lb is None else lb
        ub = self.problem.ub if ub is None else ub
        k = vs.shape[0]
        r = self.solve_objectives(lb, ub, np.concatenate([vs, vs]),
                                  np.concatenate([np.zeros(k, np.int32), np.ones(k, np.int32)]), stop_flag)
        has = bool(r["has_solution"].any())
        lo, hi = r["objective"][:k].copy(), r["objective"][k:].copy()
        if not has:
            lo[:], hi[:] = abi.POS_INF, abi.NEG_INF
        return dict(vars=vs, lb=lo, ub=hi, exact_lb=r["exhaustive"][:k].copy(), exact_ub=r["exhaustive"][k:].copy(),
                    has_solution=has, stats=r["stats"])

    def solve_supports(self, lb, ub, q_var, q_val, witnesses=0, stop_flag=None):
        """tb_solve_supports: for every query i, is there a solution of this solver's network over the union of K boxes
        ([K, nvars] int32, each a narrowing of the problem's) with q_var[i] = q_val[i]? Returns `supported` (int8 [nq]:
        1 = yes, 0 = proven no, -1 = unknown), `witness` (int32 [nq]: the row of wit_lb / wit_ub that holds the value,
        -1 = none), `wit_lb` / `wit_ub` ([nwit, nvars] solution stores; at most `witnesses` rows) and the stats. The
        problem's own objective plays no part; narrow its upper bound in the boxes to ask about (near-)optimal
        solutions."""
        n = self.problem.nvars
        lb = np.ascontiguousarray(lb, dtype=np.int32).reshape(-1, n)
        ub = np.ascontiguousarray(ub, dtype=np.int32).reshape(-1, n)
        if lb.shape != ub.shape:
            raise ValueError("lb and ub must have the same shape [K, nvars]")
        q_var = np.ascontiguousarray(q_var, dtype=np.int32).reshape(-1)
        q_val = np.ascontiguousarray(q_val, dtype=np.int32).reshape(-1)
        if q_val.shape != q_var.shape:
            raise ValueError("q_val must have one entry per query")
        m, w = q_var.shape[0], int(witnesses)
        sup = np.zeros(max(1, m), np.int32)
        wit = np.full(max(1, m), -1, np.int32)
        wlb = np.zeros((max(1, w), max(1, n)), np.int32) if w >= 0 else None
        wub = np.zeros((max(1, w), max(1, n)), np.int32) if w >= 0 else None
        nwit = np.zeros(1, np.int32)
        st = abi.TbStats()
        _check(lib().tb_solve_supports(self._h, lb.shape[0], _p(lb), _p(ub), m, _p(q_var), _p(q_val), stop_flag, _p(sup),
                                       _p(wit), w, _p(wlb), _p(wub), _p(nwit), C.byref(st)))
        k = int(nwit[0])
        return dict(supported=sup[:m].astype(np.int8), witness=wit[:m].copy(), wit_lb=wlb[:k, :n], wit_ub=wub[:k, :n],
                    stats=st.as_dict())

    # Input guard of solution_domains: one query per value, each a group of the launch with a root per box.
    MAX_DOMAIN_VALUES = 1 << 22

    def solution_domains(self, vars=None, lb=None, ub=None, witnesses=0, stop_flag=None):
        """The solution domains: for each variable of `vars` (default: every variable), the values it takes in some
        solution of the network over the union of the boxes lb / ub ([K, nvars] or [nvars]; default: the problem's
        root), as one solve_supports call with a query per value of the variable's range over the boxes. Returns, per
        variable, `supported` (the values with a solution) and `unknown` (the values neither supported nor proven
        unsupported), `exact` (every value of the variable was decided), `has_solution` (some value is supported), and
        the stats; with `witnesses` > 0 also `witness` (per variable, the pool row of each supported value, -1 = none)
        and the pool `wit_lb` / `wit_ub`. Raises ValueError on an infinite bound of a queried variable or when the
        values number more than MAX_DOMAIN_VALUES."""
        n = self.problem.nvars
        vs = np.arange(n, dtype=np.int32) if vars is None else np.asarray(vars, np.int32).reshape(-1)
        lb = np.asarray(self.problem.lb if lb is None else lb, np.int64).reshape(-1, n)
        ub = np.asarray(self.problem.ub if ub is None else ub, np.int64).reshape(-1, n)
        ranges = []
        for v in vs:
            live = lb[:, v] <= ub[:, v]
            if not live.any():
                ranges.append((0, -1))
                continue
            a, b = int(lb[live, v].min()), int(ub[live, v].max())
            if a == abi.NEG_INF or b == abi.POS_INF:
                raise ValueError(f"variable {int(v)} has an infinite bound: its solution domain cannot be enumerated")
            ranges.append((a, b))
        total = sum(b - a + 1 for a, b in ranges)
        if total > self.MAX_DOMAIN_VALUES:
            raise ValueError(f"{total} values to query, more than MAX_DOMAIN_VALUES = {self.MAX_DOMAIN_VALUES}")
        q_var = np.concatenate([np.full(b - a + 1, v, np.int32) for v, (a, b) in zip(vs, ranges)] + [np.zeros(0, np.int32)])
        q_val = np.concatenate([np.arange(a, b + 1, dtype=np.int64) for a, b in ranges] + [np.zeros(0, np.int64)])
        if total:
            r = self.solve_supports(lb, ub, q_var, q_val, witnesses, stop_flag)
        else:                                   # (every queried variable is empty in every box)
            r = dict(supported=np.zeros(0, np.int8), witness=np.zeros(0, np.int32), wit_lb=np.zeros((0, n), np.int32),
                     wit_ub=np.zeros((0, n), np.int32), stats=None)
        out = dict(vars=vs, supported=[], unknown=[], exact=np.zeros(len(vs), bool),
                   has_solution=bool((r["supported"] == 1).any()), stats=r["stats"])
        if witnesses > 0:
            out.update(witness=[], wit_lb=r["wit_lb"], wit_ub=r["wit_ub"])
        at = 0
        for i, (a, b) in enumerate(ranges):
            k = b - a + 1
            ans, vals = r["supported"][at:at + k], q_val[at:at + k]
            out["supported"].append(vals[ans == 1])
            out["unknown"].append(vals[ans == -1])
            out["exact"][i] = not (ans == -1).any()
            if witnesses > 0:
                out["witness"].append(r["witness"][at:at + k][ans == 1])
            at += k
        return out

    def solve_front(self, lb, ub, x, y, levels, maximize_x=False, maximize_y=False, stop_flag=None):
        """tb_solve_front: for every level t of `levels` (strictly ascending, finite), the best value of variable y
        (maximised when maximize_y, minimised elsewhere) over the solutions of this solver's network on the union of K
        boxes ([K, nvars] int32, each a narrowing of the problem's) with x <= t (x >= t when maximize_x), in one launch.
        Returns arrays of length nlev, shaped as solve_objectives's: row i of lb / ub is a solution with y fixed to
        the value and x fixed to the best value the row allows on the level's side; `exhaustive` says the value is
        proven. The problem's own objective plays no part."""
        n = self.problem.nvars
        lb = np.ascontiguousarray(lb, dtype=np.int32).reshape(-1, n)
        ub = np.ascontiguousarray(ub, dtype=np.int32).reshape(-1, n)
        if lb.shape != ub.shape:
            raise ValueError("lb and ub must have the same shape [K, nvars]")
        lv = np.asarray(levels, np.int64).reshape(-1)
        if ((lv < abi.NEG_INF) | (lv > abi.POS_INF)).any():
            raise ValueError("a level is outside the int32 range")
        lv = np.ascontiguousarray(lv, dtype=np.int32)
        m = lv.shape[0]
        olb = np.zeros((max(1, m), max(1, n)), np.int32)
        oub = np.zeros((max(1, m), max(1, n)), np.int32)
        has = np.zeros(max(1, m), np.int32)
        exh = np.zeros(max(1, m), np.int32)
        obj = np.zeros(max(1, m), np.int32)
        st = abi.TbStats()
        _check(lib().tb_solve_front(self._h, lb.shape[0], _p(lb), _p(ub), int(x), int(maximize_x), int(y),
                                    int(maximize_y), m, _p(lv), stop_flag, _p(olb), _p(oub), _p(has), _p(exh), _p(obj),
                                    C.byref(st)))
        return dict(lb=olb[:m, :n], ub=oub[:m, :n], has_solution=has[:m].astype(bool), exhaustive=exh[:m].astype(bool),
                    objective=obj[:m].astype(np.int64), stats=st.as_dict())

    # Input guard of pareto_front: every level is a group of the launch with a best row of the store's size.
    MAX_FRONT_LEVELS = 1 << 16

    def pareto_front(self, x, y, lb=None, ub=None, maximize_x=False, maximize_y=False, levels=None, stop_flag=None):
        """The Pareto front of objectives x and y (each minimised, or maximised where maximize_* is true) over the union
        of the boxes lb / ub ([K, nvars] or [nvars]; default: the problem's root), as one solve_front call. `levels`
        defaults to one level per value of x's range over the boxes, which makes the front exact when every level is
        exhaustive. Returns `points` [(x*, y*)] in x's preferred order, with their rows `lb` / `ub` and `proven` per
        point (its level is exhaustive), `exact` (every level is), `levels` and the stats. Raises ValueError on an
        infinite bound of x when `levels` is None, and on more than MAX_FRONT_LEVELS levels, before any launch."""
        n = self.problem.nvars
        lb = np.asarray(self.problem.lb if lb is None else lb, np.int64).reshape(-1, n)
        ub = np.asarray(self.problem.ub if ub is None else ub, np.int64).reshape(-1, n)
        if levels is None:
            live = lb[:, x] <= ub[:, x]
            a, b = (int(lb[live, x].min()), int(ub[live, x].max())) if live.any() else (0, -1)
            if a == abi.NEG_INF or b == abi.POS_INF:
                raise ValueError(f"variable {int(x)} has an infinite bound: give the levels of the front")
            if b - a + 1 > self.MAX_FRONT_LEVELS:
                raise ValueError(f"{b - a + 1} levels, more than MAX_FRONT_LEVELS = {self.MAX_FRONT_LEVELS}")
            levels = np.arange(a, b + 1, dtype=np.int64)
        levels = np.asarray(levels, np.int64).reshape(-1)
        if len(levels) > self.MAX_FRONT_LEVELS:
            raise ValueError(f"{len(levels)} levels, more than MAX_FRONT_LEVELS = {self.MAX_FRONT_LEVELS}")
        if len(levels):
            r = self.solve_front(lb, ub, x, y, levels, maximize_x, maximize_y, stop_flag)
        else:                                   # (x is empty in every box: no solution, nothing to search)
            r = dict(lb=np.zeros((0, n), np.int32), ub=np.zeros((0, n), np.int32), has_solution=np.zeros(0, bool),
                     exhaustive=np.zeros(0, bool), objective=np.zeros(0, np.int64), stats=None)
        f = front_points(r, x, maximize_x, maximize_y)
        return dict(points=f["points"], lb=f["lb"], ub=f["ub"], proven=f["proven"], exact=bool(r["exhaustive"].all()),
                    levels=levels, stats=r["stats"])

    def export_bound_handle(self):
        buf = C.create_string_buffer(64)
        _check(lib().tb_export_bound_handle(self._h, C.cast(buf, C.c_void_p)))
        return buf.raw

    def import_peer_bounds(self, handles):
        blob = b"".join(handles)
        buf = C.create_string_buffer(blob, len(blob))
        _check(lib().tb_import_peer_bounds(self._h, C.cast(buf, C.c_void_p), len(handles)))

    def stream_solutions(self, slots=16):
        """-i / -a: improving solutions also go to a ring the host can read while solve() runs (tb_stream_solutions)."""
        L = lib()
        L.tb_stream_solutions.argtypes = [C.c_void_p, C.c_int32]
        L.tb_stream_solutions.restype = C.c_int
        _check(L.tb_stream_solutions(self._h, slots))

    def poll_solution(self):
        """The newest streamed solution not returned yet, or None (call from another thread while solve() blocks)."""
        L = lib()
        i32p = C.POINTER(C.c_int32)
        L.tb_poll_solution.argtypes = [C.c_void_p, i32p, i32p, i32p, C.POINTER(C.c_int64)]
        L.tb_poll_solution.restype = C.c_int32
        n = self.problem.nvars
        lb, ub = np.zeros(max(1, n), np.int32), np.zeros(max(1, n), np.int32)
        obj, t = C.c_int32(0), C.c_int64(0)
        rc = L.tb_poll_solution(self._h, _p(lb), _p(ub), C.byref(obj), C.byref(t))
        if rc < 0:
            _check(-rc)
        return None if rc == 0 else dict(lb=lb[:n], ub=ub[:n], objective=obj.value, time_ns=t.value)

    def set_timeout(self, ms):
        L = lib()
        L.tb_set_timeout.argtypes = [C.c_void_p, C.c_uint64]
        L.tb_set_timeout.restype = C.c_int
        _check(L.tb_set_timeout(self._h, ms))

    def result_pack(self):
        """The latest solve() of this solver as bytes (tb_result_pack): what one rank contributes to the final gather."""
        L = lib()
        L.tb_result_size.argtypes = [C.c_void_p]
        L.tb_result_size.restype = C.c_size_t
        L.tb_result_pack.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.tb_result_pack.restype = C.c_int
        n = L.tb_result_size(self._h)
        buf = np.zeros(n, np.uint8)
        _check(L.tb_result_pack(self._h, buf.ctypes.data_as(C.c_void_p), n))
        return buf

    def read_bound(self):
        v = C.c_int32(0)
        _check(lib().tb_read_bound(self._h, C.byref(v)))
        return v.value


def link_peers(solvers):
    arr = (C.c_void_p * len(solvers))(*[s.handle for s in solvers])
    _check(lib().tb_link_peers(arr, len(solvers)))

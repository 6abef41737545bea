#!/usr/bin/env python
"""bench.py — throughput of the dive-and-solve hot path (BASELINE.json metric: propagations/s and
search nodes/s), measured through the C ABI of libturbo_b200.so.

A *step* is one bounded dive-and-solve pass (`tb_solve` with a per-block node budget, the
reference's `-cutnodes`) over the trains15 TNF network (BASELINE config 2, the configuration the
metric is quoted on) as the driver solves it by default: ternarised by our front-end from
benchmarks/trains15.fzn and reduced by the TNF simplifier (fixture tests/golden/simplified/trains15.npz;
`--workload trains15` is the network -disable_simplify leaves, reported as `unsimplified_network`).  `value` counts propagations (one evaluation of one TNF propagator,
the reference's `num_deductions`, include/statistics.hpp:151,354) over the device time of the solve
kernel with the network already resident in HBM; `e2e` runs the same step from host buffers
through tb_create + tb_solve + result read-back + tb_destroy.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

`--dump-outputs DIR` writes what the last timed step returned (best store lb / ub, has_solution, exhaustive,
objective) as DIR/<name>.npy in float64, so that two builds can be compared output for output on the same inputs.
When several solutions reach the best objective, which one lb / ub hold depends on which of the concurrent blocks
found it first (two runs of the default workload on one B200: objective 286 both times, stores differing in 48 of
13501 variables), so stores are compared by objective and by checking them against the network.

N > 1 is launched under torchrun (one rank per GPU): subproblems are sharded idx = k*N + rank, the
incumbent is exchanged through CUDA-IPC peer-mapped cells, torch.distributed only carries the
handles and the final reduction.  `--impl reference` times the CPU oracle (the reference itself
cannot be built offline: its arithmetic lives in un-vendored lala-* libraries, see DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# The benchmark writes nothing into the tree it runs from: without this, importing tests/, tools/, oracle/ and
# turbo_b200/ would leave __pycache__/ directories in a writable checkout.
sys.dont_write_bytecode = True

from tests import golden_io  # noqa: E402  (fixture loader only; no oracle code)
from turbo_b200 import abi  # noqa: E402

SMEM_BYTES_PER_CLK_PER_SM = 128           # nominal; B300_MICROARCH.md "smem crossbar BW 128/N B/cyc/SM"
DEFAULT_SUB = 17                          # EPS depth of the default workload on one B200 (2^17 >= 300 x 296 blocks), fixed for both arms


def sm_count(device=0):
    from turbo_b200 import engine
    return engine.device_info(device)["sm_count"]


def smem_peak(engine, device, sm_mhz, world):
    """Denominator of the roofline: the MEASURED shared-memory bandwidth (LDS.64 stream on every SM, tb_measure_smem_peak)
    scaled from the clock it ran at (the device's maximum) to the SM clock sampled under load; the nominal figure next to it."""
    info = engine.device_info(device)
    m = engine.measure_smem_peak(device)
    nominal = SMEM_BYTES_PER_CLK_PER_SM * info["sm_count"] * world * (sm_mhz or 1965.0) * 1e6 / 1e9
    bpc = m["bytes_per_clk_per_sm"]
    measured = bpc * info["sm_count"] * world * (sm_mhz or 1965.0) * 1e6 / 1e9 if bpc > 0 else m["gb_per_s"] * world
    return {"measured_gbs": measured, "measured_bytes_per_clk_per_sm": bpc, "measured_gbs_at_max_clock_one_gpu": m["gb_per_s"],
            "nominal_gbs": nominal, "sm_count": info["sm_count"]}


def recorded_traffic(workload, n_gpus):
    """DRAM bytes per launch of the solve kernel from the committed `ncu --set full` capture of this workload
    (profiles/r02_traffic.json, written by tools/ncu_summary.py): dram__bytes_read.sum + dram__bytes_write.sum."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    except (OSError, ValueError):
        return None
    rec = t.get(workload)
    return None if rec is None else rec.get("dram_bytes_per_launch")


def load_workload(name):
    if name.startswith("synthetic"):
        from turbo_b200.model import Model
        _, nv, npr = name.split(":") if ":" in name else (name, "100000", "1000000")
        m = Model.synthetic(int(nv), int(npr), 0xB200)
        return m.problem, dict(objective_kind=-1)
    if name.startswith("simplified:"):     # the network the TNF simplifier leaves (tests/golden/simplified)
        return golden_io.load_simplified_problem(name.split(":", 1)[1])
    return golden_io.load(name)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        fd, self.path = tempfile.mkstemp(suffix=".csv")
        os.close(fd)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        clocks, maxs, reasons = [], [], set()
        for line in open(self.path):
            f = [t.strip() for t in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clocks.append(float(f[1]))
                maxs.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if clocks:
            out.update(sm_mhz=float(np.median(clocks)), sm_max_mhz=float(max(maxs)), reasons=sorted(reasons), samples=len(clocks))
        return out


def reduce_over_ranks(dist, sums, maxes, device="cpu"):
    """Whole-job aggregation: counters are summed over ranks, times are the max over ranks."""
    if dist is None:
        return [float(x) for x in sums], [float(x) for x in maxes]
    import torch
    t = torch.tensor(sums, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    m = torch.tensor(maxes, dtype=torch.float64, device=device)
    dist.all_reduce(m, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()], [float(x) for x in m.tolist()]


def workload_name(workload):
    """BASELINE.json's wording for the configuration: config 2 is `benchmarks/trains15.fzn optimisation, gpu dive-and-solve`."""
    if workload.startswith("synthetic"):
        return "synthetic random TNF constraint network (BASELINE config 5)"
    simplified = workload.startswith("simplified:")
    name = workload.split(":", 1)[1] if simplified else workload
    return "benchmarks/%s.fzn optimisation, gpu dive-and-solve (%s)" % (name, "TNF after the simplifier, the driver's default" if simplified else "TNF as with -disable_simplify")


def data_description(workload):
    if workload.startswith("synthetic"):
        return "synthetic"
    if workload.startswith("simplified:"):
        return ("tests/golden/simplified fixture (TNF of the reference's benchmarks/%s.fzn after the TNF simplifier, "
                "the network the driver solves by default)" % workload.split(":", 1)[1])
    return "tests/golden fixture (TNF of the reference's benchmarks/%s.fzn, as with -disable_simplify)" % workload


def side_leg(engine, pb, opts, steps, flush, sm_mhz, world=1):
    """A short run of the same step on another network (reported next to the headline, not as it)."""
    with engine.Solver(pb, **opts) as s:
        cfg = s.config()
        ms, ded, nodes, narrowed = 0.0, 0, 0, 0
        for i in range(steps + 1):
            flush.fill_(1)
            import torch
            torch.cuda.synchronize()
            st = s.solve()["stats"]
            if i == 0:
                continue                      # warm-up
            ms += st["kernel_ms"]; ded += st["num_deductions"]; nodes += st["nodes"]; narrowed += st["bounds_narrowed"]
    secs = ms / 1e3
    peak = SMEM_BYTES_PER_CLK_PER_SM * sm_count(opts.get("device", 0)) * world * (sm_mhz or 1965.0) * 1e6 / 1e9
    return {"nvars": pb.nvars, "nprops": pb.nprops, "steps": steps, "memory_configuration": abi.MEM_NAMES.get(cfg["mem_kind"], "?"),
            "num_blocks_per_gpu": cfg["num_blocks"], "threads_per_block": cfg["threads_per_block"],
            "value": ded / secs, "unit": "propagations/s", "nodes_per_sec": nodes / secs, "ms_per_step": ms / steps,
            "roofline_frac": (24.0 * ded + 4.0 * narrowed) / secs / 1e9 / peak}


def problem_bytes(pb):
    return int(pb.lb.nbytes + pb.ub.nbytes + pb.props.nbytes + sum(v.nbytes for _, _, v in pb.strategies))


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, pb, result):
    """What tb_solve returned in the last timed step, as float64 .npy files (every int32 is exact in float64). A store
    too large for the budget is written as a fixed, seeded sample of its variables, their indices in var_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    lb, ub = np.asarray(result["lb"]), np.asarray(result["ub"])
    room = DUMP_BUDGET_BYTES - 4096                  # the three scalars and the .npy headers
    if 2 * 8 * lb.size > room:
        keep = np.sort(np.random.default_rng(0).choice(lb.size, room // (3 * 8), replace=False))
        np.save(os.path.join(out_dir, "var_index.npy"), keep.astype(np.float64))
        lb, ub = lb[keep], ub[keep]
    has = result["has_solution"]
    objective = result["lb"][pb.obj_var] if has and pb.obj_var >= 0 else np.nan      # as Solver.solve() reports it
    for name, a in (("lb", lb), ("ub", ub), ("has_solution", has), ("exhaustive", result["exhaustive"]), ("objective", objective)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    from turbo_b200 import engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if engine.device_count() <= 0:
        raise SystemExit("no CUDA device: bench.py measures the CUDA engine and has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the first communicator is created (NCCL_DEBUG=VERSION and up):
        # create it with stdout pointing at stderr, so that rank 0's stdout carries the one JSON line and nothing else
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    pb, info = load_workload(args.workload)
    sub = args.sub if args.sub is not None else (DEFAULT_SUB if args.workload == "simplified:trains15" else -1)
    opts = dict(device=local, gpu_rank=rank, gpu_world=world, cutnodes=args.cutnodes, subproblems_power=sub,
                fixpoint=abi.FP_KINDS[args.fp])
    if args.tpb:
        opts["threads_per_block"] = args.tpb
    if args.blocks:
        opts["or_blocks"] = args.blocks
    if args.mem != "auto":
        opts["mem_kind"] = {"global": abi.MEM_GLOBAL, "store_shared": abi.MEM_STORE_SHARED, "tcn_shared": abi.MEM_TCN_SHARED,
                            "store_cluster": abi.MEM_STORE_CLUSTER}[args.mem]

    def link(solver):
        """Peer-mapped incumbent / dispenser / stop cells over CUDA IPC: handles in rank order, own rank left out."""
        if world > 1:
            handles = [None] * world
            dist.all_gather_object(handles, solver.export_bound_handle())
            solver.import_peer_bounds([h for r, h in enumerate(handles) if r != rank])

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_results(solver):
        """SURVEY.md 8e: one NCCL gather of {best bound, best store, statistics} to rank 0, then reduce_blocks across GPUs."""
        if dist is None:
            return engine.result_reduce([solver.result_pack()])
        mine = torch.from_numpy(solver.result_pack()).cuda()
        got = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
        dist.gather(mine, got, dst=0)
        return engine.result_reduce([g.cpu().numpy() for g in got]) if rank == 0 else None

    solver = engine.Solver(pb, **opts)
    link(solver)
    cfg = solver.config()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step():
        flush.fill_(1)                       # evict L2 between steps
        barrier()                            # every rank starts the run together (they share the incumbent)
        return solver.solve()

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    kernel_ms, ded, nodes, narrowed, fp_ns, launches = 0.0, 0, 0, 0, 0, 0
    for _ in range(args.steps):
        r = step()
        st = r["stats"]
        kernel_ms += st["kernel_ms"]
        ded += st["num_deductions"]
        nodes += st["nodes"]
        narrowed += st["bounds_narrowed"]
        fp_ns += st["timers_ns"][abi.TIMER_FIXPOINT]
        launches += 2                        # solve_kernel + the 1-thread globaltimer probe
    barrier()
    wall_s = time.perf_counter() - t0
    clocks = sampler.stop()
    merged = gather_results(solver)          # of the last timed step: the global best and the summed statistics
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, pb, merged)

    # ---- e2e: host buffers -> tb_create (H2D) -> tb_solve -> results (D2H) -> tb_destroy -------------------
    # the drop-in call pattern (one solver per model); the split says where the time outside the kernel goes
    e2e_steps = args.steps if args.e2e_steps is None else args.e2e_steps
    solver.close()                           # its device memory goes back to the pool the e2e solvers allocate from
    barrier()
    split = dict(create=0.0, link=0.0, solve=0.0, destroy=0.0)
    e2e_ded, e2e_nodes, e2e_s = 0, 0, 0.0
    for i in range(e2e_steps + 2):           # two untimed rounds: the memory pool and the module are warm afterwards
        barrier()
        t = time.perf_counter()
        s2 = engine.Solver(pb, **opts)
        t1 = time.perf_counter()
        link(s2)
        if dist is not None:
            dist.barrier()
        t2 = time.perf_counter()
        r2 = s2.solve()                      # (returns the best store and the statistics to host buffers)
        t3 = time.perf_counter()
        s2.close()
        t4 = time.perf_counter()
        if i < 2:
            continue
        e2e_s += t4 - t
        split["create"] += t1 - t; split["link"] += t2 - t1; split["solve"] += t3 - t2; split["destroy"] += t4 - t3
        e2e_ded += r2["stats"]["num_deductions"]
        e2e_nodes += r2["stats"]["nodes"]
    h2d = problem_bytes(pb)
    d2h = int(2 * 4 * pb.nvars + abi.C.sizeof(abi.TbStats) + 128 * cfg["num_blocks"])

    # ---- strong scaling: ONE fixed instance with a FIXED number of subproblems, whatever the GPU count ---------
    strong = None
    if args.strong_ms > 0:
        sopts = dict(opts, cutnodes=0, subproblems_power=args.strong_sub, timeout_ms=args.strong_ms)
        s3 = engine.Solver(pb, **sopts)
        link(s3)
        barrier()
        r3 = s3.solve()
        m3 = gather_results(s3)
        s3.close()
        s_ms = reduce_over_ranks(dist, [0.0], [r3["stats"]["kernel_ms"]], device="cuda")[1][0]
        if rank == 0:
            st3 = m3["stats"]
            strong = {"workload": workload_name(args.workload), "subproblems_power": args.strong_sub, "budget_ms": args.strong_ms,
                      "n_gpus": world, "kernel_ms": s_ms, "exhaustive": m3["exhaustive"], "nodes": st3["nodes"],
                      "nodes_per_sec": st3["nodes"] / (s_ms / 1e3) if s_ms > 0 else 0.0,
                      "propagations_per_sec": st3["num_deductions"] / (s_ms / 1e3) if s_ms > 0 else 0.0,
                      "subproblems_solved": st3["eps_solved_subproblems"], "subproblems_skipped": st3["eps_skipped_subproblems"],
                      "subproblems_stolen": st3["eps_stolen_subproblems"], "subproblems_total": st3["eps_num_subproblems"],
                      "blocks_done": st3["num_blocks_done"], "blocks": st3["num_blocks"],
                      "first_block_idle_ms": st3["timers_ns"][abi.TIMER_FIRST_BLOCK_IDLE] / 1e6,
                      "best_objective": (golden_io.user_objective(info, m3["lb"], m3["ub"]) if m3["has_solution"] and info.get("objective_kind", -1) >= 0 else None),
                      "time_to_best_ms": st3["timers_ns"][abi.TIMER_LATEST_BEST_OBJ_FOUND] / 1e6,
                      "note": "fixed instance and subproblem count at every GPU count; a budget-bounded run measures how fast the "
                              "SAME pool of subproblems is consumed (limiters: dive cost per subproblem, starvation at the tail, start-up)"}

    # ---- reduce over ranks: sums of counters, max of times ---------------------------------------------------
    (ded, nodes, narrowed, e2e_ded, e2e_nodes), (kernel_ms, e2e_s, wall_s, sp_c, sp_l, sp_s, sp_d) = reduce_over_ranks(
        dist, [ded, nodes, narrowed, e2e_ded, e2e_nodes],
        [kernel_ms, e2e_s, wall_s, split["create"], split["link"], split["solve"], split["destroy"]], device="cuda")

    line = None
    if rank == 0:
        secs = kernel_ms / 1e3
        sm_mhz = clocks["sm_mhz"] or 0.0
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        smem_bytes = 24.0 * ded + 4.0 * narrowed          # SURVEY.md §8(d): algorithmic bytes per propagation
        achieved = smem_bytes / secs / 1e9 if secs > 0 else 0.0
        clk_for_peak = sm_mhz if sm_mhz > 0 else float(peaks.get("sm_max_mhz", 1965.0))
        pk = smem_peak(engine, local, clk_for_peak, world)
        peak = pk["measured_gbs"]
        traffic = recorded_traffic(args.workload, world)
        line = {
            "metric": "propagations/sec", "value": ded / secs if secs > 0 else 0.0, "unit": "propagations/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": kernel_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": data_description(args.workload),
            "config": {"workload": workload_name(args.workload), "workload_arg": args.workload, "nvars": pb.nvars, "nprops": pb.nprops,
                       "cutnodes_per_block": args.cutnodes,
                       "fixpoint": args.fp, "num_blocks_per_gpu": cfg["num_blocks"], "threads_per_block": cfg["threads_per_block"],
                       "memory_configuration": abi.MEM_NAMES.get(cfg["mem_kind"], "?"), "subproblems_power": cfg["subproblems_power"],
                       "l2": "flushed between steps (256 MiB write)", "parallelism": f"eps-shard x{world}"},
            "nodes_per_sec": nodes / secs if secs > 0 else 0.0,
            "nodes": nodes, "propagations": ded, "bounds_narrowed": narrowed,
            "wall_ms_per_step": wall_s * 1e3 / args.steps,
            "fixpoint_time_share": (fp_ns / 1e6 / max(1, cfg["num_blocks"])) / kernel_ms if kernel_ms > 0 else None,
            # of the last timed step, after the final gather (NCCL) and reduce_blocks across the GPUs
            "best_objective": (golden_io.user_objective(info, merged["lb"], merged["ub"]) if merged["has_solution"] and info.get("objective_kind", -1) >= 0 else None),
            "best_rank": merged["best_rank"],
            "e2e": {"value": e2e_ded / e2e_s if e2e_s > 0 else 0.0, "unit": "propagations/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "nodes_per_sec": e2e_nodes / e2e_s if e2e_s > 0 else 0.0,
                    "ms_per_step": e2e_s * 1e3 / e2e_steps,
                    "split_ms_per_step": {"tb_create": sp_c * 1e3 / e2e_steps, "link_peers": sp_l * 1e3 / e2e_steps,
                                          "tb_solve_incl_readback": sp_s * 1e3 / e2e_steps, "tb_destroy": sp_d * 1e3 / e2e_steps}},
            "gpu_launches": launches,
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
            "roofline": {"bound": "smem", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                         "traffic": traffic, "kernel": "solve_kernel (persistent dive-and-solve; fixpoint loop inside)",
                         "peak_source": "measured: LDS.64 stream on every SM (tb_measure_smem_peak), bytes/clk/SM x SMs x SM clock sampled under load",
                         "peak_measured_bytes_per_clk_per_sm": pk["measured_bytes_per_clk_per_sm"],
                         "peak_nominal_gbs": pk["nominal_gbs"], "frac_of_nominal": achieved / pk["nominal_gbs"] if pk["nominal_gbs"] else None,
                         "traffic_source": "profiles/r02_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else None,
                         "hbm_peak_gbs_measured": peaks.get("hbm_gbs")},
        }
        if strong is not None:
            line["strong_scaling"] = strong
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(pb, cfg["subproblems_power"], args)
    if rank == 0 and world == 1 and not args.no_fixpoint_leg:
        # the fixpoint kernel alone (the kernel SURVEY.md 8(d)'s shared-memory roofline is stated for): root fixpoints of
        # the FULL network (a simplified network is already at its root fixpoint: one sweep and nothing to narrow)
        from tools.fixpoint_bench import measure
        fpb, fname = pb, args.workload
        if args.workload.startswith("simplified:"):
            fname = args.workload.split(":", 1)[1]
            fpb, _ = golden_io.load(fname)
        line["fixpoint_kernel"] = measure(fpb, repeat=20, fp=args.fp, tpb=args.tpb, blocks=args.blocks, device=local,
                                          sm_mhz=clocks["sm_mhz"])
        line["fixpoint_kernel"]["network"] = fname
        line["fixpoint_kernel"]["smem_frac_of_measured_peak"] = line["fixpoint_kernel"]["smem_gbs"] / line["roofline"]["peak"]
        if args.workload.startswith("simplified:"):
            # the same step on the network as -disable_simplify leaves it (the r01 headline before the simplifier existed)
            line["unsimplified_network"] = side_leg(engine, fpb, dict(opts, subproblems_power=-1), min(args.steps, 3), flush, clocks["sm_mhz"])
        if not args.fp.endswith("_active"):
            # the same step with the active-set fixpoint (-fp wac1_active): same stores and search tree, but only the
            # propagators whose variables moved are evaluated, so nodes/s is the comparable figure, not propagations/s
            aopts = dict(opts, fixpoint=abi.FP_KINDS[args.fp + "_active"])
            line["active_set"] = side_leg(engine, pb, aopts, min(args.steps, 3), flush, clocks["sm_mhz"])
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)


def cpu_baseline(pb, depth, args, seconds=8.0):
    """The CPU oracle (kind "port") on the host cores, on a bounded sample of the same workload."""
    from oracle import oracle_py as orc
    depth = min(depth, 20)
    cores = os.cpu_count() or 1
    t = time.perf_counter()
    r1 = orc.solve(pb, depth=depth, timeout_ms=int(seconds * 1000), nthreads=1)
    s1 = time.perf_counter() - t
    t = time.perf_counter()
    rn = orc.solve(pb, depth=depth, timeout_ms=int(seconds * 1000), nthreads=cores)
    sn = time.perf_counter() - t
    return {"value": rn["stats"]["num_deductions"] / sn, "unit": "propagations/s", "cores": cores, "kind": "port",
            "sample": f"oracle dive-and-solve on the same TNF for {seconds:.0f} s (Gauss-Seidel AC1, EPS over {cores} threads)",
            "nodes_per_sec": rn["stats"]["nodes"] / sn,
            "value_1core": r1["stats"]["num_deductions"] / s1, "nodes_per_sec_1core": r1["stats"]["nodes"] / s1}


def run_reference(args):
    """--impl reference: the reference's CPU path. The reference cannot be built here (un-vendored
    lala-* dependencies), so this times the oracle port with all host threads.  Same configuration as our arm: the
    same network, the same EPS depth (--sub), the same node budget per search worker (--cutnodes; a worker is a
    host thread here and a thread block there), which also bounds the step: cores x cutnodes nodes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle_py as orc
    pb, info = load_workload(args.workload)
    cores = os.cpu_count() or 1
    depth = args.sub if args.sub is not None else (DEFAULT_SUB if args.workload == "simplified:trains15" else 12)
    for _ in range(min(args.warmup, 1)):
        orc.solve(pb, depth=depth, cutnodes=max(1, args.cutnodes // 20), nthreads=cores)
    ded, nodes, secs = 0, 0, 0.0
    for _ in range(args.steps):
        t = time.perf_counter()
        r = orc.solve(pb, depth=depth, cutnodes=args.cutnodes, timeout_ms=60000, nthreads=cores)
        secs += time.perf_counter() - t
        ded += r["stats"]["num_deductions"]
        nodes += r["stats"]["nodes"]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pb, r)
    value = ded / secs
    line = {"impl": "reference", "metric": "propagations/sec", "value": value, "unit": "propagations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs * 1e3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": data_description(args.workload),
            "config": {"workload": workload_name(args.workload), "workload_arg": args.workload, "nvars": pb.nvars, "nprops": pb.nprops,
                       "cutnodes_per_block": args.cutnodes, "subproblems_power": depth,
                       "step": f"{cores} host threads x {args.cutnodes} nodes of CPU dive-and-solve"},
            "nodes_per_sec": nodes / secs, "nodes": nodes, "propagations": ded,
            "note": "the oracle recomputes every node from the subproblem root (as the reference does) and sweeps Gauss-Seidel style, so a "
                    "CPU node costs about twice the propagations of a GPU node: nodes_per_sec is the like-for-like figure",
            "cpu_baseline": {"value": value, "unit": "propagations/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} steps of {cores} threads x {args.cutnodes} nodes of oracle dive-and-solve at EPS depth {depth}"},
            "e2e": {"value": value, "unit": "propagations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


REPORT_CONFIGS = {"1": "simplified:example_wordpress7_500", "2": "simplified:trains15", "3": "simplified:accap_a3"}


def run_report(args):
    """BASELINE.md §3: CPU-1, CPU-N and GPU-N back to back on the same TNF with the same wall budget, one table
    (`include/cpu_solving.hpp:8-48` is the shape of the CPU legs; the reference binary cannot be built, so they are the
    oracle port). Under torchrun every rank takes part in the GPU leg (sharded subproblems, shared incumbent, NCCL
    gather of the results); rank 0 alone runs the CPU legs and prints. One JSON line per leg, then the table."""
    import torch
    from turbo_b200 import engine
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    budget = args.report_ms
    cores = os.cpu_count() or 1
    rows = []
    for key in args.report.split(","):
        wl = REPORT_CONFIGS.get(key, key)
        pb, info = load_workload(wl)
        objective = lambda lb, ub: golden_io.user_objective(info, lb, ub) if info.get("objective_kind", -1) >= 0 else None

        def row(leg, r, st, secs, n):
            d = {"config": key, "workload": wl, "leg": leg, "workers": n, "budget_ms": budget,
                 "status": ("optimal" if r["exhaustive"] else "feasible") if r["has_solution"] else ("unsatisfiable" if r["exhaustive"] else "unknown"),
                 "objective": objective(r["lb"], r["ub"]) if r["has_solution"] else None, "nodes": st["nodes"],
                 "propagations": st["num_deductions"], "fixpoint_iterations": st["fixpoint_iterations"], "wall_s": secs,
                 "nodes_per_sec": st["nodes"] / secs, "propagations_per_sec": st["num_deductions"] / secs,
                 "time_to_best_s": st["timers_ns"][abi.TIMER_LATEST_BEST_OBJ_FOUND] / 1e9}
            rows.append(d)
            print(json.dumps(d), flush=True)

        if rank == 0 and not args.report_no_cpu:
            from oracle import oracle_py as orc
            for n in (1, cores):
                t = time.perf_counter()
                r = orc.solve(pb, depth=min(12, 20), timeout_ms=budget, nthreads=n)
                row(f"CPU-{n} (oracle port)", r, r["stats"], time.perf_counter() - t, n)
        if dist is not None:
            dist.barrier()
        for fp in ("wac1", "wac1_active"):
            s = engine.Solver(pb, device=local, gpu_rank=rank, gpu_world=world, timeout_ms=budget, fixpoint=abi.FP_KINDS[fp])
            if world > 1:
                handles = [None] * world
                dist.all_gather_object(handles, s.export_bound_handle())
                s.import_peer_bounds([h for q, h in enumerate(handles) if q != rank])
                dist.barrier()
            t = time.perf_counter()
            s.solve()
            secs = time.perf_counter() - t
            if world > 1:
                mine = torch.from_numpy(s.result_pack()).cuda()
                got = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
                dist.gather(mine, got, dst=0)
                m = engine.result_reduce([g.cpu().numpy() for g in got]) if rank == 0 else None
            else:
                m = engine.result_reduce([s.result_pack()])
            cfg = s.config()
            s.close()
            if rank == 0:
                row(f"GPU-{world} ({fp}, {abi.MEM_NAMES.get(cfg['mem_kind'])})", m, m["stats"], secs, world)
    if rank == 0:
        print("\n| config | leg | status | objective | nodes | nodes/s | propagations/s | time to best (s) | wall (s) |")
        print("|---|---|---|---|---|---|---|---|---|")
        for d in rows:
            print(f"| {d['config']} {d['workload']} | {d['leg']} | {d['status']} | {d['objective']} | {d['nodes']} | {d['nodes_per_sec']:.3g} | "
                  f"{d['propagations_per_sec']:.3g} | {d['time_to_best_s']:.2f} | {d['wall_s']:.1f} |")
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline and of the e2e leg; the unsimplified_network and active_set side legs "
                         "run min(steps, 3), which keeps the whole run short")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="simplified:trains15",
                    help="golden fixture name, simplified:<name> (the network the TNF simplifier leaves: what `turbo file.fzn` "
                         "solves by default, as the reference does unless -disable_simplify), or synthetic[:V:P]")
    ap.add_argument("--cutnodes", type=int, default=2000, help="node budget per search worker and step (thread block / host thread)")
    ap.add_argument("--sub", type=int, default=None, help="EPS depth; default: 17 for the default workload (both arms), else auto")
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of the e2e leg (default: --steps)")
    ap.add_argument("--strong-ms", type=int, default=3000, help="wall budget of the strong-scaling leg (0 = skip)")
    ap.add_argument("--strong-sub", type=int, default=20, help="EPS depth of the strong-scaling leg: the same at every GPU count")
    ap.add_argument("--fp", default="wac1", choices=["ac1", "wac1", "ac1_active", "wac1_active"])
    ap.add_argument("--tpb", type=int, default=0)
    ap.add_argument("--blocks", type=int, default=0)
    ap.add_argument("--mem", default="auto", choices=["auto", "global", "store_shared", "tcn_shared", "store_cluster"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fixpoint-leg", action="store_true")
    ap.add_argument("--report", default=None, help="BASELINE.md §3 table instead of the bench line: comma list of configs (1 = wordpress7_500, 2 = trains15, 3 = accap_a3, or a workload name)")
    ap.add_argument("--report-ms", type=int, default=20000, help="wall budget of every leg of --report (the reference's -t 20000)")
    ap.add_argument("--report-no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.report:
        run_report(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

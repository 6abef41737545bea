/* turbo_b200.h — C ABI of the B200-native dive-and-solve engine.
 *
 * This is the drop-in boundary for Turbo's hot path (SURVEY.md §8b).  The reference has no
 * FFI: its seam is the C++ template boundary between the host driver and the lattice-land
 * device templates.  Every entry point below names the reference interface it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions: caller owns all host buffers; the library owns device memory; status codes, no
 * exceptions, no callbacks; plain pointers and sizes only.  All integers are int32 unless noted;
 * bounds use TB_NEG_INF / TB_POS_INF as the -oo / +oo sentinels (reference: Itv = Interval<ZLB<int>>
 * with TURBO_ITV_BITS=32, include/common_solving.hpp:41-54).
 */
#ifndef TURBO_B200_H
#define TURBO_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TB_NEG_INF INT32_MIN
#define TB_POS_INF INT32_MAX

/* Operator of a ternary-normal-form propagator  x = y op z.
 * Replaces lala::Sig inside PIR's bytecode_type {op,x,y,z}
 * (include/common_solving.hpp:738-771, include/barebones_dive_and_solve.hpp:82). */
typedef enum {
  TB_OP_ADD  = 0,  /* x = y + z                                   */
  TB_OP_MUL  = 1,  /* x = y * z                                   */
  TB_OP_TDIV = 2,  /* x = y / z, truncated, z != 0 (int_div)      */
  TB_OP_TMOD = 3,  /* x = y mod z, truncated remainder (int_mod)  */
  TB_OP_MIN  = 4,  /* x = min(y, z)                               */
  TB_OP_MAX  = 5,  /* x = max(y, z)                               */
  TB_OP_EQ   = 6,  /* x = (y == z); precondition: dom(x) within 0..1 (tb_create checks) */
  TB_OP_LEQ  = 7,  /* x = (y <= z); precondition: dom(x) within 0..1               */
  TB_NUM_OPS = 8
} tb_op;

/* One propagator, 16 bytes, immutable (bytecode_type, barebones_dive_and_solve.hpp:561). */
typedef struct { int32_t op, x, y, z; } tb_prop;

/* Variable / value orders (lala::VariableOrder / ValueOrder as used in
 * barebones_dive_and_solve.hpp:193-221 and :362-387). */
typedef enum { TB_VAR_INPUT_ORDER = 0, TB_VAR_FIRST_FAIL = 1, TB_VAR_ANTI_FIRST_FAIL = 2,
               TB_VAR_SMALLEST = 3, TB_VAR_LARGEST = 4 } tb_var_order;
typedef enum { TB_VAL_MIN = 0, TB_VAL_MAX = 1, TB_VAL_SPLIT = 2, TB_VAL_REVERSE_SPLIT = 3 } tb_val_order;

/* One search strategy (StrategyType, barebones_dive_and_solve.hpp:84); n == 0 means "all store
 * variables" (:242,284). */
typedef struct { int32_t var_order, val_order, n; const int32_t* vars; } tb_strategy;

/* The root problem: what UnifiedData::root + GridData carry across the launch boundary
 * (barebones_dive_and_solve.hpp:57-78, 409-453). Host-owned, read-only to the library. */
typedef struct {
  int32_t nvars, nprops;
  const int32_t* lb;              /* [nvars] */
  const int32_t* ub;              /* [nvars] */
  const tb_prop* props;           /* [nprops] */
  int32_t nstrategies;
  const tb_strategy* strategies;
  int32_t has_eps_strategy;       /* GridData::has_eps_strategy (:434) */
  int32_t obj_var;                /* -1 = satisfaction; always minimised (:439-443) */
} tb_problem;

/* AC1 / WAC1: the reference's block fixpoints (every sweep evaluates every propagator, include/config.hpp:91-97).
 * The ..._ACTIVE kinds (SURVEY.md 8f.2; the reference's FixpointSubsetGPU idea, barebones :636,984) keep the same
 * sweeps but a warp only evaluates the chunks of 32 propagators one of whose variables changed since the chunk was
 * last evaluated; same fixpoints, same search, fewer evaluations (num_deductions counts what was evaluated). They
 * apply to the shared-memory placements and to tables of at least 128 chunks (TB_ACTIVE_MIN_CHUNKS); elsewhere they
 * behave like the plain kinds. */
typedef enum { TB_FP_AC1 = 0, TB_FP_WAC1 = 1, TB_FP_AC1_ACTIVE = 2, TB_FP_WAC1_ACTIVE = 3 } tb_fixpoint_kind;

/* Store placement (MemoryKind, include/memory_gpu.hpp:18-22) plus the B200 cluster/DSMEM tier. */
typedef enum { TB_MEM_AUTO = -1, TB_MEM_GLOBAL = 0, TB_MEM_STORE_SHARED = 1, TB_MEM_TCN_SHARED = 2,
               TB_MEM_STORE_CLUSTER = 3 } tb_mem_kind;

/* The subset of Configuration<> read on the device or by configure_gpu_barebones
 * (include/config.hpp:32-57, barebones_dive_and_solve.hpp:527-606). 0 means "auto" unless noted. */
typedef struct {
  int32_t fixpoint;             /* tb_fixpoint_kind; -fp */
  int32_t wac1_threshold;       /* -wac1_threshold */
  int32_t subproblems_power;    /* -sub; -1 = auto: smallest d with 2^d >= factor * blocks * gpus */
  int32_t subproblems_factor;   /* -subfactor (reference default 300) */
  int32_t or_blocks;            /* -or / -p; 0 = auto */
  int32_t threads_per_block;    /* 0 = auto (reference compiles 256) */
  int32_t mem_kind;             /* tb_mem_kind; TB_MEM_AUTO = placement policy; -globalmem forces GLOBAL */
  int32_t cluster_size;         /* CTAs per cluster for STORE_CLUSTER; 0 = auto */
  int32_t verbose;              /* -v count */
  int32_t max_depth;            /* decision stack capacity; 0 = 10000 (MAX_SEARCH_DEPTH, :14) */
  int32_t gpu_rank, gpu_world;  /* subproblem shard of this solver: idx = k * world + rank; 0/0 or 0/1 = all */
  int32_t device;               /* CUDA device ordinal */
  int32_t propagate_repeat;    /* tb_propagate_batch re-runs each store this many times (throughput runs); 0 = 1 */
  uint64_t timeout_ms;          /* -t; 0 = none (enforced by the caller through stop_flag and here) */
  uint64_t cutnodes;            /* -cutnodes; 0 = none (per block, barebones :1024) */
  uint64_t seed;
} tb_options;

enum { TB_TIMER_OVERALL = 0, TB_TIMER_PREPROCESSING, TB_TIMER_SEARCH, TB_TIMER_FIXPOINT,
       TB_TIMER_TRANSFER_CPU2GPU, TB_TIMER_TRANSFER_GPU2CPU, TB_TIMER_SELECT_FP_FUNCTIONS,
       TB_TIMER_WAIT_CPU, TB_TIMER_DIVE, TB_TIMER_LATEST_BEST_OBJ_FOUND, TB_TIMER_FIRST_BLOCK_IDLE,
       TB_NUM_TIMERS };

/* Every counter and timer of Statistics<> (include/statistics.hpp:137-154, Timer :13-29). */
typedef struct {
  int32_t num_blocks, depth_max, exhaustive, threads_per_block;
  int32_t mem_kind, cluster_size, subproblems_power, blocks_per_sm;
  uint64_t nodes, fails, solutions;
  uint64_t eps_num_subproblems, eps_solved_subproblems, eps_skipped_subproblems, num_blocks_done;
  uint64_t fixpoint_iterations, num_deductions;
  uint64_t bounds_narrowed;       /* successful lb/ub updates (4 B each in the roofline, SURVEY §8d) */
  uint64_t shared_bytes, store_bytes, prop_bytes;   /* memory_gpu.hpp:113-122 */
  int64_t cumulative_time_block_ns;
  int64_t timers_ns[TB_NUM_TIMERS];
  double kernel_ms;               /* device time of the solve kernel (CUDA events on its stream) */
  uint64_t eps_stolen_subproblems; /* subproblems this GPU took from a peer's shard once its own was exhausted */
  uint64_t device_bytes;          /* device memory the solver holds (the reference's heap_memory, barebones :579) */
  uint64_t eps_split_subproblems; /* subproblems given up at the tail of the search and re-split into 2^TB_SPLIT_BITS children
                                     (children can be split again; those are not counted) */
  uint64_t eps_split_parts_solved; /* children of those solved; solved + skipped + split = eps_num_subproblems when exhaustive */
  int32_t fixpoint_in_effect;     /* tb_fixpoint_kind the kernels run (an _ACTIVE request falls back to the plain kind on small
                                     tables and outside the shared-memory placements) */
  int32_t pad_;
} tb_stats;

typedef enum { TB_OK = 0, TB_ERR_INVALID = 1, TB_ERR_CUDA = 2, TB_ERR_NOMEM = 3, TB_ERR_UNSUPPORTED = 4,
               TB_ERR_NO_DEVICE = 5, TB_ERR_IO = 6, TB_ERR_PARSE = 7, TB_ERR_DEPTH = 8 } tb_status;

typedef struct tb_solver tb_solver;

/* ---- engine ------------------------------------------------------------------------------------ */

/* Copies the problem to the device, chooses blocks / subproblem depth / placement.
 * Replaces configure_gpu_barebones + UnifiedData construction + initialize_global_data
 * (barebones_dive_and_solve.hpp:479-483, 527-613). */
tb_status tb_create(tb_solver** out, const tb_problem* problem, const tb_options* options);

/* One fixpoint of all propagators on a caller-supplied store (NULL lb_in/ub_in = the root store).
 * Parity hook for `propagate()`'s fixpoint + PIR::deduce (barebones_dive_and_solve.hpp:903-966).
 * On failure (*failed = 1) the output store contents are not canonical. */
tb_status tb_propagate(tb_solver*, const int32_t* lb_in, const int32_t* ub_in,
                       int32_t* lb_out, int32_t* ub_out, int32_t* failed, tb_stats* stats);

/* Batched form: nstores independent stores, one block (or cluster) each, laid out [nstores][nvars].
 * This is the throughput-measurement entry for the fixpoint kernel. */
tb_status tb_propagate_batch(tb_solver*, int32_t nstores, const int32_t* lb_in, const int32_t* ub_in,
                             int32_t* lb_out, int32_t* ub_out, int32_t* failed, tb_stats* stats);

/* The EPS dive to subproblem `idx` at depth `depth` (barebones_dive_and_solve.hpp:663-741).
 * Outputs the store at the subproblem root *before* its first solve-propagation,
 * the remaining depth when a leaf was hit early (0 when the subproblem was reached), and whether
 * that leaf was a failure (1), a solution (2) or none (0). */
tb_status tb_dive(tb_solver*, uint64_t subproblem_idx, int32_t depth,
                  int32_t* lb_out, int32_t* ub_out, int32_t* remaining_depth, int32_t* leaf_kind);

/* Batched dive: subproblems [first, first+count), outputs laid out [count][nvars]. */
tb_status tb_dive_batch(tb_solver*, uint64_t first, int32_t count, int32_t depth,
                        int32_t* lb_out, int32_t* ub_out, int32_t* remaining_depth, int32_t* leaf_kind);

/* The whole dive-and-solve run: persistent kernel, host poll on *stop_flag / timeout, reduction.
 * Replaces gpu_barebones_solve + wait_solving_ends + reduce_blocks
 * (barebones_dive_and_solve.hpp:487-497, 620-901, 1033-1067; memory_gpu.hpp:174-196).
 * Blocks until done; safe to interrupt by writing *stop_flag != 0 from a signal handler/thread. */
tb_status tb_solve(tb_solver*, volatile int32_t* stop_flag,
                   int32_t* best_lb, int32_t* best_ub, int32_t* has_solution,
                   int32_t* exhaustive, tb_stats* stats);

/* Solves nroots problems that share this solver's network and strategies and differ in their root domains
 * (root_lb / root_ub laid out [nroots][nvars]), in one launch of the solve kernel. Each root is searched as if it
 * were the root store of its own tb_solve: its own incumbent, its own first-solution stop for satisfaction, its own
 * result. Outputs: best_lb / best_ub [nroots][nvars] (may be NULL; rows of roots without a solution are left as they
 * are), has_solution / exhaustive [nroots], objective [nroots] (value of obj_var in the returned store; TB_POS_INF
 * when there is none or the problem is a satisfaction problem), stats = the whole batch (counters summed,
 * eps_num_subproblems = nroots * 2^d). stop_flag and the solver's timeout apply to the whole batch; a root whose
 * search had ended before them stays exhaustive.
 * Every root must narrow the solver's root (root_lb >= problem lb, root_ub <= problem ub) and nroots >= 1, else
 * TB_ERR_INVALID; a root with an empty domain is legal (no solution, exhaustive). Subproblems: subproblems_power = -1
 * picks the smallest d with nroots * 2^d >= subproblems_factor * min(blocks, 4 * SMs), an explicit d applies per
 * root; d shrinks until nroots * 2^d fits 2^40. TB_ERR_UNSUPPORTED: linked or sharded solvers (gpu_world > 1), the
 * STORE_CLUSTER placement, tb_stream_solutions enabled. */
tb_status tb_solve_batch(tb_solver*, int32_t nroots, const int32_t* root_lb, const int32_t* root_ub,
                         volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                         int32_t* has_solution, int32_t* exhaustive, int32_t* objective, tb_stats* stats);

/* Solves ngroups problems in one launch, each the network over a UNION of boxes: root r (root_lb / root_ub laid out
 * [nroots][nvars], each a narrowing of the solver's root) is one box of group group_of[r]. A group's answer is what
 * tb_solve would return if its root store could be that union (a domain with holes, x != v as {x <= v-1} u {x >= v+1},
 * or one problem split into cubes): has_solution = some box has a solution; for optimisation objective = the minimum
 * over the boxes and the store a solution of one box at that objective; for satisfaction the first solution found,
 * which ends every box of its group (the group is then not exhaustive, as in tb_solve); exhaustive = every box of the
 * group was searched to its end and no block was cut while searching it. The boxes of a group share its incumbent: a
 * solution found in one prunes all of them from then on. Groups never affect each other. Boxes may overlap (only the
 * union counts). A box with an empty referenced domain is decided on the host (no solution, searched) and does not end
 * its group. Outputs per group: best_lb / best_ub [ngroups][nvars] (may be NULL; rows of groups without a solution are
 * left as they are), has_solution / exhaustive / objective [ngroups] (objective = TB_POS_INF when there is no solution
 * or the problem is a satisfaction problem); stats = the whole launch. Subproblems per root, stop_flag and the timeout
 * apply as in tb_solve_batch (nroots roots). TB_ERR_INVALID: nroots < 1, ngroups < 1, a group_of[r] outside
 * [0, ngroups), a group without a root, a root that widens the solver's root. TB_ERR_UNSUPPORTED: as tb_solve_batch.
 * tb_solve_batch is tb_solve_groups with group_of[r] = r. */
tb_status tb_solve_groups(tb_solver*, int32_t nroots, const int32_t* root_lb, const int32_t* root_ub,
                          const int32_t* group_of, int32_t ngroups, volatile int32_t* stop_flag,
                          int32_t* best_lb, int32_t* best_ub, int32_t* has_solution, int32_t* exhaustive,
                          int32_t* objective, tb_stats* stats);

/* Optimises nobj objectives of one network over one union of boxes, in one launch: objective m minimises
 * (maximize[m] == 0) or maximises (maximize[m] == 1) variable obj_var[m] over the union of nboxes boxes (box_lb /
 * box_ub laid out [nboxes][nvars], each a narrowing of the solver's root, as in tb_solve_groups). The solution hull of
 * a model - the smallest and largest value of each variable in any solution - is 2n such objectives. The problem's own
 * obj_var plays no part: to keep to optimal or near-optimal solutions, narrow its upper bound in the boxes. All the
 * objectives share the union, so every solution any of them finds is a witness for all of them: it gives every
 * objective it improves an incumbent and, where it beats that objective's best, its store. Outputs per objective
 * [nobj]: has_solution; objective = the optimum in the objective's own sense (TB_POS_INF without a solution; an
 * unbounded maximisation reports TB_POS_INF and an unbounded minimisation TB_NEG_INF, with has_solution = 1, and that
 * objective ends there, not exhaustive); exhaustive = every box was searched to its end for this objective and no block
 * was cut while doing so (a non-exhaustive objective holds a witnessed value: an inner bound of the hull); best_lb /
 * best_ub [nobj][nvars] (may be NULL) = a solution store with obj_var[m] FIXED to the objective's value, so that the
 * row's lower bounds are a point with that value (rows of objectives without a solution are left as they are).
 * Repeated objectives are legal; a box with an empty referenced domain is decided on the host, as in tb_solve_groups.
 * A box in which an objective's variable is empty but read by no propagator gives that objective no solution (its
 * search fails at every node of the box), while the other objectives search the box as usual.
 * stop_flag, the timeout and the subproblems per root apply as in tb_solve_groups, with nobj * nboxes roots.
 * TB_ERR_INVALID: nboxes < 1, nobj < 1, an obj_var outside [0, nvars), a maximize other than 0 / 1, a widening box,
 * nobj * nboxes above 2^40 (the subproblem index). TB_ERR_NOMEM: no host memory for the nobj * nboxes roots.
 * TB_ERR_UNSUPPORTED: as tb_solve_batch. */
tb_status tb_solve_objectives(tb_solver*, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                              int32_t nobj, const int32_t* obj_var, const int32_t* maximize,
                              volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                              int32_t* has_solution, int32_t* exhaustive, int32_t* objective, tb_stats* stats);

/* The solution domains of a model, in one launch: query i asks whether some solution of the network over the union of
 * nboxes boxes (box_lb / box_ub laid out [nboxes][nvars], each a narrowing of the solver's root, as in
 * tb_solve_objectives) has q_var[i] = q_val[i]. This is the set of supported values of a variable, which the hull
 * cannot give: x in [1, 9] in the hull says nothing about x = 5. Every query is a satisfaction question; the problem's
 * own obj_var plays no part (to ask about (near-)optimal solutions, narrow its upper bound in the boxes). All the
 * queries share the union, so every solution found supports every query whose value it holds, and ends it.
 * supported [nq]: 1 = a solution was found; 0 = proven that none exists (every (query, box) root was searched to its end
 * and no block was cut while doing so, or was decided on the host); -1 = unknown (stop_flag, the timeout, cutnodes, a
 * depth overflow, a node with nothing to branch on). Duplicate queries are legal and get the same answer. A query
 * whose value lies outside a box's domain of q_var, or a box with an empty referenced domain, is decided on the host for
 * that box (no solution, searched). Witnesses: solutions go to a pool of wit_cap rows, wit_lb / wit_ub
 * [wit_cap][nvars], each a solution (entailed) store; *nwit (may be NULL) = rows written. witness [nq] (may be NULL):
 * for a supported query the row w that holds q_val[i] in the domain of q_var[i] - fixing that variable to the value and
 * taking the lower bounds gives a solution point, as for tb_solve_objectives's rows - or -1: no row (the pool was full,
 * or the query is not supported). Rows of different queries may coincide. wit_cap = 0: answers only. Device memory
 * grows with the pool, not with the queries: one store image per row, none per query.
 * stop_flag, the timeout and the subproblems per root apply as in tb_solve_groups, with (distinct queries) * nboxes
 * roots. TB_ERR_INVALID: nboxes < 1, nq < 1, a q_var outside [0, nvars), a q_val equal to TB_NEG_INF or TB_POS_INF, a
 * widening box, nq * nboxes above 2^40 (the subproblem index), wit_cap < 0, wit_cap > 0 without wit_lb / wit_ub.
 * TB_ERR_NOMEM: no host memory for the roots. TB_ERR_UNSUPPORTED: as tb_solve_batch. */
tb_status tb_solve_supports(tb_solver*, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                            int32_t nq, const int32_t* q_var, const int32_t* q_val,
                            volatile int32_t* stop_flag,
                            int32_t* supported, int32_t* witness,
                            int32_t wit_cap, int32_t* wit_lb, int32_t* wit_ub, int32_t* nwit,
                            tb_stats* stats);

/* The Pareto front of two objectives, in one launch. level [nlev] is strictly ascending and finite; level i answers:
 * the best y_var, in its own sense (maximize_y), over the solutions of the network on the union of nboxes boxes
 * (box_lb / box_ub laid out [nboxes][nvars], each a narrowing of the solver's root, as in tb_solve_objectives) with
 * x_var <= level[i] (x_var >= level[i] when maximize_x = 1). The problem's own obj_var plays no part. The front is the
 * set of levels whose value strictly improves on the previous level in x's preferred order (ascending levels when x
 * is minimised, descending when maximised); with one level per value of x's range it is the exact Pareto front
 * whenever every level is exhaustive. The levels search disjoint slices of x's range - (level[i-1], level[i]] when x is
 * minimised, [level[i], level[i+1]) when maximised, the outermost slice open - and every solution is a witness for
 * every level on its side, so each part of the space is searched once. Outputs per level [nlev], shaped as in
 * tb_solve_objectives: has_solution; objective = the value (TB_POS_INF without a solution; an unbounded y reports its
 * infinity and ends that level, not exhaustive); exhaustive = the value is proven: every slice on the level's side
 * (levels 0..i when x is minimised, i..nlev-1 when maximised) was searched to its end with no block cut, or decided on
 * the host; best_lb / best_ub [nlev][nvars] (may be NULL) = a solution store with y fixed to the value and x fixed to
 * the best value the row allows on the level's side, so the row's lower bounds are the point (x*, y*) (rows of levels
 * without a solution are left as they are). A root whose box's range of x misses its slice, or whose box has an empty
 * referenced domain, is decided on the host. Device memory: the nboxes box images, 24 bytes per root (nlev * nboxes
 * roots), 48 bytes per level, and one best row of 2 * vpad int32 per level (vpad: the padded variable count).
 * stop_flag, the timeout and the subproblems per root apply as in tb_solve_groups. TB_ERR_INVALID: nboxes < 1,
 * nlev < 1, x_var or y_var outside [0, nvars), x_var == y_var, a maximize_* other than 0 / 1, levels not strictly
 * ascending, a level equal to TB_NEG_INF or TB_POS_INF, a widening box, nlev * nboxes above 2^40 (the subproblem
 * index), has_solution / exhaustive / objective NULL. TB_ERR_NOMEM: no host memory for the roots.
 * TB_ERR_UNSUPPORTED: as tb_solve_batch. */
tb_status tb_solve_front(tb_solver*, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                         int32_t x_var, int32_t maximize_x, int32_t y_var, int32_t maximize_y,
                         int32_t nlev, const int32_t* level,
                         volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                         int32_t* has_solution, int32_t* exhaustive, int32_t* objective, tb_stats* stats);

/* Intermediate solutions (-i / -a; the reference's consumer thread, gpu_dive_and_solve.hpp:100-132; its barebones
 * architecture cannot, barebones_dive_and_solve.hpp:465-467).  tb_stream_solutions (before tb_solve) makes every
 * improving solution also land in a ring of `slots` store images; tb_poll_solution, called from ANOTHER host thread
 * while tb_solve blocks (no callbacks into the host), hands out the oldest solution not handed out yet: returns 1 and
 * fills lb / ub / objective (of the minimised variable) / time_ns (since the search started), 0 when there is none,
 * a negative tb_status on error.  A consumer slower than `slots` solutions misses intermediate ones, never the last. */
tb_status tb_stream_solutions(tb_solver*, int32_t slots);
int32_t tb_poll_solution(tb_solver*, int32_t* lb, int32_t* ub, int32_t* objective, int64_t* time_ns);

/* Changes the wall budget of the next tb_solve calls (tb_options.timeout_ms; 0 = none): the driver sets what is left
 * of -t right before it starts the search, so that parsing, simplification and engine creation count against it. */
tb_status tb_set_timeout(tb_solver*, uint64_t timeout_ms);

/* Cross-GPU incumbent sharing and work stealing (SURVEY §8e; GridData::appx_best_bound / next_subproblem,
 * barebones_dive_and_solve.hpp:418,426, which the reference keeps on one device).  Each solver owns one 128-byte
 * block of device cells: its incumbent, the dispenser of its shard (idx = k * gpu_world + gpu_rank) and a stop
 * word.  Linked solvers map each other's blocks over NVLink: an improving block writes the incumbent to every
 * GPU with a system-scope atomicMin, a GPU whose shard is exhausted takes subproblems from a peer's dispenser
 * (TB_STEAL=0 keeps the shards static), the first solution of a satisfaction problem stops every GPU.
 * Same process: tb_link_peers on solvers living on different devices (peer access is enabled here).
 * Other processes (one rank per GPU): export a 64-byte CUDA IPC handle and import the peers' handles IN RANK
 * ORDER WITH THE OWN RANK LEFT OUT (npeers = gpu_world - 1).
 * Runs: every tb_solve call of a solver starts a new epoch, and every cell value carries the epoch it belongs to,
 * so nothing has to be reset between runs and a write of a peer that is still in (or already past) another run is
 * ignored.  The one requirement: linked solvers make the same sequence of tb_solve calls. */
tb_status tb_link_peers(tb_solver** solvers, int32_t n);
tb_status tb_export_bound_handle(tb_solver*, void* handle64);
tb_status tb_import_peer_bounds(tb_solver*, const void* handles64, int32_t npeers);
/* Incumbent of this solver's latest run as its own cell holds it (TB_POS_INF when none). */
tb_status tb_read_bound(tb_solver*, int32_t* bound);

/* Final gather with one process per GPU (SURVEY §8e: "one gather of {best_bound, best_store, tb_stats} to GPU 0, then
 * the reduction of reduce_blocks", barebones_dive_and_solve.hpp:1033-1067).  tb_result_pack serialises what the
 * solver's latest tb_solve returned into tb_result_size() bytes (plain bytes: the caller moves them with whatever
 * it has - an NCCL/MPI gather, a pipe); tb_result_reduce merges n such buffers laid out `stride` bytes apart:
 * counters are summed, depths and kernel times take the maximum, the first idle time the minimum, the search was
 * exhaustive if every shard was, and the best solution is the one with the smallest objective, the earliest found
 * among equals (for a satisfaction problem: the earliest found).  The driver uses the same pair for its -gpus N
 * threads. best_lb / best_ub / best_rank may be NULL. */
size_t tb_result_size(const tb_solver*);
tb_status tb_result_pack(const tb_solver*, void* buf, size_t cap);
tb_status tb_result_reduce(const void* bufs, int32_t n, size_t stride, int32_t* best_lb, int32_t* best_ub,
                           int32_t* has_solution, int32_t* exhaustive, tb_stats* total, int32_t* best_rank);

/* Fills `stats` with the launch configuration chosen by tb_create (num_blocks, mem_kind, ...). */
tb_status tb_get_config(tb_solver*, tb_stats* stats);

/* Introspection of the host layout pass that compiles the propagator table for the device (no GPU
 * needed): how many propagators fall in each device class (operator x constant operands x exact 32-bit
 * arithmetic), how the variables are placed over the shared-memory banks, and the bank model's average
 * number of wavefronts per half-warp load of an 8-byte {lb, ub} pair (1.0 = conflict free).
 * nbanks = 0 keeps the caller's numbering, 16 = bank-aware placement (16 8-byte banks). slot_of may be NULL. */
typedef struct {
  int32_t nclasses, nchunks, nslots, identity;
  int32_t class_count[32];
  uint64_t loads_per_sweep;        /* 8-byte {lb, ub} loads one sweep over the table issues */
  double wavefronts_per_load;
} tb_layout_info;
tb_status tb_layout_describe(const tb_problem* problem, int32_t nbanks, tb_layout_info* info, int32_t* slot_of);
const char* tb_layout_class_name(int32_t cls);
/* STORE_CLUSTER placement (host only): the share of the operand loads of one sweep that stay in the CTA whose warps
 * evaluate the propagator, with the layout pass's placement (variables that occur together share a CTA, a CTA gets
 * the chunks whose operands mostly live in it) and with plain striping (slot = variable index). */
tb_status tb_layout_cluster_locality(const tb_problem* problem, int32_t cluster, int32_t warps_per_cta, double* placed, double* striped);
/* Watch lists of the active-set fixpoint: for every slot of the store image the chunks (32 propagators of the device
 * table) that load it, as CSR (off has *nslots + 1 entries, list *nentries); chunk_of_prop[i] = chunk of propagator i.
 * Call with NULL buffers first to get the sizes. */
tb_status tb_layout_watch_lists(const tb_problem* problem, int32_t nbanks, int32_t* nslots, int32_t* nentries,
                                int32_t* off, int32_t* list, int32_t* slot_of, int32_t* chunk_of_prop);

void tb_destroy(tb_solver*);
const char* tb_last_error(void);
const char* tb_version(void);
/* Number of visible CUDA devices, or 0. Never fails. */
int32_t tb_device_count(void);
/* What the reference prints about the device (cuda_version: include/config.hpp:258-260; total_global_mem_bytes,
 * heap_memory, stack_memory: barebones_dive_and_solve.hpp:579-593). */
typedef struct {
  int32_t cuda_runtime_version, cuda_driver_version, sm_count, cc_major, cc_minor, pad_;
  uint64_t total_global_mem_bytes, free_global_mem_bytes, stack_limit_bytes, heap_limit_bytes;
  char name[64];
} tb_device_info;
tb_status tb_get_device_info(int32_t device, tb_device_info* info);
/* Measured shared-memory read bandwidth of the device (GB/s over all SMs; LDS.64 stream, conflict free) and the
 * bytes per clock per SM that is at the device's maximum SM clock: the measured denominator of the fixpoint
 * kernel's roofline (SURVEY.md 8d states the nominal 128 B/clk/SM). bytes_per_clk_per_sm may be NULL. */
tb_status tb_measure_smem_peak(int32_t device, double* gb_per_s, double* bytes_per_clk_per_sm);
/* -stack <KB>: per-thread stack limit of the device (cudaLimitStackSize, barebones :588-593). */
tb_status tb_set_stack_limit(int32_t device, uint64_t bytes);

/* ---- host front-end (C++ behind a C surface) ------------------------------------------------- */

typedef struct tb_model tb_model;

/* FlatZinc -> TNF.  Replaces parse_flatzinc + ternarize/normalize + interpret
 * (include/common_solving.hpp:404-439, 520-585). flags: bit0 = disable simplification. */
tb_status tb_model_load_fzn(tb_model** out, const char* path, uint32_t flags);
/* Same from a memory buffer (text need not be NUL-terminated). */
tb_status tb_model_parse_fzn(tb_model** out, const char* text, size_t len, uint32_t flags);
/* Synthetic random TNF network with a planted solution (SURVEY §8d, config 5). */
tb_status tb_model_synthetic(tb_model** out, int32_t nvars, int32_t nprops, uint64_t seed);
/* Load / save the compact binary TNF (tests/golden fixtures). */
tb_status tb_model_load_tnf(tb_model** out, const char* path);
tb_status tb_model_save_tnf(const tb_model*, const char* path);

/* Prepend the EPS strategy used while diving (-eps_var_order / -eps_value_order,
 * push_eps_strategy, common_solving.hpp:652-667). The tb_problem must be re-read afterwards. */
tb_status tb_model_push_eps_strategy(tb_model*, int32_t var_order, int32_t val_order);

const tb_problem* tb_model_problem(const tb_model*);
/* 1 when the FlatZinc model maximises (the TNF minimises __MINIMIZE_OBJ = -x, common_solving.hpp:489-510),
 * 0 minimise, -1 satisfy. */
int32_t tb_model_objective_kind(const tb_model*);
/* TNF variable holding the user's objective (not the negated one), or -1. */
int32_t tb_model_user_objective_var(const tb_model*);
int32_t tb_model_num_parsed_variables(const tb_model*);
int32_t tb_model_num_parsed_constraints(const tb_model*);
/* Root store was found inconsistent while building / preprocessing. */
int32_t tb_model_root_failed(const tb_model*);

/* ---- TNF simplifier (SURVEY.md 8f.1; replaces lala-core's Simplifier as driven by CP::preprocess_tcn,
 * include/common_solving.hpp:538-565): root fixpoint -> equivalence classes -> algebraic simplification ->
 * entailed-constraint elimination -> ICSE -> useless-variable elimination, to a fixpoint. The root fixpoint is
 * the CALLER's (the driver passes tb_propagate on the GPU), so narrowing has one implementation. Afterwards
 * tb_model_problem() is the reduced network; tb_model_check_solution / _check_tnf / _format_solution still take
 * stores of tb_model_problem() and expand them to the full network internally. */
typedef struct {
  int32_t iterations, vars_before, props_before, vars_after, props_after;
  int32_t merged_variables;        /* variables that joined another one's equivalence class */
  int32_t eliminated_equalities;   /* propagators that were equalities in disguise (algebraic simplification) */
  int32_t eliminated_entailed;     /* propagators entailed by the root store */
  int32_t eliminated_icse;         /* duplicates of another x = y op z */
  int32_t eliminated_variables;    /* classes left without any propagator */
  int32_t eliminated_functional;   /* x = y op z whose x occurs nowhere else and cannot prune: x is computed at expansion */
  int32_t root_failed;
} tb_simplify_stats;
/* In: a network and its domains in lb/ub. Out: the greatest fixpoint in lb/ub, *failed = 1 if it is empty. */
typedef tb_status (*tb_fixpoint_fn)(void* ctx, const tb_problem* pb, int32_t* lb, int32_t* ub, int32_t* failed);
tb_status tb_model_simplify(tb_model*, tb_fixpoint_fn fixpoint, void* ctx, tb_simplify_stats* stats);
/* tb_fixpoint_fn backed by tb_create + tb_propagate on CUDA device *(int32_t*)ctx (device 0 when ctx is NULL). */
tb_status tb_fixpoint_on_device(void* ctx, const tb_problem* pb, int32_t* lb, int32_t* ub, int32_t* failed);
/* Variables of the network as it was built (before simplification). */
int32_t tb_model_num_full_variables(const tb_model*);
/* Store of tb_model_problem() -> store of the full network (full_ub may be NULL). */
tb_status tb_model_expand_solution(const tb_model*, const int32_t* lb, const int32_t* ub, int32_t* full_lb, int32_t* full_ub);

/* Re-check a point (value of var v = lb[v]) against the ORIGINAL FlatZinc constraints; returns the
 * number of violated constraints (0 = valid) or -1 when the model carries no FlatZinc source
 * (synthetic / .tnf models: use tb_model_check_tnf). */
int32_t tb_model_check_solution(const tb_model*, const int32_t* lb, const int32_t* ub);
/* Check every TNF propagator at the point lb[]. Returns the number violated. */
int32_t tb_model_check_tnf(const tb_model*, const int32_t* lb);
/* Print the solution in FlatZinc output syntax (SolverOutput::print_solution,
 * common_solving.hpp:847-851) into buf; returns bytes needed (excluding NUL). */
size_t tb_model_format_solution(const tb_model*, const int32_t* lb, const int32_t* ub, char* buf, size_t cap);
void tb_model_destroy(tb_model*);

#ifdef __cplusplus
}
#endif
#endif /* TURBO_B200_H */

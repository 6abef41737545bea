// engine_internal.h — POD structures shared between the host driver and the kernels.
#pragma once
#include <stdint.h>
#include "tnf_classes.h"

// One entry of the per-block decision stack: LightBranch<Itv>
// (reference include/barebones_dive_and_solve.hpp:135,358-393). 32 bytes.
struct Decision {
  int var;
  int clb0, cub0, clb1, cub1;   // children[0], children[1]
  int rope0, rope1;             // ropes[0], ropes[1]
  int cur;                      // current_idx
};

struct DevStrategy {            // StrategyType (barebones :84)
  int var_order, val_order, n;
  const int* vars;              // device pointer; n == 0 -> all store variables
};

// Per-block statistics: Statistics<> fields written on the device (include/statistics.hpp:137-154).
struct BlockStats {
  unsigned long long nodes, fails, solutions, eps_solved, eps_skipped, eps_stolen, blocks_done;
  unsigned long long eps_split, eps_parts;     // subproblems given up and re-split at the tail / parts of them solved
  unsigned long long fixpoint_iterations, deductions, narrowed;
  long long t_fixpoint, t_dive, t_best, t_idle;
  int depth_max, exhaustive, best_bound, has_best, error, pad_;
};

// Grid cells (unsigned long long words of one GPU's cell block).
//   TB_CELL_BOUND: GridData::appx_best_bound (:426) as (~epoch << 32) | (bound ^ 0x80000000): an unsigned atomicMin keeps
//                  the newest epoch and, within it, the smallest bound;
//   TB_CELL_NEXT : GridData::next_subproblem (:418) as (epoch << 40) | k, counting this GPU's shard idx = k * world + rank;
//   TB_CELL_STOP : two ints: [0] = epoch in which a peer (or a block of this GPU) asked everybody to stop,
//                  [1] = raised by the host (UnifiedData::stop, :64) with an async copy.
#define TB_CELL_BOUND 0
#define TB_CELL_NEXT 1
#define TB_CELL_STOP 2
#define TB_CELL_STREAM 3      // number of improving solutions streamed so far in this run (tb_stream_solutions)
#define TB_CELL_SPLIT 4       // words 4..7: the control block of the tail-splitting pool (8 unsigned, TB_SPLIT_*)
#define TB_CELL_WORDS 16
// The allocation behind a cell block continues with the pool itself (TB_SPLIT_CAP entries of 32 bytes at byte 128): one
// CUDA IPC handle maps cells, control block and pool into the peers, whose idle blocks take children from it too.
#define TB_CELL_BLOCK_BYTES (TB_CELL_WORDS * 8 + TB_SPLIT_CAP * 32)
#define TB_MAX_PEERS 31
#define TB_K_BITS 40
#define TB_K_MASK ((1ull << TB_K_BITS) - 1ull)

// One record of the intermediate-solution ring (-i / -a; the consumer pattern of gpu_dive_and_solve.hpp:100-132): lives
// in pinned host memory the device writes through the mapping; seq = 1 + number of the solution (0 = empty), written last.
struct StreamRec {
  unsigned long long seq;
  int objective, block;
  long long t_ns;
};
#define TB_STREAM_MAX_SLOTS 64

// Tail splitting (adaptive EPS). The reference fixes 2^d subproblems up front (barebones :548-555); the last, hard ones
// then keep one block each busy while every other block has nothing left to do. Here a block that has worked on one
// subproblem for split_min_nodes nodes while other blocks WAIT gives the subproblem up and enters its 2^split_bits
// children (the subproblems idx * 2^e + j of depth d + e: a dive is a pure function of (root, index, depth)) into a
// pool the waiting blocks - and the block itself - take their work from. Entries can be split again.
struct SplitEntry {
  unsigned long long base;      // index of the first child at depth `depth`
  int depth;                    // dive depth of the children
  unsigned count;               // number of children (0 = entry not published yet)
  unsigned long long next;      // dispenser over the children, (epoch << 32) | next child: advanced by CAS only, so that
                                // a block of another run of a linked solver can never hand out or skip this run's children
  unsigned epoch;               // the run the entry belongs to
  unsigned pad_;
};
static_assert(sizeof(SplitEntry) == 32, "TB_CELL_BLOCK_BYTES counts 32 bytes per pool entry");
#define TB_SPLIT_CAP 16384

// tb_solve_groups / tb_solve_batch / tb_solve_objectives: what the grid shares about one root of the batch and about
// one group of roots (both written by the host before each launch). Subproblem index g = (r << d) | local; a task of
// depth D belongs to root g >> D, root r searches the box of image BatchRoot::image for group BatchRoot::group. A group
// is solved over the union of its roots' boxes: the roots share its incumbent, its stop word and its best store.
// tb_solve_batch puts every root in a group of its own; tb_solve_objectives makes objective m group m, with one root
// per box (root m * nboxes + r reads image r); tb_solve_supports makes query g group g, a satisfaction group whose
// roots g * nboxes + r read image r with one variable fixed (BatchGroup::fix); tb_solve_front makes level i group i,
// whose roots i * nboxes + r read image r with x narrowed to the level's slice.
struct BatchRoot {
  unsigned long long closed;    // weight of the root's search space closed: 2^(56 - D) per task of depth D searched to
                                // the end, 2^(56 - D + rem) per dive leaf at remaining depth rem; 2^56 = everything
  int cut;                      // a block was cut (stop, cutnodes, depth) while searching it, or stop was raised
  int skip;                     // a referenced domain is empty at the root: decided on the host, its subproblems skipped
  int group;                    // the group the root belongs to
  int image;                    // the root's box: image `image` of batch_roots (several roots may share one)
};
static_assert(sizeof(BatchRoot) == 24, "host and device agree on BatchRoot");
// The incumbent is an epoch-tagged MINIMUM of the group's key: lb(obj) when it minimises, ~ub(obj) = -ub(obj) - 1 when
// it maximises (+oo maps to the -oo key, "unbounded", and -oo to the +oo key, "none").
struct BatchGroup {
  unsigned long long bound;     // the group's incumbent, the TB_CELL_BOUND word (epoch-tagged, unsigned atomicMin)
  int stop;                     // the group is over (first solution of a satisfaction problem, unbounded objective)
  int lock;                     // one writer of the group's best image at a time
  int has;                      // the best image holds a solution
  int img_bound;                // key of the best image (TBD_PINF = none)
  int obj;                      // slot of the group's objective variable (-1 = satisfaction)
  int maximize;                 // 1: the group maximises obj
  int fix;                      // slot narrowed to [fix_lo, fix_hi] in every root of the group (-1 = none):
  int fix_lo;                   // tb_solve_supports fixes it to one value, tb_solve_front to the level's slice
  int wit;                      // tb_solve_supports: the witness row of the group (-1 = none; -2 - b while block b
                                // that won the group takes its row)
  int fix_hi;
};
static_assert(sizeof(BatchGroup) == 48, "host and device agree on BatchGroup");
#define TB_BATCH_WEIGHT_BITS 56

// words of the split control block (unsigned), which lives in the cell block (TB_CELL_SPLIT) so that the peers see it
enum { TB_SPLIT_N = 0, TB_SPLIT_WAITING = 1, TB_SPLIT_GONE = 2, TB_SPLIT_HINT = 3, TB_SPLIT_STARTED = 4, TB_SPLIT_NSLOTS = 5, TB_SPLIT_EPOCH = 6 };

// Kernel parameters: what UnifiedData + GridData carry in the reference (barebones :57-78, 409-453),
// flattened to plain device pointers (no managed memory, no device-side malloc).
struct DevParams {
  int nvars, vpad, nprops, nchunks;
  const unsigned long long* words;  // class-sorted device propagator table, nchunks * 32 words (tnf_classes.h)
  int cls_begin[TBC_NUM + 1];   // first chunk of each class
  int cls_last[TBC_NUM];        // real propagators in the last chunk of each class
  const int* slot_of;           // variable -> slot of the store image (layout.h)
  const int* var_of;            // slot -> variable, -1 for padding slots
  const unsigned char* referenced;  // per variable: appears in some propagator
  int root_failed, pad1_;       // a referenced variable is empty in the root store
  const int* root_store;        // image of the root store, same layout as a block store
  int nstrategies, has_eps_strategy, obj_var, fixpoint_kind, wac1_threshold, subproblems_power;
  const DevStrategy* strategies;
  unsigned long long num_subproblems, cutnodes, t_start;
  int rank, world, max_depth, npeers;
  int observe_stop, pad3_;      // 0 for the parity hooks (tb_propagate / tb_dive): the stop cells are neither read nor raised
  unsigned epoch, steal;        // tb_solve call number of this solver (tags the grid cells); stealing from peers enabled
  int cluster_size, cluster_log2, vc, pad7_;   // STORE_CLUSTER: CTAs per cluster, its log2, variables per CTA slice
  // per-block scratch in global memory, [slot] major
  int* block_root;              // snapshot of the subproblem root (root_store, barebones :89)
  int* block_best;              // best solution of the block (best_store, :92)
  int* block_store;             // current store when it does not live in shared memory
  Decision* decisions;
  BlockStats* stats;
  // snapshot ring (copying instead of recomputation on backtrack): store image of the node where decision j was taken,
  // kept in slot j % nsnap of the block; snap_tag says which j a slot holds (-1 = none)
  int* block_snap;              // [slot][nsnap] images of 2 * vpad ints
  int* snap_tag;                // [slot][nsnap]
  unsigned* snap_flags;         // [slot][nsnap][nwarps * act_fpw / 4]: the chunks' entailment cache at the snapshot (active set)
  int nsnap, pad2_;
  // grid-shared cells: one 128-byte block per GPU (TB_CELL_*), the peers' blocks mapped over NVLink.  The incumbent and
  // the dispenser carry the epoch (the solver's tb_solve call number) in their high bits, so that a write that belongs
  // to another run of a linked solver can never prune or hand out work in this one (no reset protocol between runs).
  unsigned long long* cells;             // this GPU's block
  unsigned long long* peer_cells[TB_MAX_PEERS];   // the other GPUs' blocks (peer-mapped)
  int peer_rank[TB_MAX_PEERS];           // whose shard a peer's dispenser counts (idx = k * world + peer_rank)
  // active-set fixpoint (TB_FP_*_ACTIVE): slot -> chunks that load it (CSR), and where its flags live in shared memory
  const int* watch_off;                  // vpad + 1 offsets into watch_list
  const int* watch_list;                 // chunk ids, ascending per slot
  const unsigned long long* watch_inline; // per slot: its first three watchers as 16-bit chunk ids (0xFFFF = none), top 16 bits 0xFFFE = more in the CSR list
  // tail splitting (see SplitEntry)
  SplitEntry* split_pool;                // [TB_SPLIT_CAP], behind this GPU's cell block
  unsigned* split_ctl;                   // entries appended / blocks waiting for work / blocks gone / lowest open entry / ...
  int split_bits, split_min_nodes;       // e (0 = off) and the node count after which a subproblem may be given up
  int share_split, pad5_;                // idle blocks also take children from the peers' pools
  // intermediate solutions (tb_stream_solutions): ring of store images in device memory + records in mapped host memory
  int* stream_img;                       // [stream_slots] images of 2 * vpad ints
  StreamRec* stream_rec;                 // [stream_slots], pinned host memory
  int* stream_lock;                      // [TB_STREAM_MAX_SLOTS] one writer per slot at a time
  int stream_slots, pad4_;
  // the propagator table in TENSOR MEMORY (STORE_SHARED, dense kinds): the first tmem_visits visits of every warp read
  // their words from the CTA's TMEM columns instead of L2; tmem_cols = columns the CTA allocates (0 = off)
  int tmem_cols, tmem_visits;
  int act_off;                           // byte offset of the active-set area in dynamic shared memory
  int act_fpw;                           // chunk flags per warp (multiple of 32): chunk ch is flag (ch / nwarps) of warp (ch % nwarps)
  // tb_solve_groups (read by the BATCH kernels only): num_subproblems = nroots << subproblems_power
  const int* batch_roots;                // [nimages][2 * vpad] root images, layout of a block store
  int* batch_best;                       // [ngroups][2 * vpad] best store of each group
  BatchRoot* batch_state;                // [nroots]
  int batch_max_depth;                   // deepest task: root bits + depth fit the 64-bit index, at most 56
  int batch_share;                       // tb_solve_objectives: ngroups, every solution is a witness for all of them;
                                         // 0 = a solution counts for its own group only
  BatchGroup* batch_groups;              // [ngroups]
  // tb_solve_supports: the queries as a CSR over the queried slots, values ascending per slot; the query at position k
  // of batch_qval is group k. batch_nqslots = 0: every other batch call (a solution counts for the groups as above)
  const int* batch_qslot;                // [nqslots] queried slots
  const int* batch_qoff;                 // [nqslots + 1] their ranges in batch_qval
  const int* batch_qval;                 // [ngroups]
  int* batch_wit;                        // [wit_cap][2 * vpad] witness pool, one row per solution that won a query
  unsigned* batch_wit_n;                 // rows taken (may run past wit_cap: those solutions keep no row)
  int batch_nqslots, batch_wit_cap;
  // tb_solve_front: 0 = off (every other call), 1 = the front minimises x, 2 = it maximises x; batch_front_x = x's
  // slot. The two words keep the size a multiple of 16: the kernel arguments behind DevParams keep their alignment, so
  // their loads keep their width
  int batch_front, batch_front_x;
};

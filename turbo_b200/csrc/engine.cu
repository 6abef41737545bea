// engine.cu — B200-native dive-and-solve engine behind the C ABI of include/turbo_b200.h.
//
// Replaces the device hot path of the reference's barebones architecture
// (include/barebones_dive_and_solve.hpp:620-1067) and its launch glue (:464-606,
// include/memory_gpu.hpp).  Design (DESIGN.md has the full story):
//   * one persistent CTA per search worker; the interval store lives in shared memory
//     (STORE_SHARED / TCN_SHARED), striped over a thread-block cluster's distributed shared memory
//     (STORE_CLUSTER, cluster.cu) or in L2-resident global memory (GLOBAL);
//   * propagators are immutable, sorted into classes (tnf_classes.h) and packed to one 64-bit word of three
//     21-bit fields, streamed coalesced (one 64-bit load per lane) from L2, or staged once into shared memory;
//   * the fixpoint loop publishes narrowed bounds with shared-memory atomicMax/atomicMin, detects
//     "changed / failed / not entailed" with a warp REDUX + one atomicOr per warp into a rotating
//     three-slot flag word: one __syncthreads per sweep; entailment (`ask`) is fused into the
//     final sweep instead of a separate pass;
//   * snapshot / restore-from-root / best-store copies are TMA bulk copies (cp.async.bulk) between
//     global and shared memory, completion tracked by an mbarrier;
//   * branching, the decision stack with ropes, the EPS dive and the subproblem dispenser all run
//     in the kernel: no host round trip per node;
//   * backtracking reloads the fixpoint of the node where the decision was taken from a ring of store images in
//     HBM (copying instead of the reference's recomputation from the subproblem root; same stores, same tree);
//   * the *_ACTIVE fixpoint kinds only evaluate the chunks whose variables moved (same fixpoints, fewer evaluations).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <algorithm>
#include <mutex>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/turbo_b200.h"
#include "engine_internal.h"
#include "tnf_device.cuh"
#include "layout.h"

// ================================================================================================
// device helpers
// ================================================================================================

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ unsigned smem_u32(const void* p) {
  return (unsigned)__cvta_generic_to_shared(p);
}

// ---- TMA bulk copies (SASS: UBLKCP) -------------------------------------------------------------
__device__ __forceinline__ void mbar_init(unsigned long long* mbar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* mbar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* mbar, unsigned phase) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(mbar)), "r"(phase) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bulk_g2s_issue(void* sdst, const void* gsrc, unsigned bytes, unsigned long long* mbar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(sdst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g_issue(void* gdst, const void* ssrc, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
// The issuing thread may overwrite the shared source as soon as the copy engine has READ it; the global writes are
// only waited for (bulk_wait_all) by whoever reads an image back or leaves the kernel.
__device__ __forceinline__ void bulk_commit_wait_read() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- tensor memory as a table cache ----------------------------------------------------------------------------
// The fixpoint never touches the tensor cores, so the SM's 256 KB of tensor memory (512 columns x 128 lanes x 32 bit)
// are free. A warp can reach the 32 lanes of its quarter (warp index mod 4) at any column: lane l of the warp keeps
// ITS propagator word of visit k in columns 2k, 2k+1 of its own TMEM lane. tcgen05.st fills them once per launch,
// one tcgen05.ld per visit reads them back with a latency of a dozen cycles instead of an L2 round trip, and the
// table stream leaves the L2 -> SM path altogether.
__device__ __forceinline__ void tmem_alloc(unsigned* smem_dst, unsigned ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned taddr, unsigned ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_st64(unsigned taddr, unsigned long long v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"((unsigned)v), "r"((unsigned)(v >> 32)) : "memory");
}
__device__ __forceinline__ unsigned long long tmem_ld64(unsigned taddr) {
  unsigned lo, hi;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
  return ((unsigned long long)hi << 32) | lo;
}

// The bulk-copy unit takes sizes that are multiples of 16 B; one instruction moves at most this
// many bytes so that the mbarrier transaction count (20 bits) never overflows.
#define BULK_CHUNK (128u * 1024u)

// Threads per CTA: every thread evaluates TBC_U propagators per chunk visit, which takes up to 128 registers
// for TBC_U = 2, so a CTA has at most 512 threads (1024 at 64 registers when TBC_U = 1).
#ifndef TB_MAX_THREADS
#define TB_MAX_THREADS (TBC_U >= 2 ? 512 : 1024)
#endif

// ================================================================================================
// block context
// ================================================================================================

struct Ctl {                       // per-CTA control block in static shared memory
  unsigned long long mbar;
  unsigned long long sel_key[2];   // arg-min key of the variable selection (two cells, used in turn)
  unsigned long long task_idx;     // the subproblem being solved: dive to index task_idx at depth task_depth
  int task_depth;                  // P.subproblems_power, or deeper for a child of a subproblem that was split at the tail
  int task_entry;                  // -1, or the pool entry the child comes from
  int task_src;                    // whose pool that is: -1 this GPU's, else the peer's index
  unsigned task_j;                 // its number inside that entry
  int have_task;                   // next_subproblem() found work
  unsigned task_nodes;             // nodes spent on this subproblem so far
  int abandon;                     // the subproblem is being given up (tail splitting)
  int counted_idle;                // this block is counted among the waiting blocks
  int flags[3];                    // rotating fixpoint flag words
  int sel_first[2];
  int stop, leaf, failed;
  int remaining_depth, depth, cur_strategy, next_unassigned, snap_strategy, snap_next_unassigned;
  int best_bound;
  int pushed;
  int dirty_all;                   // active-set fixpoint: the store was rewritten, every chunk must be evaluated
  long long t_mark;
  unsigned tmem_base;              // tensor-memory address of the CTA's columns (tcgen05.alloc writes it here)
  unsigned long long stream_seq;   // number of the solution being streamed (tb_stream_solutions)
  int stream_slot;                 // and the ring slot it goes to
};

// The block store: one {lb, ub} pair of int32 per slot.  All accesses are volatile inline PTX on explicit
// addresses: the fixpoint loop re-reads bounds other warps narrow concurrently, so a load must never be
// cached in a register across iterations, and the 32-bit shared address of a slot is one LEA.
template <int MEM>
struct StoreRef {           // STORE_SHARED / TCN_SHARED: shared memory of this CTA
  unsigned base;            // shared::cta address of slot 0
  __device__ __forceinline__ unsigned addr(int v) const {
    unsigned r;            // one IMAD; opaque so that the mask of the field decode is not re-associated around it
    asm("mad.lo.u32 %0, %1, 8, %2;" : "=r"(r) : "r"((unsigned)v), "r"(base));
    return r;
  }
  __device__ __forceinline__ void ld(int v, int& l, int& u) const {
    asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(l), "=r"(u) : "r"(addr(v)));
  }
  __device__ __forceinline__ void set(int v, int l, int u) const {
    asm volatile("st.shared.v2.s32 [%0], {%1, %2};" ::"r"(addr(v)), "r"(l), "r"(u) : "memory");
  }
  // Publish a bound if it moved (n != old) and count it: three predicated instructions, no branch.
  __device__ __forceinline__ void tell_lb(int v, int n, int old, unsigned& count) const {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, %3;\n\t@p red.shared.max.s32 [%1], %2;\n\t@p add.u32 %0, %0, 1;\n\t}"
                 : "+r"(count) : "r"(addr(v)), "r"(n), "r"(old) : "memory");
  }
  __device__ __forceinline__ void tell_ub(int v, int n, int old, unsigned& count) const {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, %3;\n\t@p red.shared.min.s32 [%1+4], %2;\n\t@p add.u32 %0, %0, 1;\n\t}"
                 : "+r"(count) : "r"(addr(v)), "r"(n), "r"(old) : "memory");
  }
  // VStore::embed (barebones :707,761-764,805,846,853): in-place meet, returns "changed"
  __device__ __forceinline__ bool embed(int v, int l, int u) const {
    int ol, ou;
    asm volatile("atom.shared.max.s32 %0, [%1], %2;" : "=r"(ol) : "r"(addr(v)), "r"(l) : "memory");
    asm volatile("atom.shared.min.s32 %0, [%1+4], %2;" : "=r"(ou) : "r"(addr(v)), "r"(u) : "memory");
    return l > ol || u < ou;
  }
};

// The same shared-memory store addressed by ABSOLUTE shared addresses: the all-in-tensor-memory kernels rewrite the slot
// fields of their propagator words to `base + 8 * slot` when they fill tensor memory (ctx_init), so the sweep's three
// address computations per evaluation disappear. Only the sweep uses this view; everything else works on slots.
struct StoreAbs {
  __device__ __forceinline__ void ld(int a, int& l, int& u) const {
    asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(l), "=r"(u) : "r"((unsigned)a));
  }
  __device__ __forceinline__ void tell_lb(int a, int n, int old, unsigned& count) const {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, %3;\n\t@p red.shared.max.s32 [%1], %2;\n\t@p add.u32 %0, %0, 1;\n\t}"
                 : "+r"(count) : "r"((unsigned)a), "r"(n), "r"(old) : "memory");
  }
  __device__ __forceinline__ void tell_ub(int a, int n, int old, unsigned& count) const {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %2, %3;\n\t@p red.shared.min.s32 [%1+4], %2;\n\t@p add.u32 %0, %0, 1;\n\t}"
                 : "+r"(count) : "r"((unsigned)a), "r"(n), "r"(old) : "memory");
  }
};

template <>
struct StoreRef<TB_MEM_GLOBAL> {   // L2-resident global memory (ld.cg: never through the non-coherent L1)
  int2* p;
  __device__ __forceinline__ void ld(int v, int& l, int& u) const {
    asm volatile("ld.global.cg.v2.s32 {%0, %1}, [%2];" : "=r"(l), "=r"(u) : "l"(p + v));
  }
  __device__ __forceinline__ void set(int v, int l, int u) const {
    asm volatile("st.global.cg.v2.s32 [%0], {%1, %2};" ::"l"(p + v), "r"(l), "r"(u) : "memory");
  }
  __device__ __forceinline__ void tell_lb(int v, int n, int old, unsigned& count) const { if (n != old) { atomicMax(&p[v].x, n); ++count; } }
  __device__ __forceinline__ void tell_ub(int v, int n, int old, unsigned& count) const { if (n != old) { atomicMin(&p[v].y, n); ++count; } }
  __device__ __forceinline__ bool embed(int v, int l, int u) const {
    int ol = atomicMax(&p[v].x, l), ou = atomicMin(&p[v].y, u);
    return l > ol || u < ou;
  }
};

// Store striped over the distributed shared memory of a thread-block cluster: slot v lives in
// CTA (v mod C) at local index (v div C); every CTA's slice is vc {lb, ub} pairs at the same shared
// offset, reached with mapa + ld/red/atom.shared::cluster.
template <>
struct StoreRef<TB_MEM_STORE_CLUSTER> {
  unsigned base;   // shared::cta address of this CTA's slice
  int lc;          // log2(C)
  unsigned cmask;  // C - 1
  __device__ __forceinline__ unsigned addr(int v) const {
    unsigned r;
    asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(base + (((unsigned)v >> lc) << 3)), "r"((unsigned)v & cmask));
    return r;
  }
  __device__ __forceinline__ void ld(int v, int& l, int& u) const {
    asm volatile("ld.shared::cluster.v2.s32 {%0, %1}, [%2];" : "=r"(l), "=r"(u) : "r"(addr(v)));
  }
  __device__ __forceinline__ void set(int v, int l, int u) const {
    asm volatile("st.shared::cluster.v2.s32 [%0], {%1, %2};" ::"r"(addr(v)), "r"(l), "r"(u) : "memory");
  }
  __device__ __forceinline__ void tell_lb(int v, int n, int old, unsigned& count) const {
    if (n != old) { asm volatile("red.shared::cluster.max.s32 [%0], %1;" ::"r"(addr(v)), "r"(n) : "memory"); ++count; }
  }
  __device__ __forceinline__ void tell_ub(int v, int n, int old, unsigned& count) const {
    if (n != old) { asm volatile("red.shared::cluster.min.s32 [%0], %1;" ::"r"(addr(v) + 4u), "r"(n) : "memory"); ++count; }
  }
  __device__ __forceinline__ bool embed(int v, int l, int u) const {
    const unsigned a = addr(v);
    int ol, ou;
    asm volatile("atom.shared::cluster.max.s32 %0, [%1], %2;" : "=r"(ol) : "r"(a), "r"(l) : "memory");
    asm volatile("atom.shared::cluster.min.s32 %0, [%1], %2;" : "=r"(ou) : "r"(a + 4u), "r"(u) : "memory");
    return l > ol || u < ou;
  }
};

template <int MEM>
__device__ __forceinline__ void init_store_ref(StoreRef<MEM>& st, const DevParams&, unsigned char* dyn, int) {
  // volatile: keep the base in a register instead of re-deriving it (4 instructions) at every chunk
  asm volatile("mov.u32 %0, %1;" : "=r"(st.base) : "r"(smem_u32(dyn)));
}
template <>
__device__ __forceinline__ void init_store_ref<TB_MEM_GLOBAL>(StoreRef<TB_MEM_GLOBAL>& st, const DevParams& P, unsigned char*, int slot) {
  st.p = (int2*)(P.block_store + (size_t)slot * 2 * P.vpad);
}
template <>
__device__ __forceinline__ void init_store_ref<TB_MEM_STORE_CLUSTER>(StoreRef<TB_MEM_STORE_CLUSTER>& st, const DevParams& P, unsigned char* dyn, int) {
  st.base = smem_u32(dyn); st.lc = P.cluster_log2; st.cmask = (unsigned)P.cluster_size - 1u;
}

// A device propagator word with its slot fields rewritten to absolute shared addresses (`base` = address of slot 0);
// constants and unused fields stay as they are. `cls` is the class of the word's chunk.
__device__ __forceinline__ unsigned long long word_to_abs(unsigned long long wd, int cls, unsigned base) {
  unsigned long long a = wd & TBC_FIELD_MASK, b = (wd >> TBC_FIELD_BITS) & TBC_FIELD_MASK, cc = (wd >> (2 * TBC_FIELD_BITS)) & TBC_FIELD_MASK;
  constexpr unsigned kNoX = (1u << TBC_ADD_XK) | (1u << TBC_EQ_T) | (1u << TBC_EQ_F) | (1u << TBC_LEQ_T) | (1u << TBC_LEQ_F);
  constexpr unsigned kNoZ = (1u << TBC_ADD_ZK) | (1u << TBC_EQ_ZK) | (1u << TBC_LEQ_ZK);
  if (!((kNoX >> cls) & 1u)) a = base + 8u * (unsigned)a;
  b = base + 8u * (unsigned)b;
  if (!((kNoZ >> cls) & 1u)) cc = base + 8u * (unsigned)cc;
  return a | (b << TBC_FIELD_BITS) | (cc << (2 * TBC_FIELD_BITS));
}

// The three 21-bit fields of a device propagator word (tnf_classes.h); constants are sign-extended.
template <int CLS>
__device__ __forceinline__ void decode_word(unsigned long long w, int& a, int& b, int& c) {
  const unsigned lo = (unsigned)w, hi = (unsigned)(w >> 32);
  a = (int)(lo & TBC_FIELD_MASK);
  b = (int)(__funnelshift_r(lo, hi, TBC_FIELD_BITS) & TBC_FIELD_MASK);
  c = (int)(hi >> (2 * TBC_FIELD_BITS - 32));          // bit 63 of a word is zero
  if (CLS == TBC_ADD_XK) a = (a << (32 - TBC_FIELD_BITS)) >> (32 - TBC_FIELD_BITS);
  if (!tbd::cls_loads_z(CLS)) c = (c << (32 - TBC_FIELD_BITS)) >> (32 - TBC_FIELD_BITS);
}

// The class that owns chunk `ch`: the table is sorted by class, so it is the largest cls with cls_begin[cls] <= ch
// (empty classes are skipped by the <=).
__device__ __forceinline__ int chunk_class(const DevParams& P, int ch) {
  int cls = 0;
#pragma unroll
  for (int step = 16; step > 0; step >>= 1)
    if (cls + step < TBC_NUM && ch >= P.cls_begin[cls + step]) cls += step;
  return cls;
}

// Per-CTA state of the BATCH kernels only (a function-scope __shared__ object: the other kernels never reference it).
// Set by thread 0 when a task starts: `group`, the group of the task's root, its objective slot `obj` (-1 =
// satisfaction) and sense `maximize`, `image`, the root's box, and the group's fixing `fix` in [fix_lo, fix_hi] (-1 =
// none). `pick` / `key`: witness sharing (batch_share_witness, batch_support_witness).
struct BatchCtl { int won; int group; int obj; int maximize; int image; int pick; int key; int fix; int fix_lo; int fix_hi; };
__device__ __forceinline__ BatchCtl& batch_ctl() { __shared__ BatchCtl b; return b; }

// The incumbent's key of a solution's objective domain [l, u]: l when minimising, ~u = -u - 1 when maximising. The
// incumbent is the minimum key in both senses. The one's complement is a decreasing bijection of the int32 range that
// swaps the sentinels (~TBD_PINF = TBD_NINF, the key of an unbounded objective; ~TBD_NINF = TBD_PINF, "none") and keeps
// every finite bound finite: -u would turn u = INT32_MIN + 1 into TBD_PINF, a solution never recorded.
__device__ __forceinline__ int objective_key(int l, int u, int maximize) { return maximize ? ~u : l; }

// TMALL: every visit of every warp finds its propagator word in tensor memory (the table fits): the sweep is compiled
// without the L2 path and without the test that chooses between the two.
// BATCH: tb_solve_groups - subproblem g of depth D belongs to root g >> D, which has its image and closed-weight counter
// (BatchRoot); its group has the objective, the incumbent, the stop word and the best store (BatchGroup); every
// batch-only branch is `if constexpr`.
template <int MEM, bool ACT = false, bool TMALL = false, bool BATCH = false>
struct Ctx {
  const DevParams& P;
  Ctl& c;
  StoreRef<MEM> store;
  unsigned char* sdyn;     // dynamic shared memory: the store image of this CTA (shared placements)
  const unsigned long long* words;   // the propagator table: global (L2) or shared (TCN_SHARED)
  unsigned mbar_phase;
  unsigned tm_warp;        // tensor-memory address of this warp's table words (tm_visits of them; 0 = none)
  int tm_visits;
  unsigned fp_rot;         // rotation of the three fixpoint flag words, kept across calls (dense fixpoint)
  int sel_par;             // which selection cell the next split() uses
  unsigned narrowed;       // per-thread count of published bounds
  unsigned long long deductions;     // per-warp (lane-uniform) count of propagator evaluations
  int* g_root;             // this block's snapshot (global, same layout as the store)
  int* g_snap;             // this block's snapshot ring (P.nsnap images) and its tags
  int* g_snap_tag;
  unsigned* g_snap_flags;
  int* g_best;
  Decision* dec;
  BlockStats* st;
  Ctl* lc;                 // this CTA's own control block (owns the mbarrier used by its bulk copies)
  int tid, T;              // thread index / thread count of the worker (a CTA, or a whole cluster)
  int slot, nslots;        // worker index / number of workers in the grid
  int cta_rank;            // rank of this CTA inside its cluster (0 without clusters)

  __device__ Ctx(const DevParams& P_, Ctl& c_) : P(P_), c(c_) {}

  // Worker-wide barrier: the CTA barrier, or the cluster barrier when the store is striped over DSMEM.
  __device__ __forceinline__ void sync() const {
    if (MEM == TB_MEM_STORE_CLUSTER) {
      asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
      asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    } else __syncthreads();
  }

  // ---- grid cells (engine_internal.h): incumbent, dispenser, stop; thread 0 only -----------------
  __device__ __forceinline__ unsigned long long bound_word(int b) const {
    return ((unsigned long long)(~P.epoch) << 32) | (unsigned long long)((unsigned)b ^ 0x80000000u);
  }
  // ---- tb_solve_groups: the root of the current task, its group and their cells (thread 0) --------------------------
  __device__ __forceinline__ BatchRoot& batch_root() const { return P.batch_state[c.task_idx >> c.task_depth]; }
  __device__ __forceinline__ BatchGroup& batch_group() const { return P.batch_groups[batch_ctl().group]; }
  __device__ __forceinline__ bool batch_group_over() const { return *(volatile int*)&batch_group().stop != 0; }
  __device__ __forceinline__ void batch_cut() const { *(volatile int*)&batch_root().cut = 1; }
  // the objective slot of the current task (-1 = satisfaction) and its sense: the problem's (minimise), or (BATCH) its
  // group's; every BATCH read of the objective goes through these two
  __device__ __forceinline__ int obj_slot() const {
    if constexpr (BATCH) return batch_ctl().obj;
    else return P.obj_var;
  }
  __device__ __forceinline__ bool maximizes() const {
    if constexpr (BATCH) return batch_ctl().maximize != 0;
    else return false;
  }
  __device__ __forceinline__ unsigned long long* bound_cell() const {
    if constexpr (BATCH) return &batch_group().bound;
    else return P.cells + TB_CELL_BOUND;
  }
  // GridData::appx_best_bound (:426): this GPU's copy; a word left by another run reads as "no incumbent"
  __device__ __forceinline__ int read_bound() const {
    const unsigned long long v = *(volatile unsigned long long*)bound_cell();
    return (unsigned)(v >> 32) == ~P.epoch ? (int)((unsigned)v ^ 0x80000000u) : TBD_PINF;
  }
  // an improving solution goes to this GPU's cell and to every peer's over NVLink (:997 + SURVEY 8e)
  __device__ __forceinline__ void publish_bound(int l) const {
    const unsigned long long w = bound_word(l);
    atomicMin(bound_cell(), w);
    for (int g = 0; g < P.npeers; ++g) atomicMin_system(P.peer_cells[g] + TB_CELL_BOUND, w);
  }
  __device__ __forceinline__ bool stop_raised() const {
    if (!P.observe_stop) return false;
    volatile int* f = (volatile int*)(P.cells + TB_CELL_STOP);
    return f[0] == (int)P.epoch || f[1] != 0;
  }
  // everywhere: the whole job is over (first solution of a satisfaction problem, unbounded objective)
  __device__ __forceinline__ void raise_stop(bool everywhere) const {
    if (!P.observe_stop) return;
    *(volatile int*)(P.cells + TB_CELL_STOP) = (int)P.epoch;
    if (everywhere) for (int g = 0; g < P.npeers; ++g) *(volatile int*)(P.peer_cells[g] + TB_CELL_STOP) = (int)P.epoch;
  }
  // Monotone max on the dispenser of rank q's shard: nobody hands out a counter value below k any more (subtree skip,
  // :732-734). The own cell always carries this run's epoch; a peer's may belong to another run and is left alone then.
  __device__ __forceinline__ void dispenser_skip_to(int peer, unsigned long long k) const {
    const unsigned long long tag = (unsigned long long)P.epoch << TB_K_BITS;
    if (peer < 0) { atomicMax(P.cells + TB_CELL_NEXT, tag | k); return; }
    unsigned long long* cell = P.peer_cells[peer] + TB_CELL_NEXT;
    unsigned long long v = *(volatile unsigned long long*)cell;
    while ((v >> TB_K_BITS) == (unsigned long long)P.epoch && (v & TB_K_MASK) < k) {
      const unsigned long long old = atomicCAS_system(cell, v, tag | k);
      if (old == v) break;
      v = old;
    }
  }
  // The control block and the pool behind a cell block (this GPU's or a peer's).
  __device__ __forceinline__ static unsigned* split_ctl_of(unsigned long long* cb) { return (unsigned*)(cb + TB_CELL_SPLIT); }
  __device__ __forceinline__ static SplitEntry* split_pool_of(unsigned long long* cb) { return (SplitEntry*)(cb + TB_CELL_WORDS); }

  // One child of a split subproblem from the pool behind `cb` (src = -1: this GPU's; else peer `src`'s, over NVLink).
  __device__ __forceinline__ bool take_split_from(unsigned long long* cb, int src) {
    unsigned* ctl = split_ctl_of(cb);
    if (src >= 0 && *(volatile unsigned*)(ctl + TB_SPLIT_EPOCH) != P.epoch) return false;      // the peer is in another run
    SplitEntry* pool = split_pool_of(cb);
    const unsigned n = min(*(volatile unsigned*)(ctl + TB_SPLIT_N), (unsigned)TB_SPLIT_CAP);
    unsigned first_open = n;
    for (unsigned i = *(volatile unsigned*)(ctl + TB_SPLIT_HINT); i < n; ++i) {
      SplitEntry* e = pool + i;
      const unsigned cnt = *(volatile unsigned*)&e->count;
      if (cnt == 0) { first_open = min(first_open, i); continue; }            // being written
      unsigned long long v = *(volatile unsigned long long*)&e->next;
      if ((unsigned)v >= cnt) continue;
      first_open = min(first_open, i);
      // (a CAS, as on the peers' dispensers: the counter of another run is never advanced)
      while ((unsigned)(v >> 32) == P.epoch && (unsigned)v < cnt) {
        const unsigned long long old = src < 0 ? atomicCAS(&e->next, v, v + 1ull) : atomicCAS_system(&e->next, v, v + 1ull);
        if (old == v) {
          const unsigned j = (unsigned)v;
          c.task_idx = e->base + (unsigned long long)j; c.task_depth = e->depth; c.task_entry = (int)i; c.task_j = j; c.task_src = src;
          c.have_task = 1;
          return true;
        }
        v = old;
      }
    }
    if (first_open > *(volatile unsigned*)(ctl + TB_SPLIT_HINT)) {
      if (src < 0) atomicMax(ctl + TB_SPLIT_HINT, first_open); else atomicMax_system(ctl + TB_SPLIT_HINT, first_open);
    }
    return false;
  }
  __device__ __forceinline__ bool take_split(bool peers = true) {
    if (!P.split_bits) return false;
    if (take_split_from(P.cells, -1)) return true;
    if (P.share_split && peers)
      for (int t = 0; t < P.npeers; ++t) { const int g = (slot + t) % P.npeers; if (take_split_from(P.peer_cells[g], g)) return true; }
    return false;
  }
  // Somebody - on this GPU or on a linked one - is waiting for work.
  __device__ __forceinline__ bool somebody_waits() const {
    if (*(volatile unsigned*)(P.split_ctl + TB_SPLIT_WAITING) > 0u) return true;
    if (P.share_split)
      for (int g = 0; g < P.npeers; ++g) {
        volatile unsigned* ctl = split_ctl_of(P.peer_cells[g]);
        if (ctl[TB_SPLIT_EPOCH] == P.epoch && ctl[TB_SPLIT_WAITING] > 0u) return true;
      }
    return false;
  }
  // Every block of every linked GPU (of this run) is waiting or gone: the search is over. A peer whose control block
  // carries an OLDER epoch has not started this run yet - linked solvers make the same sequence of tb_solve calls, so it
  // will: during `grace` it counts as busy. One with a newer epoch has left this run behind.
  __device__ __forceinline__ bool everybody_idle(bool grace) const {
    if (*(volatile unsigned*)(P.split_ctl + TB_SPLIT_WAITING) + *(volatile unsigned*)(P.split_ctl + TB_SPLIT_GONE) < (unsigned)nslots) return false;
    if (P.share_split)
      for (int g = 0; g < P.npeers; ++g) {
        volatile unsigned* ctl = split_ctl_of(P.peer_cells[g]);
        const unsigned pe = ctl[TB_SPLIT_EPOCH];
        if (pe != P.epoch) { if (grace && pe < P.epoch) return false; continue; }
        if (ctl[TB_SPLIT_WAITING] + ctl[TB_SPLIT_GONE] < ctl[TB_SPLIT_NSLOTS]) return false;
      }
    return true;
  }

  // The subproblem this block has been working on becomes 2^split_bits children in the pool (thread 0).
  __device__ __forceinline__ bool push_split() {
    const unsigned i = atomicAdd(P.split_ctl + TB_SPLIT_N, 1u);
    if (i >= (unsigned)TB_SPLIT_CAP) return false;
    SplitEntry* e = P.split_pool + i;
    e->base = c.task_idx << P.split_bits; e->depth = c.task_depth + P.split_bits; e->next = (unsigned long long)P.epoch << 32; e->epoch = P.epoch;
    __threadfence_system();
    *(volatile unsigned*)&e->count = 1u << P.split_bits;
    if (c.task_entry < 0) st->eps_split += 1;      // (a child that is split again is counted with neither)
    return true;
  }

  // G (:873-885) generalised: the next subproblem of this GPU's shard; once that is exhausted a child of a subproblem
  // that was split at the tail, then a subproblem of a peer's shard (work stealing through the peer-mapped dispensers; a
  // CAS, so that a dispenser of another run is never advanced). With nothing to take the block WAITS (that is what makes
  // the busy blocks split), until work appears or every block of the grid is waiting or gone. Thread 0.
  __device__ __forceinline__ void next_subproblem() {
    const unsigned long long world = (unsigned long long)P.world;
    c.have_task = 0; c.task_entry = -1; c.task_src = -1; c.task_depth = P.subproblems_power;
    const unsigned long long k = atomicAdd(P.cells + TB_CELL_NEXT, 1ull) & TB_K_MASK;
    if (k * world + (unsigned long long)P.rank < P.num_subproblems) { c.task_idx = k * world + (unsigned long long)P.rank; c.have_task = 1; return; }
    if (take_split()) return;
    if (P.steal) {
      for (int t = 0; t < P.npeers; ++t) {
        const int g = (slot + t) % P.npeers;
        unsigned long long* cell = P.peer_cells[g] + TB_CELL_NEXT;
        unsigned long long v = *(volatile unsigned long long*)cell;
        while ((v >> TB_K_BITS) == (unsigned long long)P.epoch &&
               (v & TB_K_MASK) * world + (unsigned long long)P.peer_rank[g] < P.num_subproblems) {
          const unsigned long long old = atomicCAS_system(cell, v, v + 1ull);
          if (old == v) {
            c.task_idx = (v & TB_K_MASK) * world + (unsigned long long)P.peer_rank[g]; c.have_task = 1;
            st->eps_stolen += 1;
            return;
          }
          v = old;
        }
      }
    }
    if (!P.split_bits) return;
    // Waiting is only safe while every CTA of the grid is running: a CTA that has not started yet (the device is shared
    // with another kernel) needs the slot of one that leaves.
    // (A grid launched on a free device is complete within microseconds: give it 50 of them.)
    for (int t = 0; t < 50 && *(volatile unsigned*)(P.split_ctl + TB_SPLIT_STARTED) < (unsigned)nslots; ++t) __nanosleep(1000);
    if (*(volatile unsigned*)(P.split_ctl + TB_SPLIT_STARTED) < (unsigned)nslots) return;
    atomicAdd(P.split_ctl + TB_SPLIT_WAITING, 1u);
    c.counted_idle = 1;
    // (this GPU's pool is polled every 2 us, the peers' - over NVLink - every 16 us)
    const unsigned long long t0 = globaltimer_ns();
    for (unsigned it = 0;; ++it) {
      if (stop_raised()) return;
      const bool far = (it & 7u) == 0u;
      if (take_split(far)) { atomicSub(P.split_ctl + TB_SPLIT_WAITING, 1u); c.counted_idle = 0; return; }
      // (grace: one second for a peer whose host has not launched this run yet - first-run allocations, process skew)
      if ((far || !P.share_split) && everybody_idle(globaltimer_ns() - t0 < 1000000000ull)) return;
      __nanosleep(2000);
    }
  }

  // ---- copies between the block store and a global image of it ---------------------------------
  // An image is P.vpad * 8 bytes; with a cluster it is C slices of vc * 8 bytes, one per CTA, and every
  // CTA moves its own slice with its own mbarrier.
  __device__ __forceinline__ void load_store(const int* gsrc) {
    sync();
    if (ACT && threadIdx.x == 0) c.dirty_all = 1;       // (read after the next barrier, at the start of a fixpoint)
    if (MEM == TB_MEM_GLOBAL) {
      const unsigned bytes = (unsigned)P.vpad * 8u;
      const int4* s4 = (const int4*)gsrc; int4* d4 = (int4*)(MEM == TB_MEM_GLOBAL ? (void*)P.block_store + (size_t)slot * 8 * P.vpad : (void*)sdyn);
      for (unsigned i = tid; i < bytes / 16; i += T) d4[i] = __ldcg(s4 + i);
      sync();
    } else {
      const unsigned bytes = (unsigned)(MEM == TB_MEM_STORE_CLUSTER ? P.vc : P.vpad) * 8u;
      const char* src = (const char*)gsrc + (size_t)cta_rank * bytes;
      if (threadIdx.x == 0) {
        bulk_wait_all();                 // the image may be one this thread wrote a moment ago
        fence_proxy_async();
        mbar_expect_tx(&lc->mbar, bytes);
        for (unsigned off = 0; off < bytes; off += BULK_CHUNK)
          bulk_g2s_issue((char*)sdyn + off, src + off, min(BULK_CHUNK, bytes - off), &lc->mbar);
      }
      while (!mbar_try_wait(&lc->mbar, mbar_phase)) {}
      mbar_phase ^= 1;
      if (MEM == TB_MEM_STORE_CLUSTER) sync();     // every slice has landed before anybody gathers from it
    }
  }
  // `synced`: a worker-wide barrier has passed since the last write to the store (the caller just came out of one).
  // `settle`: end with a barrier, after which anybody may write to the store again. Without it (single-CTA shared
  // placements only) the issuing thread 0 alone may, because it has waited for the copy engine to read the image.
  __device__ __forceinline__ void save_store(int* gdst, const bool synced = false, bool settle = true) {
    if (MEM == TB_MEM_GLOBAL || MEM == TB_MEM_STORE_CLUSTER) settle = true;
    if (!synced) sync();
    if (MEM == TB_MEM_GLOBAL) {
      const unsigned bytes = (unsigned)P.vpad * 8u;
      const int4* s4 = (const int4*)(MEM == TB_MEM_GLOBAL ? (const void*)P.block_store + (size_t)slot * 8 * P.vpad : (const void*)sdyn); int4* d4 = (int4*)gdst;
      for (unsigned i = tid; i < bytes / 16; i += T) d4[i] = __ldcg(s4 + i);
    } else if (threadIdx.x == 0) {
      const unsigned bytes = (unsigned)(MEM == TB_MEM_STORE_CLUSTER ? P.vc : P.vpad) * 8u;
      char* dst = (char*)gdst + (size_t)cta_rank * bytes;
      fence_proxy_async();
      for (unsigned off = 0; off < bytes; off += BULK_CHUNK)
        bulk_s2g_issue(dst + off, (const char*)sdyn + off, min(BULK_CHUNK, bytes - off));
      bulk_commit_wait_read();
    }
    if (settle) sync();
  }

  // ---- fixpoint (BlockAsynchronousFixpointGPU::fixpoint + warp_fixpoint, barebones :925-965) ---
  // What the sweeps touch, copied out of the context into registers for the duration of one fixpoint: the
  // context itself lives in local memory whenever a kernel calls the fixpoint from more than one place, and the
  // volatile accesses of the loop would otherwise re-read its fields from there at every evaluation.
  // (TMALL: the words in tensor memory carry absolute shared addresses, see StoreAbs)
  static constexpr bool kAbs = !ACT && TBC_U == 1 && ((TMALL && MEM == TB_MEM_STORE_SHARED) || MEM == TB_MEM_TCN_SHARED);
  struct HotSlots { StoreRef<MEM> store; const unsigned long long* words; unsigned narrowed; unsigned tm; int tm_visits; };
  struct HotAbs { StoreAbs store; const unsigned long long* words; unsigned narrowed; unsigned tm; int tm_visits; };
  struct Hot : std::conditional<kAbs, HotAbs, HotSlots>::type {};

  // One lane's TBC_U words of a chunk (adjacent in the table: one vector load).
  struct Words { unsigned long long w[TBC_U]; };

  // A warp requests the words of its next chunk before it knows whether the sweep goes on: the global table is followed
  // by padding chunks (tb_create), so the request needs no bound check; the shared copy (TCN_SHARED) is not, and clamps.
  __device__ __forceinline__ Words load_words(const unsigned long long* words, int i) const {
    Words r;
    if (MEM == TB_MEM_TCN_SHARED) i = min(i, (P.nchunks * 32 - 1) * TBC_U);
    if (TBC_U == 2) {
      const ulonglong2 t = MEM == TB_MEM_TCN_SHARED ? *(const ulonglong2*)(words + i) : __ldg((const ulonglong2*)(words + i));
      r.w[0] = t.x; r.w[TBC_U - 1] = t.y;
    } else {
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) r.w[u] = MEM == TB_MEM_TCN_SHARED ? words[i + u] : __ldg(words + i + u);
    }
    return r;
  }

  // Orders this thread's published bounds before its re-reads (see tbd::emptied).
  // (Promptness, not correctness: a re-read that misses the thread's own update finds "work" again and republishes the
  // same bounds; an empty interval is found by the next evaluation that loads it; the sweep barrier publishes everything.
  // With a cluster the fence is MEMBAR + ERRBAR + CCTL.IVALL, 12 % of the stall samples; dropping it gained 0.5 %.)
  __device__ __forceinline__ void publish_fence() const {
    if (MEM == TB_MEM_STORE_CLUSTER) asm volatile("fence.sc.cluster;" ::: "memory");
    else asm volatile("fence.sc.cta;" ::: "memory");
  }

  // ---- the dense fixpoint -----------------------------------------------------------------------------------------
  // A sweep: a warp walks the whole table ch = warp, warp + nwarps, ... (so the classes load-balance together and the
  // next chunk's words are always requested ahead, across class boundaries too); the table is sorted by class, so the
  // walk is a chain of per-class loops in each of which the operator is a compile-time constant. A chunk is 32 * TBC_U
  // propagators of one class, TBC_U per lane. With WAC1 (`warp_fixpoint`, :951-962) the warp iterates the chunk to a
  // warp-local fixpoint before moving on. Every branch is warp-uniform (votes), so the hot path carries no reconvergence bookkeeping.
  // Nine visits out of ten find nothing to do, and the loop is shaped for them:
  //   * the work path is one cold block: after publishing, ONE re-read of the operands is both the emptiness check
  //     (failure detection, tbd::emptied) and the snapshot of the next warp-local iteration; failure leaves the
  //     sweep from there, so the hot loop carries no `dead` / `late change` flags;
  //   * evaluations are counted as visits (derived from the walk) + re-evaluations (counted in the work path);
  //   * the `ask` (:972-982) is fused into the sweeps, evaluated on the last snapshot, which in the sweep where nothing
  //     changed is the final store; it stops at the first non-entailed propagator the warp sees in a sweep: the node then
  //     cannot be a solution, whatever the other chunks say (all-entailed sweeps still check every chunk);
  //   * every flag the warp reports is warp-uniform: no REDUX before the atomicOr;
  //   * the three flag words keep rotating across calls, so a fixpoint ends on its last sweep's barrier.
  struct Walk {
    int ch;                       // current chunk of this warp (uniform)
    int widx;                     // index of this lane's first word of the chunk the warp visits next
    Words cur;                    // this lane's words of the current chunk (requested at the end of the previous visit)
    unsigned extra;               // evaluations beyond one per visit (WAC1 re-evaluations)
    unsigned pad_evals;           // propagator evaluations spent on padding lanes
    int changed;                  // some visit published a bound
    int notent;                   // per lane: non-zero iff some propagator of this lane is not entailed
    unsigned ta;                  // tensor-memory address of the next request's words (two columns per visit)
  };

  // The words of the chunk the warp visits next: from tensor memory when they are there.
  __device__ __forceinline__ Words next_words(const Hot& h, Walk& w) const {
    Words r;
    if (TBC_U == 1 && MEM == TB_MEM_STORE_SHARED && (TMALL || w.ta < h.tm + 2u * (unsigned)h.tm_visits)) r.w[0] = tmem_ld64(w.ta);
    else r = load_words(h.words, w.widx);
    w.ta += 2u;
    return r;
  }

  // The part of one sweep that falls in class CLS. Returns true when the store failed (the sweep is over for this warp).
  template <int CLS>
  __device__ __forceinline__ bool sweep_class(Hot& h, Walk& w, const bool wac1, const int nwarps, const int stride) {
    const auto& store = h.store;
    const int ce = P.cls_begin[CLS + 1];
    unsigned last_extra = 0;      // re-evaluations of the latest visit that had work, and which chunk that was
    int last_work_ch = -1;
    do {
      int fa[TBC_U], fb[TBC_U], fc[TBC_U];
      tbd::Snap s[TBC_U];
      bool work = false;
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) decode_word<CLS>(w.cur.w[u], fa[u], fb[u], fc[u]);
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) tbd::load_snap<CLS>(store, fa[u], fb[u], fc[u], s[u]);
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) work |= tbd::has_work<CLS>(s[u]);
      if (__builtin_expect(__any_sync(0xffffffffu, work), 0)) {
        unsigned n = 0;
        for (;;) {
#pragma unroll
          for (int u = 0; u < TBC_U; ++u) {
            tbd::Snap nb;
            tbd::narrow<CLS>(s[u], nb);
            tbd::publish<CLS>(store, fa[u], fb[u], fc[u], s[u], nb, h.narrowed);
          }
          publish_fence();
          bool empty = false;
          work = false;
#pragma unroll
          for (int u = 0; u < TBC_U; ++u) {
            tbd::load_snap<CLS>(store, fa[u], fb[u], fc[u], s[u]);
            empty |= tbd::snapshot_empty<CLS>(s[u]);
          }
          ++n;
          if (__any_sync(0xffffffffu, empty)) { w.changed = 1; w.extra += wac1 ? n : 0u; return true; }
          if (!wac1) break;
#pragma unroll
          for (int u = 0; u < TBC_U; ++u) work |= tbd::has_work<CLS>(s[u]);
          if (!__any_sync(0xffffffffu, work)) break;
        }
        w.changed = 1;
        last_extra = wac1 ? n : 0u; last_work_ch = w.ch;
        w.extra += last_extra;
      }
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) w.notent |= tbd::not_entailed_bits<CLS>(s[u]);
      w.ch += nwarps;
      // (One word in flight, not two: ptxas schedules the copy of a second, prefetched word right behind its request, so
      // a two-deep register queue has no more distance than this - measured, as is the variant that pins the copy to the
      // end of the visit: profiles/r02_ab_dense_variants.md. From tensor memory the word is a dozen cycles away anyway.)
      w.cur = next_words(h, w);
      w.widx += stride;
    } while (w.ch < ce);
    // the class's last chunk is padded with copies of its last propagator: do not count those lanes
    if (w.ch - nwarps == ce - 1) w.pad_evals += (1u + (last_work_ch == ce - 1 ? last_extra : 0u)) * (unsigned)(32 * TBC_U - P.cls_last[CLS]);
    return false;
  }

  // Returns the OR of the flag bits of the last sweep; `iters` = number of block sweeps.
  __device__ __forceinline__ int fixpoint(int& iters) {
    // (broadcast from lane 0: tells the compiler the warp index is warp-uniform, so the walk's loop control
    // lives in uniform registers and its branches need no reconvergence bookkeeping)
    const int lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), nwarps = T >> 5;
    const int stride = nwarps * 32 * TBC_U;
    const bool wac1 = P.fixpoint_kind == TB_FP_WAC1 && P.nprops > P.wac1_threshold;
    Hot h;
    if constexpr (!kAbs) h.store = store;
    h.words = words; h.narrowed = narrowed;
    // (broadcast from lane 0: the address is warp-uniform, tcgen05.ld takes it from a uniform register)
    h.tm = __shfl_sync(0xffffffffu, tm_warp, 0); h.tm_visits = tm_visits;
    unsigned long long ded = 0;
    unsigned rot = fp_rot;
    int it = 0, f;
    for (;; ++it) {
      Walk w;
      w.ch = warp; w.extra = w.pad_evals = 0; w.changed = 0; w.notent = 0;
      w.widx = (warp * 32 + lane) * TBC_U;
      w.ta = h.tm;
      w.cur = next_words(h, w);
      w.widx += stride;
      bool failed = false;
#define TB_SWEEP(CLS) if (!failed && w.ch < P.cls_begin[CLS + 1]) failed = sweep_class<CLS>(h, w, wac1, nwarps, stride);
      TB_SWEEP(TBC_ADD_S) TB_SWEEP(TBC_ADD_XK) TB_SWEEP(TBC_ADD_ZK) TB_SWEEP(TBC_ADD_G)
      TB_SWEEP(TBC_MUL) TB_SWEEP(TBC_TDIV) TB_SWEEP(TBC_TMOD) TB_SWEEP(TBC_MIN) TB_SWEEP(TBC_MAX)
      TB_SWEEP(TBC_EQ_S) TB_SWEEP(TBC_EQ_T) TB_SWEEP(TBC_EQ_F) TB_SWEEP(TBC_EQ_ZK) TB_SWEEP(TBC_EQ_G)
      TB_SWEEP(TBC_LEQ_S) TB_SWEEP(TBC_LEQ_T) TB_SWEEP(TBC_LEQ_F) TB_SWEEP(TBC_LEQ_ZK) TB_SWEEP(TBC_LEQ_G)
#undef TB_SWEEP
      // one evaluation per completed visit, one more for the visit a failure interrupted, plus the re-evaluations
      const unsigned visits = (unsigned)(w.ch - warp) / (unsigned)nwarps + (failed ? 1u : 0u);
      ded += (unsigned long long)(visits + w.extra) * (unsigned long long)(32 * TBC_U) - (unsigned long long)w.pad_evals;
      const int bits = (w.changed ? F_CHANGED : 0) | (failed ? F_FAILED : 0) | (__any_sync(0xffffffffu, w.notent != 0) ? F_NOT_ENTAILED : 0);
      const unsigned slot = rot % 3u;
      if (lane == 0 && bits) atomicOr(&c.flags[slot], bits);
      if (tid == 0) c.flags[(rot + 1u) % 3u] = 0;
      sync();
      f = c.flags[slot];
      ++rot;
      if (!(f & F_CHANGED) || (f & F_FAILED)) break;
    }
    fp_rot = rot;
    iters = it + 1;
    narrowed = h.narrowed;
    deductions += ded;
    return f;
  }

  // ---- active-set fixpoint (TB_FP_*_ACTIVE; SURVEY 8f.2, the idea of FixpointSubsetGPU, barebones :636,984) ------
  // The same warp-local WAC1 iteration and the same flag bits as the dense fixpoint, but a warp only evaluates the chunks
  // one of whose variables moved since the chunk was last evaluated.  State in dynamic shared memory (P.act_off):
  //   vbits  : one bit per slot, set (red.or) by whoever moves a bound of the slot;
  //   dirty  : one byte per chunk, grouped per owning warp (chunk ch = flag ch / nwarps of warp ch % nwarps), set in
  //            the marking phase between two sweeps from vbits and the slot -> chunks watch lists (global, L2), cleared
  //            by the owning warp when it evaluates the chunk;
  //   notent : one byte per chunk, the fused `ask` of its last evaluation (valid while the chunk is clean).
  // Markers only write `dirty` between the two barriers of the marking phase and owners only during a sweep, so the
  // flags need no atomics.  A chunk that is clean has seen no change since it was found at its local fixpoint, so a
  // sweep that publishes nothing ends at the same greatest fixpoint as the dense sweeps.
  __device__ __forceinline__ unsigned* act_vbits() const { return (unsigned*)(sdyn + P.act_off); }

  // A bound of `slot` was moved outside the fixpoint (decision, incumbent): its watchers are due.
  __device__ __forceinline__ void mark_var(int slot) const {
    if (ACT) atomicOr(act_vbits() + (slot >> 5), 1u << (slot & 31));
  }

  // The chunks that load `slot` are due: set their flags in `dirty` (chunk ch is flag ch >> lw of warp ch & (nwarps - 1)).
  // One 64-bit word names a slot's first three watchers, the few slots with more continue through the CSR list.
  __device__ __forceinline__ void mark_watchers(int slot, unsigned char* dirty, int nwarps, int lw, int FPW) const {
    const unsigned long long wd = __ldg(P.watch_inline + slot);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const unsigned id = (unsigned)(wd >> (16 * k)) & 0xFFFFu;
      if (id != 0xFFFFu) dirty[(id & (unsigned)(nwarps - 1)) * FPW + (id >> lw)] = 1;
    }
    if ((unsigned)(wd >> 48) == 0xFFFEu) {
      const int e = __ldg(P.watch_off + slot + 1);
      for (int k = __ldg(P.watch_off + slot) + 3; k < e; ++k) {
        const int ch = __ldg(P.watch_list + k);
        dirty[(ch & (nwarps - 1)) * FPW + (ch >> lw)] = 1;
      }
    }
  }

  template <int CLS>
  __device__ __forceinline__ void active_visit(Hot& h, const Words& cur, const bool wac1, const int ch, unsigned* vbits,
                                               unsigned char* ne_slot, unsigned& evals, unsigned& pad_evals, int& late_chg, int& failed) {
    const StoreRef<MEM>& store = h.store;
    int fa[TBC_U], fb[TBC_U], fc[TBC_U];
#pragma unroll
    for (int u = 0; u < TBC_U; ++u) decode_word<CLS>(cur.w[u], fa[u], fb[u], fc[u]);
    tbd::Snap s[TBC_U];
    const unsigned e0 = evals;
    bool dead = false;
    for (;;) {
      bool chg = false;
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) tbd::load_snap<CLS>(store, fa[u], fb[u], fc[u], s[u]);
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) chg |= tbd::has_work<CLS>(s[u]);
      ++evals;
      if (!__any_sync(0xffffffffu, chg)) break;
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) {
        tbd::Snap n;
        tbd::narrow<CLS>(s[u], n);
        tbd::publish<CLS>(store, fa[u], fb[u], fc[u], s[u], n, h.narrowed);
        if (tbd::cls_loads_x(CLS) && ((n.xl != s[u].xl) | (n.xu != s[u].xu))) atomicOr(vbits + (fa[u] >> 5), 1u << (fa[u] & 31));
        if ((n.yl != s[u].yl) | (n.yu != s[u].yu)) atomicOr(vbits + (fb[u] >> 5), 1u << (fb[u] & 31));
        if (tbd::cls_loads_z(CLS) && ((n.zl != s[u].zl) | (n.zu != s[u].zu))) atomicOr(vbits + (fc[u] >> 5), 1u << (fc[u] & 31));
      }
      bool fail = false;
#pragma unroll
      for (int u = 0; u < TBC_U; ++u) fail |= tbd::emptied<CLS>(store, fa[u], fb[u], fc[u]);
      dead = __any_sync(0xffffffffu, fail);
      if (dead | !wac1) { late_chg = 1; break; }
    }
    int ne = 0;
#pragma unroll
    for (int u = 0; u < TBC_U; ++u) ne |= tbd::not_entailed_bits<CLS>(s[u]);
    const bool any_ne = __any_sync(0xffffffffu, ne != 0);
    if ((tid & 31) == 0) *ne_slot = any_ne ? 1 : 0;
    if (dead) failed = 1;
    if (ch == P.cls_begin[CLS + 1] - 1) pad_evals += (evals - e0) * (unsigned)(32 * TBC_U - P.cls_last[CLS]);
  }

  __device__ __forceinline__ int fixpoint_active(int& iters) {
    const int lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), nwarps = T >> 5;
    const int lw = 31 - __clz(nwarps);
    const bool wac1 = P.fixpoint_kind == TB_FP_WAC1 && P.nprops > P.wac1_threshold;
    unsigned* vbits = act_vbits();
    const int nvw = P.vpad >> 5, FPW = P.act_fpw;
    unsigned char* dirty = (unsigned char*)(vbits + nvw);
    unsigned char* mydirty = dirty + warp * FPW;
    unsigned char* mynotent = dirty + nwarps * FPW + warp * FPW;
    Hot h;
    h.store = store; h.words = words; h.narrowed = narrowed;
    h.tm = __shfl_sync(0xffffffffu, tm_warp, 0); h.tm_visits = tm_visits;
    unsigned long long ded = 0;
    int it = 0, f;
    for (;; ++it) {
      // ---- marking phase: moved slots -> dirty chunks
      if (c.dirty_all) {
        for (int i = tid; i < nwarps * FPW; i += T) { const int w = i / FPW, k = i - w * FPW; dirty[i] = (k * nwarps + w) < P.nchunks ? 1 : 0; }
        for (int i = tid; i < nvw; i += T) vbits[i] = 0;
      } else {
        // every thread follows the watchers of the moved slots of its own words (moved slots are spread thinly over the
        // words, so the lanes of a warp work on different slots at the same time: one L2 round trip per round of bits)
        for (int i = tid; i < nvw; i += T) {
          unsigned m = vbits[i];
          if (m) {
            vbits[i] = 0;
            do {
              const int v = (i << 5) + __ffs((int)m) - 1;
              m &= m - 1;
              mark_watchers(v, dirty, nwarps, lw, FPW);
            } while (m);
          }
        }
      }
      sync();
      if (tid == 0) {
        c.dirty_all = 0;
        c.flags[(it + 1) % 3] = 0;
      }
      // ---- sweep: this warp's dirty chunks
      unsigned evals = 0, pad_evals = 0, visits = 0;
      int late_chg = 0, failed = 0;
      for (int g = 0; g < FPW && !failed; g += 32) {
        unsigned mask = __ballot_sync(0xffffffffu, mydirty[g + lane] != 0);
        if (mask) mydirty[g + lane] = 0;
        while (mask && !failed) {
          const int k = g + __ffs((int)mask) - 1;
          mask &= mask - 1;
          const int ch = k * nwarps + warp;
          Words cur;
          // (the k-th chunk of this warp: its words are in tensor memory when the table fits, a dozen cycles away
          // instead of an L2 round trip on the critical path of a sweep that visits one or two chunks)
          if (TBC_U == 1 && MEM == TB_MEM_STORE_SHARED && k < h.tm_visits) cur.w[0] = tmem_ld64(h.tm + 2u * (unsigned)k);
          else cur = load_words(h.words, (ch * 32 + lane) * TBC_U);
          switch (chunk_class(P, ch)) {                         // warp-uniform
#define TB_CASE(CLS) case CLS: active_visit<CLS>(h, cur, wac1, ch, vbits, mynotent + k, evals, pad_evals, late_chg, failed); break;
            TB_CASE(TBC_ADD_S) TB_CASE(TBC_ADD_XK) TB_CASE(TBC_ADD_ZK) TB_CASE(TBC_ADD_G)
            TB_CASE(TBC_MUL) TB_CASE(TBC_TDIV) TB_CASE(TBC_TMOD) TB_CASE(TBC_MIN) TB_CASE(TBC_MAX)
            TB_CASE(TBC_EQ_S) TB_CASE(TBC_EQ_T) TB_CASE(TBC_EQ_F) TB_CASE(TBC_EQ_ZK) TB_CASE(TBC_EQ_G)
            TB_CASE(TBC_LEQ_S) TB_CASE(TBC_LEQ_T) TB_CASE(TBC_LEQ_F) TB_CASE(TBC_LEQ_ZK) TB_CASE(TBC_LEQ_G)
#undef TB_CASE
            default: break;
          }
          ++visits;
        }
      }
      __syncwarp();
      int ne = 0;
      for (int g = 0; g < FPW; g += 32) ne |= mynotent[g + lane];
      ded += (unsigned long long)evals * (unsigned long long)(32 * TBC_U) - (unsigned long long)pad_evals;
      const bool changed = evals > visits || late_chg;
      int bits = (changed ? F_CHANGED : 0) | (failed ? F_FAILED : 0) | (ne ? F_NOT_ENTAILED : 0);
      bits = __reduce_or_sync(0xffffffffu, bits);
      const int slot = it % 3;
      if (lane == 0 && bits) atomicOr(&c.flags[slot], bits);
      sync();
      f = c.flags[slot];
      if (!(f & F_CHANGED) || (f & F_FAILED)) break;
    }
    iters = it + 1;
    narrowed = h.narrowed;
    deductions += ded;
    // leave slot 0 clean for the next call (nobody reads flags until the next fixpoint's barrier)
    sync();
    if (tid < 3) c.flags[tid] = 0;
    sync();
    return f;
  }

  // ---- intermediate solutions (-i / -a) --------------------------------------------------------------------------
  // An improving solution also goes into a ring of images the host reads WHILE the kernel runs (tb_poll_solution from
  // another host thread; the reference's consumer thread, gpu_dive_and_solve.hpp:100-132): the image first, then a
  // record in pinned host memory whose sequence number is written last. A slot is reused after stream_slots more
  // solutions; a consumer that lags that far simply misses intermediate solutions (it re-checks the record). A slot
  // has one writer at a time (several blocks may find their first solutions in the same microsecond): a lock per slot,
  // taken by walking the ring from the solution's own slot to the first free one.
  __device__ __forceinline__ void stream_solution(int objective) {
    if (tid == 0) {
      const unsigned long long q = atomicAdd(P.cells + TB_CELL_STREAM, 1ull);
      int s0 = (int)(q % (unsigned long long)P.stream_slots);
      while (atomicCAS(P.stream_lock + s0, 0, 1) != 0) s0 = s0 + 1 == P.stream_slots ? 0 : s0 + 1;
      c.stream_seq = q; c.stream_slot = s0;
      P.stream_rec[s0].seq = 0ull;                  // the slot is being rewritten
      __threadfence_system();
    }
    sync();
    const unsigned long long seq = c.stream_seq;
    const int sl = c.stream_slot;
    save_store(P.stream_img + (size_t)sl * 2 * P.vpad);
    if (threadIdx.x == 0) bulk_wait_all();
    __threadfence_system();
    sync();
    if (tid == 0) {
      StreamRec* r = P.stream_rec + sl;
      r->objective = objective; r->block = slot; r->t_ns = (long long)(globaltimer_ns() - P.t_start);
      __threadfence_system();
      *(volatile unsigned long long*)&r->seq = seq + 1ull;
      __threadfence_system();
      atomicExch(P.stream_lock + sl, 0);
    }
  }

  // ---- tb_solve_groups: the best store of group `grp` -----------------------------------------------------------
  // Optimisation: the block takes the group's lock and writes the image only if its key still beats the image's; the
  // copy has landed before the lock is released, so two writers never interleave. Satisfaction: only the block that won
  // the group's stop word gets here, and writes without the lock.
  __device__ __forceinline__ void batch_save_best(int grp, int bound, bool optimise) {
    BatchCtl& b = batch_ctl();
    if (tid == 0) {
      BatchGroup& g = P.batch_groups[grp];
      if (optimise) {
        while (atomicCAS(&g.lock, 0, 1) != 0) __nanosleep(64);
        __threadfence();
        b.won = bound < *(volatile int*)&g.img_bound;
      } else b.won = 1;
    }
    sync();
    const bool won = b.won != 0;
    if (won) {
      save_store(P.batch_best + (size_t)grp * 2 * P.vpad, true);
      if (threadIdx.x == 0) bulk_wait_all();
      __threadfence();
      sync();
    }
    if (tid == 0) {
      BatchGroup& g = P.batch_groups[grp];
      if (won) { *(volatile int*)&g.img_bound = bound; *(volatile int*)&g.has = 1; }
      __threadfence();
      if (optimise) atomicExch(&g.lock, 0);
    }
  }

  // ---- tb_solve_objectives: a solution is a witness for every group ----------------------------------------------
  // The groups optimise over the same union of boxes, so a solution of one is a solution of every group whose objective
  // variable is not empty in it (see below). The threads split the
  // other groups (the task's own group went through propagate()): each computes the group's key from the store,
  // publishes it where it beats the group's incumbent, and asks for the image where it beats the group's best image.
  // The block then writes the image into those rows one group at a time, as batch_save_best does, so it holds one lock
  // at a time. An unbounded key ends its group, as it ends the group that finds it.
  // tb_solve_front: group i asks for the best y with x <= level[i] (x >= level[i] when maximising x), and level[i] is
  // its fix_hi (fix_lo). A store with x in [l, u] is a witness for group i iff l <= level[i] (u >= level[i]): the levels
  // ascend, so those groups are a suffix (a prefix) of the groups, found by a binary search. This is the dominance cut:
  // a solution of a low slice is the incumbent of every level above it.
  __device__ __forceinline__ void batch_share_witness() {
    BatchCtl& b = batch_ctl();
    const int own = b.group;
    int first = 0, n = P.batch_share;
    if (P.batch_front) {
      int l, u; store.ld(P.batch_front_x, l, u);
      const bool min_x = P.batch_front == 1;
      int lo = 0, hi = n;                       // the first group whose level the store does not reach from below
      while (lo < hi) {                         // (min x) / reaches (max x)
        const int m = (lo + hi) >> 1;
        const BatchGroup& g = P.batch_groups[m];
        if (min_x ? g.fix_hi < l : g.fix_lo <= u) lo = m + 1; else hi = m;
      }
      if (min_x) first = lo; else n = lo;
    }
    for (int base = first; base < n; base += T) {
      const int grp = base + tid;
      int key = TBD_PINF;
      bool want = false;
      if (grp < n && grp != own) {
        BatchGroup& g = P.batch_groups[grp];
        int l, u; store.ld(g.obj, l, u);
        // (an objective variable the propagators do not see can be empty in a box whose other variables have
        // solutions: that group fails every node of the box, as its own search does, and the store is no witness for it)
        if (l <= u) {
          key = objective_key(l, u, g.maximize);
          const unsigned long long w = bound_word(key);
          if (w < *(volatile unsigned long long*)&g.bound) atomicMin(&g.bound, w);
          if (key == TBD_NINF) *(volatile int*)&g.stop = 1;
          want = key < *(volatile int*)&g.img_bound;
        }
      }
      for (;;) {                                // one row per round: the lowest thread that still wants one
        if (tid == 0) b.pick = T;
        if (!__syncthreads_or(want)) break;
        if (want) atomicMin(&b.pick, tid);
        __syncthreads();
        const int t = b.pick;
        if (tid == t) { b.key = key; want = false; }
        __syncthreads();
        batch_save_best(base + t, b.key, true);
      }
    }
  }

  // ---- tb_solve_supports: a solution is a witness for every query value it holds ----------------------------------
  // Every group asks whether some solution of the union has one slot at one value, so a solution store supports every
  // query (slot, v) with v in the store's [l, u] of that slot (an entailed box: any value of it extends to a point). The
  // threads split the queried slots; for each, a binary search finds the first value >= l and the walk goes up to u. A
  // group that is still open is won with a CAS on its stop word: it is supported, and its blocks leave at their next
  // node. A block that won something takes one row of the pool, writes its store there once and names that row as the
  // witness of every group it won: the winner marks each won group with -2 - slot in the first walk and replaces the
  // mark by the row (or -1, the pool being full) in the second. Nobody else writes a won group's `wit`, and the store
  // does not change between the walks, so both walks meet the same groups. The task's own group is one of the queries.
  // Returns (uniformly) whether the block won a group.
  __device__ __forceinline__ bool batch_support_witness() {
    BatchCtl& b = batch_ctl();
    const int mark = -2 - slot;
    if (!__syncthreads_or(support_walk(mark, 0, true))) return false;
    if (tid == 0) {
      const unsigned r = atomicAdd(P.batch_wit_n, 1u);
      b.pick = r < (unsigned)P.batch_wit_cap ? (int)r : -1;
    }
    sync();
    const int row = b.pick;
    if (row >= 0) {
      save_store(P.batch_wit + (size_t)row * 2 * P.vpad, true);
      if (threadIdx.x == 0) bulk_wait_all();
      __threadfence();
      sync();
    }
    support_walk(mark, row, false);
    __threadfence();
    return true;
  }
  // One walk of batch_support_witness over this thread's query slots: claim the open groups (returns whether it won
  // one), or give the groups marked `mark` their witness `row`.
  __device__ __forceinline__ bool support_walk(int mark, int row, bool claim) {
    bool mine = false;
    for (int q = tid; q < P.batch_nqslots; q += T) {
      int l, u; store.ld(__ldg(P.batch_qslot + q), l, u);
      int lo = __ldg(P.batch_qoff + q), hi = __ldg(P.batch_qoff + q + 1);
      const int end = hi;
      while (lo < hi) {                         // the first value >= l
        const int m = (lo + hi) >> 1;
        if (__ldg(P.batch_qval + m) < l) lo = m + 1; else hi = m;
      }
      for (int k = lo; k < end && __ldg(P.batch_qval + k) <= u; ++k) {
        BatchGroup& g = P.batch_groups[k];
        if (claim) {
          if (*(volatile int*)&g.stop == 0 && atomicCAS(&g.stop, 0, 1) == 0) { *(volatile int*)&g.wit = mark; mine = true; }
        } else if (*(volatile int*)&g.wit == mark) {
          *(volatile int*)&g.wit = row; *(volatile int*)&g.has = 1;
        }
      }
    }
    return mine;
  }

  // ---- propagate() (barebones :903-1031) -----------------------------------------------------------
  // Runs the fixpoint, classifies the node, records solutions, updates counters and the stop flag.
  // Sets c.leaf / c.failed / c.stop uniformly (valid after return).
  __device__ __forceinline__ void propagate() {
    unsigned long long t0 = 0;
    if (tid == 0) t0 = globaltimer_ns();
    int iters = 0, f;
    bool pre_failed = P.root_failed != 0;       // a referenced variable is already empty in the root store
    if (obj_slot() >= 0) { int l, u; store.ld(obj_slot(), l, u); pre_failed |= l > u; }
    if (pre_failed) f = F_FAILED;
    else if constexpr (ACT) f = fixpoint_active(iters);
    else f = fixpoint(iters);
    const bool failed = (f & F_FAILED) != 0;
    const bool solution = !failed && !(f & F_NOT_ENTAILED);
    unsigned long long t1 = 0;
    if (tid == 0) t1 = globaltimer_ns();
    bool improved = false;
    if (solution) {
      if (obj_slot() >= 0) {
        int l, u; store.ld(obj_slot(), l, u);
        if constexpr (BATCH) l = objective_key(l, u, maximizes());   // (the group's key)
        improved = c.best_bound > l;           // uniform: same smem word read by everybody
        sync();
        if (improved && tid == 0) {
          c.best_bound = l;
          publish_bound(l);
          st->t_best = (long long)(globaltimer_ns() - P.t_start);
          st->best_bound = l;
        }
      } else {
        if constexpr (BATCH) {                  // satisfaction: the first solution of the GROUP wins
          if (P.batch_nqslots) {                // (supports: of every group it holds; no best row is written)
            if (batch_support_witness() && tid == 0) { st->solutions++; st->has_best = 1; }
          } else {
            if (tid == 0) batch_ctl().won = atomicCAS(&batch_group().stop, 0, 1) == 0;
            sync();
            improved = batch_ctl().won != 0;
          }
        } else {
          improved = st->solutions == 0;          // satisfaction: first solution wins
          sync();
        }
        if (tid == 0) st->t_best = (long long)(globaltimer_ns() - P.t_start);
      }
      if (improved) {
        if constexpr (BATCH) batch_save_best(batch_ctl().group, obj_slot() >= 0 ? c.best_bound : 0, obj_slot() >= 0);
        else save_store(g_best);
        if (tid == 0) { st->solutions++; st->has_best = 1; }
        if constexpr (!BATCH) { if (P.stream_slots) stream_solution(P.obj_var >= 0 ? c.best_bound : 0); }
      }
      if constexpr (BATCH) { if (P.batch_share) batch_share_witness(); }
    }
    if (tid == 0) {
      c.leaf = failed || solution;
      c.failed = failed;
      st->fixpoint_iterations += (unsigned long long)iters;
      st->nodes++;
      st->fails += failed ? 1 : 0;
      if (c.depth > st->depth_max) st->depth_max = c.depth;
      st->t_fixpoint += (long long)(t1 - t0);
      if (solution && obj_slot() < 0) {      // satisfaction: stop everybody after the first solution
        st->exhaustive = 0;
        // (batch: the group's stop word is raised, the blocks of its roots move on; the root that found the group's
        // first solution is never exhaustive, whatever weight the task that found it closes, so neither is the group)
        if constexpr (BATCH) batch_cut();
        else {
          c.stop = 1;
          raise_stop(true);
        }
      }
      if ((P.cutnodes && st->nodes >= P.cutnodes) || stop_raised()) {
        st->exhaustive = 0;
        c.stop = 1;
        if constexpr (BATCH) batch_cut();
      }
    }
    sync();
  }

  // ---- branching (BlockData::split / push_decision, barebones :187-405) ----------------------------
  __device__ __forceinline__ unsigned long long sel_key(int order, int l, int u, int i) const {
    unsigned hi;
    switch (order) {
      case TB_VAR_INPUT_ORDER:     hi = 0u; break;
      case TB_VAR_FIRST_FAIL:      hi = (unsigned)u - (unsigned)l; break;
      case TB_VAR_ANTI_FIRST_FAIL: hi = ~((unsigned)u - (unsigned)l); break;
      case TB_VAR_SMALLEST:        hi = (unsigned)l ^ 0x80000000u; break;
      default:                     hi = ~((unsigned)u ^ 0x80000000u); break;   // LARGEST
    }
    return ((unsigned long long)hi << 32) | (unsigned)i;
  }

  // thread 0 only
  __device__ __forceinline__ void push_decision(int val_order, int var) {
    if (c.depth >= P.max_depth) {
      st->error = TB_ERR_DEPTH; st->exhaustive = 0; c.stop = 1; raise_stop(false); c.pushed = 0;
      if constexpr (BATCH) batch_cut();
      return;
    }
    int l, u; store.ld(var, l, u);
    Decision d;
    d.var = var; d.cur = -1;
    int mid = (int)((long long)l + ((long long)u - (long long)l) / 2);
    switch (val_order) {
      case TB_VAL_MIN:   d.clb0 = l; d.cub0 = l; d.clb1 = l + 1; d.cub1 = u; break;
      case TB_VAL_MAX:   d.clb0 = u; d.cub0 = u; d.clb1 = l; d.cub1 = u - 1; break;
      case TB_VAL_SPLIT: d.clb0 = l; d.cub0 = mid; d.clb1 = mid + 1; d.cub1 = u; break;
      default:           d.clb0 = mid + 1; d.cub0 = u; d.clb1 = l; d.cub1 = mid; break;
    }
    d.rope0 = c.depth + 1;
    if (c.depth > 0) { const Decision& p = dec[c.depth - 1]; d.rope1 = p.cur == 0 ? p.rope0 : p.rope1; }
    else d.rope1 = -1;
    dec[c.depth] = d;
    c.depth++;
    c.pushed = 1;
  }

  // Returns (uniformly) whether a decision was pushed at dec[depth-1].
  __device__ __forceinline__ bool split() {
    const int lane = tid & 31;
    for (;;) {
      const int s = c.cur_strategy;       // uniform (barrier before every read)
      if (s >= P.nstrategies) return false;
      const DevStrategy strat = P.strategies[s];
      const bool in_store = strat.n == 0;
      const int n = in_store ? P.nvars : strat.n;
      unsigned long long key = ~0ull;
      int first = INT32_MAX;
      for (int i = c.next_unassigned + tid; i < n; i += T) {
        int v = in_store ? i : __ldg(strat.vars + i);
        int l, u; store.ld(v, l, u);
        if (l != u && l != TBD_NINF && u != TBD_PINF) {
          if (first == INT32_MAX) first = i;
          unsigned long long k = sel_key(strat.var_order, l, u, i);
          if (k < key) key = k;
          if (strat.var_order == TB_VAR_INPUT_ORDER) break;
        }
      }
      first = __reduce_min_sync(0xffffffffu, first);
      for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
        if (other < key) key = other;
      }
      // two selection cells used in turn: thread 0 re-arms the other one while everybody reads this one
      const int par = sel_par;
      sel_par ^= 1;
      if (lane == 0 && key != ~0ull) { atomicMin(&c.sel_key[par], key); atomicMin(&c.sel_first[par], first); }
      sync();
      const unsigned long long best = c.sel_key[par];
      if (tid == 0) {
        if (best != ~0ull) {
          c.next_unassigned = c.sel_first[par];
          int i = (int)(unsigned)(best & 0xffffffffu);
          push_decision(strat.val_order, in_store ? i : strat.vars[i]);
        } else {
          c.cur_strategy = s + 1;
          c.next_unassigned = 0;
        }
        c.sel_key[par ^ 1] = ~0ull; c.sel_first[par ^ 1] = INT32_MAX;
      }
      sync();
      if (best != ~0ull) return c.pushed != 0;
    }
  }

  // ---- EPS dive (barebones :663-741) ------------------------------------------------------------------
  // One step of the dive below a node that propagate() left open: branch, and take the child that bit
  // remaining_depth - 1 of `idx` names (decisions are not recorded while diving). A node with nothing left to
  // branch on is a leaf.
  __device__ __forceinline__ void dive_step(unsigned long long idx) {
    if (c.leaf) return;
    bool pushed = split();
    if (tid == 0) {
      if (!pushed) { c.leaf = 1; st->exhaustive = 0; if constexpr (BATCH) batch_cut(); }
      else {
        --c.remaining_depth;
        --c.depth;
        const Decision& d = dec[0];
        int bit = (int)((idx >> c.remaining_depth) & 1ull);
        store.embed(d.var, bit ? d.clb1 : d.clb0, bit ? d.cub1 : d.cub0);
        mark_var(d.var);
      }
    }
  }

  // Dives from the problem root following the bits of `idx`. Returns remaining depth (uniform).
  __device__ __forceinline__ int dive(unsigned long long idx, int depth_power) {
    if (tid == 0) {
      c.cur_strategy = 0; c.next_unassigned = 0; c.depth = 0;
      c.remaining_depth = depth_power; c.leaf = 0; c.failed = 0;
      c.t_mark = (long long)globaltimer_ns();
    }
    load_store(P.root_store);
    sync();
    while (c.remaining_depth > 0 && !c.leaf && !c.stop) {
      sync();
      propagate();
      dive_step(idx);
      sync();
    }
    if (tid == 0) st->t_dive += (long long)globaltimer_ns() - c.t_mark;
    sync();
    return c.remaining_depth;
  }

  // ---- the whole search of one worker (barebones :656-886) -----------------------------------------------
  // Main loop B-G of gpu_barebones_solve: take a subproblem, dive to it (steps C-D, :663-714), skip its
  // subtree if the dive hit a leaf (E, :718-741), otherwise solve it by depth-first branch and bound with
  // restore-from-root + decision replay (F, :742-871), then ask the dispenser for the next one (G, :873-885).
  // Written as one flat state machine around a SINGLE propagate() call: with one call site the whole node
  // step is inlined, the context stays in registers and the kernel parameters stay in the constant bank
  // (two call sites cost ~25 % of the node rate: the fixpoint went out of line and re-read both from memory).
  __device__ __forceinline__ void search() {
    enum { M_START, M_DIVE, M_SOLVE, M_SOLVE_END, M_NEXT };
    const unsigned long long nsub = P.num_subproblems;
    const unsigned long long world = (unsigned long long)P.world, rank = (unsigned long long)P.rank;
    unsigned long long idx = 0;
    int mode = M_START;
    for (;;) {
      if (mode == M_START) {
        if (!c.have_task || c.stop) break;
        idx = c.task_idx;
        sync();
        if (tid == 0) {
          c.cur_strategy = 0; c.next_unassigned = 0; c.depth = 0;
          c.remaining_depth = c.task_depth; c.leaf = 0; c.failed = 0;
          c.task_nodes = 0; c.abandon = 0;
          c.t_mark = (long long)globaltimer_ns();
          if constexpr (BATCH) {
            c.best_bound = TBD_PINF;          // the incumbent of ANOTHER group must never prune this one
            const BatchRoot& r = batch_root();
            const BatchGroup& g = P.batch_groups[r.group];
            BatchCtl& b = batch_ctl();
            b.group = r.group; b.image = r.image; b.obj = g.obj; b.maximize = g.maximize;
            b.fix = g.fix; b.fix_lo = g.fix_lo; b.fix_hi = g.fix_hi;
            c.abandon = r.skip || batch_group_over();   // (nothing left to do for a root that is over)
          }
        }
        if constexpr (BATCH) sync();
        if (BATCH && c.abandon) mode = M_NEXT;
        else {
          for (int i = tid; i < P.nsnap; i += T) g_snap_tag[i] = -1;       // snapshots belong to one subproblem
          if constexpr (BATCH) {
            load_store(P.batch_roots + (size_t)batch_ctl().image * 2 * P.vpad);
            // The group's fixing (tb_solve_supports, tb_solve_front), marked for the active set before the first
            // propagation. This is the only place a batch root store is built: the dive starts here, g_root and the
            // snapshots are saved from stores below it, and a tail-split child is a task that starts here again, so
            // all of them hold it.
            if (tid == 0 && batch_ctl().fix >= 0) {
              store.embed(batch_ctl().fix, batch_ctl().fix_lo, batch_ctl().fix_hi);
              mark_var(batch_ctl().fix);
            }
          } else load_store(P.root_store);
          sync();
          mode = M_DIVE;
        }
      }
      if (mode == M_DIVE && !(c.remaining_depth > 0 && !c.leaf && !c.stop)) {
        // the dive is over: at the subproblem (remaining depth 0), or at a leaf above it
        if (tid == 0) st->t_dive += (long long)globaltimer_ns() - c.t_mark;
        sync();
        const int remaining = c.remaining_depth;
        if (c.leaf && !c.stop) {
          // E. a leaf above the subproblem depth: skip the whole subtree (:718-741)
          if (tid == 0 && c.task_entry >= 0) {
            // a child of a split subproblem: its siblings below the same leaf need no dive either
            SplitEntry* e = split_pool_of(c.task_src < 0 ? P.cells : P.peer_cells[c.task_src]) + c.task_entry;
            if (remaining < 31) {
              // (the entry's epoch is in the high half of the word: a max can only move this run's counter)
              const unsigned long long to = ((unsigned long long)P.epoch << 32) | min(e->count, ((c.task_j >> remaining) + 1u) << remaining);
              unsigned long long v = *(volatile unsigned long long*)&e->next;
              while ((unsigned)(v >> 32) == P.epoch && v < to) {
                const unsigned long long old = atomicCAS_system(&e->next, v, to);
                if (old == v) break;
                v = old;
              }
            }
          } else if (tid == 0) {
            // nobody needs to dive into [idx, next) any more: advance every shard's dispenser past it
            const unsigned long long next = ((idx >> remaining) + 1ull) << remaining;
            dispenser_skip_to(-1, next <= rank ? 0ull : (next - rank + world - 1ull) / world);
            for (int g = 0; g < P.npeers && P.steal; ++g) {
              const unsigned long long q = (unsigned long long)P.peer_rank[g];
              dispenser_skip_to(g, next <= q ? 0ull : (next - q + world - 1ull) / world);
            }
            if ((idx & ((1ull << remaining) - 1ull)) == 0ull) st->eps_skipped += next - idx;
          }
          // the leaf closes the 2^remaining tasks of depth D below it: counted once, by the task aligned on them
          if constexpr (BATCH) {
            if (tid == 0 && (idx & ((1ull << remaining) - 1ull)) == 0ull)
              atomicAdd(&batch_root().closed, 1ull << (TB_BATCH_WEIGHT_BITS - c.task_depth + remaining));
          }
          mode = M_NEXT;
        } else if (!c.stop) {
          if (tid == 0 && P.has_eps_strategy) { c.cur_strategy = max(1, c.cur_strategy); c.next_unassigned = 0; }
          sync();
          mode = M_SOLVE;
        } else mode = M_NEXT;
      }
      if (mode == M_SOLVE) {
        if (c.stop) mode = M_SOLVE_END;
        else {
          // I. inject the incumbent bound (thread 0), detect an unconstrained objective
          // (batch, a group that maximises: the incumbent is the key ~ub, so lb narrows to ~key + 1)
          if (tid == 0 && obj_slot() >= 0) {
            int appx = read_bound();
            if (appx != TBD_PINF) {
              bool moved;
              if (maximizes()) {
                moved = store.embed(obj_slot(), tbd::succ(~appx), TBD_PINF);
                moved |= store.embed(obj_slot(), tbd::succ(~c.best_bound), TBD_PINF);
              } else {
                moved = store.embed(obj_slot(), TBD_NINF, tbd::pred(appx));
                moved |= store.embed(obj_slot(), TBD_NINF, tbd::pred(c.best_bound));
              }
              if (moved) mark_var(obj_slot());
            }
            if (appx == TBD_NINF) {
              if constexpr (BATCH) { *(volatile int*)&batch_group().stop = 1; batch_cut(); }   // this group only
              else { c.stop = 1; raise_stop(true); }
            }
          }
          // batch: a group that is over (see propagate) is left at the next node, by every block working on it
          bool over = false;
          if constexpr (BATCH) { if (tid == 0) over = batch_group_over(); }
          // tail splitting: somebody is waiting for work and this subproblem has been going on for a while
          if (tid == 0 && !over && P.split_bits && ++c.task_nodes >= (unsigned)P.split_min_nodes && (c.task_nodes & 255u) == 0u &&
              somebody_waits() && c.task_depth + P.split_bits <= (BATCH ? P.batch_max_depth : 56) &&
              *(volatile unsigned*)(P.split_ctl + TB_SPLIT_N) < (unsigned)TB_SPLIT_CAP)
            c.abandon = push_split() ? 1 : 0;
          if constexpr (BATCH) { if (over) c.abandon = 1; }
          sync();
          if (c.stop) mode = M_SOLVE_END;
          else if (c.abandon) mode = M_NEXT;          // its children are in the pool now; this block takes one of them
        }
      }
      if (mode == M_SOLVE_END) {
        sync();
        if (tid == 0 && !(P.cutnodes && st->nodes >= P.cutnodes) && !stop_raised()) { if (c.task_entry < 0) st->eps_solved += 1; else st->eps_parts += 1; }
        // (a block that was cut marked the root in propagate / push_decision)
        if constexpr (BATCH) {
          if (tid == 0 && !c.stop) atomicAdd(&batch_root().closed, 1ull << (TB_BATCH_WEIGHT_BITS - c.task_depth));
        }
        mode = M_NEXT;
      }
      if (mode == M_NEXT) {
        sync();
        if (tid == 0 && !c.stop) next_subproblem();
        sync();
        mode = M_START;
        continue;
      }

      // II. one node
      if (mode == M_DIVE) sync();
      propagate();

      if (mode == M_DIVE) {
        dive_step(idx);
        sync();
      } else {
        // III. branch
        if (!c.leaf) {
          if (c.depth == 0) {
            save_store(g_root);
            if (tid == 0) { c.snap_strategy = c.cur_strategy; c.snap_next_unassigned = c.next_unassigned; }
            sync();
          }
          bool pushed = split();
          if (pushed && P.nsnap) {
            // copying instead of recomputation: keep this node's fixpoint, so that the right branch of the decision
            // restarts from here (one changed variable) instead of from the subproblem root plus a replay
            const int j = c.depth - 1;
            // (split() ended on a barrier; the decision below is applied by the thread that waited for the copy engine)
            save_store(g_snap + (size_t)(j % P.nsnap) * 2 * P.vpad, true, false);
            if (tid == 0) g_snap_tag[j % P.nsnap] = j;
            if (ACT) {
              // the fixpoint has just converged: no moved bit, no dirty chunk; keep the entailment cache with the image
              const int fw = (T >> 5) * P.act_fpw / 4;
              const unsigned* ne = act_vbits() + (P.vpad >> 5) + fw;
              unsigned* g = g_snap_flags + (size_t)(j % P.nsnap) * fw;
              for (int i = tid; i < fw; i += T) g[i] = ne[i];
            }
          }
          if (tid == 0) {
            if (!pushed) { c.leaf = 1; st->exhaustive = 0; if constexpr (BATCH) batch_cut(); }
            else {
              Decision& d = dec[c.depth - 1];
              d.cur = 0;
              store.embed(d.var, d.clb0, d.cub0);
              mark_var(d.var);
            }
          }
          sync();
        }
        // IV. backtrack: follow the rope, restore from the subproblem root, replay the decisions
        if (c.leaf) {
          if (c.depth == 0) { mode = M_SOLVE_END; continue; }
          sync();
          if (tid == 0) { const Decision& d = dec[c.depth - 1]; c.depth = d.cur == 0 ? d.rope0 : d.rope1; }
          sync();
          const int depth = c.depth;
          if (depth == -1) { mode = M_SOLVE_END; continue; }
          // the node where decision depth-1 was taken is in the snapshot ring unless a deeper level has reused its slot
          const bool snap = P.nsnap && *(volatile int*)(g_snap_tag + (depth - 1) % P.nsnap) == depth - 1;      // uniform (global, written before a barrier)
          if (snap) {
            load_store(g_snap + (size_t)((depth - 1) % P.nsnap) * 2 * P.vpad);
            if (ACT) {
              // back at a converged node: every chunk is clean, its entailment cache is the one saved with the image,
              // and only the watchers of the decision variable (marked below) are due
              const int fw = (T >> 5) * P.act_fpw / 4, nvw = P.vpad >> 5;
              unsigned* vb = act_vbits();
              const unsigned* g = g_snap_flags + (size_t)((depth - 1) % P.nsnap) * fw;
              for (int i = tid; i < nvw + fw; i += T) vb[i] = 0u;
              for (int i = tid; i < fw; i += T) vb[nvw + fw + i] = __ldcg(g + i);
              if (tid == 0) c.dirty_all = 0;
              sync();
            }
          } else {
            load_store(g_root);
            for (int i = tid; i < depth - 1; i += T) {
              const Decision d = dec[i];
              store.embed(d.var, d.cur == 0 ? d.clb0 : d.clb1, d.cur == 0 ? d.cub0 : d.cub1);
            }
          }
          if (tid == 0) {
            Decision& d = dec[depth - 1];
            d.cur += 1;
            store.embed(d.var, d.cur == 0 ? d.clb0 : d.clb1, d.cur == 0 ? d.cub0 : d.cub1);
            mark_var(d.var);
            c.cur_strategy = c.snap_strategy; c.next_unassigned = c.snap_next_unassigned;
          }
          sync();
        }
      }
    }
  }
};

// ---- context construction shared by the three kernels -----------------------------------------------
__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_nctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }

// The control block every CTA of the worker reads: its own, or CTA 0's through DSMEM.
template <int MEM>
__device__ __forceinline__ Ctl* shared_ctl(Ctl* local) {
  if (MEM != TB_MEM_STORE_CLUSTER) return local;
  unsigned long long g = (unsigned long long)local, r;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(r) : "l"(g), "r"(0u));
  return (Ctl*)r;
}

template <int MEM, bool ACT, bool TMALL, bool BATCH>
__device__ __forceinline__ void ctx_init(Ctx<MEM, ACT, TMALL, BATCH>& k, Ctl* local, unsigned char* dyn) {
  const DevParams& P = k.P;
  k.lc = local;
  if (MEM == TB_MEM_STORE_CLUSTER) {
    const unsigned csize = cluster_nctarank();
    k.cta_rank = (int)cluster_ctarank();
    k.tid = k.cta_rank * (int)blockDim.x + (int)threadIdx.x;
    k.T = (int)(blockDim.x * csize);
    k.slot = (int)(blockIdx.x / csize);
    k.nslots = (int)(gridDim.x / csize);
  } else {
    k.cta_rank = 0; k.tid = threadIdx.x; k.T = blockDim.x; k.slot = blockIdx.x; k.nslots = gridDim.x;
  }
  const int slot = k.slot;
  const size_t store_bytes = (size_t)P.vpad * 8;
  init_store_ref(k.store, P, dyn, slot);
  k.sdyn = dyn;
  k.words = P.words;
  k.mbar_phase = 0;
  k.fp_rot = 0;
  k.sel_par = 0;
  k.narrowed = 0;
  k.deductions = 0;
  k.g_root = P.block_root + (size_t)slot * 2 * P.vpad;
  k.g_best = P.block_best + (size_t)slot * 2 * P.vpad;
  k.g_snap = P.nsnap ? P.block_snap + (size_t)slot * P.nsnap * 2 * P.vpad : nullptr;
  k.g_snap_tag = P.nsnap ? P.snap_tag + (size_t)slot * P.nsnap : nullptr;
  k.g_snap_flags = (ACT && P.nsnap) ? P.snap_flags + (size_t)slot * P.nsnap * ((blockDim.x >> 5) * P.act_fpw / 4) : nullptr;
  k.dec = P.decisions + (size_t)slot * P.max_depth;
  k.st = P.stats + slot;
  if (threadIdx.x == 0) {
    mbar_init(&local->mbar, 1);
    local->flags[0] = local->flags[1] = local->flags[2] = 0;
    local->sel_key[0] = local->sel_key[1] = ~0ull; local->sel_first[0] = local->sel_first[1] = INT32_MAX;
    local->stop = 0; local->leaf = 0; local->failed = 0; local->depth = 0; local->pushed = 0;
    local->cur_strategy = 0; local->next_unassigned = 0; local->snap_strategy = 0; local->snap_next_unassigned = 0;
    local->best_bound = TBD_PINF; local->remaining_depth = 0;
    local->dirty_all = 1;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (ACT) {
    // vbits, dirty and notent flags start clear; the first fixpoint evaluates everything (dirty_all)
    const int words_ = (P.vpad >> 5) + ((2 * (int)(blockDim.x >> 5) * P.act_fpw + 3) >> 2);
    unsigned* a = (unsigned*)(dyn + P.act_off);
    for (int i = threadIdx.x; i < words_; i += blockDim.x) a[i] = 0u;
  }
  k.sync();
  k.tm_warp = 0; k.tm_visits = 0;
  if (MEM == TB_MEM_STORE_SHARED && TBC_U == 1 && !P.tmem_cols && threadIdx.x < 32) {
    // A CTA of a kernel that carries tensor-memory code holds the SM's allocation permit until it gives it up, and no
    // second CTA starts on the SM meanwhile (measured: TB_TMEM=0 ran one CTA per SM): give it up at once.
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (MEM == TB_MEM_STORE_SHARED && TBC_U == 1 && P.tmem_cols) {
    // the table goes to tensor memory: one warp allocates the CTA's columns, every warp stores the words of its own
    // first tmem_visits visits into its quarter of the lanes (chunk ch = warp + k * nwarps at columns 2k, 2k + 1)
    const int warp = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31), nwarps = (int)(blockDim.x >> 5);
    if (warp == 0) tmem_alloc(&local->tmem_base, (unsigned)P.tmem_cols);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    k.sync();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned cols_per_warp = (unsigned)P.tmem_cols / (unsigned)((nwarps + 3) / 4);
    k.tm_warp = local->tmem_base + ((unsigned)(32 * (warp & 3)) << 16) + (unsigned)(warp >> 2) * cols_per_warp;
    k.tm_visits = P.tmem_visits;
    for (int v = 0; v < P.tmem_visits; ++v) {
      const int ch = warp + v * nwarps;
      // (the table is padded behind its end: a chunk index past nchunks reads zeros that are never evaluated)
      unsigned long long wd = __ldg(P.words + (size_t)ch * 32 + lane);
      if (Ctx<MEM, ACT, TMALL, BATCH>::kAbs && ch < P.nchunks) wd = word_to_abs(wd, chunk_class(P, ch), smem_u32(dyn));
      tmem_st64(k.tm_warp + 2u * (unsigned)v, wd);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  if (MEM == TB_MEM_TCN_SHARED) {
    // stage the propagator table once: TMA bulk copy global -> shared
    unsigned char* sprops = dyn + store_bytes;
    const unsigned bytes = (unsigned)((size_t)P.nchunks * 32 * TBC_U * 8);
    if (threadIdx.x == 0 && bytes) {
      fence_proxy_async();
      mbar_expect_tx(&local->mbar, bytes);
      for (unsigned off = 0; off < bytes; off += BULK_CHUNK)
        bulk_g2s_issue(sprops + off, (const char*)P.words + off, min(BULK_CHUNK, bytes - off), &local->mbar);
    }
    if (bytes) { while (!mbar_try_wait(&local->mbar, k.mbar_phase)) {} k.mbar_phase ^= 1; }
    k.words = (const unsigned long long*)sprops;
    if (Ctx<MEM, ACT, TMALL, BATCH>::kAbs) {
      // the staged copy is this CTA's own: rewrite its slot fields to absolute shared addresses (see StoreAbs)
      unsigned long long* tw = (unsigned long long*)sprops;
      for (int i = threadIdx.x; i < P.nchunks * 32; i += blockDim.x) {
        const int cls = chunk_class(P, i >> 5);
        tw[i] = word_to_abs(tw[i], cls, smem_u32(dyn));
      }
      k.sync();
    }
  }
}

template <int MEM, bool ACT, bool TMALL, bool BATCH>
__device__ __forceinline__ void ctx_finish(Ctx<MEM, ACT, TMALL, BATCH>& k) {
  // fold the per-thread / per-warp counters into the block statistics
  unsigned n = k.narrowed;
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&k.st->narrowed, (unsigned long long)n);
    if (k.deductions) atomicAdd(&k.st->deductions, k.deductions);
  }
  if (threadIdx.x == 0) bulk_wait_all();     // images still on their way to global memory (best store, snapshots)
  k.sync();        // with a cluster: nobody leaves while a peer may still touch its shared memory
  if (MEM == TB_MEM_STORE_SHARED && TBC_U == 1 && k.P.tmem_cols && threadIdx.x < 32)
    tmem_dealloc(k.lc->tmem_base, (unsigned)k.P.tmem_cols);
}

// ================================================================================================
// kernels
// ================================================================================================

// The persistent dive-and-solve kernel (gpu_barebones_solve, barebones :620-901). BATCH: tb_solve_groups.
template <int MEM, bool ACT = false, bool TMALL = false, bool BATCH = false>
__global__ void __launch_bounds__(TB_MAX_THREADS) solve_kernel(const __grid_constant__ DevParams P) {
  extern __shared__ __align__(128) unsigned char dyn[];
  __shared__ Ctl c_local;
  Ctl& c = *shared_ctl<MEM>(&c_local);
  Ctx<MEM, ACT, TMALL, BATCH> k(P, c);
  ctx_init(k, &c_local, dyn);
  const int tid = k.tid;
  BlockStats* st = k.st;
  if (tid == 0) {
    c.task_idx = (unsigned long long)k.slot * (unsigned long long)P.world + (unsigned long long)P.rank;
    c.task_depth = P.subproblems_power; c.task_entry = -1; c.task_src = -1; c.task_j = 0; c.counted_idle = 0; c.abandon = 0; c.task_nodes = 0;
    c.have_task = c.task_idx < P.num_subproblems;
    if (P.split_bits) atomicAdd(P.split_ctl + TB_SPLIT_STARTED, 1u);
    if (!c.have_task) k.next_subproblem();       // more blocks than subproblems: wait for the tail to be split
    // this run's epoch enters the incumbent cell: whatever an earlier run (of this solver or of a peer) left is void
    atomicMin(P.cells + TB_CELL_BOUND, k.bound_word(TBD_PINF));
  }
  k.sync();
  k.search();
  if (tid == 0) {
    if (P.split_bits && !c.counted_idle) atomicAdd(P.split_ctl + TB_SPLIT_GONE, 1u);      // (waiting blocks stay counted as such)
    if (!(P.cutnodes && st->nodes >= P.cutnodes) && !k.stop_raised()) st->blocks_done = 1;
    st->t_idle = (long long)(globaltimer_ns() - P.t_start);
  }
  ctx_finish(k);
}

// One fixpoint per block on caller-provided stores (tb_propagate / tb_propagate_batch).
template <int MEM, bool ACT = false, bool TMALL = false>
__global__ void __launch_bounds__(TB_MAX_THREADS) propagate_kernel(const __grid_constant__ DevParams P, int nstores,
                                                         const int* in_lb, const int* in_ub,
                                                         int* out_lb, int* out_ub, int* out_failed, int repeat) {
  extern __shared__ __align__(128) unsigned char dyn[];
  __shared__ Ctl c_local;
  Ctl& c = *shared_ctl<MEM>(&c_local);
  Ctx<MEM, ACT, TMALL> k(P, c);
  ctx_init(k, &c_local, dyn);
  const int tid = k.tid, T = k.T;
  for (int s = k.slot; s < nstores; s += k.nslots) {
    int f = 0, iters = 0;
    for (int r = 0; r < repeat; ++r) {
      k.sync();
      // load the caller's store into the block store (slot order); a referenced variable that is already
      // empty fails the store before any propagation, as the oracle's deduce does
      if (tid == 0) { c.leaf = 0; c.dirty_all = 1; }
      k.sync();
      int empty_seen = 0;
      if (P.vpad != P.nvars) {                 // padding slots hold the singleton 0
        for (int sl = tid; sl < P.vpad; sl += T) if (P.var_of[sl] < 0) k.store.set(sl, 0, 0);
      }
      for (int v = tid; v < P.nvars; v += T) {
        const int l = in_lb[(size_t)s * P.nvars + v], u = in_ub[(size_t)s * P.nvars + v];
        empty_seen |= (l > u) & (int)P.referenced[v];
        k.store.set(P.slot_of[v], l, u);
      }
      if (empty_seen) atomicOr(&c.leaf, 1);
      k.sync();
      if (c.leaf) { f = F_FAILED; iters = 0; k.sync(); }
      else if constexpr (ACT) f = k.fixpoint_active(iters);
      else f = k.fixpoint(iters);
      if (tid == 0) {
        k.st->fixpoint_iterations += (unsigned long long)iters;
        k.st->nodes++;
      }
    }
    k.sync();
    for (int v = tid; v < P.nvars; v += T) {
      int l, u; k.store.ld(P.slot_of[v], l, u);
      out_lb[(size_t)s * P.nvars + v] = l; out_ub[(size_t)s * P.nvars + v] = u;
    }
    if (tid == 0) out_failed[s] = (f & F_FAILED) ? 1 : 0;
  }
  ctx_finish(k);
}

// EPS dive only (tb_dive / tb_dive_batch).
template <int MEM, bool ACT = false, bool TMALL = false>
__global__ void __launch_bounds__(TB_MAX_THREADS) dive_kernel(const __grid_constant__ DevParams P, unsigned long long first, int count,
                                                    int depth, int* out_lb, int* out_ub, int* out_remaining, int* out_kind) {
  extern __shared__ __align__(128) unsigned char dyn[];
  __shared__ Ctl c_local;
  Ctl& c = *shared_ctl<MEM>(&c_local);
  Ctx<MEM, ACT, TMALL> k(P, c);
  ctx_init(k, &c_local, dyn);
  const int tid = k.tid, T = k.T;
  for (int s = k.slot; s < count; s += k.nslots) {
    k.sync();
    int remaining = k.dive(first + (unsigned long long)s, depth);
    k.sync();
    for (int v = tid; v < P.nvars; v += T) {
      int l, u; k.store.ld(P.slot_of[v], l, u);
      out_lb[(size_t)s * P.nvars + v] = l; out_ub[(size_t)s * P.nvars + v] = u;
    }
    if (tid == 0) { out_remaining[s] = remaining; out_kind[s] = c.leaf ? (c.failed ? 1 : 2) : 0; }
  }
  ctx_finish(k);
}

// ================================================================================================
// host side
// ================================================================================================

struct tb_solver;
static void unpack_store(const tb_solver* s, const int* img, int32_t* lb, int32_t* ub);
static inline size_t img_lb(const tb_solver* s, int v);
static inline size_t img_ub(const tb_solver* s, int v);
static thread_local std::string g_last_error;
static void set_error(const std::string& s) { g_last_error = s; }
extern "C" const char* tb_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* tb_version(void) { return "turbo-b200 0.1.0 (sm_100a)"; }
void tb_set_error_internal(const char* s) { set_error(s); }

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                          \
      return TB_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

extern "C" int32_t tb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

extern "C" tb_status tb_get_device_info(int32_t device, tb_device_info* info) {
  if (!info) { set_error("null argument"); return TB_ERR_INVALID; }
  memset(info, 0, sizeof(*info));
  if (tb_device_count() <= device || device < 0) { set_error("no such CUDA device"); return TB_ERR_NO_DEVICE; }
  cudaDeviceProp dp;
  CU(cudaGetDeviceProperties(&dp, device));
  CU(cudaRuntimeGetVersion(&info->cuda_runtime_version));
  CU(cudaDriverGetVersion(&info->cuda_driver_version));
  info->sm_count = dp.multiProcessorCount; info->cc_major = dp.major; info->cc_minor = dp.minor;
  info->total_global_mem_bytes = dp.totalGlobalMem;
  int prev = 0;
  CU(cudaGetDevice(&prev));
  CU(cudaSetDevice(device));
  size_t fr = 0, tot = 0, lim = 0;
  if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) info->free_global_mem_bytes = fr;
  if (cudaDeviceGetLimit(&lim, cudaLimitStackSize) == cudaSuccess) info->stack_limit_bytes = lim;
  if (cudaDeviceGetLimit(&lim, cudaLimitMallocHeapSize) == cudaSuccess) info->heap_limit_bytes = lim;
  cudaGetLastError();
  cudaSetDevice(prev);
  strncpy(info->name, dp.name, sizeof(info->name) - 1);
  return TB_OK;
}

extern "C" tb_status tb_set_stack_limit(int32_t device, uint64_t bytes) {
  if (tb_device_count() <= device || device < 0) { set_error("no such CUDA device"); return TB_ERR_NO_DEVICE; }
  int prev = 0;
  CU(cudaGetDevice(&prev));
  CU(cudaSetDevice(device));
  cudaError_t e = cudaDeviceSetLimit(cudaLimitStackSize, (size_t)bytes);
  cudaSetDevice(prev);
  if (e != cudaSuccess) { set_error(std::string("cudaDeviceSetLimit(stack): ") + cudaGetErrorString(e)); cudaGetLastError(); return TB_ERR_CUDA; }
  return TB_OK;
}

struct tb_solver {
  DevParams P;
  tb_options opt;
  int device = 0;
  int nvars = 0, nprops = 0, root_obj_var = -1;
  int mem_kind = TB_MEM_GLOBAL, threads = 256, num_blocks = 1, blocks_per_sm = 1, cluster = 1;
  TnfLayout layout;                   // device table + variable placement (layout.h)
  std::vector<int32_t> root_lb, root_ub;   // the root domains (precondition check of tb_propagate)
  size_t shared_bytes = 0, store_bytes = 0, prop_bytes = 0;
  bool tmall = false;                 // every table word of every warp fits in tensor memory (kernel variant without the L2 path)
  bool want_active = false, active = false;   // TB_FP_*_ACTIVE requested / in effect (shared-memory placements)
  int num_sms = 0;
  size_t device_bytes = 0;            // what the solver holds on the device
  cudaStream_t stream = nullptr, copy_stream = nullptr, poll_stream = nullptr;
  // intermediate-solution ring (tb_stream_solutions / tb_poll_solution)
  StreamRec* h_stream_rec = nullptr;  // pinned, mapped
  int* h_stream_img = nullptr;        // pinned staging buffer for one image
  unsigned long long stream_read = 0; // 1 + number of the latest solution handed to the caller
  std::mutex poll_mutex;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
  std::vector<void*> allocs;
  std::vector<unsigned long long*> peer_cells;   // device pointers to the other GPUs' cell blocks (engine_internal.h)
  std::vector<int> peer_ranks;        // the shard (gpu_rank) each of them dispenses
  std::vector<void*> ipc_opened;
  unsigned long long* d_cells = nullptr;   // this GPU's cell block: incumbent, dispenser, stop
  unsigned epoch = 0;                 // number of tb_solve calls so far: tags the cells of the current run
  // what the latest tb_solve returned (tb_result_pack)
  tb_stats last_stats;
  int last_has = 0, last_exhaustive = 0, last_valid = 0;
  std::vector<int32_t> last_lb, last_ub;
  int scratch_blocks = 0;             // number of per-block scratch slots allocated
  // batch buffers (grown on demand)
  int *d_in_lb = nullptr, *d_in_ub = nullptr, *d_out_lb = nullptr, *d_out_ub = nullptr, *d_out_i0 = nullptr, *d_out_i1 = nullptr;
  size_t batch_cap = 0;
  // tb_solve_groups buffers (grown on demand): root images, BatchRoot cells, best images and BatchGroup cells; for
  // tb_solve_supports the query table (the pool's row counter, then the CSR) and the witness pool
  int *d_batch_roots = nullptr, *d_batch_best = nullptr, *d_batch_query = nullptr, *d_batch_wit = nullptr;
  BatchRoot* d_batch_state = nullptr;
  BatchGroup* d_batch_groups = nullptr;
  size_t batch_images_cap = 0, batch_roots_cap = 0, batch_groups_cap = 0, batch_best_cap = 0, batch_query_cap = 0,
         batch_wit_cap = 0;
  int32_t* h_pinned_one = nullptr;
};

// Device memory comes from the device's stream-ordered pool with the release threshold lifted, so that
// creating and destroying solvers (the drop-in call pattern: one solver per model) does not pay
// cudaMalloc / cudaFree every time: cudaFree of the per-block scratch alone took up to 0.7 s.
static void retain_pool_memory(int device) {
  static bool done[64] = {false};
  if (device < 0 || device >= 64 || done[device]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  cudaGetLastError();
  done[device] = true;
}

template <class T>
static tb_status dev_alloc(tb_solver* s, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = std::max<size_t>(count * sizeof(T), 16);
  retain_pool_memory(s->device);
  cudaError_t e = cudaMallocAsync(&q, bytes, (cudaStream_t)0);
  if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)0);   // usable from the solver's own streams
  if (e != cudaSuccess) { set_error(std::string("cudaMallocAsync: ") + cudaGetErrorString(e)); cudaGetLastError(); return e == cudaErrorMemoryAllocation ? TB_ERR_NOMEM : TB_ERR_CUDA; }
  s->allocs.push_back(q);
  s->device_bytes += bytes;
  *p = (T*)q;
  return TB_OK;
}

// Cell blocks (engine_internal.h) are plain cudaMalloc allocations (CUDA IPC cannot export pool memory), and cudaFree
// synchronises the device and costs tens of milliseconds: a destroyed solver's block goes to a per-device free list
// instead and serves the next solver (the drop-in call pattern creates and destroys one solver per model).
static std::mutex g_cells_mutex;
static std::vector<unsigned long long*> g_free_cells[64];
static unsigned long long* acquire_cells(int device) {
  {
    std::lock_guard<std::mutex> lock(g_cells_mutex);
    if (device >= 0 && device < 64 && !g_free_cells[device].empty()) {
      unsigned long long* p = g_free_cells[device].back();
      g_free_cells[device].pop_back();
      return p;
    }
  }
  unsigned long long* p = nullptr;
  if (cudaMalloc((void**)&p, TB_CELL_BLOCK_BYTES) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
static void release_cells(int device, unsigned long long* p) {
  if (!p) return;
  if (device < 0 || device >= 64) { cudaFree(p); return; }
  std::lock_guard<std::mutex> lock(g_cells_mutex);
  g_free_cells[device].push_back(p);
}

// TB_TRACE_TIMING=1: where tb_create / tb_destroy spend their time (stderr)
struct PhaseTimer {
  bool on; double t0; const char* what;
  static double now() { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e3 + t.tv_nsec * 1e-6; }
  explicit PhaseTimer(const char* w) : on(getenv("TB_TRACE_TIMING") != nullptr), t0(now()), what(w) {}
  void mark(const char* phase) { if (on) { const double t = now(); fprintf(stderr, "[tb timing] %s: %s %.3f ms\n", what, phase, t - t0); t0 = t; } }
};

// One pinned word holding the constant 1 (source of the asynchronous "stop" copy), shared by all solvers.
static int32_t* pinned_one() {
  static int32_t* p = nullptr;
  static std::once_flag once;               // solvers of several GPUs may be created from concurrent host threads
  std::call_once(once, [] {
    if (cudaHostAlloc((void**)&p, 64, cudaHostAllocPortable) != cudaSuccess) { p = nullptr; cudaGetLastError(); }
    else *p = 1;
  });
  return p;
}

// kernel dispatch over the placement
template <class F>
static tb_status dispatch(const tb_solver* s, F&& f) {
  using Dense = std::false_type;
  using Active = std::true_type;          // active-set fixpoint: shared-memory placements only
  using Mixed = std::false_type;          // table words from tensor memory where they fit, from L2 beyond
  using AllTm = std::true_type;           // the whole table is in tensor memory (s->tmall)
  switch (s->mem_kind) {
    case TB_MEM_GLOBAL: return f(std::integral_constant<int, TB_MEM_GLOBAL>{}, Dense{}, Mixed{});
    case TB_MEM_STORE_SHARED:
      if (s->active) return f(std::integral_constant<int, TB_MEM_STORE_SHARED>{}, Active{}, Mixed{});
      return s->tmall ? f(std::integral_constant<int, TB_MEM_STORE_SHARED>{}, Dense{}, AllTm{}) : f(std::integral_constant<int, TB_MEM_STORE_SHARED>{}, Dense{}, Mixed{});
    case TB_MEM_TCN_SHARED:
      return s->active ? f(std::integral_constant<int, TB_MEM_TCN_SHARED>{}, Active{}, Mixed{}) : f(std::integral_constant<int, TB_MEM_TCN_SHARED>{}, Dense{}, Mixed{});
    case TB_MEM_STORE_CLUSTER: return f(std::integral_constant<int, TB_MEM_STORE_CLUSTER>{}, Dense{}, Mixed{});
    default: break;
  }
  set_error("unsupported memory kind");
  return TB_ERR_UNSUPPORTED;
}

// Launch `workers` workers: one CTA each, or one cluster of s->cluster CTAs each (STORE_CLUSTER).
template <class... KArgs, class... Args>
static cudaError_t launch_workers(const tb_solver* s, void (*kernel)(KArgs...), int workers, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3((unsigned)s->threads);
  cfg.dynamicSmemBytes = s->shared_bytes;
  cfg.stream = s->stream;
  cudaLaunchAttribute attr[1];
  if (s->mem_kind == TB_MEM_STORE_CLUSTER) {
    cfg.gridDim = dim3((unsigned)(workers * s->cluster));
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)s->cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
  } else cfg.gridDim = dim3((unsigned)workers);
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// cudaGetDeviceProperties costs 10-20 ms a call: asked once per device
static const cudaDeviceProp* device_props(int device) {
  static cudaDeviceProp props[64];
  static bool have[64] = {false};
  static std::mutex m;
  if (device < 0 || device >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(m);
  if (!have[device]) {
    if (cudaGetDeviceProperties(&props[device], device) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    have[device] = true;
  }
  return &props[device];
}

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

// The sweep assigns chunk ch to warp (ch mod nwarps) with a mask: the warp count is a power of two.
static int pow2_threads(int t) {
  int p = 32;
  while (p * 2 <= std::min(t, TB_MAX_THREADS)) p *= 2;
  return p;
}

// Placement policy: MemoryConfig (memory_gpu.hpp:43-84) + configure_gpu_barebones (barebones :527-606),
// solved together with occupancy (the reference queries occupancy with 0 dynamic smem, SURVEY App. A).
static tb_status configure(tb_solver* s) {
  const cudaDeviceProp* dpp = device_props(s->device);
  if (!dpp) { set_error("cudaGetDeviceProperties failed"); return TB_ERR_CUDA; }
  const cudaDeviceProp& dp = *dpp;
  s->num_sms = dp.multiProcessorCount;
  const size_t max_block_smem = dp.sharedMemPerBlockOptin;               // 227 KB on sm_100
  const size_t sm_smem = dp.sharedMemPerMultiprocessor;                  // 228 KB
  const size_t reserved = dp.reservedSharedMemPerBlock + sizeof(Ctl) + 64;
  // the active-set fixpoint keeps one bit per slot and two bytes per chunk next to the store (upper bound here, the
  // exact figure needs the thread count: place_active)
  const size_t act_b = s->want_active ? (s->store_bytes / 64 + 2 * ((size_t)s->P.nchunks + 1024) + 64) : 0;
  const size_t store_b = s->store_bytes + act_b, prop_b = s->prop_bytes;
  auto blocks_for = [&](size_t dyn) -> int {
    if (dyn + sizeof(Ctl) + 64 > max_block_smem) return 0;
    return (int)std::min<size_t>(32, sm_smem / (dyn + reserved));
  };
  int kind = s->opt.mem_kind;
  const int b_tcn = blocks_for(store_b + prop_b), b_store = blocks_for(store_b);
  // cluster tier: smallest power-of-two cluster whose slice (vc * 8 bytes per CTA) fits one SM
  auto slice_vars = [&](int c) { return ((s->nvars + c - 1) / c + 3) / 4 * 4; };
  int cluster = 0;
  for (int c = 2; c <= 16; c *= 2)
    if (blocks_for((size_t)std::max(4, slice_vars(c)) * 8) >= 1) { cluster = c; break; }
  if (s->opt.cluster_size > 0) {
    cluster = s->opt.cluster_size;
    if ((cluster & (cluster - 1)) != 0 || cluster > 16 || blocks_for((size_t)std::max(4, slice_vars(cluster)) * 8) < 1) {
      set_error("cluster_size must be a power of two <= 16 whose slice fits in shared memory"); return TB_ERR_INVALID;
    }
  }
  const bool shape_v1 = env_int("TB_SHAPE_V1", 0) != 0;      // round 1's placement and block shape, for A/B runs
  if (kind == TB_MEM_AUTO) {
    // The store in shared memory whenever it fits, the table in tensor memory or L2: shared memory then holds more
    // blocks, and independent blocks are what hides the barriers and the one-thread sections of the search (round 1
    // already found 2 x 512 threads with the table in L2 faster than 1 x 1024 with the table in shared memory on
    // trains15; with small single-warp blocks the same holds for the small networks - accap_a3: 42.4 M nodes/s with
    // 24 x 32 threads per SM and the table in L2 against 27.6 M with 8 x 128 and the table in shared memory,
    // profiles/r02_block_shapes.md). TCN_SHARED stays available on request.
    if (shape_v1 && b_tcn >= 1 && !(b_tcn == 1 && b_store >= 2) && (b_tcn >= 4 || b_tcn * 2 >= std::min(b_store, 8))) kind = TB_MEM_TCN_SHARED;
    else if (b_store >= 1) kind = TB_MEM_STORE_SHARED;
    else if (cluster >= 2) kind = TB_MEM_STORE_CLUSTER;    // the store is larger than one SM: stripe it over DSMEM
    else kind = TB_MEM_GLOBAL;
  }
  if (kind == TB_MEM_TCN_SHARED && b_tcn < 1) { set_error("TCN_SHARED does not fit in shared memory"); return TB_ERR_INVALID; }
  if (kind == TB_MEM_STORE_SHARED && b_store < 1) { set_error("STORE_SHARED does not fit in shared memory"); return TB_ERR_INVALID; }
  if (kind == TB_MEM_STORE_CLUSTER) {
    if (cluster < 2) { set_error("STORE_CLUSTER: no cluster size up to 16 holds this store"); return TB_ERR_INVALID; }
    s->cluster = cluster;
    s->P.cluster_size = cluster;
    s->P.cluster_log2 = 0;
    while ((1 << s->P.cluster_log2) < cluster) ++s->P.cluster_log2;
    s->P.vc = std::max(4, slice_vars(cluster));
    s->P.vpad = s->P.vc * cluster;               // an image is `cluster` slices of vc variables
    s->store_bytes = (size_t)s->P.vpad * 8;
    s->mem_kind = kind;
    s->shared_bytes = (size_t)s->P.vc * 8;
    s->threads = s->opt.threads_per_block > 0 ? pow2_threads(s->opt.threads_per_block) : TB_MAX_THREADS;
    s->blocks_per_sm = 1;
    // how many clusters can be co-resident is asked from the driver once the kernel attributes are set
    s->num_blocks = std::max(1, s->num_sms / cluster);
    return TB_OK;
  }
  s->mem_kind = kind;
  s->shared_bytes = kind == TB_MEM_TCN_SHARED ? store_b + prop_b : (kind == TB_MEM_STORE_SHARED ? store_b : 0);
  int bps = kind == TB_MEM_TCN_SHARED ? b_tcn : (kind == TB_MEM_STORE_SHARED ? b_store : 8);
  // Threads: keep ~1024 resident threads per SM at <= 64 registers (the reference compiles 256/block).
  int threads = s->opt.threads_per_block;
  if (threads <= 0 && (shape_v1 || s->P.nchunks < 16)) {
    // Round 1's shape: 1024 resident threads per SM spread over up to 8 blocks. Still the choice for the tiniest
    // networks (under 16 chunks, i.e. 500 propagators): their nodes are all search bookkeeping, and 32 single-warp
    // blocks per SM, each somewhere else in a 150 KB kernel, run it 2-3 x slower than 8 blocks of 4 warps (pat1, pat10,
    // pat11: profiles/r02_block_shapes.md).
    bps = std::min(bps, 8);
    threads = bps >= 8 ? 128 : (bps >= 4 ? 256 : (bps >= 2 ? 512 : 1024));
    threads = std::min(threads, TB_MAX_THREADS);
    while (threads > 128 && threads / 2 >= s->P.nchunks * 32) threads /= 2;   // at least one chunk per warp
  } else if (threads <= 0) {
    // As many blocks as shared memory holds (up to 32 per SM), each with as FEW warps as keeps (a) about 24 warps
    // resident per SM and (b) a warp's share of a sweep around 24 chunks or more: a sweep costs every warp some 300
    // instructions of class entry / exit and flag handling whatever it visits, and every block-wide barrier waits
    // for the slowest warp, so few long warps beat many short ones - down to single-warp blocks, whose barriers are
    // free (accap_a3, 40 chunks: 24 x 32 threads per SM; trains15, 440 chunks, 2 blocks fit: 2 x 512; wordpress: 1 x 1024).
    bps = std::min(bps, 32);
    int warps = 1;
    while (warps < 32 && warps * bps < 24) warps *= 2;
    while (warps < 32 && warps * 2 * 24 <= s->P.nchunks) warps *= 2;
    threads = std::min(32 * warps, TB_MAX_THREADS);
    bps = std::max(1, std::min(bps, 1024 / threads));                          // 64 registers per thread
  }
  threads = pow2_threads(threads);
  bps = std::max(1, std::min(bps, 2048 / threads));
  s->threads = threads;
  s->blocks_per_sm = bps;
  int blocks = bps * s->num_sms;
  if (s->opt.or_blocks > 0) blocks = std::min(blocks, s->opt.or_blocks);
  s->num_blocks = std::max(1, blocks);
  s->blocks_per_sm = (s->num_blocks + s->num_sms - 1) / s->num_sms;
  return TB_OK;
}

// Active-set fixpoint: exact size and position of its flags once the layout pass has fixed the store image and the
// placement policy the thread count.  Shared-memory placements only; elsewhere the plain sweeps run.
static void place_active(tb_solver* s) {
  s->active = s->want_active && (s->mem_kind == TB_MEM_STORE_SHARED || s->mem_kind == TB_MEM_TCN_SHARED);
  s->P.act_off = 0; s->P.act_fpw = 0;
  if (!s->active) return;
  const int nwarps = s->threads / 32;
  const int per_warp = (s->P.nchunks + nwarps - 1) / nwarps;
  s->P.act_fpw = std::max(32, (per_warp + 31) / 32 * 32);
  const size_t table = s->mem_kind == TB_MEM_TCN_SHARED ? (size_t)s->P.nchunks * 32 * TBC_U * 8 : 0;
  s->P.act_off = (int)(s->store_bytes + table);
  const size_t act = (size_t)s->P.vpad / 8 + (size_t)2 * nwarps * s->P.act_fpw;     // moved bits, dirty, cached ask
  s->shared_bytes = (size_t)s->P.act_off + (act + 15) / 16 * 16;
}

static tb_status set_smem_attr(tb_solver* s) {
  return dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
    constexpr int m = decltype(M)::value;
    constexpr bool act = decltype(A)::value;
    constexpr bool tmall = decltype(TM)::value;
    if (s->shared_bytes) {
      CU(cudaFuncSetAttribute(solve_kernel<m, act, tmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->shared_bytes));
      CU(cudaFuncSetAttribute(propagate_kernel<m, act, tmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->shared_bytes));
      CU(cudaFuncSetAttribute(dive_kernel<m, act, tmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->shared_bytes));
    }
    if (m == TB_MEM_STORE_CLUSTER) {
      if (s->cluster > 8) {
        CU(cudaFuncSetAttribute(solve_kernel<m, act, tmall>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        CU(cudaFuncSetAttribute(propagate_kernel<m, act, tmall>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        CU(cudaFuncSetAttribute(dive_kernel<m, act, tmall>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      }
      cudaLaunchConfig_t cfg = {};
      cfg.blockDim = dim3((unsigned)s->threads);
      cfg.gridDim = dim3((unsigned)(s->cluster * s->num_sms));
      cfg.dynamicSmemBytes = s->shared_bytes;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)s->cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      int nclusters = 0;
      CU(cudaOccupancyMaxActiveClusters(&nclusters, solve_kernel<m, act, tmall>, &cfg));
      if (nclusters < 1) { set_error("the device cannot host a cluster of this size"); return TB_ERR_UNSUPPORTED; }
      int workers = nclusters;
      if (s->opt.or_blocks > 0) workers = std::min(workers, s->opt.or_blocks);
      s->num_blocks = std::max(1, workers);
    } else {
      // registers limit the resident CTAs too: ask the driver what really fits (persistent kernel: one wave)
      int per_sm = 0;
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, solve_kernel<m, act, tmall>, s->threads, s->shared_bytes));
      if (getenv("TB_TRACE_TIMING")) {
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, solve_kernel<m, act, tmall>) == cudaSuccess)
          fprintf(stderr, "[tb config] solve_kernel<%d,%d>: %d threads, dynamic smem %zu, static smem %zu, %d registers, local %zu B -> %d CTAs per SM by the occupancy API (policy wanted %d)\n",
                  m, (int)act, s->threads, s->shared_bytes, fa.sharedSizeBytes, fa.numRegs, fa.localSizeBytes, per_sm, s->blocks_per_sm);
      }
      if (per_sm < 1) { set_error("the solve kernel does not fit on an SM with this configuration"); return TB_ERR_UNSUPPORTED; }
      // The occupancy API answers "one CTA per SM" for every kernel that contains tcgen05.alloc, whatever it allocates
      // (measured). The policy above already keeps to 1024 resident threads per SM at 64 registers (__launch_bounds__)
      // and to the shared memory of the SM, and the CTAs split the 512 tensor-memory columns between them (tb_create):
      // for those kernels its own arithmetic stands.
      if ((m == TB_MEM_STORE_SHARED && TBC_U == 1) || env_int("TB_IGNORE_OCCUPANCY_API", 0)) {
        // (own arithmetic: shared memory was accounted for by configure(); registers and threads here. The grid MUST be
        // co-resident: blocks that find no work wait for the others - tail splitting - and a CTA that cannot start
        // because its SM is full of waiting CTAs would never let them finish.)
        cudaFuncAttributes fa;
        CU(cudaFuncGetAttributes(&fa, solve_kernel<m, act, tmall>));
        const cudaDeviceProp* dp = device_props(s->device);
        const int regs_per_cta = std::max(1, fa.numRegs) * ((s->threads + 31) / 32 * 32);
        const int by_regs = dp ? std::max(1, dp->regsPerMultiprocessor / regs_per_cta) : 1;
        const int by_threads = dp ? std::max(1, dp->maxThreadsPerMultiProcessor / s->threads) : 1;
        per_sm = std::max(per_sm, std::min(s->blocks_per_sm, std::min(by_regs, by_threads)));
      }
      if (per_sm < s->blocks_per_sm) {
        s->blocks_per_sm = per_sm;
        int blocks = per_sm * s->num_sms;
        if (s->opt.or_blocks > 0) blocks = std::min(blocks, s->opt.or_blocks);
        s->num_blocks = std::max(1, blocks);
      }
    }
    return TB_OK;
  });
}

static tb_status ensure_scratch(tb_solver* s, int slots) {
  if (slots <= s->scratch_blocks) return TB_OK;
  DevParams& P = s->P;
  tb_status rc;
  const size_t img = (size_t)2 * P.vpad;
  if ((rc = dev_alloc(s, &P.block_root, img * slots))) return rc;
  if ((rc = dev_alloc(s, &P.block_best, img * slots))) return rc;
  if (s->mem_kind == TB_MEM_GLOBAL) { if ((rc = dev_alloc(s, &P.block_store, img * slots))) return rc; }
  if ((rc = dev_alloc(s, &P.decisions, (size_t)P.max_depth * slots))) return rc;
  {
    // snapshot ring: as many levels as a memory budget allows (TB_SNAPSHOT_MB, default 4096 MB per GPU; 0 disables),
    // at most 64 per block (TB_SNAPSHOT_LEVELS lowers that: the tests run rings of 2 and 3 levels to exercise slot reuse)
    const size_t budget = (size_t)std::max(0, env_int("TB_SNAPSHOT_MB", 4096)) << 20;
    const size_t per_level = img * sizeof(int) * (size_t)slots;
    int n = (int)std::min<size_t>((size_t)std::max(0, std::min(64, env_int("TB_SNAPSHOT_LEVELS", 64))), per_level ? budget / per_level : 0);
    if (s->opt.max_depth > 0) n = std::min(n, s->opt.max_depth);
    P.nsnap = 0; P.block_snap = nullptr; P.snap_tag = nullptr;
    if (n >= 2) {
      if (dev_alloc(s, &P.block_snap, img * (size_t)slots * (size_t)n) == TB_OK && dev_alloc(s, &P.snap_tag, (size_t)slots * (size_t)n) == TB_OK) {
        if (cudaMemset(P.snap_tag, 0xff, (size_t)slots * (size_t)n * sizeof(int)) != cudaSuccess) { set_error("memset snapshot tags"); return TB_ERR_CUDA; }
        P.nsnap = n;
        if (s->active) {
          const size_t fw = (size_t)(s->threads / 32) * (size_t)P.act_fpw / 4;
          if (dev_alloc(s, &P.snap_flags, std::max<size_t>(1, fw * (size_t)slots * (size_t)n)) != TB_OK) { cudaGetLastError(); P.nsnap = 0; }
        }
      } else { cudaGetLastError(); P.block_snap = nullptr; P.snap_tag = nullptr; }    // no room: recompute on backtrack as the reference does
    }
  }
  if ((rc = dev_alloc(s, &P.stats, (size_t)slots))) return rc;
  if (!P.split_pool) {
    // (control block and pool live in the cell block's allocation: the peers map them with the same IPC handle)
    P.split_ctl = (unsigned*)(s->d_cells + TB_CELL_SPLIT);
    P.split_pool = (SplitEntry*)(s->d_cells + TB_CELL_WORDS);
    P.split_bits = std::max(0, std::min(12, env_int("TB_SPLIT_BITS", 6)));
    P.split_min_nodes = std::max(256, env_int("TB_SPLIT_MIN_NODES", 4096));
  }
  s->scratch_blocks = slots;
  return TB_OK;
}

extern "C" tb_status tb_create(tb_solver** out, const tb_problem* pb, const tb_options* opt_in) {
  if (!out || !pb) { set_error("null argument"); return TB_ERR_INVALID; }
  *out = nullptr;
  if (pb->nvars < 0 || pb->nprops < 0 || (pb->nvars && (!pb->lb || !pb->ub)) || (pb->nprops && !pb->props)) {
    set_error("malformed tb_problem"); return TB_ERR_INVALID;
  }
  for (int i = 0; i < pb->nprops; ++i) {
    const tb_prop& p = pb->props[i];
    if (p.op < 0 || p.op >= TB_NUM_OPS || p.x < 0 || p.y < 0 || p.z < 0 || p.x >= pb->nvars || p.y >= pb->nvars || p.z >= pb->nvars) {
      set_error("propagator " + std::to_string(i) + " has an invalid operator or variable index"); return TB_ERR_INVALID;
    }
    if ((p.op == TB_OP_EQ || p.op == TB_OP_LEQ) && (pb->lb[p.x] < 0 || pb->ub[p.x] > 1)) {
      set_error("propagator " + std::to_string(i) + ": the result variable of EQ/LEQ must have a domain within 0..1"); return TB_ERR_INVALID;
    }
  }
  if (pb->obj_var >= pb->nvars) { set_error("obj_var out of range"); return TB_ERR_INVALID; }
  for (int i = 0; i < pb->nstrategies; ++i) {
    const tb_strategy& st = pb->strategies[i];
    if (st.n < 0 || (st.n && !st.vars)) { set_error("malformed strategy"); return TB_ERR_INVALID; }
    for (int j = 0; j < st.n; ++j) if (st.vars[j] < 0 || st.vars[j] >= pb->nvars) { set_error("strategy variable out of range"); return TB_ERR_INVALID; }
  }
  if (tb_device_count() <= 0) { set_error("no CUDA device visible: the engine has no CPU fallback"); return TB_ERR_NO_DEVICE; }
  PhaseTimer pt("tb_create");

  tb_options opt;
  memset(&opt, 0, sizeof(opt));
  if (opt_in) opt = *opt_in;
  else { opt.fixpoint = TB_FP_WAC1; opt.subproblems_power = -1; opt.subproblems_factor = 300; opt.mem_kind = TB_MEM_AUTO; opt.gpu_world = 1; }
  if (opt.gpu_world <= 0) { opt.gpu_world = 1; opt.gpu_rank = 0; }
  if (opt.gpu_rank < 0 || opt.gpu_rank >= opt.gpu_world) { set_error("gpu_rank out of range"); return TB_ERR_INVALID; }
  if (opt.subproblems_factor <= 0) opt.subproblems_factor = 300;

  tb_solver* s = new tb_solver();
  s->opt = opt;
  s->device = opt.device;
  tb_status rc = TB_OK;
  auto fail = [&](tb_status r) { tb_destroy(s); return r; };
  if (cudaSetDevice(s->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return fail(TB_ERR_CUDA); }
  DevParams& P = s->P;
  memset(&P, 0, sizeof(P));
  s->nvars = pb->nvars; s->nprops = pb->nprops;
  P.nvars = pb->nvars; P.nprops = pb->nprops;
  P.obj_var = pb->obj_var;
  s->root_obj_var = pb->obj_var;
  P.has_eps_strategy = pb->has_eps_strategy;
  P.fixpoint_kind = (opt.fixpoint == TB_FP_AC1 || opt.fixpoint == TB_FP_AC1_ACTIVE) ? TB_FP_AC1 : TB_FP_WAC1;
  s->want_active = opt.fixpoint == TB_FP_AC1_ACTIVE || opt.fixpoint == TB_FP_WAC1_ACTIVE;
  P.wac1_threshold = opt.wac1_threshold;
  P.cutnodes = opt.cutnodes;
  P.rank = opt.gpu_rank; P.world = opt.gpu_world;
  P.max_depth = opt.max_depth > 0 ? opt.max_depth : 10000;
  if (pb->nvars > TBC_MAX_VARS) { set_error("more than 2^21 variables: the device propagator word has 21-bit fields"); return fail(TB_ERR_UNSUPPORTED); }
  s->root_lb.assign(pb->lb, pb->lb + pb->nvars);
  s->root_ub.assign(pb->ub, pb->ub + pb->nvars);

  // ---- placement, then the layout pass for that placement (layout.h) ----------------------------------
  {
    // sizes the placement policy needs: the table is padded per class to whole chunks of 32
    int per_class[TBC_NUM] = {0};
    for (int i = 0; i < pb->nprops; ++i) { bool sw; ++per_class[tb_classify(pb->props[i], pb->lb, pb->ub, &sw)]; }
    int nchunks = 0;
    for (int c = 0; c < TBC_NUM; ++c) nchunks += (per_class[c] + 32 * TBC_U - 1) / (32 * TBC_U);
    P.nchunks = nchunks;
    s->prop_bytes = (size_t)nchunks * 32 * TBC_U * 8;
    s->store_bytes = (size_t)std::max(32, (pb->nvars + 31) / 32 * 32) * 8;     // shared placements pad to the 32 banks
  }
  // Small tables are cheaper to sweep densely than to track (accap_a3, 32 chunks: 25 M nodes/s dense, 13.5 M active;
  // trains15, 420 chunks: 5.7 M dense, 8.4 M active): below TB_ACTIVE_MIN_CHUNKS (default 128) the plain kind runs
  // and no flag area is reserved. Chunk ids must fit the 16-bit fields of the watch words.
  if (P.nchunks < env_int("TB_ACTIVE_MIN_CHUNKS", 128) || P.nchunks >= 0xFFFE) s->want_active = false;
  pt.mark("validate, classify");
  if ((rc = configure(s)) != TB_OK) return fail(rc);
  pt.mark("configure");
  {
    TnfLayoutOptions lo;
    const bool shared_store = s->mem_kind == TB_MEM_STORE_SHARED || s->mem_kind == TB_MEM_TCN_SHARED;
    lo.nbanks = shared_store && env_int("TB_NO_BANK_LAYOUT", 0) == 0 ? 16 : 0;
    lo.slot_align = shared_store ? 32 : (s->mem_kind == TB_MEM_STORE_CLUSTER ? 4 * s->cluster : 4);
    if (s->mem_kind == TB_MEM_STORE_CLUSTER && env_int("TB_CLUSTER_LOCALITY", 1) != 0) { lo.cluster = s->cluster; lo.cluster_warps = s->threads / 32; }
    std::string err;
    if ((rc = tb_build_layout(pb, lo, &s->layout, &err)) != TB_OK) { set_error(err); return fail(rc); }
    const TnfLayout& L = s->layout;
    if (s->mem_kind == TB_MEM_STORE_CLUSTER && getenv("TB_TRACE_TIMING"))
      fprintf(stderr, "[tb config] store_cluster x%d: %.1f %% of the operand loads of a sweep stay in the evaluating CTA (striped placement: %.1f %%)\n",
              s->cluster, 100.0 * L.cluster_local_fraction, 100.0 / s->cluster);
    P.vpad = L.nslots;
    if (s->mem_kind == TB_MEM_STORE_CLUSTER && P.vpad != P.vc * s->cluster) { set_error("internal: cluster slice size mismatch"); return fail(TB_ERR_INVALID); }
    s->store_bytes = (size_t)P.vpad * 8;
    P.nchunks = L.cls_begin[TBC_NUM];
    for (int c = 0; c <= TBC_NUM; ++c) P.cls_begin[c] = L.cls_begin[c];
    for (int c = 0; c < TBC_NUM; ++c) P.cls_last[c] = L.cls_last[c];
    if (pb->obj_var >= 0) P.obj_var = L.slot_of[pb->obj_var];
    for (int v = 0; v < pb->nvars; ++v) if (L.referenced[v] && pb->lb[v] > pb->ub[v]) P.root_failed = 1;
  }
  pt.mark("layout pass");
  place_active(s);
  if ((rc = set_smem_attr(s)) != TB_OK) return fail(rc);
  // Tensor memory as the table cache (STORE_SHARED, dense kinds): the resident CTAs of an SM share its 512 columns, a
  // CTA's warps share the CTA's columns by quarter (warp index mod 4), a visit takes two columns. TB_TMEM=0: off.
  P.tmem_cols = 0; P.tmem_visits = 0;
  if (TBC_U == 1 && s->mem_kind == TB_MEM_STORE_SHARED && env_int("TB_TMEM", 1) != 0 && P.nchunks > 0) {
    int cols = 32;
    while (cols * 2 * s->blocks_per_sm <= 512) cols *= 2;
    const int nwarps = s->threads / 32, per_quarter = (nwarps + 3) / 4;
    const int visits_fit = cols / per_quarter / 2, visits_needed = (P.nchunks + nwarps - 1) / nwarps;
    if (cols * s->blocks_per_sm <= 512 && visits_fit >= 1) { P.tmem_cols = cols; P.tmem_visits = std::min(visits_fit, visits_needed); }
    s->tmall = P.tmem_cols && !s->active && visits_fit >= visits_needed;
    // (set_smem_attr ran for the mixed variant above; the all-in-TMEM kernels that will be launched need theirs too)
    if (s->tmall && (rc = set_smem_attr(s)) != TB_OK) return fail(rc);
  }
  pt.mark("kernel attributes, occupancy");

  // ---- device images ---------------------------------------------------------------------------------
  {
    std::vector<int> img((size_t)2 * P.vpad, 0);
    for (int v = 0; v < pb->nvars; ++v) { img[img_lb(s, v)] = pb->lb[v]; img[img_ub(s, v)] = pb->ub[v]; }
    int* d = nullptr;
    if ((rc = dev_alloc(s, &d, img.size()))) return fail(rc);
    if (cudaMemcpy(d, img.data(), img.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("H2D root store"); return fail(TB_ERR_CUDA); }
    P.root_store = d;
  }
  {
    const TnfLayout& L = s->layout;
    unsigned long long* d = nullptr;
    // Padding behind the table: a warp requests the words of its next chunk (ch + nwarps) before it knows whether the sweep
    // goes on, without a bound check, so up to nwarps chunks past the end are read (never used); 2 * nwarps + 1 chunks of
    // padding cover that. nwarps is the warp count of a whole worker: threads * cluster / 32, up to 512 with a cluster of 16.
    const size_t pad_words = (size_t)(2 * (s->threads * std::max(1, s->cluster) / 32) + 1) * 32 * TBC_U;
    if ((rc = dev_alloc(s, &d, L.words.size() + pad_words))) return fail(rc);
    if (cudaMemset(d, 0, (L.words.size() + pad_words) * 8) != cudaSuccess ||
        (L.words.size() && cudaMemcpy(d, L.words.data(), L.words.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess)) { set_error("H2D props"); return fail(TB_ERR_CUDA); }
    P.words = d;
    if (s->active) {
      int *wo = nullptr, *wl = nullptr;
      if ((rc = dev_alloc(s, &wo, L.watch_off.size()))) return fail(rc);
      if ((rc = dev_alloc(s, &wl, std::max<size_t>(1, L.watch_list.size())))) return fail(rc);
      if (cudaMemcpy(wo, L.watch_off.data(), L.watch_off.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess ||
          (L.watch_list.size() && cudaMemcpy(wl, L.watch_list.data(), L.watch_list.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess)) { set_error("H2D watch lists"); return fail(TB_ERR_CUDA); }
      P.watch_off = wo; P.watch_list = wl;
      unsigned long long* wi = nullptr;
      if ((rc = dev_alloc(s, &wi, std::max<size_t>(1, L.watch_inline.size())))) return fail(rc);
      if (L.watch_inline.size() && cudaMemcpy(wi, L.watch_inline.data(), L.watch_inline.size() * 8, cudaMemcpyHostToDevice) != cudaSuccess) { set_error("H2D watch words"); return fail(TB_ERR_CUDA); }
      P.watch_inline = wi;
    }
    std::vector<int> var_of((size_t)P.vpad, -1);
    for (int v = 0; v < pb->nvars; ++v) var_of[L.slot_of[v]] = v;
    int *dslot = nullptr, *dvar = nullptr;
    unsigned char* dref = nullptr;
    if ((rc = dev_alloc(s, &dslot, L.slot_of.size()))) return fail(rc);
    if ((rc = dev_alloc(s, &dvar, var_of.size()))) return fail(rc);
    if ((rc = dev_alloc(s, &dref, L.referenced.size()))) return fail(rc);
    if ((pb->nvars && cudaMemcpy(dslot, L.slot_of.data(), L.slot_of.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) ||
        cudaMemcpy(dvar, var_of.data(), var_of.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess ||
        (pb->nvars && cudaMemcpy(dref, L.referenced.data(), L.referenced.size(), cudaMemcpyHostToDevice) != cudaSuccess)) {
      set_error("H2D layout tables"); return fail(TB_ERR_CUDA);
    }
    P.slot_of = dslot; P.var_of = dvar; P.referenced = dref;
  }
  {
    std::vector<DevStrategy> hs((size_t)std::max(1, pb->nstrategies));
    const TnfLayout& L = s->layout;
    for (int i = 0; i < pb->nstrategies; ++i) {
      const tb_strategy& st = pb->strategies[i];
      hs[i].var_order = st.var_order; hs[i].val_order = st.val_order; hs[i].n = st.n; hs[i].vars = nullptr;
      // the device works on slots: translate the list; "all variables in index order" (n == 0) becomes an
      // explicit list once the placement is not the identity, so that ties still break on the caller's order
      std::vector<int> slots;
      if (st.n) { slots.resize((size_t)st.n); for (int j = 0; j < st.n; ++j) slots[j] = L.slot_of[st.vars[j]]; }
      else if (!L.identity && pb->nvars) { slots = L.slot_of; hs[i].n = pb->nvars; }
      if (!slots.empty()) {
        int* dv = nullptr;
        if ((rc = dev_alloc(s, &dv, slots.size()))) return fail(rc);
        if (cudaMemcpy(dv, slots.data(), slots.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("H2D strategy"); return fail(TB_ERR_CUDA); }
        hs[i].vars = dv;
      }
    }
    DevStrategy* d = nullptr;
    if ((rc = dev_alloc(s, &d, hs.size()))) return fail(rc);
    if (cudaMemcpy(d, hs.data(), hs.size() * sizeof(DevStrategy), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("H2D strategies"); return fail(TB_ERR_CUDA); }
    P.strategies = d; P.nstrategies = pb->nstrategies;
  }
  // the cell block is exported to other processes (CUDA IPC): that needs a plain cudaMalloc allocation
  {
    unsigned long long init[TB_CELL_WORDS] = {0};
    init[TB_CELL_BOUND] = ~0ull;            // epoch 0, no incumbent
    if ((s->d_cells = acquire_cells(s->device)) == nullptr ||
        cudaMemcpy(s->d_cells, init, sizeof(init), cudaMemcpyHostToDevice) != cudaSuccess) {
      set_error("cudaMalloc (grid cells) failed"); cudaGetLastError(); return fail(TB_ERR_CUDA);
    }
  }
  P.cells = s->d_cells; P.npeers = 0; P.steal = 0; P.epoch = 0; P.observe_stop = 1;
  pt.mark("uploads");
  if ((rc = ensure_scratch(s, s->num_blocks))) return fail(rc);
  pt.mark("per-block scratch");
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&s->ev_start) != cudaSuccess || cudaEventCreate(&s->ev_stop) != cudaSuccess ||
      (s->h_pinned_one = pinned_one()) == nullptr) {
    set_error("stream/event creation failed"); return fail(TB_ERR_CUDA);
  }

  // The propagator table is what every block streams from L2 in every sweep, next to the snapshot images that flow
  // through L2 once: TB_L2_PERSIST=1 asks for the table's lines to persist (access policy window on the solver's stream). Best effort: a device without the feature just keeps its normal policy.
  // Measured (profiles/r02_ab_dense_variants.md): no effect on the solve kernel (320.6 against 320.8 Gprop/s: the table
  // never leaves L2 anyway) and 30-110 ms per tb_create for the two API calls, so it is OFF unless TB_L2_PERSIST=1.
  if (env_int("TB_L2_PERSIST", 0) != 0 && s->mem_kind != TB_MEM_TCN_SHARED && s->layout.words.size()) {
    const cudaDeviceProp* dpp = device_props(s->device);
    if (dpp && dpp->persistingL2CacheMaxSize > 0 && dpp->accessPolicyMaxWindowSize > 0) {
      const cudaDeviceProp& dp = *dpp;
      const size_t bytes = std::min<size_t>(s->layout.words.size() * 8, (size_t)dp.accessPolicyMaxWindowSize);
      size_t cur = 0;
      cudaDeviceGetLimit(&cur, cudaLimitPersistingL2CacheSize);
      const size_t want = std::min<size_t>((size_t)dp.persistingL2CacheMaxSize, std::max<size_t>(bytes * 2, 4u << 20));
      if (cur < want) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want);
      cudaStreamAttrValue av;
      memset(&av, 0, sizeof(av));
      av.accessPolicyWindow.base_ptr = (void*)P.words;
      av.accessPolicyWindow.num_bytes = bytes;
      av.accessPolicyWindow.hitRatio = 1.0f;
      av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      av.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
      cudaStreamSetAttribute(s->stream, cudaStreamAttributeAccessPolicyWindow, &av);
      cudaGetLastError();
    }
  }

  // II. number of subproblems (barebones :548-555), generalised to the GPU count (SURVEY §8e)
  int d = opt.subproblems_power;
  if (d < 0) {
    d = 0;
    // (per block up to 4 blocks per SM: the single-warp blocks of the small networks come 24 to an SM, and a dive per
    // subproblem is what a small search tree then mostly consists of - pat10: 30 M nodes for 2^21 subproblems, 7.5 M for
    // 2^19; the blocks that run out of subproblems split the ones that are left, see tail splitting)
    const unsigned long long per_gpu = (unsigned long long)std::min(s->num_blocks, 4 * s->num_sms);
    const unsigned long long want = (unsigned long long)opt.subproblems_factor * per_gpu * (unsigned long long)opt.gpu_world;
    while ((1ull << d) < want && d < 62) ++d;
  }
  pt.mark("streams, L2 window");
  if (d > TB_K_BITS) d = TB_K_BITS;          // the dispenser word keeps its high bits for the epoch
  P.subproblems_power = d;
  P.num_subproblems = 1ull << d;
  *out = s;
  return TB_OK;
}

extern "C" void tb_destroy(tb_solver* s) {
  if (!s) return;
  PhaseTimer pt("tb_destroy");
  cudaSetDevice(s->device);
  for (void* h : s->ipc_opened) cudaIpcCloseMemHandle(h);
  pt.mark("ipc close");
  if (s->stream) cudaStreamSynchronize(s->stream);
  pt.mark("stream sync");
  for (void* p : s->allocs) cudaFreeAsync(p, (cudaStream_t)0);     // back to the pool, which keeps it
  pt.mark("free async");
  release_cells(s->device, s->d_cells);
  cudaGetLastError();
  if (s->poll_stream) cudaStreamDestroy(s->poll_stream);
  if (s->h_stream_rec) cudaFreeHost(s->h_stream_rec);
  if (s->h_stream_img) cudaFreeHost(s->h_stream_img);
  if (s->stream) cudaStreamDestroy(s->stream);
  if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
  if (s->ev_start) cudaEventDestroy(s->ev_start);
  if (s->ev_stop) cudaEventDestroy(s->ev_stop);
  pt.mark("streams, events");
  delete s;
  pt.mark("delete");
}

static void fill_config(const tb_solver* s, tb_stats* st) {
  st->num_blocks = s->num_blocks; st->threads_per_block = s->threads; st->mem_kind = s->mem_kind;
  st->cluster_size = s->cluster; st->subproblems_power = s->P.subproblems_power; st->blocks_per_sm = s->blocks_per_sm;
  st->shared_bytes = s->shared_bytes; st->store_bytes = s->store_bytes; st->prop_bytes = s->prop_bytes;
  st->eps_num_subproblems = s->P.num_subproblems;
  st->device_bytes = s->device_bytes;
  st->fixpoint_in_effect = (s->P.fixpoint_kind == TB_FP_AC1 ? TB_FP_AC1 : TB_FP_WAC1) + (s->active ? 2 : 0);
}

// ---- intermediate solutions (-i / -a; SURVEY 8f.3, gpu_dive_and_solve.hpp:100-132) ---------------------------------
extern "C" tb_status tb_stream_solutions(tb_solver* s, int32_t slots) {
  if (!s || slots < 0 || slots > TB_STREAM_MAX_SLOTS) { set_error("tb_stream_solutions: slots must be within 0..64"); return TB_ERR_INVALID; }
  CU(cudaSetDevice(s->device));
  std::lock_guard<std::mutex> lock(s->poll_mutex);
  if (slots == 0) { s->P.stream_slots = 0; return TB_OK; }
  if (s->h_stream_rec) { set_error("tb_stream_solutions: already enabled"); return TB_ERR_INVALID; }
  tb_status rc;
  if ((rc = dev_alloc(s, &s->P.stream_img, (size_t)slots * 2 * (size_t)s->P.vpad))) return rc;
  if ((rc = dev_alloc(s, &s->P.stream_lock, (size_t)TB_STREAM_MAX_SLOTS))) return rc;
  CU(cudaMemset(s->P.stream_lock, 0, sizeof(int) * TB_STREAM_MAX_SLOTS));
  CU(cudaHostAlloc((void**)&s->h_stream_rec, sizeof(StreamRec) * (size_t)slots, cudaHostAllocMapped | cudaHostAllocPortable));
  CU(cudaHostAlloc((void**)&s->h_stream_img, sizeof(int) * 2 * (size_t)s->P.vpad, cudaHostAllocPortable));
  memset(s->h_stream_rec, 0, sizeof(StreamRec) * (size_t)slots);
  StreamRec* dptr = nullptr;
  CU(cudaHostGetDevicePointer((void**)&dptr, s->h_stream_rec, 0));
  CU(cudaStreamCreateWithFlags(&s->poll_stream, cudaStreamNonBlocking));
  s->P.stream_rec = dptr;
  s->P.stream_slots = slots;
  s->stream_read = 0;
  return TB_OK;
}

extern "C" int32_t tb_poll_solution(tb_solver* s, int32_t* lb, int32_t* ub, int32_t* objective, int64_t* time_ns) {
  if (!s || !lb || !ub) { set_error("null argument"); return -TB_ERR_INVALID; }
  std::lock_guard<std::mutex> lock(s->poll_mutex);
  if (!s->P.stream_slots || !s->h_stream_rec) return 0;
  if (cudaSetDevice(s->device) != cudaSuccess) { set_error("cudaSetDevice failed"); return -TB_ERR_CUDA; }
  for (int attempt = 0; attempt < 4; ++attempt) {
    // the oldest record not handed out yet (solutions come out in the order they were found)
    int best = -1; unsigned long long best_seq = ~0ull;
    for (int i = 0; i < s->P.stream_slots; ++i) {
      const unsigned long long q = *(volatile unsigned long long*)&s->h_stream_rec[i].seq;
      if (q > s->stream_read && q < best_seq) { best_seq = q; best = i; }
    }
    if (best < 0) return 0;
    StreamRec rec;
    memcpy(&rec, (const void*)&s->h_stream_rec[best], sizeof(rec));
    const size_t bytes = sizeof(int) * 2 * (size_t)s->P.vpad;
    if (cudaMemcpyAsync(s->h_stream_img, s->P.stream_img + (size_t)best * 2 * s->P.vpad, bytes, cudaMemcpyDeviceToHost, s->poll_stream) != cudaSuccess ||
        cudaStreamSynchronize(s->poll_stream) != cudaSuccess) { set_error("tb_poll_solution: copy failed"); cudaGetLastError(); return -TB_ERR_CUDA; }
    // the slot may have been rewritten while it was being copied: then look again
    if (*(volatile unsigned long long*)&s->h_stream_rec[best].seq != best_seq) continue;
    unpack_store(s, s->h_stream_img, lb, ub);
    if (objective) *objective = rec.objective;
    if (time_ns) *time_ns = rec.t_ns;
    s->stream_read = best_seq;
    return 1;
  }
  return 0;
}

extern "C" tb_status tb_set_timeout(tb_solver* s, uint64_t timeout_ms) {
  if (!s) { set_error("null solver"); return TB_ERR_INVALID; }
  s->opt.timeout_ms = timeout_ms;
  return TB_OK;
}

extern "C" tb_status tb_get_config(tb_solver* s, tb_stats* st) {
  if (!s || !st) { set_error("null argument"); return TB_ERR_INVALID; }
  memset(st, 0, sizeof(*st));
  st->exhaustive = 1;
  fill_config(s, st);
  return TB_OK;
}

static tb_status reset_stats(tb_solver* s, int slots) {
  std::vector<BlockStats> z((size_t)slots);
  memset(z.data(), 0, z.size() * sizeof(BlockStats));
  for (auto& b : z) { b.exhaustive = 1; b.best_bound = TBD_PINF; }
  CU(cudaMemcpyAsync(s->P.stats, z.data(), z.size() * sizeof(BlockStats), cudaMemcpyHostToDevice, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  return TB_OK;
}

// Sum the per-block statistics (reduce_blocks, barebones :1033-1067, done on the host: B is small).
static void reduce_stats(const std::vector<BlockStats>& bs, tb_stats* st, int* best_block) {
  int best = -1; int best_bound = TBD_PINF; long long best_time = 0;
  long long first_idle = -1;
  for (size_t i = 0; i < bs.size(); ++i) {
    const BlockStats& b = bs[i];
    st->nodes += b.nodes; st->fails += b.fails; st->solutions += b.solutions;
    st->depth_max = std::max(st->depth_max, b.depth_max);
    st->exhaustive = st->exhaustive && b.exhaustive;
    st->eps_solved_subproblems += b.eps_solved; st->eps_skipped_subproblems += b.eps_skipped;
    st->eps_stolen_subproblems += b.eps_stolen;
    st->eps_split_subproblems += b.eps_split; st->eps_split_parts_solved += b.eps_parts;
    st->num_blocks_done += b.blocks_done;
    st->fixpoint_iterations += b.fixpoint_iterations; st->num_deductions += b.deductions;
    st->bounds_narrowed += b.narrowed;
    st->cumulative_time_block_ns += b.t_idle;
    st->timers_ns[TB_TIMER_FIXPOINT] += b.t_fixpoint;
    st->timers_ns[TB_TIMER_DIVE] += b.t_dive;
    st->timers_ns[TB_TIMER_SEARCH] += b.t_idle - b.t_fixpoint;
    if (first_idle < 0 || b.t_idle < first_idle) first_idle = b.t_idle;
    if (b.has_best) {
      if (best < 0 || b.best_bound < best_bound || (b.best_bound == best_bound && b.t_best <= best_time)) {
        best = (int)i; best_bound = b.best_bound; best_time = b.t_best;
      }
    }
  }
  st->timers_ns[TB_TIMER_FIRST_BLOCK_IDLE] = std::max<long long>(first_idle, 0);
  st->timers_ns[TB_TIMER_LATEST_BEST_OBJ_FOUND] = best >= 0 ? best_time : 0;
  if (best_block) *best_block = best;
}

// Position of lb[v] / ub[v] inside a store image: slot = layout.slot_of[v]; one {lb, ub} pair per slot, or
// cluster slices of vc pairs per CTA with slot s in CTA (s mod C) at local index (s div C).
static inline size_t img_lb(const tb_solver* s, int v) {
  const int sl = s->layout.slot_of[v];
  if (s->mem_kind == TB_MEM_STORE_CLUSTER) { const int c = s->cluster, vc = s->P.vc; return (size_t)(sl % c) * 2 * vc + 2 * (size_t)(sl / c); }
  return 2 * (size_t)sl;
}
static inline size_t img_ub(const tb_solver* s, int v) { return img_lb(s, v) + 1; }
static void unpack_store(const tb_solver* s, const int* img, int32_t* lb, int32_t* ub) {
  for (int v = 0; v < s->nvars; ++v) { lb[v] = img[img_lb(s, v)]; ub[v] = img[img_ub(s, v)]; }
}

static unsigned long long host_globaltimer_probe(tb_solver* s);

__global__ void read_globaltimer_kernel(unsigned long long* out) { *out = globaltimer_ns(); }

static unsigned long long host_globaltimer_probe(tb_solver* s) {
  unsigned long long* d = s->d_cells + TB_CELL_WORDS - 1;    // a spare word of the cell block
  read_globaltimer_kernel<<<1, 1, 0, s->stream>>>(d);
  unsigned long long h = 0;
  cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, s->stream);
  cudaStreamSynchronize(s->stream);
  return h;
}

static double now_ms() {
  struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t);
  return t.tv_sec * 1e3 + t.tv_nsec * 1e-6;
}

// What tb_solve and tb_solve_batch share: a new epoch, the grid cells and the split pool reset, the launch (`launch`
// starts the solve kernel on P), the poll loop on *stop_flag / the timeout (wait_solving_ends, memory_gpu.hpp:174-196)
// and the block statistics.
struct SearchRun {
  bool interrupted = false;          // the host raised the stop word (stop_flag or timeout)
  float kernel_ms = 0.f;
  std::vector<BlockStats> blocks;
};
template <class Launch>
static tb_status run_search(tb_solver* s, DevParams& P, double t_begin, volatile int32_t* stop_flag, Launch&& launch, SearchRun& run) {
  tb_status rc;
  if ((rc = reset_stats(s, s->num_blocks))) return rc;
  P.t_start = host_globaltimer_probe(s);
  // A new run = a new epoch (linked solvers make the same sequence of tb_solve calls, so their epochs agree): the
  // incumbent of the previous run, a late write of a peer that is still in it, a stale stop request are all void
  // without any reset protocol between the processes. The kernel enters the epoch into the incumbent cell itself.
  P.epoch = ++s->epoch;
  const int zero = 0;
  const unsigned long long first_free = ((unsigned long long)P.epoch << TB_K_BITS) | (unsigned long long)s->num_blocks;
  CU(cudaMemcpyAsync((int*)(s->d_cells + TB_CELL_STOP) + 1, &zero, sizeof(int), cudaMemcpyHostToDevice, s->stream));
  if (P.stream_slots) {
    std::lock_guard<std::mutex> lock(s->poll_mutex);
    const unsigned long long z = 0;
    CU(cudaMemcpyAsync(s->d_cells + TB_CELL_STREAM, &z, sizeof(z), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemsetAsync(s->P.stream_lock, 0, sizeof(int) * TB_STREAM_MAX_SLOTS, s->stream));
    memset(s->h_stream_rec, 0, sizeof(StreamRec) * (size_t)P.stream_slots);
    s->stream_read = 0;
  }
  if (P.split_bits) {
    CU(cudaMemsetAsync(P.split_ctl, 0, 8 * sizeof(unsigned), s->stream));
    CU(cudaMemsetAsync(P.split_pool, 0, sizeof(SplitEntry) * (size_t)TB_SPLIT_CAP, s->stream));
    const unsigned who[2] = {(unsigned)s->num_blocks, P.epoch};          // TB_SPLIT_NSLOTS, TB_SPLIT_EPOCH: written last
    CU(cudaMemcpyAsync(P.split_ctl + TB_SPLIT_NSLOTS, who, sizeof(who), cudaMemcpyHostToDevice, s->stream));
  }
  CU(cudaMemcpyAsync(s->d_cells + TB_CELL_NEXT, &first_free, sizeof(first_free), cudaMemcpyHostToDevice, s->stream));
  CU(cudaEventRecord(s->ev_start, s->stream));
  if ((rc = launch(P))) return rc;
  CU(cudaEventRecord(s->ev_stop, s->stream));
  while (true) {
    cudaError_t q = cudaEventQuery(s->ev_stop);
    if (q == cudaSuccess) break;
    if (q != cudaErrorNotReady) { set_error(std::string("kernel failed: ") + cudaGetErrorString(q)); return TB_ERR_CUDA; }
    bool must = (stop_flag && *stop_flag) || (s->opt.timeout_ms && now_ms() - t_begin >= (double)s->opt.timeout_ms);
    if (must && !run.interrupted) {
      run.interrupted = true;
      CU(cudaMemcpyAsync((int*)(s->d_cells + TB_CELL_STOP) + 1, s->h_pinned_one, sizeof(int), cudaMemcpyHostToDevice, s->copy_stream));
    }
    struct timespec ts = {0, 200000};
    nanosleep(&ts, nullptr);
  }
  CU(cudaStreamSynchronize(s->stream));
  CU(cudaEventElapsedTime(&run.kernel_ms, s->ev_start, s->ev_stop));
  run.blocks.resize((size_t)s->num_blocks);
  CU(cudaMemcpy(run.blocks.data(), P.stats, run.blocks.size() * sizeof(BlockStats), cudaMemcpyDeviceToHost));
  return TB_OK;
}

extern "C" tb_status tb_solve(tb_solver* s, volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                              int32_t* has_solution, int32_t* exhaustive, tb_stats* stats) {
  if (!s) { set_error("null solver"); return TB_ERR_INVALID; }
  CU(cudaSetDevice(s->device));
  DevParams& P = s->P;
  const double t_begin = now_ms();
  SearchRun run;
  tb_status rc = run_search(s, P, t_begin, stop_flag, [&](const DevParams& Pl) {
    return dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
      CU(launch_workers(s, solve_kernel<decltype(M)::value, decltype(A)::value, decltype(TM)::value>, s->num_blocks, Pl));
      CU(cudaGetLastError());
      return TB_OK;
    });
  }, run);
  if (rc) return rc;
  const std::vector<BlockStats>& bs = run.blocks;
  tb_stats st; memset(&st, 0, sizeof(st));
  st.exhaustive = 1;
  fill_config(s, &st);
  int best_block = -1;
  reduce_stats(bs, &st, &best_block);
  for (auto& b : bs) if (b.error) { set_error("decision stack overflow (raise max_depth)"); rc = (tb_status)b.error; }
  if (run.interrupted) st.exhaustive = 0;
  st.kernel_ms = run.kernel_ms;
  st.timers_ns[TB_TIMER_OVERALL] = (int64_t)((now_ms() - t_begin) * 1e6);
  if (has_solution) *has_solution = best_block >= 0;
  s->last_lb.assign((size_t)std::max(1, s->nvars), 0); s->last_ub.assign((size_t)std::max(1, s->nvars), 0);
  if (best_block >= 0) {
    std::vector<int> img((size_t)2 * P.vpad);
    CU(cudaMemcpy(img.data(), P.block_best + (size_t)best_block * 2 * P.vpad, img.size() * sizeof(int), cudaMemcpyDeviceToHost));
    unpack_store(s, img.data(), s->last_lb.data(), s->last_ub.data());
    if (best_lb && best_ub && s->nvars) { memcpy(best_lb, s->last_lb.data(), (size_t)s->nvars * 4); memcpy(best_ub, s->last_ub.data(), (size_t)s->nvars * 4); }
  }
  if (exhaustive) *exhaustive = st.exhaustive;
  if (stats) *stats = st;
  s->last_stats = st; s->last_has = best_block >= 0; s->last_exhaustive = st.exhaustive; s->last_valid = 1;
  return rc;
}

static tb_status ensure_batch_buffers(tb_solver* s, size_t nimages, size_t nroots, size_t ngroups, size_t nbest,
                                      size_t nquery, size_t nwit) {
  tb_status rc;
  const size_t img = (size_t)2 * s->P.vpad;
  if (nimages > s->batch_images_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_roots, nimages * img))) return rc;
    s->batch_images_cap = nimages;
  }
  if (nroots > s->batch_roots_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_state, nroots))) return rc;
    s->batch_roots_cap = nroots;
  }
  if (ngroups > s->batch_groups_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_groups, ngroups))) return rc;
    s->batch_groups_cap = ngroups;
  }
  if (nbest > s->batch_best_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_best, nbest * img))) return rc;
    s->batch_best_cap = nbest;
  }
  if (nquery > s->batch_query_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_query, nquery))) return rc;
    s->batch_query_cap = nquery;
  }
  if (nwit > s->batch_wit_cap) {
    if ((rc = dev_alloc(s, &s->d_batch_wit, nwit * img))) return rc;
    s->batch_wit_cap = nwit;
  }
  return TB_OK;
}

// The fixing of tb_solve_supports and tb_solve_front: group g narrows variable var[g] to [lo[g], hi[g]] in every root
// (a query's value; a level's slice of x). A root whose box's range of that variable misses the interval is decided on
// the host, as an empty box is. `front` (tb_solve_front: 1 = the front minimises x, 2 = it maximises x; 0 = none):
// every group narrows x, its level is hi[g] (lo[g]), a solution is a witness for every level it reaches, and each
// returned row also has x fixed to the best value the row allows on the level's side.
struct GroupFixing {
  const int32_t *var, *lo, *hi;
  int front;
};

// tb_solve_supports's part of solve_groups. The groups fix one variable each (GroupFixing, lo = hi = the value) and are
// sorted by (slot, value), so their values are the value list of the CSR over the queried slots qslot / qoff.
// Solutions go to a pool of wit_cap rows (*nwit of them written, wit_lb / wit_ub [wit_cap][nvars]); wit_of [ngroups]
// receives each group's row (-1 = none).
struct SupportQueries {
  std::vector<int32_t> qslot, qoff;
  int32_t wit_cap;
  int32_t *wit_lb, *wit_ub, *nwit, *wit_of;
};

// The one host path of the BATCH kernel: tb_solve_groups, tb_solve_batch, tb_solve_objectives, tb_solve_supports and
// tb_solve_front. `nimages` boxes (box_lb / box_ub [nimages][nvars]); root r searches box image_of[r] for group
// group_of[r] (nroots entries); group g optimises variable obj_of[g] (-1 = satisfaction) in the sense maximize[g]
// (ngroups entries). `objectives` (tb_solve_objectives, tb_solve_front): every solution is a witness for every group
// (for the groups whose level it reaches, with a front `fix`), each returned row has the group's objective variable
// fixed to its value, and an unbounded objective is never exhaustive. `fix`: each group's fixing (GroupFixing).
// `sup` (tb_solve_supports, with `fix`): every group is a satisfaction group with one variable fixed, every solution is
// a witness for every group it holds, and there are no best rows (best_lb / best_ub / objective are NULL), only the
// witness pool. `fn` names the entry point in errors.
static tb_status solve_groups(tb_solver* s, const char* fn, int32_t nimages, const int32_t* box_lb, const int32_t* box_ub,
                              long long nroots, const int32_t* image_of, const int32_t* group_of, int32_t ngroups,
                              const int32_t* obj_of, const int32_t* maximize, bool objectives, const GroupFixing* fix,
                              const SupportQueries* sup, volatile int32_t* stop_flag, int32_t* best_lb,
                              int32_t* best_ub, int32_t* has_solution, int32_t* exhaustive, int32_t* objective,
                              tb_stats* stats) {
  const std::string name(fn);
  if (!s || nimages < 1 || nroots < 1 || ngroups < 1 || !group_of || (s->nvars && (!box_lb || !box_ub))) {
    set_error(name + ": needs nroots >= 1, ngroups >= 1, root_lb / root_ub and group_of"); return TB_ERR_INVALID;
  }
  if (!s->peer_cells.empty() || s->opt.gpu_world > 1) { set_error(name + ": a batch runs on one GPU (linked or sharded solvers are not supported)"); return TB_ERR_UNSUPPORTED; }
  if (s->mem_kind == TB_MEM_STORE_CLUSTER) { set_error(name + ": the STORE_CLUSTER placement is not supported"); return TB_ERR_UNSUPPORTED; }
  if (s->P.stream_slots) { set_error(name + ": intermediate solutions (tb_stream_solutions) are not supported"); return TB_ERR_UNSUPPORTED; }
  // the subproblem index (r << d) | local is counted by the dispenser's TB_K_BITS field
  if ((unsigned long long)nroots > (1ull << TB_K_BITS)) {
    set_error(name + ": " + std::to_string(nroots) + " roots do not fit the subproblem index (at most 2^40)"); return TB_ERR_INVALID;
  }
  std::vector<char> has_root((size_t)ngroups, 0);
  for (long long r = 0; r < nroots; ++r) {
    if (group_of[r] < 0 || group_of[r] >= ngroups) {
      set_error(name + ": root " + std::to_string(r) + " names group " + std::to_string(group_of[r]) + ", outside [0, ngroups)");
      return TB_ERR_INVALID;
    }
    has_root[(size_t)group_of[r]] = 1;
  }
  for (int32_t g = 0; g < ngroups; ++g)
    if (!has_root[(size_t)g]) { set_error(name + ": group " + std::to_string(g) + " has no root"); return TB_ERR_INVALID; }
  // Every box narrows the solver's root: the layout pass chose each propagator's device class (folded constants, exact
  // 32-bit arithmetic) from the root bounds, which stays valid under narrowing only.
  const size_t nv = (size_t)s->nvars;
  for (size_t r = 0; r < (size_t)nimages; ++r)
    for (size_t v = 0; v < nv; ++v)
      if (box_lb[r * nv + v] < s->root_lb[v] || box_ub[r * nv + v] > s->root_ub[v]) {
        set_error(name + ": root " + std::to_string(r) + " widens the solver's domain of variable " + std::to_string(v));
        return TB_ERR_INVALID;
      }
  CU(cudaSetDevice(s->device));
  const double t_begin = now_ms();
  // subproblems per root: -sub -1 is the tb_create rule with the roots folded in; the index (r << d) | local must fit
  // the dispenser's TB_K_BITS
  int d = s->opt.subproblems_power;
  if (d < 0) {
    d = 0;
    const unsigned long long want = (unsigned long long)s->opt.subproblems_factor * (unsigned long long)std::min(s->num_blocks, 4 * s->num_sms);
    while (((unsigned long long)nroots << d) < want && d < TB_K_BITS) ++d;
  }
  while (d > 0 && ((unsigned long long)nroots << d) > (1ull << TB_K_BITS)) --d;
  int root_bits = 0;
  while ((1ull << root_bits) < (unsigned long long)nroots) ++root_bits;
  tb_status rc;
  // (tb_solve_supports: no best row per group - the groups may be many more than the solutions - only the pool)
  const size_t nqslots = sup ? sup->qslot.size() : 0;
  const size_t nquery = sup ? 1 + nqslots + (nqslots + 1) + (size_t)ngroups : 0;
  if ((rc = ensure_batch_buffers(s, (size_t)nimages, (size_t)nroots, (size_t)ngroups, sup ? 0 : (size_t)ngroups, nquery,
                                 sup ? (size_t)sup->wit_cap : 0))) return rc;
  DevParams P = s->P;
  const size_t img = (size_t)2 * P.vpad;
  // box images in the slot layout; a box with an empty referenced variable fails before any search, as tb_solve's
  // root does: the subproblems of its roots are skipped, and their groups go on with their other roots
  std::vector<int> images((size_t)nimages * img, 0);
  std::vector<char> empty((size_t)nimages, 0);
  for (size_t r = 0; r < (size_t)nimages; ++r) {
    int* im = images.data() + r * img;
    for (size_t v = 0; v < nv; ++v) {
      const int l = box_lb[r * nv + v], u = box_ub[r * nv + v];
      im[img_lb(s, (int)v)] = l; im[img_ub(s, (int)v)] = u;
      if (l > u && s->layout.referenced[v]) empty[r] = 1;
    }
  }
  std::vector<BatchRoot> state((size_t)nroots);
  for (size_t r = 0; r < (size_t)nroots; ++r) {
    BatchRoot& b = state[r];
    memset(&b, 0, sizeof(b));
    b.group = group_of[r];
    b.image = image_of[r];
    b.skip = empty[(size_t)b.image];
    if (fix) {                                         // (a fixing that misses the box: decided on the host, as empty)
      const size_t at = (size_t)b.image * nv + (size_t)fix->var[b.group];
      b.skip |= std::max(fix->lo[b.group], box_lb[at]) > std::min(fix->hi[b.group], box_ub[at]);
    }
  }
  std::vector<BatchGroup> groups((size_t)ngroups);
  for (size_t g = 0; g < (size_t)ngroups; ++g) {
    BatchGroup& G = groups[g];
    memset(&G, 0, sizeof(G));
    G.bound = ~0ull;                                   // epoch 0, no incumbent (as the cell at tb_create)
    G.img_bound = TBD_PINF;
    G.obj = obj_of[g] >= 0 ? s->layout.slot_of[obj_of[g]] : -1;
    G.maximize = maximize[g];
    G.fix = fix ? s->layout.slot_of[fix->var[g]] : -1;
    G.fix_lo = fix ? fix->lo[g] : 0;
    G.fix_hi = fix ? fix->hi[g] : 0;
    G.wit = -1;
  }
  CU(cudaMemcpyAsync(s->d_batch_roots, images.data(), images.size() * sizeof(int), cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemcpyAsync(s->d_batch_state, state.data(), state.size() * sizeof(BatchRoot), cudaMemcpyHostToDevice, s->stream));
  CU(cudaMemcpyAsync(s->d_batch_groups, groups.data(), groups.size() * sizeof(BatchGroup), cudaMemcpyHostToDevice, s->stream));
  P.batch_roots = s->d_batch_roots; P.batch_best = s->d_batch_best; P.batch_state = s->d_batch_state;
  P.batch_groups = s->d_batch_groups;
  P.batch_share = objectives && ngroups > 1 ? ngroups : 0;   // (one objective has nobody to share with)
  P.batch_nqslots = (int)nqslots;
  P.batch_front = fix ? fix->front : 0;
  P.batch_front_x = fix && fix->front ? s->layout.slot_of[fix->var[0]] : 0;
  if (sup) {
    // the query table: the pool's row counter (0), then qslot, qoff and the values
    std::vector<int32_t> q(nquery, 0);
    std::copy(sup->qslot.begin(), sup->qslot.end(), q.begin() + 1);
    std::copy(sup->qoff.begin(), sup->qoff.end(), q.begin() + 1 + nqslots);
    std::copy(fix->lo, fix->lo + ngroups, q.begin() + 1 + 2 * nqslots + 1);
    CU(cudaMemcpyAsync(s->d_batch_query, q.data(), q.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s->stream));
    P.batch_wit_n = (unsigned*)s->d_batch_query;
    P.batch_qslot = s->d_batch_query + 1;
    P.batch_qoff = P.batch_qslot + nqslots;
    P.batch_qval = P.batch_qoff + nqslots + 1;
    P.batch_wit = s->d_batch_wit;
    P.batch_wit_cap = sup->wit_cap;
    P.batch_best = nullptr;
  }
  P.subproblems_power = d;
  P.num_subproblems = (unsigned long long)nroots << d;
  P.batch_max_depth = std::min(TB_BATCH_WEIGHT_BITS, 64 - root_bits);
  // (the BATCH kernel has the registers of the others - __launch_bounds__ caps them all - and a few bytes more of
  // static shared memory, which the 64 bytes configure() reserves beside Ctl cover: the grid of tb_create fits)
  rc = dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
    if constexpr (decltype(M)::value != TB_MEM_STORE_CLUSTER) {
      if (s->shared_bytes)
        CU(cudaFuncSetAttribute(solve_kernel<decltype(M)::value, decltype(A)::value, decltype(TM)::value, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->shared_bytes));
    }
    return TB_OK;
  });
  if (rc) return rc;
  SearchRun run;
  rc = run_search(s, P, t_begin, stop_flag, [&](const DevParams& Pl) {
    return dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
      if constexpr (decltype(M)::value == TB_MEM_STORE_CLUSTER) { set_error(name + ": STORE_CLUSTER"); return TB_ERR_UNSUPPORTED; }
      else {
        CU(launch_workers(s, solve_kernel<decltype(M)::value, decltype(A)::value, decltype(TM)::value, true>, s->num_blocks, Pl));
        CU(cudaGetLastError());
        return TB_OK;
      }
    });
  }, run);
  if (rc) return rc;
  CU(cudaMemcpy(state.data(), s->d_batch_state, state.size() * sizeof(BatchRoot), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(groups.data(), s->d_batch_groups, groups.size() * sizeof(BatchGroup), cudaMemcpyDeviceToHost));
  bool any = false;
  for (auto& g : groups) any |= g.has != 0 && !sup;
  std::vector<int> best(any ? (size_t)ngroups * img : 0);
  if (any) CU(cudaMemcpy(best.data(), s->d_batch_best, best.size() * sizeof(int), cudaMemcpyDeviceToHost));
  tb_stats st; memset(&st, 0, sizeof(st));
  st.exhaustive = 1;
  fill_config(s, &st);
  st.subproblems_power = d;
  st.eps_num_subproblems = P.num_subproblems;
  reduce_stats(run.blocks, &st, nullptr);
  for (auto& b : run.blocks) if (b.error) { set_error("decision stack overflow (raise max_depth)"); rc = (tb_status)b.error; }
  // per root: exhausted iff all of its search space was closed and no block was cut while searching it (roots that
  // finished before a stop or a timeout stay exhausted); a skipped root is exhausted without a solution. A group is
  // exhaustive iff all of its roots are.
  const unsigned long long all = 1ull << TB_BATCH_WEIGHT_BITS;
  std::vector<int> exh((size_t)ngroups, 1);
  for (const BatchRoot& b : state) exh[(size_t)b.group] &= b.skip ? 1 : (b.closed == all && !b.cut);
  int all_exhaustive = 1;
  std::vector<int32_t> lb(std::max<size_t>(1, nv)), ub(std::max<size_t>(1, nv));
  for (size_t g = 0; g < (size_t)ngroups; ++g) {
    const bool has = groups[g].has != 0;
    const int x = obj_of[g];
    if (has && !sup) {
      unpack_store(s, best.data() + g * img, lb.data(), ub.data());
      // the value is lb(x) of the best store when minimising, ub(x) when maximising; tb_solve_objectives returns the
      // point's side: x fixed to that value (a sub-box of an entailed box is entailed)
      if (objectives) {
        const int val = maximize[g] ? ub[(size_t)x] : lb[(size_t)x];
        lb[(size_t)x] = ub[(size_t)x] = val;
        if (val == (maximize[g] ? TB_POS_INF : TB_NEG_INF)) exh[g] = 0;     // unbounded: the objective ended there
      }
      // tb_solve_front: x at the best value of the row, which is on the level's side: the row is the group's own
      // solution, inside its slice, or a witness, whose x reaches the level (batch_share_witness)
      if (fix && fix->front) {
        const size_t xv = (size_t)fix->var[g];
        if (fix->front == 1) ub[xv] = lb[xv]; else lb[xv] = ub[xv];
      }
    }
    all_exhaustive &= exh[g];
    if (has_solution) has_solution[g] = has;
    if (exhaustive) exhaustive[g] = exh[g];
    if (objective) objective[g] = TB_POS_INF;
    if (!has) continue;
    if (objective && x >= 0) objective[g] = maximize[g] ? ub[(size_t)x] : lb[(size_t)x];
    if (best_lb && nv) memcpy(best_lb + g * nv, lb.data(), nv * 4);
    if (best_ub && nv) memcpy(best_ub + g * nv, ub.data(), nv * 4);
  }
  if (sup) {
    for (size_t g = 0; g < (size_t)ngroups; ++g) sup->wit_of[g] = groups[g].has && groups[g].wit >= 0 ? groups[g].wit : -1;
    unsigned taken = 0;
    CU(cudaMemcpy(&taken, s->d_batch_query, sizeof(unsigned), cudaMemcpyDeviceToHost));
    const size_t rows = std::min<size_t>(taken, (size_t)sup->wit_cap);
    std::vector<int> pool(rows * img);
    if (rows) CU(cudaMemcpy(pool.data(), s->d_batch_wit, pool.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (size_t w = 0; w < rows && nv; ++w) unpack_store(s, pool.data() + w * img, sup->wit_lb + w * nv, sup->wit_ub + w * nv);
    if (sup->nwit) *sup->nwit = (int32_t)rows;
  }
  st.exhaustive = all_exhaustive;
  st.kernel_ms = run.kernel_ms;
  st.timers_ns[TB_TIMER_OVERALL] = (int64_t)((now_ms() - t_begin) * 1e6);
  if (stats) *stats = st;
  return rc;
}

// tb_solve_objectives, tb_solve_supports and tb_solve_front: group g's root g * nboxes + r searches box r
static void roots_per_box(int32_t nboxes, long long nroots, std::vector<int32_t>& image_of, std::vector<int32_t>& group_of) {
  image_of.resize((size_t)nroots);
  group_of.resize((size_t)nroots);
  for (size_t i = 0; i < (size_t)nroots; ++i) { image_of[i] = (int32_t)(i % (size_t)nboxes); group_of[i] = (int32_t)(i / (size_t)nboxes); }
}

// tb_solve_groups and tb_solve_batch: one root per box, every group optimises the problem's objective
static tb_status solve_boxes(tb_solver* s, const char* fn, int32_t nroots, const int32_t* root_lb, const int32_t* root_ub,
                             const int32_t* group_of, int32_t ngroups, volatile int32_t* stop_flag, int32_t* best_lb,
                             int32_t* best_ub, int32_t* has_solution, int32_t* exhaustive, int32_t* objective,
                             tb_stats* stats) try {
  std::vector<int32_t> own((size_t)std::max(0, nroots));
  for (size_t r = 0; r < own.size(); ++r) own[r] = (int32_t)r;
  const int32_t obj = s ? s->root_obj_var : -1;
  std::vector<int32_t> obj_of((size_t)std::max(0, ngroups), obj), minimize((size_t)std::max(0, ngroups), 0);
  return solve_groups(s, fn, nroots, root_lb, root_ub, nroots, own.data(), group_of ? group_of : own.data(), ngroups,
                      obj_of.data(), minimize.data(), false, nullptr, nullptr, stop_flag, best_lb, best_ub, has_solution, exhaustive,
                      objective, stats);
} catch (const std::bad_alloc&) {             // (the per-root host arrays: nothing may unwind through the C ABI)
  set_error(std::string(fn) + ": out of host memory for the roots");
  return TB_ERR_NOMEM;
}

extern "C" tb_status tb_solve_groups(tb_solver* s, int32_t nroots, const int32_t* root_lb, const int32_t* root_ub,
                                     const int32_t* group_of, int32_t ngroups, volatile int32_t* stop_flag,
                                     int32_t* best_lb, int32_t* best_ub, int32_t* has_solution, int32_t* exhaustive,
                                     int32_t* objective, tb_stats* stats) {
  if (!group_of) { set_error("tb_solve_groups: needs nroots >= 1, ngroups >= 1, root_lb / root_ub and group_of"); return TB_ERR_INVALID; }
  return solve_boxes(s, "tb_solve_groups", nroots, root_lb, root_ub, group_of, ngroups, stop_flag, best_lb, best_ub,
                     has_solution, exhaustive, objective, stats);
}

extern "C" tb_status tb_solve_batch(tb_solver* s, int32_t nroots, const int32_t* root_lb, const int32_t* root_ub,
                                    volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                                    int32_t* has_solution, int32_t* exhaustive, int32_t* objective, tb_stats* stats) {
  return solve_boxes(s, "tb_solve_batch", nroots, root_lb, root_ub, nullptr, nroots, stop_flag, best_lb, best_ub,
                     has_solution, exhaustive, objective, stats);
}

extern "C" tb_status tb_solve_objectives(tb_solver* s, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                                         int32_t nobj, const int32_t* obj_var, const int32_t* maximize,
                                         volatile int32_t* stop_flag, int32_t* best_lb, int32_t* best_ub,
                                         int32_t* has_solution, int32_t* exhaustive, int32_t* objective, tb_stats* stats) {
  const std::string name("tb_solve_objectives");
  if (!s || nboxes < 1 || nobj < 1 || !obj_var || !maximize) {
    set_error(name + ": needs nboxes >= 1, nobj >= 1, obj_var and maximize"); return TB_ERR_INVALID;
  }
  for (int32_t m = 0; m < nobj; ++m) {
    if (obj_var[m] < 0 || obj_var[m] >= s->nvars) {
      set_error(name + ": objective " + std::to_string(m) + " names variable " + std::to_string(obj_var[m]) + ", outside [0, nvars)");
      return TB_ERR_INVALID;
    }
    if (maximize[m] != 0 && maximize[m] != 1) {
      set_error(name + ": maximize[" + std::to_string(m) + "] is neither 0 nor 1"); return TB_ERR_INVALID;
    }
  }
  const long long nroots = (long long)nobj * nboxes;
  if ((unsigned long long)nroots > (1ull << TB_K_BITS)) {     // (before the per-root arrays are allocated)
    set_error(name + ": nobj * nboxes = " + std::to_string(nroots) + " roots do not fit the subproblem index (at most 2^40)");
    return TB_ERR_INVALID;
  }
  // objective m is group m
  try {
    std::vector<int32_t> image_of, group_of;
    roots_per_box(nboxes, nroots, image_of, group_of);
    return solve_groups(s, "tb_solve_objectives", nboxes, box_lb, box_ub, nroots, image_of.data(), group_of.data(), nobj,
                        obj_var, maximize, true, nullptr, nullptr, stop_flag, best_lb, best_ub, has_solution, exhaustive,
                        objective, stats);
  } catch (const std::bad_alloc&) {           // (the per-root host arrays: nothing may unwind through the C ABI)
    set_error(name + ": out of host memory for " + std::to_string(nroots) + " roots");
    return TB_ERR_NOMEM;
  }
}

extern "C" tb_status tb_solve_supports(tb_solver* s, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                                       int32_t nq, const int32_t* q_var, const int32_t* q_val,
                                       volatile int32_t* stop_flag, int32_t* supported, int32_t* witness,
                                       int32_t wit_cap, int32_t* wit_lb, int32_t* wit_ub, int32_t* nwit,
                                       tb_stats* stats) {
  const std::string name("tb_solve_supports");
  if (!s || nboxes < 1 || nq < 1 || !q_var || !q_val || !supported) {
    set_error(name + ": needs nboxes >= 1, nq >= 1, q_var, q_val and supported"); return TB_ERR_INVALID;
  }
  if (wit_cap < 0 || (wit_cap > 0 && (!wit_lb || !wit_ub))) {
    set_error(name + ": needs wit_cap >= 0, and wit_lb / wit_ub when wit_cap > 0"); return TB_ERR_INVALID;
  }
  for (int32_t i = 0; i < nq; ++i) {
    if (q_var[i] < 0 || q_var[i] >= s->nvars) {
      set_error(name + ": query " + std::to_string(i) + " names variable " + std::to_string(q_var[i]) + ", outside [0, nvars)");
      return TB_ERR_INVALID;
    }
    if (q_val[i] == TB_NEG_INF || q_val[i] == TB_POS_INF) {
      set_error(name + ": query " + std::to_string(i) + " asks for an infinite value"); return TB_ERR_INVALID;
    }
  }
  const long long nqroots = (long long)nq * nboxes;
  if ((unsigned long long)nqroots > (1ull << TB_K_BITS)) {    // (before the per-root arrays are allocated)
    set_error(name + ": nq * nboxes = " + std::to_string(nqroots) + " roots do not fit the subproblem index (at most 2^40)");
    return TB_ERR_INVALID;
  }
  try {
    // the distinct queries sorted by (slot, value): group g is the g-th of them, and its values are the CSR's
    std::vector<int32_t> order((size_t)nq);
    for (int32_t i = 0; i < nq; ++i) order[(size_t)i] = i;
    auto key = [&](int32_t i) { return std::make_pair(s->layout.slot_of[q_var[i]], q_val[i]); };
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return key(a) < key(b); });
    std::vector<int32_t> group_of_query((size_t)nq), fix_var, fix_val;
    SupportQueries sup;
    for (int32_t i : order) {
      if (fix_var.empty() || key(i) != std::make_pair(s->layout.slot_of[fix_var.back()], fix_val.back())) {
        if (sup.qslot.empty() || sup.qslot.back() != key(i).first) {
          sup.qslot.push_back(key(i).first);
          sup.qoff.push_back((int32_t)fix_var.size());
        }
        fix_var.push_back(q_var[i]); fix_val.push_back(q_val[i]);
      }
      group_of_query[(size_t)i] = (int32_t)fix_var.size() - 1;
    }
    sup.qoff.push_back((int32_t)fix_var.size());
    const int32_t ngroups = (int32_t)fix_var.size();
    const GroupFixing fix{fix_var.data(), fix_val.data(), fix_val.data(), 0};
    sup.wit_cap = wit_cap; sup.wit_lb = wit_lb; sup.wit_ub = wit_ub; sup.nwit = nwit;
    std::vector<int32_t> wit_of((size_t)ngroups, -1);
    sup.wit_of = wit_of.data();
    const long long nroots = (long long)ngroups * nboxes;
    std::vector<int32_t> image_of, group_of, obj_of((size_t)ngroups, -1), maximize((size_t)ngroups, 0),
        has((size_t)ngroups), exh((size_t)ngroups);
    roots_per_box(nboxes, nroots, image_of, group_of);
    if (nwit) *nwit = 0;
    const tb_status rc = solve_groups(s, "tb_solve_supports", nboxes, box_lb, box_ub, nroots, image_of.data(),
                                      group_of.data(), ngroups, obj_of.data(), maximize.data(), false, &fix, &sup,
                                      stop_flag, nullptr, nullptr, has.data(), exh.data(), nullptr, stats);
    if (rc != TB_OK && rc != TB_ERR_DEPTH) return rc;
    // 1: a solution holds the value; 0: every root of the query was searched to its end uncut or decided on the host
    for (int32_t i = 0; i < nq; ++i) {
      const int32_t g = group_of_query[(size_t)i];
      supported[i] = has[(size_t)g] ? 1 : exh[(size_t)g] ? 0 : -1;
      if (witness) witness[i] = wit_of[(size_t)g];
    }
    return rc;
  } catch (const std::bad_alloc&) {           // (the per-query and per-root host arrays)
    set_error(name + ": out of host memory for " + std::to_string(nqroots) + " roots");
    return TB_ERR_NOMEM;
  }
}

extern "C" tb_status tb_solve_front(tb_solver* s, int32_t nboxes, const int32_t* box_lb, const int32_t* box_ub,
                                    int32_t x_var, int32_t maximize_x, int32_t y_var, int32_t maximize_y,
                                    int32_t nlev, const int32_t* level, volatile int32_t* stop_flag, int32_t* best_lb,
                                    int32_t* best_ub, int32_t* has_solution, int32_t* exhaustive, int32_t* objective,
                                    tb_stats* stats) {
  const std::string name("tb_solve_front");
  if (!s || nboxes < 1 || nlev < 1 || !level || !has_solution || !exhaustive || !objective) {
    set_error(name + ": needs nboxes >= 1, nlev >= 1, level, has_solution, exhaustive and objective"); return TB_ERR_INVALID;
  }
  if (x_var < 0 || x_var >= s->nvars || y_var < 0 || y_var >= s->nvars || x_var == y_var) {
    set_error(name + ": x_var = " + std::to_string(x_var) + " and y_var = " + std::to_string(y_var) +
              " must be two different variables of [0, nvars)");
    return TB_ERR_INVALID;
  }
  if ((maximize_x != 0 && maximize_x != 1) || (maximize_y != 0 && maximize_y != 1)) {
    set_error(name + ": maximize_x and maximize_y must be 0 or 1"); return TB_ERR_INVALID;
  }
  for (int32_t i = 0; i < nlev; ++i) {
    if (level[i] == TB_NEG_INF || level[i] == TB_POS_INF) {
      set_error(name + ": level " + std::to_string(i) + " is infinite"); return TB_ERR_INVALID;
    }
    if (i && level[i] <= level[i - 1]) {
      set_error(name + ": the levels are not strictly ascending at level " + std::to_string(i)); return TB_ERR_INVALID;
    }
  }
  const long long nroots = (long long)nlev * nboxes;
  if ((unsigned long long)nroots > (1ull << TB_K_BITS)) {     // (before the per-root arrays are allocated)
    set_error(name + ": nlev * nboxes = " + std::to_string(nroots) + " roots do not fit the subproblem index (at most 2^40)");
    return TB_ERR_INVALID;
  }
  try {
    // Level i is group i, optimising y over its slice of x: (level[i-1], level[i]] when the front minimises x, the
    // first slice open below; [level[i], level[i+1]) when it maximises x, the last open above. The slices partition x's
    // range, so every part of the space is searched once, and a solution of a slice is a witness for every level on
    // its side (batch_share_witness).
    std::vector<int32_t> var((size_t)nlev, x_var), lo((size_t)nlev), hi((size_t)nlev), obj_of((size_t)nlev, y_var),
        maximize((size_t)nlev, maximize_y), image_of, group_of;
    for (int32_t i = 0; i < nlev; ++i) {
      if (maximize_x) { lo[(size_t)i] = level[i]; hi[(size_t)i] = i + 1 < nlev ? level[i + 1] - 1 : TB_POS_INF; }
      else { lo[(size_t)i] = i ? level[i - 1] + 1 : TB_NEG_INF; hi[(size_t)i] = level[i]; }
    }
    const GroupFixing fix{var.data(), lo.data(), hi.data(), maximize_x ? 2 : 1};
    roots_per_box(nboxes, nroots, image_of, group_of);
    const tb_status rc = solve_groups(s, "tb_solve_front", nboxes, box_lb, box_ub, nroots, image_of.data(), group_of.data(),
                                      nlev, obj_of.data(), maximize.data(), true, &fix, nullptr, stop_flag, best_lb,
                                      best_ub, has_solution, exhaustive, objective, stats);
    if (rc != TB_OK && rc != TB_ERR_DEPTH) return rc;
    // A level's value is the best over its own slice and every witness on its side, so it is proven when every slice on
    // its side was searched to its end (or decided on the host): groups 0..i when minimising x, i..last when maximising.
    if (maximize_x) for (int32_t i = nlev - 2; i >= 0; --i) exhaustive[i] &= exhaustive[i + 1];
    else for (int32_t i = 1; i < nlev; ++i) exhaustive[i] &= exhaustive[i - 1];
    return rc;
  } catch (const std::bad_alloc&) {           // (the per-level and per-root host arrays)
    set_error(name + ": out of host memory for " + std::to_string(nroots) + " roots");
    return TB_ERR_NOMEM;
  }
}

// ---- final gather across processes (SURVEY §8e; reduce_blocks, barebones :1033-1067, across GPUs) -------------------
struct ResultHeader {
  uint32_t magic; int32_t nvars, obj_var, has_solution, exhaustive, objective;
  int64_t t_best_ns;
  tb_stats stats;
};
static const uint32_t kResultMagic = 0x54425232u;   // "TBR2"

extern "C" size_t tb_result_size(const tb_solver* s) {
  return s ? sizeof(ResultHeader) + (size_t)2 * (size_t)s->nvars * sizeof(int32_t) : 0;
}

extern "C" tb_status tb_result_pack(const tb_solver* s, void* buf, size_t cap) {
  if (!s || !buf) { set_error("null argument"); return TB_ERR_INVALID; }
  if (!s->last_valid) { set_error("tb_result_pack: no tb_solve has completed on this solver"); return TB_ERR_INVALID; }
  if (cap < tb_result_size(s)) { set_error("tb_result_pack: buffer too small"); return TB_ERR_INVALID; }
  ResultHeader h;
  memset(&h, 0, sizeof(h));
  h.magic = kResultMagic; h.nvars = s->nvars; h.obj_var = s->root_obj_var; h.has_solution = s->last_has; h.exhaustive = s->last_exhaustive;
  h.objective = (s->last_has && s->root_obj_var >= 0) ? s->last_lb[(size_t)s->root_obj_var] : TBD_PINF;
  h.t_best_ns = s->last_stats.timers_ns[TB_TIMER_LATEST_BEST_OBJ_FOUND];
  h.stats = s->last_stats;
  char* p = (char*)buf;
  memcpy(p, &h, sizeof(h));
  if (s->nvars) {
    memcpy(p + sizeof(h), s->last_lb.data(), (size_t)s->nvars * 4);
    memcpy(p + sizeof(h) + (size_t)s->nvars * 4, s->last_ub.data(), (size_t)s->nvars * 4);
  }
  return TB_OK;
}

extern "C" tb_status tb_result_reduce(const void* bufs, int32_t n, size_t stride, int32_t* best_lb, int32_t* best_ub,
                                      int32_t* has_solution, int32_t* exhaustive, tb_stats* total, int32_t* best_rank) {
  if (!bufs || n <= 0 || stride < sizeof(ResultHeader)) { set_error("tb_result_reduce: invalid argument"); return TB_ERR_INVALID; }
  tb_stats t;
  memset(&t, 0, sizeof(t));
  t.exhaustive = 1;
  int best = -1;
  ResultHeader hb;
  memset(&hb, 0, sizeof(hb));
  for (int r = 0; r < n; ++r) {
    ResultHeader h;
    memcpy(&h, (const char*)bufs + (size_t)r * stride, sizeof(h));
    if (h.magic != kResultMagic || (r && h.nvars != hb.nvars && best >= 0)) { set_error("tb_result_reduce: malformed buffer"); return TB_ERR_INVALID; }
    if (stride < sizeof(ResultHeader) + (size_t)2 * (size_t)h.nvars * 4) { set_error("tb_result_reduce: stride smaller than a result"); return TB_ERR_INVALID; }
    const tb_stats& s = h.stats;
    if (r == 0) {                      // the launch configuration is the same on every GPU
      t.threads_per_block = s.threads_per_block; t.mem_kind = s.mem_kind; t.cluster_size = s.cluster_size;
      t.subproblems_power = s.subproblems_power; t.blocks_per_sm = s.blocks_per_sm; t.eps_num_subproblems = s.eps_num_subproblems;
      t.shared_bytes = s.shared_bytes; t.store_bytes = s.store_bytes; t.prop_bytes = s.prop_bytes;
      t.fixpoint_in_effect = s.fixpoint_in_effect;
      t.timers_ns[TB_TIMER_FIRST_BLOCK_IDLE] = s.timers_ns[TB_TIMER_FIRST_BLOCK_IDLE];
    }
    t.num_blocks += s.num_blocks;
    t.nodes += s.nodes; t.fails += s.fails; t.solutions += s.solutions;
    t.depth_max = std::max(t.depth_max, s.depth_max);
    t.exhaustive = t.exhaustive && s.exhaustive && h.exhaustive;
    t.eps_solved_subproblems += s.eps_solved_subproblems; t.eps_skipped_subproblems += s.eps_skipped_subproblems;
    t.eps_stolen_subproblems += s.eps_stolen_subproblems;
    t.eps_split_subproblems += s.eps_split_subproblems; t.eps_split_parts_solved += s.eps_split_parts_solved;
    t.num_blocks_done += s.num_blocks_done;
    t.fixpoint_iterations += s.fixpoint_iterations; t.num_deductions += s.num_deductions; t.bounds_narrowed += s.bounds_narrowed;
    t.cumulative_time_block_ns += s.cumulative_time_block_ns;
    t.device_bytes += s.device_bytes;
    for (int k = 0; k < TB_NUM_TIMERS; ++k)
      if (k != TB_TIMER_LATEST_BEST_OBJ_FOUND && k != TB_TIMER_FIRST_BLOCK_IDLE && k != TB_TIMER_OVERALL) t.timers_ns[k] += s.timers_ns[k];
    t.timers_ns[TB_TIMER_OVERALL] = std::max(t.timers_ns[TB_TIMER_OVERALL], s.timers_ns[TB_TIMER_OVERALL]);
    t.timers_ns[TB_TIMER_FIRST_BLOCK_IDLE] = std::min(t.timers_ns[TB_TIMER_FIRST_BLOCK_IDLE], s.timers_ns[TB_TIMER_FIRST_BLOCK_IDLE]);
    t.kernel_ms = std::max(t.kernel_ms, s.kernel_ms);
    if (h.has_solution) {
      const bool better = best < 0 || (h.obj_var >= 0 ? (h.objective < hb.objective || (h.objective == hb.objective && h.t_best_ns <= hb.t_best_ns))
                                                      : h.t_best_ns < hb.t_best_ns);
      if (better) { best = r; hb = h; }
    } else if (best < 0) hb.nvars = h.nvars;
  }
  if (best >= 0) {
    t.timers_ns[TB_TIMER_LATEST_BEST_OBJ_FOUND] = hb.t_best_ns;
    const char* p = (const char*)bufs + (size_t)best * stride + sizeof(ResultHeader);
    if (best_lb && hb.nvars) memcpy(best_lb, p, (size_t)hb.nvars * 4);
    if (best_ub && hb.nvars) memcpy(best_ub, p + (size_t)hb.nvars * 4, (size_t)hb.nvars * 4);
  }
  if (has_solution) *has_solution = best >= 0;
  if (exhaustive) *exhaustive = t.exhaustive;
  if (total) *total = t;
  if (best_rank) *best_rank = best;
  return TB_OK;
}

static tb_status ensure_batch(tb_solver* s, size_t n) {
  if (n <= s->batch_cap) return TB_OK;
  tb_status rc;
  size_t cap = std::max<size_t>(n, 1);
  size_t cells = cap * (size_t)std::max(1, s->nvars);
  if ((rc = dev_alloc(s, &s->d_in_lb, cells))) return rc;
  if ((rc = dev_alloc(s, &s->d_in_ub, cells))) return rc;
  if ((rc = dev_alloc(s, &s->d_out_lb, cells))) return rc;
  if ((rc = dev_alloc(s, &s->d_out_ub, cells))) return rc;
  if ((rc = dev_alloc(s, &s->d_out_i0, cap))) return rc;
  if ((rc = dev_alloc(s, &s->d_out_i1, cap))) return rc;
  s->batch_cap = cap;
  return TB_OK;
}

extern "C" tb_status tb_propagate_batch(tb_solver* s, int32_t nstores, const int32_t* lb_in, const int32_t* ub_in,
                                        int32_t* lb_out, int32_t* ub_out, int32_t* failed, tb_stats* stats) {
  if (!s || nstores < 0) { set_error("invalid argument"); return TB_ERR_INVALID; }
  if (nstores == 0) return TB_OK;
  CU(cudaSetDevice(s->device));
  tb_status rc;
  if ((rc = ensure_batch(s, (size_t)nstores))) return rc;
  const int grid = std::min(nstores, s->num_blocks);
  if ((rc = reset_stats(s, grid))) return rc;
  const size_t nv = (size_t)s->nvars, cells = nv * (size_t)nstores;
  std::vector<int32_t> tmp;
  const int32_t *hl = lb_in, *hu = ub_in;
  if (!lb_in || !ub_in) {          // NULL = the root store, replicated
    tmp.resize(2 * cells);
    for (int b = 0; b < nstores; ++b) {
      std::copy(s->root_lb.begin(), s->root_lb.end(), tmp.begin() + b * nv);
      std::copy(s->root_ub.begin(), s->root_ub.end(), tmp.begin() + cells + b * nv);
    }
    hl = tmp.data(); hu = tmp.data() + cells;
  } else {
    // Precondition: every store is contained in the root store the solver was created with (the device
    // table is specialised on the root domains: constants are folded, 32-bit arithmetic is proven exact).
    for (int b = 0; b < nstores; ++b)
      for (size_t v = 0; v < nv; ++v)
        if (lb_in[b * nv + v] < s->root_lb[v] || ub_in[b * nv + v] > s->root_ub[v]) {
          set_error("tb_propagate: store " + std::to_string(b) + " is not contained in the root store (variable " + std::to_string(v) + ")");
          return TB_ERR_INVALID;
        }
  }
  if (cells) {
    CU(cudaMemcpyAsync(s->d_in_lb, hl, cells * sizeof(int), cudaMemcpyHostToDevice, s->stream));
    CU(cudaMemcpyAsync(s->d_in_ub, hu, cells * sizeof(int), cudaMemcpyHostToDevice, s->stream));
  }
  const int repeat = std::max(1, s->opt.propagate_repeat);
  CU(cudaEventRecord(s->ev_start, s->stream));
  rc = dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
    CU(launch_workers(s, propagate_kernel<decltype(M)::value, decltype(A)::value, decltype(TM)::value>, grid, s->P, nstores,
                      (const int*)s->d_in_lb, (const int*)s->d_in_ub, s->d_out_lb, s->d_out_ub, s->d_out_i0, repeat));
    CU(cudaGetLastError());
    return TB_OK;
  });
  if (rc) return rc;
  CU(cudaEventRecord(s->ev_stop, s->stream));
  if (cells && lb_out) CU(cudaMemcpyAsync(lb_out, s->d_out_lb, cells * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  if (cells && ub_out) CU(cudaMemcpyAsync(ub_out, s->d_out_ub, cells * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  if (failed) CU(cudaMemcpyAsync(failed, s->d_out_i0, (size_t)nstores * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  if (stats) {
    float kms = 0.f;
    CU(cudaEventElapsedTime(&kms, s->ev_start, s->ev_stop));
    std::vector<BlockStats> bs((size_t)grid);
    CU(cudaMemcpy(bs.data(), s->P.stats, bs.size() * sizeof(BlockStats), cudaMemcpyDeviceToHost));
    memset(stats, 0, sizeof(*stats));
    stats->exhaustive = 1;
    fill_config(s, stats);
    reduce_stats(bs, stats, nullptr);
    stats->num_blocks = grid;
    stats->kernel_ms = kms;
  }
  return TB_OK;
}

extern "C" tb_status tb_propagate(tb_solver* s, const int32_t* lb_in, const int32_t* ub_in, int32_t* lb_out, int32_t* ub_out,
                                  int32_t* failed, tb_stats* stats) {
  return tb_propagate_batch(s, 1, lb_in, ub_in, lb_out, ub_out, failed, stats);
}

extern "C" tb_status tb_dive_batch(tb_solver* s, uint64_t first, int32_t count, int32_t depth, int32_t* lb_out, int32_t* ub_out,
                                   int32_t* remaining_depth, int32_t* leaf_kind) {
  if (!s || count < 0 || depth < 0 || depth > 62) { set_error("invalid argument"); return TB_ERR_INVALID; }
  if (count == 0) return TB_OK;
  CU(cudaSetDevice(s->device));
  tb_status rc;
  if ((rc = ensure_batch(s, (size_t)count))) return rc;
  const int grid = std::min(count, s->num_blocks);
  if ((rc = reset_stats(s, grid))) return rc;
  DevParams P = s->P;
  P.cutnodes = 0;
  P.t_start = 0;
  P.npeers = 0; P.steal = 0; P.observe_stop = 0;     // a dive is a pure function of (root, idx): no incumbent, no stop
  rc = dispatch(s, [&](auto M, auto A, auto TM) -> tb_status {
    CU(launch_workers(s, dive_kernel<decltype(M)::value, decltype(A)::value, decltype(TM)::value>, grid, P,
                      (unsigned long long)first, count, depth, s->d_out_lb, s->d_out_ub, s->d_out_i0, s->d_out_i1));
    CU(cudaGetLastError());
    return TB_OK;
  });
  if (rc) return rc;
  const size_t cells = (size_t)s->nvars * (size_t)count;
  if (cells && lb_out) CU(cudaMemcpyAsync(lb_out, s->d_out_lb, cells * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  if (cells && ub_out) CU(cudaMemcpyAsync(ub_out, s->d_out_ub, cells * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  if (remaining_depth) CU(cudaMemcpyAsync(remaining_depth, s->d_out_i0, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  if (leaf_kind) CU(cudaMemcpyAsync(leaf_kind, s->d_out_i1, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  CU(cudaStreamSynchronize(s->stream));
  return TB_OK;
}

extern "C" tb_status tb_dive(tb_solver* s, uint64_t idx, int32_t depth, int32_t* lb_out, int32_t* ub_out,
                             int32_t* remaining_depth, int32_t* leaf_kind) {
  return tb_dive_batch(s, idx, 1, depth, lb_out, ub_out, remaining_depth, leaf_kind);
}

// ---- cross-GPU grid cells (SURVEY §8e): incumbent exchange and work stealing ----------------------------------
static tb_status publish_peers(tb_solver* s) {
  DevParams& P = s->P;
  P.npeers = 0; P.steal = 0;
  if (s->peer_cells.empty()) return TB_OK;
  if (s->peer_cells.size() > TB_MAX_PEERS) { set_error("too many peers"); return TB_ERR_UNSUPPORTED; }
  for (size_t i = 0; i < s->peer_cells.size(); ++i) { P.peer_cells[i] = s->peer_cells[i]; P.peer_rank[i] = s->peer_ranks[i]; }
  P.npeers = (int)s->peer_cells.size();
  // stealing needs every other shard's dispenser (TB_STEAL=0 keeps the static shards)
  P.steal = (P.npeers == P.world - 1 && env_int("TB_STEAL", 1) != 0) ? 1u : 0u;
  // ... and the tail: idle blocks take children of subproblems a peer has split (TB_SHARE_SPLIT=0: every GPU its own tail)
  P.share_split = (P.steal && env_int("TB_SHARE_SPLIT", 1) != 0) ? 1 : 0;
  return TB_OK;
}

extern "C" tb_status tb_link_peers(tb_solver** solvers, int32_t n) {
  if (!solvers || n <= 0) { set_error("invalid argument"); return TB_ERR_INVALID; }
  for (int i = 0; i < n; ++i) {
    tb_solver* a = solvers[i];
    a->peer_cells.clear(); a->peer_ranks.clear();
    CU(cudaSetDevice(a->device));
    for (int j = 0; j < n; ++j) {
      if (i == j) continue;
      tb_solver* b = solvers[j];
      if (a->device != b->device) {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, a->device, b->device));
        if (!can) { set_error("devices cannot access each other's memory"); return TB_ERR_UNSUPPORTED; }
        cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { set_error(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e)); return TB_ERR_CUDA; }
        cudaGetLastError();
      }
      a->peer_cells.push_back(b->d_cells);
      a->peer_ranks.push_back(b->opt.gpu_rank);
    }
  }
  for (int i = 0; i < n; ++i) { tb_status rc = publish_peers(solvers[i]); if (rc) return rc; }
  return TB_OK;
}

extern "C" tb_status tb_export_bound_handle(tb_solver* s, void* handle64) {
  if (!s || !handle64) { set_error("null argument"); return TB_ERR_INVALID; }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
  CU(cudaSetDevice(s->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, s->d_cells));
  memcpy(handle64, &h, 64);
  return TB_OK;
}

extern "C" tb_status tb_import_peer_bounds(tb_solver* s, const void* handles64, int32_t npeers) {
  if (!s || (npeers && !handles64) || npeers < 0) { set_error("invalid argument"); return TB_ERR_INVALID; }
  CU(cudaSetDevice(s->device));
  s->peer_cells.clear(); s->peer_ranks.clear();
  for (int i = 0; i < npeers; ++i) {
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles64 + (size_t)i * 64, 64);
    // A peer's cell block is recycled by its solvers (acquire_cells), so the same handle comes back with every solver of
    // a create / solve / destroy cycle: the mapping is opened once per process and kept (cudaIpcCloseMemHandle alone
    // took 80 ms of every tb_destroy; profiles/r02_multi_gpu_bench_n2.json).
    void* p = nullptr;
    {
      static std::mutex m;
      static std::vector<std::pair<std::string, void*>> opened[64];
      std::lock_guard<std::mutex> lock(m);
      const std::string key((const char*)&h, 64);
      auto& tab = opened[s->device >= 0 && s->device < 64 ? s->device : 0];
      for (auto& kv : tab) if (kv.first == key) { p = kv.second; break; }
      if (!p) {
        CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        tab.emplace_back(key, p);
      }
    }
    s->peer_cells.push_back((unsigned long long*)p);
    // handles come in rank order with this solver's own rank left out
    s->peer_ranks.push_back(i < s->opt.gpu_rank ? i : i + 1);
  }
  return publish_peers(s);
}

extern "C" tb_status tb_read_bound(tb_solver* s, int32_t* bound) {
  if (!s || !bound) { set_error("null argument"); return TB_ERR_INVALID; }
  CU(cudaSetDevice(s->device));
  unsigned long long w = ~0ull;
  CU(cudaMemcpy(&w, s->d_cells + TB_CELL_BOUND, sizeof(w), cudaMemcpyDeviceToHost));
  *bound = (unsigned)(w >> 32) == ~s->epoch ? (int32_t)((unsigned)w ^ 0x80000000u) : TBD_PINF;
  return TB_OK;
}

// ---- the engine's fixpoint as a tb_fixpoint_fn (root fixpoint of the TNF simplifier, tnf_simplify.cpp) ------
extern "C" tb_status tb_fixpoint_on_device(void* ctx, const tb_problem* pb, int32_t* lb, int32_t* ub, int32_t* failed) {
  if (!pb || !lb || !ub || !failed) { set_error("tb_fixpoint_on_device: null argument"); return TB_ERR_INVALID; }
  tb_options o;
  memset(&o, 0, sizeof(o));
  o.fixpoint = TB_FP_WAC1; o.subproblems_power = 0; o.subproblems_factor = 300; o.mem_kind = TB_MEM_AUTO; o.gpu_world = 1;
  o.or_blocks = 1;
  o.device = ctx ? *(const int32_t*)ctx : 0;
  tb_problem q = *pb;
  q.lb = lb; q.ub = ub;
  tb_solver* s = nullptr;
  tb_status rc = tb_create(&s, &q, &o);
  if (rc != TB_OK) return rc;
  std::vector<int32_t> olb((size_t)std::max(1, pb->nvars)), oub((size_t)std::max(1, pb->nvars));
  tb_stats st;
  rc = tb_propagate(s, nullptr, nullptr, olb.data(), oub.data(), failed, &st);
  tb_destroy(s);
  if (rc != TB_OK) return rc;
  if (!*failed && pb->nvars) { memcpy(lb, olb.data(), (size_t)pb->nvars * 4); memcpy(ub, oub.data(), (size_t)pb->nvars * 4); }
  return TB_OK;
}

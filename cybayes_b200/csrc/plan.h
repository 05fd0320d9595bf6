// Evaluation planner (host only, no CUDA): turns the op lists of one evaluation into an EvalPlan -- which ops run
// (cherries folded away), in which order, in which ranges and launches, where every child comes from, which results
// are stored.  See plan.cpp.
#pragma once
#include <stdint.h>

#include <vector>

#include "cb_types.cuh"

namespace cb {

int fail(const char* fmt, ...);  // records the message for cb_last_error() and returns 1 (defined by the library)
#define REQUIRE(cond, ...) do { if (!(cond)) return fail(__VA_ARGS__); } while (0)

// ---- snapshot bookkeeping (host-side reference counts; the partial buffers themselves are the library's)
struct Snapshot {
  std::vector<int32_t> buf_of_node;     // index by node id; -1 = absent
  std::vector<int32_t> cherry_of_node;  // 2-state family: record of a folded cherry (never materialised), or -1
  int refs = 0;
};
// A small subtree kept by a snapshot as a RECORD instead of a stored partial: its two children and, in the library's own
// P pool at slots [rec * 2C, (rec + 1) * 2C), copies of the P matrices of its two child edges (child 0: C slots, child 1:
// C slots).  A cherry (both children tips) is folded into its parent's lookup table; a node whose children are tips or
// cherries (3 or 4 tips below it; tiled kernel only) is recomputed on the fly when a later dirty path needs it as a
// sibling -- two table look-ups and a product per site instead of 68 bytes of HBM per site.  child[k] <= n_taxa: a tip;
// otherwise the node id of a cherry that the same snapshot holds as a record.
struct CherryRec {
  int32_t tip[2] = {0, 0};   // (children; named tip for the common case)
  int refs = 0;
};

// ---- what the planner reads of the context (filled by plan_config in cybayes_b200.cu)
struct PlanConfig {
  int n_taxa, n_cats, code_bytes;
  int64_t P, buffer_bytes;       // padded pattern count; bytes of one stored partial with its exponents
  int sm_count;
  bool family_s2, dmma_rc;       // 2-state kernels (cherries fold); register-carried DMMA kernel (always walks)
  bool s2_tiled;                 // tiled 2-state kernel: stack slots, canonical child order, inlined subtrees, records
  int s2t_slots;                 // its shared-memory stack slots per tile
  bool s2t_bulk, s2t_prefetch, s2t_small_recs;   // its staging-buffer stores, dirty-path prefetch, small-subtree records
  bool stream_stores;            // partials nobody reads back in the evaluation are stored with the streaming hint
  // launch geometry behind the split walk's limit: sites per block tile, blocks per tile (general family: one per rate
  // category), resident blocks per SM
  int64_t tile_sites; int tile_blocks, blocks_per_sm;
};

// ---- plans
struct PlanChild {
  int32_t kind;  // SrcKind
  int32_t ref;   // SRC_TIP: tip id.  SRC_BUFFER: position of the producing op, or ~node (< 0) when the input snapshot
                 // holds it.  SRC_CHERRY: caller's op index of the folded cherry, or ~node for a record of the input
                 // snapshot.  SRC_STACK: tile buffer.  SRC_SMALL: position of its descriptor.  SRC_CARRIED: unused.
  int32_t edge;  // 2 * (caller's op index) + child: where this edge's P slots sit in the caller's arrays; < 0: the edge
                 // belongs to a record of the input snapshot, its P copies start at library slot ~edge
};
struct PlanOp {
  int32_t node;
  PlanChild ch[2];
  int32_t out_buf;               // tiled kernel: shared-memory tile buffer of the result, or -1
  int32_t pf_buf;                // tiled kernel: tile buffer a stored child is prefetched into, or -1
  uint8_t is_root, keep, stream, spill, pushed;
  uint8_t make_rec;              // not stored: the returned snapshot keeps the node as a record (small subtree)
  uint8_t synthetic;             // not in the caller's list: a record of the input snapshot recomputed as a sibling
};
struct PlanLaunch { int r_begin, r_end, max_ops, n_bufs; };
struct EvalPlan {
  // key (full evaluations only); split_env: CYBAYES_WALK_SPLIT, > 0 forces the split walk's limit
  int flags = 0, n_lists = 0, split_env = 0;
  std::vector<int32_t> key_offsets, key_nodes, key_children;
  // compiled form
  std::vector<PlanOp> ops;
  std::vector<RangeDesc> ranges;
  std::vector<PlanLaunch> launches;
  int64_t bytes_written = 0, bytes_read = 0;
  int n_stored = 0, n_buffer_reads = 0, n_stack = 0, n_spills = 0, n_cherries = 0, n_small_recs = 0;
  int n_inlined = 0;   // ops computed inside their parent's op (SRC_SMALL): in `ops` for their descriptor, in no range
  uint64_t stamp = 0;
  void clear_compiled() {
    ops.clear(), ranges.clear(), launches.clear();
    bytes_written = bytes_read = n_stored = n_buffer_reads = n_stack = n_spills = n_cherries = n_small_recs = n_inlined = 0;
  }
};
constexpr int PLAN_FLAG_MASK = CB_EVAL_WANT_SNAPSHOT | CB_EVAL_STORE_ROOT | CB_EVAL_FORCE_LEVELS | CB_EVAL_FORCE_WALK | CB_EVAL_NO_FOLD;
constexpr int PLAN_CACHE_SIZE = 6;
constexpr int MAX_CHAIN_OPS = 4096;          // longer dirty paths fall back to the level schedule
constexpr int64_t WALK_MIN_SITES_S2 = 32768; // below this a site tile cannot fill the GPU: use levels
constexpr int64_t WALK_MIN_SITES_GENERAL = 32768;

// Schedules (all run the same per-node arithmetic, so results are bit-identical):
//   CHAIN  a dirty path: one launch, one block range walks the ops, the on-path partial is
//          carried in registers / shared memory                        (ML_gamma.pyx:99-114)
//   WALK   a whole (sub)tree in ONE launch; every block walks all ops for its site tile depth-first.  The child
//          finished last is carried on chip; the other child of a node with two internal children is pushed on a
//          stack in shared memory (tiled 2-state kernel: K tile buffers per warp) or, when the stack is full or the
//          kernel has none, written to its buffer and read back.  The visiting order minimises those read-backs
//          (dynamic programme over the tree; ties: heavier subtree first, so a read-back finds its line in L2).
//   LEVELS one launch per tree level, grid.y = nodes of the level: the latency schedule for
//          small alignments where a site tile alone cannot fill the GPU.
enum Schedule { SCHED_CHAIN = 0, SCHED_WALK = 1, SCHED_LEVELS = 2 };

// Compiles n_lists op lists (list li: ops [offsets[li], offsets[li + 1]) of the caller's nodes / children, as cb_eval
// takes them) against the input snapshot `sin` (nullptr: none; `recs`: the library's records) into `plan`, whose
// split_env is read.  Returns 0, or 1 after fail().
int build_plan(const PlanConfig& cfg, const Snapshot* sin, const std::vector<CherryRec>& recs, int n_lists,
               const int32_t* offsets, const int32_t* nodes, const int32_t* children, int flags, EvalPlan& plan);

// The plan of a FULL evaluation depends only on the op list and the flags, so it is cached per topology (a handful of
// trees are alive at a time in an MCMC run: the current one and the proposals); executing a cached plan only refills
// buffer pointers and P slots.  Evaluations against a snapshot are planned into the scratch plan on every call.
struct PlanCache {
  std::vector<EvalPlan> plans;
  EvalPlan scratch_plan;
  uint64_t plan_clock = 0;
  bool no_plan_cache = false;   // CYBAYES_NO_PLAN_CACHE: build every plan anew
};
// The plan of this evaluation, looked up or built (least recently used evicted); nullptr after fail().
EvalPlan* plan_for(PlanCache& cache, const PlanConfig& cfg, const Snapshot* sin, const std::vector<CherryRec>& recs,
                   int n_lists, const int32_t* offsets, const int32_t* nodes, const int32_t* children, int flags);

}  // namespace cb

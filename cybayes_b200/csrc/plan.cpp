// Evaluation planner (see plan.h): build_plan compiles each op list in named passes over one ListWork.
#include "plan.h"

#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <numeric>
#include <utility>

namespace cb {
namespace {

// the input snapshot holds node nd as a record (a folded cherry or a small subtree)
bool snap_rec(const Snapshot* sin, int nd) { return sin && nd < (int)sin->cherry_of_node.size() && sin->cherry_of_node[nd] >= 0; }

// An op that runs.  caller: its index in the caller's arrays, or ~record for a synthetic op; folded[k]: caller's index
// of the folded cherry that child k is, or -1.
struct LOp { int32_t node, caller; int32_t child[2], folded[2]; };

// The evaluation's inputs, and the state of the op list being compiled (rebuilt by the passes for each list).  Ops are
// indexed j in list order, positions p in visiting order.
struct ListWork {
  const PlanConfig& cfg;
  const Snapshot* sin;
  const std::vector<CherryRec>& recs;
  const int32_t *offsets, *nodes, *children;
  int n_lists, flags, split_env, N;
  // small_recs: small subtrees (children: tips / cherries) of a cache-kept pass are kept as records, not stored
  bool fold, want_snap, store_root, small_recs;
  int li = 0, n = 0, n_inl = 0, base = 0;   // base: plan.ops index of position 0
  std::vector<LOp> L;
  std::vector<int> kid[2];              // op -> producer of child k in this list, or -1 (tip, folded cherry, snapshot)
  Schedule sched = SCHED_CHAIN;
  std::vector<int> n_sub;               // walk: ops in each op's subtree
  std::vector<int> cut;                 // split walk: roots of the cut subtrees, biggest first; empty: no cut
  std::vector<int> seg_of;              // op -> segment (0 = top / whole list, s + 1 = cut subtree s)
  std::vector<int> small_of;            // op -> its child (0 / 1) that it computes itself (SRC_SMALL), or -1
  std::vector<char> inlined;            // op -> computed inside its parent's op
  std::vector<int> order, pos_of;       // position -> op and back; positions [n - n_inl, n) hold the inlined ops
  std::vector<int> push_slot;           // op -> stack slot its result is pushed into, or -1
  std::vector<std::pair<int, int>> segs;  // split walk: positions of the cut segments
  std::vector<int> range_id;            // position -> range of the list (0: the top / whole list, s + 1: segment s)
  std::vector<char> read_back;          // op -> read from memory by a later op (2: inside one launch, a spill)
  int n_exec() const { return n - n_inl; }
  bool same_range(int p0, int p1) const { return sched != SCHED_LEVELS && range_id[p0] == range_id[p1]; }
};

// Cherry folding (2-state family): an op whose two children are tips is not run: its parent (always in the list) takes
// it as a SRC_CHERRY child and looks the cherry's 3 x 3 possible partials up.
int fold_cherries(ListWork& w, EvalPlan& plan) {
  const int N = w.N, b_in = w.offsets[w.li], e_in = w.offsets[w.li + 1];
  std::vector<int32_t> parent_op(2 * N, -1), folded_at(2 * N, -1);   // by node id: ids 1 .. 2N-1
  w.L.clear();
  for (int i = b_in; i < e_in; ++i)
    for (int kx = 0; kx < 2; ++kx) {
      const int ch = w.children[2 * i + kx];
      REQUIRE((ch >= 1 && ch <= N) || (ch > N && ch < 2 * N), "op %d: bad child id %d", i, ch);
      if (ch > N) parent_op[ch] = i;
    }
  for (int i = b_in; i < e_in; ++i) {
    const int node = w.nodes[i], c0 = w.children[2 * i], c1 = w.children[2 * i + 1];
    REQUIRE(node > N && node < 2 * N, "op %d: node %d is not an internal node", i, node);
    if (w.fold && c0 <= N && c1 <= N && i != e_in - 1 && parent_op[node] > i) {
      folded_at[node] = i;
      plan.n_cherries++;
      continue;
    }
    w.L.push_back(LOp{node, i, {c0, c1}, {c0 > N ? folded_at[c0] : -1, c1 > N ? folded_at[c1] : -1}});
  }
  return 0;
}

// Children that the input snapshot holds as records of small subtrees (not cherries) are recomputed here: one synthetic
// op each, placed before the caller's ops; the walk pushes / carries its result like any other child.
void add_record_ops(ListWork& w) {
  if (!w.sin || !w.cfg.s2_tiled) return;
  std::vector<LOp> syn;
  for (const LOp& o : w.L)
    for (int kx = 0; kx < 2; ++kx) {
      const int ch = o.child[kx];
      if (ch <= w.N || o.folded[kx] >= 0 || !snap_rec(w.sin, ch)) continue;
      const int rec = w.sin->cherry_of_node[ch];
      const CherryRec& r = w.recs[rec];
      if (r.tip[0] <= w.N && r.tip[1] <= w.N) continue;   // a cherry: folded into the parent's table
      if (std::none_of(w.L.begin(), w.L.end(), [&](const LOp& q) { return q.node == ch; }))
        syn.push_back(LOp{ch, ~rec, {r.tip[0], r.tip[1]}, {-1, -1}});
    }
  w.L.insert(w.L.begin(), syn.begin(), syn.end());
}

// Producers of the children inside the list; every other internal child is a folded cherry or in the input snapshot.
int link_producers(ListWork& w) {
  const int n = w.n = (int)w.L.size();
  std::vector<int32_t> op_of_node(2 * w.N, -1);
  for (int j = 0; j < n; ++j) {
    REQUIRE(op_of_node[w.L[j].node] < 0, "op %d: node %d is computed twice", w.L[j].caller, w.L[j].node);
    op_of_node[w.L[j].node] = j;
  }
  for (auto& k : w.kid) k.assign(n, -1);
  for (int j = 0; j < n; ++j)
    for (int kx = 0; kx < 2; ++kx) {
      const int ch = w.L[j].child[kx], a = ch > w.N ? op_of_node[ch] : -1;
      if (ch <= w.N || w.L[j].folded[kx] >= 0) continue;
      REQUIRE(a < j, "op %d: child %d is computed after its parent", w.L[j].caller, ch);
      REQUIRE(a >= 0 || (w.sin && ch < (int)w.sin->buf_of_node.size() && w.sin->buf_of_node[ch] >= 0) || snap_rec(w.sin, ch),
              "op %d: child %d is neither recomputed nor in the input snapshot", w.L[j].caller, ch);
      w.kid[kx][j] = a;
    }
  return 0;
}

// Chain when every op after the first consumes exactly the previous op and nothing else of the list; otherwise a walk
// or levels.  A walk needs every op under the last one (and gets the subtree sizes).
int choose_schedule(ListWork& w) {
  const int n = w.n;
  bool chain = !(w.flags & CB_EVAL_FORCE_LEVELS) && n <= MAX_CHAIN_OPS;
  for (int j = 0; j < n && chain; ++j) {
    const int a0 = w.kid[0][j], a1 = w.kid[1][j];
    if (j == 0) chain = (a0 < 0 && a1 < 0);
    else chain = (a0 == j - 1) != (a1 == j - 1) && (a0 < 0 || a0 == j - 1) && (a1 < 0 || a1 == j - 1);
  }
  w.sched = SCHED_CHAIN;
  if (chain) return 0;
  // the register-carried kernel only pays off when the partial is carried: its alignments always walk;
  // candidates of a batch always walk (one range per candidate)
  const bool big = w.cfg.dmma_rc || w.cfg.P >= (w.cfg.family_s2 ? WALK_MIN_SITES_S2 : WALK_MIN_SITES_GENERAL);
  w.sched = ((big || w.n_lists > 1 || (w.flags & CB_EVAL_FORCE_WALK)) && !(w.flags & CB_EVAL_FORCE_LEVELS)) ? SCHED_WALK : SCHED_LEVELS;
  REQUIRE(w.n_lists == 1 || w.sched == SCHED_WALK, "cb_eval_batch: candidate %d is not a chain (level schedule forced)", w.li);
  if (w.sched != SCHED_WALK) return 0;
  w.n_sub.assign(n, 1);   // subtree sizes in ops (children precede parents in the caller's order)
  for (int j = 0; j < n; ++j)
    for (int kx = 0; kx < 2; ++kx)
      if (w.kid[kx][j] >= 0) w.n_sub[j] += w.n_sub[w.kid[kx][j]];
  if (w.n_sub[n - 1] != n) {
    REQUIRE(w.n_lists == 1, "cb_eval_batch: candidate %d has ops that are not under its root", w.li);
    w.sched = SCHED_LEVELS;
  }
  return 0;
}

// append j and the ops under it (children: kid_of(k, op), -1 for none) to `out`, depth first
template <typename F> void subtree(int j, F kid_of, std::vector<int>& stack, std::vector<int>& out) {
  for (stack.push_back(j); !stack.empty();) {
    const int x = stack.back();
    stack.pop_back();
    out.push_back(x);
    for (int kx = 0; kx < 2; ++kx)
      if (kid_of(kx, x) >= 0) stack.push_back(kid_of(kx, x));
  }
}

// Split walk.  When the alignment gives too few site tiles to fill the GPU for a whole sequential walk (small shards),
// the tree is cut into independent subtrees of at most `limit` ops that run as parallel ranges of a first launch; the
// ops above the cut follow in a second launch.
void cut_segments(ListWork& w) {
  const int n = w.n;
  w.seg_of.assign(n, 0);
  w.cut.clear();
  if (w.sched != SCHED_WALK || w.n_lists != 1) return;
  int limit = n + 1;
  const int64_t blocks = (w.cfg.P + w.cfg.tile_sites - 1) / w.cfg.tile_sites * w.cfg.tile_blocks;
  const int64_t slots = (int64_t)w.cfg.sm_count * w.cfg.blocks_per_sm;
  // Every block walks the whole list (0.7 ms on C4, 3 ms on a C5 shard), so a ragged last wave is expensive even
  // at many waves: 2-3 % at 8.8 waves, 12 % at 4.4 and 5.3.  Measured: C4 6.07 -> 5.91 ms on 1 GPU and 3.28 ->
  // 2.98 ms per GPU on 2; the C5 shard of an 8-GPU run (25 000 patterns x 64 states) 17.7 -> 15.9 ms.
  // Under one wave the cut is there for parallelism (about 8 waves of ranges); from one wave up it only has to
  // even out the tail, and a small limit costs more in the launch of the ops above the cut (16 ops at limit 93
  // on a 125 000-pattern shard: 65 us of 800) than it gains: a third of the tree per range measured best there
  // (0.794 -> 0.77 ms).
  if (blocks < 16 * slots && n >= 64 && !(w.flags & CB_EVAL_FORCE_WALK)) {
    int lim = (int)(n * blocks / (8 * slots)) + 1;
    if (blocks >= slots) lim = std::max(lim, n / 3);
    limit = std::max(16, std::min(256, lim));
  }
  if (w.split_env > 0) limit = std::max(2, w.split_env);
  if (limit >= n) return;  // nothing to cut
  // walk down from the root: ops with a subtree above the limit stay in the top segment
  std::vector<int> stack, under;
  subtree(n - 1, [&](int kx, int j) { return w.n_sub[j] <= limit ? -1 : w.kid[kx][j]; }, stack, under);
  for (int j : under)
    if (w.n_sub[j] <= limit) w.cut.push_back(j);
  std::stable_sort(w.cut.begin(), w.cut.end(), [&](int x, int y) { return w.n_sub[x] > w.n_sub[y]; });  // big first
  for (size_t s = 0; s < w.cut.size(); ++s) {   // everything under a cut root belongs to that root's segment
    under.clear();
    subtree(w.cut[s], [&](int kx, int j) { return w.kid[kx][j]; }, stack, under);
    for (int j : under) w.seg_of[j] = (int)s + 1;
  }
}

// Tiled kernel: a (tip, cherry) subtree that is not stored is computed inside its parent's op (SRC_SMALL) when the
// parent runs in the same range and its other child is a tip or the op carried into it -- the same arithmetic
// without an op of its own (image, dispatch, rescale, loop iteration) and without a stack slot.  In a chain only the
// first op can be such a subtree; its parent takes it beside a tip.
void pick_inlined(ListWork& w) {
  const int N = w.N, n = w.n;
  w.small_of.assign(n, -1);
  w.inlined.assign(n, 0);
  w.n_inl = 0;
  if (!w.cfg.s2_tiled || w.sched == SCHED_LEVELS) return;
  auto is_cherry = [&](int j, int kx) {   // the child resolves to SRC_CHERRY (resolve_children)
    const int ch = w.L[j].child[kx];
    return ch > N && (w.L[j].folded[kx] >= 0 || (w.kid[kx][j] < 0 && w.fold && snap_rec(w.sin, ch)));
  };
  for (int j = 0; j < n; ++j)
    for (int kx = 1; kx >= 0 && w.small_of[j] < 0; --kx) {
      const int s = w.kid[kx][j], o = w.kid[1 - kx][j];
      if (s < 0 || w.seg_of[s] != w.seg_of[j]) continue;
      const bool tip_cherry = (w.L[s].child[0] <= N && is_cherry(s, 1)) || (w.L[s].child[1] <= N && is_cherry(s, 0));
      // not stored: likelihood-only pass, a recomputed record, or kept as a record (decide_storage; checked there)
      const bool unstored = !w.want_snap || w.L[s].caller < 0 || w.small_recs;
      const bool sibling_ok = w.L[j].child[1 - kx] <= N || (o >= 0 && w.seg_of[o] == w.seg_of[j]);
      if (tip_cherry && unstored && sibling_ok) {
        w.small_of[j] = kx;
        w.inlined[s] = 1;
        w.n_inl++;
      }
    }
}

// Visiting order.  Chain and levels: the caller's order.  Walk: per segment (cut subtrees first, biggest first, then
// the top), the order that needs the fewest read-backs, found by a dynamic programme; it also assigns the stack slots.
// Inlined ops go last either way: their descriptors are in no range.
int visit_order(ListWork& w) {
  const int n = w.n;
  const int K = w.cfg.s2_tiled ? w.cfg.s2t_slots : 0;            // stack slots of the kernel
  const int slot_base = w.cfg.s2t_bulk ? S2T_STAGING : 0;        // tile buffers below it are the staging buffers of the bulk-store path
  w.order.resize(n);
  std::iota(w.order.begin(), w.order.end(), 0);
  w.push_slot.assign(n, -1);
  w.segs.clear();
  if (w.sched != SCHED_WALK) {
    std::stable_partition(w.order.begin(), w.order.end(), [&](int j) { return !w.inlined[j]; });
    return 0;
  }
  // children the walk visits: a cut root lives in another launch and is read from its buffer; an inlined subtree
  // is computed by its parent, like a tip
  auto walk_kid = [&](int kx, int j) {
    const int a = w.kid[kx][j];
    return a >= 0 && w.seg_of[a] == w.seg_of[j] && !w.inlined[a] ? a : -1;
  };
  // f(j, k) = fewest read-backs in j's subtree (inside its segment) with k free stack slots; of two internal children
  // the first visited is pushed (or read back when k == 0), the second carried.  first(j, k): bit 0 which child goes
  // first, bit 1 the third choice below
  std::vector<int> fv((size_t)n * (K + 1), 0), first_kid((size_t)n * (K + 1), 0);
  auto f = [&](int j, int k) -> int& { return fv[(size_t)j * (K + 1) + k]; };
  auto first = [&](int j, int k) -> int& { return first_kid[(size_t)j * (K + 1) + k]; };
  for (int j = 0; j < n; ++j) {
    const int a = walk_kid(0, j), b = walk_kid(1, j);
    for (int kk = 0; kk <= K; ++kk) {
      if (a >= 0 && b >= 0) {
        const int k1 = kk > 0 ? kk - 1 : 0, miss = kk == 0 ? 1 : 0;
        const int ca = f(a, kk) + miss + f(b, k1), cb = f(b, kk) + miss + f(a, k1);
        const bool a_first = ca < cb || (ca == cb && w.n_sub[a] >= w.n_sub[b]);
        f(j, kk) = a_first ? ca : cb;
        first(j, kk) = a_first ? 0 : 1;
        // third choice: read the first child back although a slot is free, so that the second keeps all kk slots
        // (one read-back here instead of one at every fork of a subtree left with too few slots)
        const int cs = f(a, kk) + 1 + f(b, kk);
        if (kk > 0 && cs < f(j, kk)) {
          f(j, kk) = cs;
          first(j, kk) = (w.n_sub[a] >= w.n_sub[b] ? 0 : 1) | 2;
        }
      } else if (a >= 0 || b >= 0) {
        f(j, kk) = f(a >= 0 ? a : b, kk);
      }
    }
  }
  std::vector<int> out;
  out.reserve(n);
  struct Frame { int j, k, phase; };
  std::vector<Frame> fr;
  auto emit = [&](int root_op) {
    for (fr.push_back({root_op, K, 0}); !fr.empty();) {
      Frame& t = fr.back();
      const int j = t.j, kk = t.k;
      const int a = walk_kid(0, j), b = walk_kid(1, j);
      if (a >= 0 && b >= 0) {
        const int fk = first(j, kk);
        const bool push = kk > 0 && !(fk & 2);
        const int x = (fk & 1) == 0 ? a : b, y = (fk & 1) == 0 ? b : a;
        if (t.phase == 0) { t.phase = 1; fr.push_back({x, kk, 0}); continue; }
        if (t.phase == 1) {
          w.push_slot[x] = push ? slot_base + (K - kk) : -1;
          t.phase = 2;
          fr.push_back({y, push ? kk - 1 : kk, 0});
          continue;
        }
      } else if ((a >= 0 || b >= 0) && t.phase == 0) {
        t.phase = 2;
        fr.push_back({a >= 0 ? a : b, kk, 0});
        continue;
      }
      out.push_back(j);
      fr.pop_back();
    }
  };
  for (int r : w.cut) {
    const int b0 = (int)out.size();
    emit(r);
    w.segs.push_back({b0, (int)out.size()});
  }
  emit(n - 1);
  REQUIRE((int)out.size() == w.n_exec(), "internal error: walk order covers %d of %d ops", (int)out.size(), w.n_exec());
  for (int j = 0; j < n; ++j)
    if (w.inlined[j]) out.push_back(j);
  w.order.swap(out);
  return 0;
}

// Where each child comes from, and which ops a later op reads back from memory.  Appends the list's ops to the plan.
int resolve_children(ListWork& w, EvalPlan& plan) {
  const int N = w.N, C = w.cfg.n_cats, n = w.n, base = w.base = (int)plan.ops.size();
  const int64_t tip_row_bytes = w.cfg.P * w.cfg.code_bytes;
  w.pos_of.assign(n, 0);
  for (int p = 0; p < n; ++p) w.pos_of[w.order[p]] = p;
  w.range_id.assign(n, 0);
  for (size_t si = 0; si < w.segs.size(); ++si)
    for (int p = w.segs[si].first; p < w.segs[si].second; ++p) w.range_id[p] = (int)si + 1;
  w.read_back.assign(n, 0);
  plan.ops.resize(base + n);   // value-initialised: every flag 0
  for (int p = 0; p < n; ++p) {
    const int j = w.order[p];
    const LOp& o = w.L[j];
    PlanOp& po = plan.ops[base + p];
    po.node = o.node;
    po.is_root = (j == n - 1);
    REQUIRE(!po.is_root || p == w.n_exec() - 1, "internal error: root is not last");
    po.synthetic = o.caller < 0 ? 1 : 0;
    po.out_buf = po.pf_buf = -1;
    for (int kx = 0; kx < 2; ++kx) {
      PlanChild& pc = po.ch[kx];
      const int ch = o.child[kx], jj = w.kid[kx][j], pp = jj >= 0 ? w.pos_of[jj] : -1;
      pc.edge = o.caller >= 0 ? 2 * o.caller + kx : ~((~o.caller) * 2 * C + kx * C);
      if (ch <= N) {
        pc = {SRC_TIP, ch, pc.edge};
        plan.bytes_read += tip_row_bytes;
      } else if (o.folded[kx] >= 0) {
        pc = {SRC_CHERRY, o.folded[kx], pc.edge};
        plan.bytes_read += 2 * tip_row_bytes;
      } else if (w.small_of[j] == kx) {
        pc = {SRC_SMALL, base + pp, pc.edge};   // its descriptor
      } else if (jj >= 0 && w.same_range(pp, p) && pp == p - 1) {
        pc = {SRC_CARRIED, 0, pc.edge};
      } else if (jj >= 0 && w.same_range(pp, p) && w.push_slot[jj] >= 0) {
        pc = {SRC_STACK, w.push_slot[jj], pc.edge};
        plan.n_stack++;
      } else if (jj >= 0) {
        REQUIRE(pp < p, "internal error: producer of node %d runs after its consumer", ch);
        pc = {SRC_BUFFER, base + pp, pc.edge};
        w.read_back[jj] = w.same_range(pp, p) ? 2 : 1;   // 2: inside one launch (a spill)
        plan.bytes_read += w.cfg.buffer_bytes;
        plan.n_buffer_reads++;
      } else {
        const bool rec = w.fold && snap_rec(w.sin, ch);
        pc = {rec ? SRC_CHERRY : SRC_BUFFER, ~ch, pc.edge};
        plan.bytes_read += rec ? 2 * tip_row_bytes : w.cfg.buffer_bytes;
        plan.n_buffer_reads += !rec;
      }
    }
    // the tiled kernel wants the children in canonical order (products and exponent sums commute exactly)
    if (w.cfg.s2_tiled && s2t_rank(po.ch[1].kind) < s2t_rank(po.ch[0].kind)) std::swap(po.ch[0], po.ch[1]);
    REQUIRE(!w.cfg.s2_tiled || s2t_combo(po.ch[0].kind, po.ch[1].kind) >= 0,
            "internal error: op of node %d has children of kinds %d, %d", po.node, po.ch[0].kind, po.ch[1].kind);
  }
  plan.bytes_read += w.cfg.P * 8;  // pattern weights at the root
  return 0;
}

// Which results are stored (kept by the returned snapshot or read back), with which store, which are kept as records,
// and the tile buffers of pushed results and of the bulk-store path's staging.
int decide_storage(ListWork& w, EvalPlan& plan) {
  int staging_rr = 0;
  for (int p = 0; p < w.n; ++p) {
    const int j = w.order[p];
    PlanOp& po = plan.ops[w.base + p];
    po.keep = po.is_root ? (w.want_snap && w.store_root) : ((w.want_snap && !po.synthetic) || w.read_back[j] != 0);
    po.spill = (w.read_back[j] == 2) ? 1 : 0;
    // small subtrees (children: tips / cherries) are not stored: the returned snapshot keeps a record
    if (w.small_recs && po.keep && !po.is_root && !po.synthetic && w.read_back[j] == 0 &&
        (po.ch[0].kind == SRC_TIP || po.ch[0].kind == SRC_CHERRY) && po.ch[1].kind == SRC_CHERRY) {
      po.keep = 0;
      po.make_rec = 1;
      plan.n_small_recs++;
    }
    po.stream = (po.keep && w.read_back[j] == 0 && w.cfg.stream_stores) ? 1 : 0;
    plan.n_stored += po.keep;
    plan.n_spills += po.keep && po.spill;
    plan.bytes_written += po.keep ? w.cfg.buffer_bytes : 0;
    // an inlined op has no store of its own: a buffer given to it would enter the snapshot unwritten
    REQUIRE(!w.inlined[j] || !po.keep, "internal error: inlined node %d would be stored", po.node);
    if (w.cfg.s2_tiled && w.push_slot[j] >= 0 && !po.is_root) { po.out_buf = w.push_slot[j]; po.pushed = 1; }
    else if (w.cfg.s2_tiled && w.cfg.s2t_bulk && po.keep && !po.spill) { po.out_buf = staging_rr; staging_rr ^= 1; }
  }
  return 0;
}

// Dirty paths and other lists with a shallow stack: a stored partial that comes from the input snapshot (or an
// earlier launch) and is read beside a carried child is prefetched into a tile buffer two ops ahead (three rotating
// buffers above the stack slots in use) and then read like a stack slot: the path keeps three sibling tiles per
// warp in flight instead of exposing one DRAM latency per op.
void add_prefetch(ListWork& w, EvalPlan& plan) {
  const int max_slot = w.n ? *std::max_element(w.push_slot.begin(), w.push_slot.end()) : -1;
  if (!w.cfg.s2_tiled || !w.cfg.s2t_prefetch || max_slot >= 2 || w.cfg.s2t_bulk) return;
  for (int p = 0, rr = 0; p < w.n; ++p) {
    PlanOp& po = plan.ops[w.base + p];
    if (po.ch[0].kind != SRC_CARRIED || po.ch[1].kind != SRC_BUFFER) continue;
    const int ref = po.ch[1].ref;
    const bool other_launch = ref < 0 || !w.same_range(ref - w.base, p);
    if (!other_launch) continue;
    po.ch[1].kind = SRC_STACK;     // read from the tile buffer; po.ch[1].ref keeps naming the stored partial
    po.pf_buf = max_slot + 1 + rr;
    rr = (rr + 1) % 3;
  }
}

// shared-memory tile buffers per warp that plan ops [p0, p1) name
int bufs_of(const EvalPlan& plan, int p0, int p1) {
  int nb = 0;
  for (int p = p0; p < p1; ++p) {
    const PlanOp& po = plan.ops[p];
    nb = std::max(nb, std::max(po.out_buf, po.pf_buf) + 1);
    for (int kx = 0; kx < 2; ++kx)
      if (po.ch[kx].kind == SRC_STACK && po.pf_buf < 0) nb = std::max(nb, po.ch[kx].ref + 1);
  }
  return nb;
}

// Ranges of the list.  A split walk gets two launches (cut segments, then the top) and levels one launch per level;
// the ranges of every other list share one launch, added by build_plan at the end.
void add_ranges(ListWork& w, EvalPlan& plan) {
  const int base = w.base, n = w.n, n_exec = w.n_exec();
  if (w.sched == SCHED_WALK && !w.segs.empty()) {
    const int start = (int)plan.ranges.size();
    int mx = 1, nb = 0;
    for (auto& sg : w.segs) {
      plan.ranges.push_back(RangeDesc{base + sg.first, base + sg.second, -1, 0});
      mx = std::max(mx, sg.second - sg.first);
      nb = std::max(nb, bufs_of(plan, base + sg.first, base + sg.second));
    }
    plan.launches.push_back({start, (int)plan.ranges.size(), mx, nb});
    const int tb = w.segs.back().second;
    plan.ranges.push_back(RangeDesc{base + tb, base + n_exec, w.li, 0});
    plan.launches.push_back({(int)plan.ranges.size() - 1, (int)plan.ranges.size(), n_exec - tb, bufs_of(plan, base + tb, base + n_exec)});
  } else if (w.sched != SCHED_LEVELS) {
    plan.ranges.push_back(RangeDesc{base, base + n_exec, w.li, 0});
  } else {   // one range per op (order is the identity for this schedule), one launch per level
    std::vector<int> level_of(n, 1), by_level(n);
    for (int j = 0; j < n; ++j) {
      by_level[j] = j;
      for (int kx = 0; kx < 2; ++kx)
        if (w.kid[kx][j] >= 0) level_of[j] = std::max(level_of[j], level_of[w.kid[kx][j]] + 1);
    }
    std::stable_sort(by_level.begin(), by_level.end(), [&](int x, int y) { return level_of[x] < level_of[y]; });
    for (int q = 0; q < n; ++q) {
      const int j = by_level[q];
      if (q == 0 || level_of[j] != level_of[by_level[q - 1]]) plan.launches.push_back({(int)plan.ranges.size(), 0, 1, 0});
      plan.ranges.push_back(RangeDesc{base + j, base + j + 1, (j == n - 1) ? w.li : -1, 0});
      plan.launches.back().r_end = (int)plan.ranges.size();
      plan.launches.back().n_bufs = std::max(plan.launches.back().n_bufs, bufs_of(plan, base + j, base + j + 1));
    }
  }
}

}  // namespace

int build_plan(const PlanConfig& cfg, const Snapshot* sin, const std::vector<CherryRec>& recs, int n_lists,
               const int32_t* offsets, const int32_t* nodes, const int32_t* children, int flags, EvalPlan& plan) {
  const bool want_snap = (flags & CB_EVAL_WANT_SNAPSHOT) != 0;
  ListWork w{cfg, sin, recs, offsets, nodes, children, n_lists, flags, plan.split_env, cfg.n_taxa,
             cfg.family_s2 && !(flags & CB_EVAL_NO_FOLD), want_snap, (flags & CB_EVAL_STORE_ROOT) != 0,
             cfg.s2_tiled && cfg.s2t_small_recs && want_snap};   // small_recs: see ListWork
  plan.clear_compiled();
  for (w.li = 0; w.li < n_lists; ++w.li) {
    REQUIRE(offsets[w.li + 1] > offsets[w.li], "empty op list %d", w.li);
    if (fold_cherries(w, plan)) return 1;
    add_record_ops(w);
    if (link_producers(w) || choose_schedule(w)) return 1;
    cut_segments(w);
    pick_inlined(w);
    if (visit_order(w) || resolve_children(w, plan) || decide_storage(w, plan)) return 1;
    plan.n_inlined += w.n_inl;
    add_prefetch(w, plan);
    add_ranges(w, plan);
  }
  if (plan.launches.empty()) {  // no split walk, no levels: every range in one launch
    int mx = 0;
    for (const RangeDesc& r : plan.ranges) mx = std::max(mx, r.end - r.begin);
    plan.launches.push_back({0, (int)plan.ranges.size(), mx, bufs_of(plan, 0, (int)plan.ops.size())});
  }
  return 0;
}

EvalPlan* plan_for(PlanCache& cache, const PlanConfig& cfg, const Snapshot* sin, const std::vector<CherryRec>& recs,
                   int n_lists, const int32_t* offsets, const int32_t* nodes, const int32_t* children, int flags) {
  const char* env = getenv("CYBAYES_WALK_SPLIT");   // read on every evaluation: tests change it between them
  const int split_env = env ? atoi(env) : 0, total = offsets[n_lists];
  EvalPlan* plan = nullptr;
  if (sin || cache.no_plan_cache) {
    plan = &cache.scratch_plan;
    plan->split_env = split_env;
    return build_plan(cfg, sin, recs, n_lists, offsets, nodes, children, flags, *plan) ? nullptr : plan;
  }
  for (auto& p : cache.plans)
    if (!plan && p.n_lists == n_lists && p.flags == (flags & PLAN_FLAG_MASK) && p.split_env == split_env &&
        (int)p.key_nodes.size() == total && memcmp(p.key_offsets.data(), offsets, (size_t)(n_lists + 1) * 4) == 0 &&
        memcmp(p.key_nodes.data(), nodes, (size_t)total * 4) == 0 && memcmp(p.key_children.data(), children, (size_t)total * 8) == 0)
      plan = &p;
  if (!plan) {
    if ((int)cache.plans.size() < PLAN_CACHE_SIZE) plan = &cache.plans.emplace_back();
    else plan = &*std::min_element(cache.plans.begin(), cache.plans.end(),   // evict the least recently used
                                   [](const EvalPlan& x, const EvalPlan& y) { return x.stamp < y.stamp; });
    plan->n_lists = 0;  // invalid while it is rebuilt
    plan->split_env = split_env;
    if (build_plan(cfg, sin, recs, n_lists, offsets, nodes, children, flags, *plan)) { plan->key_nodes.clear(); return nullptr; }
    plan->n_lists = n_lists;
    plan->flags = flags & PLAN_FLAG_MASK;
    plan->key_offsets.assign(offsets, offsets + n_lists + 1);
    plan->key_nodes.assign(nodes, nodes + total);
    plan->key_children.assign(children, children + 2 * (size_t)total);
  }
  plan->stamp = ++cache.plan_clock;
  return plan;
}

}  // namespace cb

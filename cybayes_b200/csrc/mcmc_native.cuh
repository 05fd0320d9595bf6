// Native Metropolis-Hastings generation loop (SURVEY 8f rank 1): the reference's driver loop
// (mat_mcmc_gamma.py:97-221) and its proposal generators (mcmc_gamma.pyx:40-198) restated in C++, so that a
// generation costs no Python: proposal -> P matrices of the touched branches -> dirty-path / full evaluation on the
// GPU -> accept test, all inside one cb_chain_run call for as many generations as the caller asks for.
//
// The TRACE is the contract: for a fixed seed the chain takes the moves and makes the accept / reject decisions of
// the reference, generation by generation.  That pins
//   * both random streams -- Python's `random` (MT19937: random() = 53-bit double from two draws, getrandbits,
//     _randbelow by rejection on bit_length bits, choice, randint, sample, uniform) and NumPy's legacy global
//     generator (MT19937: random_sample) -- which are imported from / exported to the interpreter as raw MT states,
//   * the insertion order of the tree dict (it feeds random.choice(list(tree)) and the edge post-order), kept here
//     as a vector of edges with Python-dict semantics (delete = erase in place, insert = append),
//   * the host arithmetic of the moves (libm exp, as the reference's c_exp).
// What is not restated but called back into the interpreter, because bit-exactness depends on SciPy / BLAS:
// the discrete-Gamma rates (mcmc_gamma.pyx:596-602), beta = 1 / (1 - pi.pi) (numpy dot), the GTR eigensystem.
// Those are needed only by pi / rates / alpha moves (12 % of the generations).
//
// The likelihood side is reached through a small backend table: by default the CUDA context's own cb_pmat_build /
// cb_eval / cb_snapshot_release; tests substitute callbacks into the NumPy oracle to check the trace on CPU.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/cybayes_b200.h"

namespace cbm {

struct MT19937 {
  uint32_t mt[624];
  int pos = 624;
  uint32_t next32() {
    if (pos >= 624) {
      for (int kk = 0; kk < 624; ++kk) {
        const uint32_t y = (mt[kk] & 0x80000000u) | (mt[(kk + 1) % 624] & 0x7fffffffu);
        mt[kk] = mt[(kk + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      pos = 0;
    }
    uint32_t y = mt[pos++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
  }
  // genrand_res53 (CPython random_random) == rk_double (NumPy legacy random_sample)
  double res53() {
    const uint32_t a = next32() >> 5, b = next32() >> 6;
    return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0);
  }
  // CPython Random.getrandbits(k), 1 <= k <= 32, and Random._randbelow_with_getrandbits(n), n > 0
  uint32_t getrandbits(int k) { return next32() >> (32 - k); }
  uint32_t randbelow(uint32_t n) {
    int k = 0;
    for (uint32_t v = n; v; v >>= 1) ++k;
    uint32_t r = getrandbits(k);
    while (r >= n) r = getrandbits(k);
    return r;
  }
};

struct Edge {
  int32_t p, c;
  double t;
  int32_t slot[CB_MAX_CATS];
};

enum Param { P_PI = 0, P_RATES = 1, P_TREE = 2, P_BL = 3, P_SRATES = 4 };
// trace ids of the moves (tests/golden/make_golden.py C1_MOVES order, then the rates slider)
enum Move { MV_SCALE_EDGE = 0, MV_NODE_SLIDER = 1, MV_NNI = 2, MV_SPR = 3, MV_PI = 4, MV_ALPHA = 5, MV_RATES = 6, MV_COUNT = 7 };

constexpr double BL_EXP_SCALE = 0.1;  // mcmc_gamma.pyx:21
constexpr double SCALER_ALPHA = 1.0;  // mcmc_gamma.pyx:22

struct Chain {
  cb_ctx* ctx = nullptr;
  cb_chain_backend be;
  int n_taxa = 0, S = 0, C = 0, model = 0, root = 0, host_exp_max = 4096;
  bool binary = false;
  std::vector<int> param_ids;
  std::vector<double> params_cdf, tree_cdf, bl_cdf;
  // state
  std::vector<Edge> tree;
  std::vector<double> pi, rates, site_rates, gtr;  // gtr: eigensystem of (pi, rates) for the GTR builder
  double alpha = 0.0, beta = 0.0, lnl = 0.0;
  int snap = -1;
  MT19937 py, np_;
  std::vector<int32_t> free_slots;
  int64_t n_moves[MV_COUNT] = {0}, n_accepts[MV_COUNT] = {0};
  // Full-table proposals (pi / rates / alpha) on a large alignment: a rejected one needs no cache, and a pass that
  // keeps none is cheaper (C4: 4.9 instead of 5.9 ms).  While such proposals are rarely accepted the chain asks for the
  // likelihood only and repeats the pass with the cache on the rare acceptance (same operands, same bits -- checked).
  // lnl_first: -1 = decide from the context and the acceptance count, 0 = never, 1 = always (CYBAYES_CHAIN_LNL_FIRST).
  int lnl_first = -1;
  int64_t full_props = 0, full_accepts = 0;
  std::string err;
  // scratch
  std::vector<int32_t> nodes, children, pslots, kid0, kid1, parent_of, index_of, order_nodes;
  std::vector<std::pair<int32_t, int32_t>> post;
};

static int chain_fail(Chain* ch, const char* msg) {
  ch->err = msg;
  return 1;
}

// ---- backend shims -------------------------------------------------------------------------------------------
static int be_build(Chain* ch, int model, const double* pi, double beta, const double* gtr, int count, const int32_t* slots,
                    const double* d, const double* x) {
  if (ch->be.pmat_build) return ch->be.pmat_build(ch->be.user, model, pi, beta, gtr, count, slots, d, x);
  return cb_pmat_build(ch->ctx, model, pi, beta, gtr, count, slots, d, x);
}
static int be_eval(Chain* ch, int snap_in, int n_ops, const int32_t* nodes, const int32_t* children, const int32_t* pslots,
                   const double* pi, int* snap_out, double* lnl, bool keep_cache = true) {
  const int flags = keep_cache ? CB_EVAL_WANT_SNAPSHOT : 0;
  *snap_out = -1;
  if (ch->be.eval) return ch->be.eval(ch->be.user, snap_in, n_ops, nodes, children, pslots, pi, flags, snap_out, lnl);
  return cb_eval(ch->ctx, snap_in, n_ops, nodes, children, pslots, pi, flags, snap_out, lnl);
}
static int be_eval_sites(Chain* ch, int snap_in, int n_ops, const int32_t* nodes, const int32_t* children,
                         const int32_t* pslots, const double* pi, double* lnl, double* site_lnl, double* cat_post) {
  int snap_out = -1;
  if (ch->be.eval_sites)
    return ch->be.eval_sites(ch->be.user, snap_in, n_ops, nodes, children, pslots, pi, 0, &snap_out, lnl, site_lnl, cat_post);
  if (ch->be.eval || !ch->ctx)
    return chain_fail(ch, "native chain: per-site terms need an eval_sites callback when evaluation goes through callbacks");
  return cb_eval_sites(ch->ctx, snap_in, n_ops, nodes, children, pslots, pi, 0, &snap_out, lnl, site_lnl, cat_post);
}
static void be_release(Chain* ch, int snap) {
  if (snap < 0) return;
  if (ch->be.snapshot_release) ch->be.snapshot_release(ch->be.user, snap);
  else cb_snapshot_release(ch->ctx, snap);
}

// ---- tree helpers (tree.py / mcmc_gamma.pyx:200-242) -----------------------------------------------------------
// children lists in insertion order; parent map
static void build_kids(const Chain* ch, const std::vector<Edge>& tree, std::vector<int32_t>& k0, std::vector<int32_t>& k1,
                       std::vector<int32_t>& parent_of) {
  const int n_nodes = 2 * ch->n_taxa;
  k0.assign(n_nodes, -1);
  k1.assign(n_nodes, -1);
  parent_of.assign(n_nodes, -1);
  for (const Edge& e : tree) {
    if (k0[e.p] < 0) k0[e.p] = e.c; else k1[e.p] = e.c;
    parent_of[e.c] = e.p;
  }
}
static int find_edge(const std::vector<Edge>& tree, int p, int c) {
  for (size_t i = 0; i < tree.size(); ++i)
    if (tree[i].p == p && tree[i].c == c) return (int)i;
  return -1;
}
// The node-operation list of an edge post-order (likelihood._Plan): postorder(kids, root)[::-1] walked in order, a
// node is completed when its second edge is seen.  Fills ch->order_nodes (completion order) and index_of.
static void plan_nodes(Chain* ch, const std::vector<int32_t>& k0, const std::vector<int32_t>& k1) {
  const int N = ch->n_taxa;
  ch->post.clear();
  std::vector<int32_t> stack;
  stack.push_back(ch->root);
  while (!stack.empty()) {
    const int nd = stack.back();
    stack.pop_back();
    const int a = k0[nd], b = k1[nd];
    ch->post.push_back({nd, a});
    ch->post.push_back({nd, b});
    if (b > N) stack.push_back(b);
    if (a > N) stack.push_back(a);
  }
  // reversed list: the parent is completed at its second appearance
  ch->order_nodes.clear();
  ch->index_of.assign(2 * N, -1);
  std::vector<char> seen(2 * N, 0);
  for (size_t i = ch->post.size(); i-- > 0;) {
    const int p = ch->post[i].first;
    if (seen[p]) {
      ch->index_of[p] = (int)ch->order_nodes.size();
      ch->order_nodes.push_back(p);
    } else {
      seen[p] = 1;
    }
  }
}
// children of a node in the order the reversed post-order presents its two edges: (second-listed, first-listed)
static inline void op_children(const std::vector<int32_t>& k0, const std::vector<int32_t>& k1, int node, int& c_first, int& c_second) {
  // postorder() lists (node, k0) then (node, k1); reversed, (node, k1) comes first
  c_first = k1[node];
  c_second = k0[node];
}

// The op list of `todo` nodes (in plan order) on `tree` into ch->nodes / children / pslots.
static void fill_ops(Chain* ch, const std::vector<Edge>& tree, const std::vector<int32_t>& k0, const std::vector<int32_t>& k1,
                     const std::vector<int32_t>& todo) {
  const int C = ch->C, n = (int)todo.size();
  ch->nodes.resize(n);
  ch->children.resize(2 * (size_t)n);
  ch->pslots.resize(2 * (size_t)n * C);
  // slots by child id (every child has one parent edge)
  static thread_local std::vector<int32_t> edge_of_child;
  edge_of_child.assign(2 * ch->n_taxa, -1);
  for (size_t i = 0; i < tree.size(); ++i) edge_of_child[tree[i].c] = (int32_t)i;
  for (int i = 0; i < n; ++i) {
    const int node = todo[i];
    int c[2];
    op_children(k0, k1, node, c[0], c[1]);
    ch->nodes[i] = node;
    for (int kx = 0; kx < 2; ++kx) {
      ch->children[2 * i + kx] = c[kx];
      const Edge& e = tree[edge_of_child[c[kx]]];
      for (int q = 0; q < C; ++q) ch->pslots[(size_t)(2 * i + kx) * C + q] = e.slot[q];
    }
  }
}
// Evaluate the op list of `todo` nodes (in plan order) on `tree`; snap_in < 0 = full evaluation.
static int evaluate(Chain* ch, const std::vector<Edge>& tree, const std::vector<int32_t>& k0, const std::vector<int32_t>& k1,
                    const std::vector<int32_t>& todo, int snap_in, const double* pi, int* snap_out, double* lnl,
                    bool keep_cache = true) {
  fill_ops(ch, tree, k0, k1, todo);
  return be_eval(ch, snap_in, (int)todo.size(), ch->nodes.data(), ch->children.data(), ch->pslots.data(), pi, snap_out, lnl,
                 keep_cache);
}
// Per-site terms of the current state: the root op alone against the chain's snapshot (cb_chain_site_lnl).
static int site_lnl(Chain* ch, double* out, double* cat_post) {
  std::vector<int32_t> k0, k1, par;
  build_kids(ch, ch->tree, k0, k1, par);
  fill_ops(ch, ch->tree, k0, k1, std::vector<int32_t>{ch->root});
  double lnl = 0.0;
  return be_eval_sites(ch, ch->snap, 1, ch->nodes.data(), ch->children.data(), ch->pslots.data(), ch->pi.data(), &lnl, out,
                       cat_post);
}

// likelihood first, cache on acceptance?  Only where keeping the cache costs real bandwidth (a cache of 1 GB and more:
// the reference datasets are latency-bound either way) and only while full-table proposals are accepted less than
// one time in eight (the repeat costs a whole pass).  The decision depends on the chain's own history only, so the
// ranks of a sharded chain take it alike.
static bool lnl_first_now(const Chain* ch) {
  if (ch->lnl_first >= 0) return ch->lnl_first != 0;
  if (!ch->ctx) return false;
  const double cache_bytes = (double)ch->ctx->P * ch->C * ch->S * 8.0 * (ch->n_taxa - 1);
  if (cache_bytes < 1e9) return false;
  return ch->full_props >= 8 && ch->full_accepts * 8 < ch->full_props;
}

// ---- P matrices (subst._queue) -----------------------------------------------------------------------------
static int alloc_slots(Chain* ch, int n, int32_t* out) {
  if ((int)ch->free_slots.size() < n) return chain_fail(ch, "native chain: P-slot pool exhausted");
  for (int i = 0; i < n; ++i) {
    out[i] = ch->free_slots.back();
    ch->free_slots.pop_back();
  }
  return 0;
}
static void free_slots(Chain* ch, const int32_t* s, int n) {
  for (int i = 0; i < n; ++i) ch->free_slots.push_back(s[i]);
}
static int build_pmats(Chain* ch, const double* pi, double beta, const double* gtr, int count, const int32_t* slots, const double* d) {
  if (count == 0) return 0;
  if (ch->model == 2 /* GTR */) return be_build(ch, CB_MODEL_GTR_EIG, pi, 0.0, gtr, count, slots, d, nullptr);
  std::vector<double> x;
  if (count <= ch->host_exp_max) {  // exp(-beta d) from the host libm: matrices bit-identical to the reference's
    x.resize(count);
    const double nb = -beta;
    for (int i = 0; i < count; ++i) x[i] = exp(nb * d[i]);
  }
  const int m = ch->model == 0 ? CB_MODEL_JC : (ch->binary ? CB_MODEL_F81_BINARY : CB_MODEL_F81);
  return be_build(ch, m, pi, beta, nullptr, count, slots, d, x.empty() ? nullptr : x.data());
}
// all edges x categories into fresh slots of `tree` (get_prob_t_all); d[k][e] = t_e * r_k
static int build_all(Chain* ch, std::vector<Edge>& tree, const double* pi, double beta, const double* gtr, const double* site_rates) {
  const int C = ch->C, E = (int)tree.size();
  std::vector<int32_t> slots((size_t)E * C);
  std::vector<double> d((size_t)E * C);
  if (alloc_slots(ch, E * C, slots.data())) return 1;
  for (int k = 0; k < C; ++k)
    for (int e = 0; e < E; ++e) {
      d[(size_t)k * E + e] = site_rates[k] * tree[e].t;
      tree[e].slot[k] = slots[(size_t)k * E + e];
    }
  return build_pmats(ch, pi, beta, gtr, E * C, slots.data(), d.data());
}

// ---- the moves (mcmc_gamma.pyx:40-198 as restated in moves.py) ----------------------------------------------------
static inline void multiplier(Chain* ch, double& log_c, double& c) {
  log_c = SCALER_ALPHA * (ch->py.res53() - 0.5);
  c = exp(log_c);
}

static void path_to_root(const std::vector<int32_t>& parent_of, int node, int root, std::vector<int32_t>& out) {
  while (true) {
    node = parent_of[node];
    out.push_back(node);
    if (node == root) return;
  }
}
static void sort_by_plan(const Chain* ch, std::vector<int32_t>& todo, int root) {
  todo.push_back(root);
  std::sort(todo.begin(), todo.end(), [&](int a, int b) { return ch->index_of[a] < ch->index_of[b]; });
  todo.erase(std::unique(todo.begin(), todo.end()), todo.end());
}

static int run(Chain* ch, int64_t n_gens, int8_t* t_move, int8_t* t_acc, double* t_cur, double* t_prop, double* t_ratio, double* t_logu) {
  const int C = ch->C, N = ch->n_taxa, root = ch->root;
  std::vector<Edge> prop;
  std::vector<int32_t> k0, k1, parent_of, pk0, pk1, pparent, todo, new_slots, old_slots;
  std::vector<double> pi_prop, rates_prop, sr_prop, gtr_prop, d;
  for (int64_t it = 0; it < n_gens; ++it) {
    pi_prop = ch->pi;
    rates_prop = ch->rates;
    double hr = 0.0, pr_ratio = 0.0;
    const double u0 = ch->np_.res53();
    const int pidx = (int)(std::upper_bound(ch->params_cdf.begin(), ch->params_cdf.end(), u0) - ch->params_cdf.begin());
    if (pidx >= (int)ch->param_ids.size()) return chain_fail(ch, "native chain: bad parameter weights");
    const int param = ch->param_ids[pidx];
    int move;
    if (param == P_TREE) {
      const double u1 = ch->np_.res53();
      move = (std::upper_bound(ch->tree_cdf.begin(), ch->tree_cdf.end(), u1) - ch->tree_cdf.begin()) == 0 ? MV_NNI : MV_SPR;
    } else if (param == P_BL) {
      const double u1 = ch->np_.res53();
      move = (std::upper_bound(ch->bl_cdf.begin(), ch->bl_cdf.end(), u1) - ch->bl_cdf.begin()) == 0 ? MV_SCALE_EDGE : MV_NODE_SLIDER;
    } else {
      move = param == P_PI ? MV_PI : param == P_RATES ? MV_RATES : MV_ALPHA;  // np.random.randint(0, 1): no draw
    }
    ch->n_moves[move]++;

    build_kids(ch, ch->tree, k0, k1, parent_of);
    double proposed = 0.0, new_alpha = ch->alpha, beta_prop = ch->beta;
    int prop_snap = -1;
    bool tree_changed = false, full_tables = false;
    new_slots.clear();
    old_slots.clear();
    std::vector<int> changed_edges;  // indices into ch->tree whose slots were swapped (bl moves)
    std::vector<int32_t> saved;

    if (move == MV_SCALE_EDGE || move == MV_NODE_SLIDER) {
      const int E = (int)ch->tree.size();
      int ei, ui = -1;
      double new_t = 0.0, new_up = 0.0;
      if (move == MV_SCALE_EDGE) {
        ei = (int)ch->py.randbelow((uint32_t)E);
        const double old = ch->tree[ei].t;
        double log_c, c;
        multiplier(ch, log_c, c);
        new_t = old * c;
        pr_ratio = -(new_t - old) / BL_EXP_SCALE;
        hr = log_c;
        changed_edges.push_back(ei);
      } else {
        while (true) {
          ei = (int)ch->py.randbelow((uint32_t)E);
          if (ch->tree[ei].p != root) break;
        }
        ui = find_edge(ch->tree, parent_of[ch->tree[ei].p], ch->tree[ei].p);
        const double total = ch->tree[ui].t + ch->tree[ei].t;
        double log_c, c;
        multiplier(ch, log_c, c);
        const double new_total = total * c;
        new_up = new_total * ch->py.res53();
        new_t = new_total - new_up;
        pr_ratio = -(new_total - total) / BL_EXP_SCALE;
        hr = log_c;
        changed_edges.push_back(ei);
        changed_edges.push_back(ui);
      }
      // new P matrices of the changed branches, all categories (driver.py: for rate in site_rates for e in changed)
      const int nc = (int)changed_edges.size();
      new_slots.resize((size_t)nc * C);
      d.resize((size_t)nc * C);
      if (alloc_slots(ch, nc * C, new_slots.data())) return 1;
      for (int k = 0; k < C; ++k)
        for (int j = 0; j < nc; ++j) d[(size_t)k * nc + j] = (j == 0 ? new_t : new_up) * ch->site_rates[k];
      if (build_pmats(ch, pi_prop.data(), ch->beta, ch->gtr.data(), nc * C, new_slots.data(), d.data())) return 1;
      saved.resize((size_t)nc * C);
      for (int j = 0; j < nc; ++j)
        for (int k = 0; k < C; ++k) {
          saved[(size_t)j * C + k] = ch->tree[changed_edges[j]].slot[k];
          ch->tree[changed_edges[j]].slot[k] = new_slots[(size_t)k * nc + j];
        }
      todo.clear();
      path_to_root(parent_of, ch->tree[ei].c, root, todo);
      plan_nodes(ch, k0, k1);
      sort_by_plan(ch, todo, root);
      if (evaluate(ch, ch->tree, k0, k1, todo, ch->snap, pi_prop.data(), &prop_snap, &proposed)) return 1;
      // keep the new lengths aside; committed on acceptance
      prop.clear();
      prop.push_back(Edge{0, 0, new_t, {0}});
      prop.push_back(Edge{0, 0, new_up, {0}});
    } else if (move == MV_NNI) {
      prop = ch->tree;
      const int E = (int)prop.size();
      std::vector<int> order(E);
      for (int i = 0; i < E; ++i) order[i] = i;
      for (int i = E - 1; i > 0; --i) {  // random.shuffle
        const int r = (int)ch->py.randbelow((uint32_t)(i + 1));
        std::swap(order[i], order[r]);
      }
      int a = -1, b = -1;
      for (int i = 0; i < E; ++i)
        if (prop[order[i]].c > N) { a = prop[order[i]].p; b = prop[order[i]].c; break; }
      if (a < 0) return chain_fail(ch, "native chain: tree has no internal edge");
      const int src = (k0[a] == b) ? k1[a] : k0[a];
      const int tgt = (ch->py.randbelow(2u) == 0) ? k0[b] : k1[b];
      const int i_src = find_edge(prop, a, src), i_tgt = find_edge(prop, b, tgt);
      Edge e_src = prop[i_src], e_tgt = prop[i_tgt];
      // del tree[a, src], tree[b, tgt]; tree[a, tgt] = tgt_bl; tree[b, src] = src_bl   (P matrices travel with the branches)
      prop.erase(prop.begin() + std::max(i_src, i_tgt));
      prop.erase(prop.begin() + std::min(i_src, i_tgt));
      e_tgt.p = a;
      e_src.p = b;
      prop.push_back(e_tgt);
      prop.push_back(e_src);
      build_kids(ch, prop, pk0, pk1, pparent);
      plan_nodes(ch, pk0, pk1);
      todo.clear();
      todo.push_back(b);
      path_to_root(pparent, b, root, todo);
      sort_by_plan(ch, todo, root);
      if (evaluate(ch, prop, pk0, pk1, todo, ch->snap, pi_prop.data(), &prop_snap, &proposed)) return 1;
      tree_changed = true;
    } else if (move == MV_SPR) {
      prop = ch->tree;
      const int E = (int)prop.size();
      const int leaf = 1 + (int)ch->py.randbelow((uint32_t)N);   // random.randint(1, N)
      const int hub = parent_of[leaf];
      const int ti = (int)ch->py.randbelow((uint32_t)E);         // random.choice(list(tree))
      const int tp = prop[ti].p, tc = prop[ti].c;
      bool moved = false;
      if (!(hub == root || hub == tp || hub == tc || parent_of[hub] == tp || parent_of[hub] == tc)) {
        const int up = parent_of[hub];
        const int other = (k0[hub] == leaf) ? k1[hub] : k0[hub];
        const int i_x = find_edge(prop, up, hub), i_y = find_edge(prop, hub, other);
        const double x = prop[i_x].t, y = prop[i_y].t, r = prop[ti].t;
        // the three deleted branches give their slots back if the proposal is accepted
        for (int idx : {i_x, i_y, ti})
          for (int k = 0; k < C; ++k) old_slots.push_back(prop[idx].slot[k]);
        int del[3] = {i_x, i_y, ti};
        std::sort(del, del + 3);
        for (int j = 2; j >= 0; --j) prop.erase(prop.begin() + del[j]);
        const double u = ch->py.res53();
        Edge e1{tp, hub, r * u, {0}}, e2{hub, tc, r * (1.0 - u), {0}}, e3{up, other, x + y, {0}};
        hr = r / (x + y);   // the ratio itself, not its log (SURVEY F7)
        new_slots.resize((size_t)3 * C);
        d.resize((size_t)3 * C);
        if (alloc_slots(ch, 3 * C, new_slots.data())) return 1;
        Edge* ne[3] = {&e1, &e2, &e3};
        for (int j = 0; j < 3; ++j)
          for (int k = 0; k < C; ++k) {
            d[(size_t)j * C + k] = ne[j]->t * ch->site_rates[k];
            ne[j]->slot[k] = new_slots[(size_t)j * C + k];
          }
        if (build_pmats(ch, pi_prop.data(), ch->beta, ch->gtr.data(), 3 * C, new_slots.data(), d.data())) return 1;
        prop.push_back(e1);
        prop.push_back(e2);
        prop.push_back(e3);
        moved = true;
      }
      build_kids(ch, prop, pk0, pk1, pparent);
      plan_nodes(ch, pk0, pk1);
      todo.clear();
      if (moved) {
        // nodes whose child set or child branch changed, and all their ancestors in the new tree (driver._spr_dirty_nodes)
        std::vector<char> mark(2 * N, 0);
        for (const Edge& e : prop)
          if (parent_of[e.c] != e.p) mark[e.p] = 1;
        for (int cnode = 1; cnode < 2 * N; ++cnode)
          if (parent_of[cnode] >= 0 && pparent[cnode] != parent_of[cnode]) mark[parent_of[cnode]] = 1;
        for (int nd = N + 1; nd < 2 * N; ++nd) {
          if (!mark[nd]) continue;
          if (pparent[nd] < 0 && nd != root) continue;
          int x2 = nd;
          todo.push_back(x2);
          while (x2 != root) {
            x2 = pparent[x2];
            todo.push_back(x2);
          }
        }
      }
      sort_by_plan(ch, todo, root);
      if (evaluate(ch, prop, pk0, pk1, todo, ch->snap, pi_prop.data(), &prop_snap, &proposed)) return 1;
      tree_changed = true;
    } else {
      // pi / rates / alpha: every P matrix changes -> rebuild all tables, full pass (mat_mcmc_gamma.py:167-169)
      sr_prop = ch->site_rates;
      gtr_prop = ch->gtr;
      if (move == MV_PI || move == MV_RATES) {
        std::vector<double>& v = (move == MV_PI) ? pi_prop : rates_prop;
        const uint32_t n = (uint32_t)v.size();
        if (n < 2) return chain_fail(ch, "Sample larger than population or is negative");   // the reference's crash (SURVEY F5)
        uint32_t i, j;
        if (n <= 21) {  // random.sample(range(n), 2): pool branch
          i = ch->py.randbelow(n);
          uint32_t jj = ch->py.randbelow(n - 1);
          // pool[i] was replaced by pool[n - 1]
          j = (jj == i) ? n - 1 : jj;
        } else {        // set branch
          i = ch->py.randbelow(n);
          j = ch->py.randbelow(n);
          while (j == i) j = ch->py.randbelow(n);
        }
        const double total = v[i] + v[j];
        const double x = total * ch->py.res53();
        v[i] = x;
        v[j] = total - x;
        hr = 0.0;
        if (ch->model == 1 && ch->be.f81_beta(ch->be.user, pi_prop.data(), ch->S, &beta_prop)) return chain_fail(ch, "f81_beta callback failed");
        if (ch->model == 2) {
          gtr_prop.resize((size_t)ch->S + 2 * (size_t)ch->S * ch->S);
          if (ch->be.gtr_eig(ch->be.user, pi_prop.data(), rates_prop.data(), gtr_prop.data())) return chain_fail(ch, "gtr_eig callback failed");
        }
      } else {  // scale_alpha (mcmc_gamma.pyx:94-99): alpha is a C float on entry
        const double a32 = (double)(float)ch->alpha;
        double log_c, c;
        multiplier(ch, log_c, c);
        new_alpha = a32 * c;
        hr = log_c;
        pr_ratio = -(new_alpha - a32);
        if (ch->be.site_rates(ch->be.user, new_alpha, sr_prop.data())) return chain_fail(ch, "site_rates callback failed");
      }
      prop = ch->tree;
      if (build_all(ch, prop, pi_prop.data(), beta_prop, gtr_prop.data(), sr_prop.data())) return 1;
      for (const Edge& e : prop)
        for (int k = 0; k < C; ++k) new_slots.push_back(e.slot[k]);
      plan_nodes(ch, k0, k1);
      if (evaluate(ch, prop, k0, k1, ch->order_nodes, -1, pi_prop.data(), &prop_snap, &proposed, !lnl_first_now(ch))) return 1;
      full_tables = true;
      ch->full_props++;
    }

    const double current = ch->lnl;
    double ll_ratio = proposed - current + pr_ratio;
    ll_ratio += hr;
    const double log_u = log(ch->py.res53());
    const bool accepted = log_u <= ll_ratio;
    if (accepted && full_tables) {
      ch->full_accepts++;
      if (prop_snap < 0) {  // the likelihood-only pass was accepted: the same pass again, this time keeping its cache
        double again = 0.0;
        if (evaluate(ch, prop, k0, k1, ch->order_nodes, -1, pi_prop.data(), &prop_snap, &again)) return 1;
        if (again != proposed || prop_snap < 0) return chain_fail(ch, "native chain: the repeated full pass gave another likelihood");
      }
    }
    if (accepted) {
      if (move == MV_SCALE_EDGE || move == MV_NODE_SLIDER) {
        ch->tree[changed_edges[0]].t = prop[0].t;
        if (changed_edges.size() > 1) ch->tree[changed_edges[1]].t = prop[1].t;
        free_slots(ch, saved.data(), (int)saved.size());
      } else if (tree_changed) {
        ch->tree.swap(prop);
        free_slots(ch, old_slots.data(), (int)old_slots.size());
      } else if (full_tables) {
        for (const Edge& e : ch->tree) free_slots(ch, e.slot, C);
        ch->tree.swap(prop);
        ch->pi = pi_prop;
        ch->rates = rates_prop;
        ch->beta = beta_prop;
        if (move == MV_ALPHA) {
          ch->alpha = new_alpha;
          ch->site_rates = sr_prop;
        }
        ch->gtr = gtr_prop;
      }
      ch->lnl = proposed;
      be_release(ch, ch->snap);
      ch->snap = prop_snap;
      ch->n_accepts[move]++;
    } else {
      if (move == MV_SCALE_EDGE || move == MV_NODE_SLIDER) {
        for (size_t j = 0; j < changed_edges.size(); ++j)
          for (int k = 0; k < C; ++k) ch->tree[changed_edges[j]].slot[k] = saved[j * C + k];
      }
      free_slots(ch, new_slots.data(), (int)new_slots.size());
      be_release(ch, prop_snap);
    }
    if (t_move) t_move[it] = (int8_t)move;
    if (t_acc) t_acc[it] = accepted ? 1 : 0;
    if (t_cur) t_cur[it] = current;
    if (t_prop) t_prop[it] = proposed;
    if (t_ratio) t_ratio[it] = ll_ratio;
    if (t_logu) t_logu[it] = log_u;
  }
  return 0;
}

}  // namespace cbm

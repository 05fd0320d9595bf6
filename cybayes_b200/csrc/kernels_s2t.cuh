// Two-state pruning kernel for LARGE alignments on sm_100a: tile-interleaved partials, a shared-memory
// stack for the walk, bulk-async (TMA) stores -- the HBM-write-bound version of kernels_s2.cuh.
//
// Same arithmetic as prune_s2_kernel (ML_gamma.pyx:24-38 + the exact power-of-two rescale), bit for bit;
// what changes is where the bytes live and how they move:
//
//   * Layout.  A partial buffer is cut into TILES of 32 sites (one warp).  A tile is one contiguous block of
//     32 * (2C * 8 + 4) bytes (2176 for C = 4): 2C rows of 32 doubles ([category][state][site]) followed by the
//     32 rescale exponents.  The same image is used in global memory and in shared memory, so a warp moves a
//     node's tile with ONE bulk-async copy (cp.async.bulk, SASS UBLKCP) issued by an elected lane: no per-row
//     64-bit address arithmetic, no 9 STG per thread and op, and DRAM sees 2 KB bursts instead of 256-byte
//     pieces 8 MB apart.
//   * Walk with a stack in shared memory.  A warp walks the whole op range for its tile depth-first.  The
//     child finished last is carried in registers (as before); the other child of a node with two internal
//     children is PUSHED into one of K tile buffers in shared memory and popped by its parent -- it is never
//     read back from L2/HBM.  The host orders the walk (dynamic programme over the tree, cybayes_b200.cu) so
//     that almost every such child fits the K slots (C4: 1 of 210 misses with K = 4, 31 with K = 3); the
//     misses ("spills") go through global memory with plain stores/loads.  In steady state the kernel issues
//     NO register-destination global loads: the tip codes (1 byte per site and tip) arrive in shared memory through
//     4-byte cp.async copies issued two ops ahead (a load into a register would tie the op to a scoreboard that
//     unrelated instructions end up waiting on -- measured: 13 % of all stall samples on one integer add).
//   * Op images.  Everything a block used to recompute per op while staging (P rows with the missing-data
//     column, the 9-row lookup tables of folded cherries) is built ONCE per evaluation by s2t_image_kernel
//     into a 1408-byte image per op; the main kernel streams the images of its range through a two-chunk ring
//     in shared memory with bulk-async loads completing on mbarriers (the warp that finishes a chunk last
//     issues the refill: no producer warp, no block-wide barrier in the op loop).
#pragma once
#include "cb_types.cuh"
#include "kernels_s2.cuh"

namespace cb {

constexpr int S2T_W = 32;          // sites per tile
constexpr int S2T_WARPS = 8;       // tiles per block (a warp owns V consecutive tiles: 8 / V warps per block)
constexpr int S2T_THREADS = S2T_W * S2T_WARPS;
constexpr int S2T_RING_OPS = 4;    // op images per ring chunk
__host__ __device__ constexpr int s2t_ring_stages(int minb) { return minb >= 3 ? 3 : 4; }  // chunks in the ring: a refill has
                                                                                         // (stages - 1) chunks of slack
constexpr int S2T_STAGING = 2;     // bulk-store path only: tile buffers 0..1 per warp rotate as store staging, stack slots follow

__host__ __device__ constexpr int s2t_tile_bytes(int C) { return S2T_W * (2 * C * 8 + 4); }

// One op as the main kernel consumes it from shared memory.
struct S2TImage {
  double tab[2][s2_child_stage(CB_S2_MAX_CATS)];  // per child: see s2_child_stage (P rows / tip rows / cherry table)
  char* dst;                 // tile-layout partial buffer, or nullptr (not stored)
  const char* src[2];        // SRC_BUFFER: tile-layout partial buffer; SRC_TIP: code row
  const void* rows[4];       // code rows the op reads, at fixed positions: child 0 -> [0] (tip / cherry tip a), [1] (cherry
                             // tip b); child 1 -> [2], [3] (SRC_SMALL: see s2t_rank); unused positions point at a valid
                             // row (loaded, ignored)
  int32_t kind[2];           // canonical order (s2t_rank): the host swaps the children when needed
  int32_t is_root;
  int32_t combo;             // S2TCombo: the pair of child kinds, selects the specialised op body
  int32_t out_buf;           // shared-memory tile buffer that receives the result (-1: registers only)
  int32_t in_buf[2];         // SRC_STACK: tile buffer holding the child
  int32_t store_mode;        // S2TStore
  int32_t pf_buf;            // >= 0: child 1 is a stored partial that is PREFETCHED into this tile buffer two ops ahead
  int32_t pad_;              //       (cp.async, no destination registers) and then read like a stack slot
};
static_assert(sizeof(S2TImage) == 1408, "S2TImage must stay 1408 bytes (a multiple of 16)");

// Children of an op are kept in a canonical order (products and exponent sums commute exactly), which leaves twelve
// possible pairs of child kinds; each has its own straight-line op body in the kernel.
//
// An inlined (tip, cherry) subtree (SRC_SMALL) is always child 1, beside a carried child or a tip.  Its op image holds
// three children's worth of tables: tab[0] = child 0's P rows (4C doubles), the parent's P rows for the subtree (4C),
// the subtree's P rows for its tip (4C); tab[1] = the subtree's cherry table.  Code rows: [0] child 0's tip, [1] the
// subtree's tip, [2] and [3] the tips of its cherry.
__host__ __device__ constexpr int s2t_rank(int kind) {
  return kind == SRC_CARRIED ? 0 : kind == SRC_STACK ? 1 : kind == SRC_BUFFER ? 2 : kind == SRC_TIP ? 3 : kind == SRC_CHERRY ? 4 : 5;
}
enum S2TCombo : int32_t {
  S2T_CARRIED_STACK = 0, S2T_CARRIED_BUFFER, S2T_CARRIED_TIP, S2T_CARRIED_CHERRY, S2T_BUFFER_BUFFER, S2T_BUFFER_TIP,
  S2T_BUFFER_CHERRY, S2T_TIP_TIP, S2T_TIP_CHERRY, S2T_CHERRY_CHERRY, S2T_CARRIED_SMALL, S2T_TIP_SMALL, S2T_N_COMBOS
};
// does an op whose children have kinds k0, k1 (canonical order) read code row q of its image?
__host__ __device__ inline bool s2t_row_used(int k0, int k1, int q) {
  return q == 0 ? (k0 == SRC_TIP || k0 == SRC_CHERRY) : q == 1 ? (k0 == SRC_CHERRY || k1 == SRC_SMALL)
                                                               : (k1 == SRC_CHERRY || k1 == SRC_SMALL || (q == 2 && k1 == SRC_TIP));
}
__host__ __device__ inline int s2t_combo(int k0, int k1) {   // kinds in canonical order; -1: not a pair the walk produces
  if (k0 == SRC_CARRIED) return k1 == SRC_STACK ? S2T_CARRIED_STACK : k1 == SRC_BUFFER ? S2T_CARRIED_BUFFER : k1 == SRC_TIP ? S2T_CARRIED_TIP : k1 == SRC_CHERRY ? S2T_CARRIED_CHERRY : k1 == SRC_SMALL ? S2T_CARRIED_SMALL : -1;
  if (k0 == SRC_BUFFER) return k1 == SRC_BUFFER ? S2T_BUFFER_BUFFER : k1 == SRC_TIP ? S2T_BUFFER_TIP : k1 == SRC_CHERRY ? S2T_BUFFER_CHERRY : -1;
  if (k0 == SRC_TIP) return k1 == SRC_TIP ? S2T_TIP_TIP : k1 == SRC_CHERRY ? S2T_TIP_CHERRY : k1 == SRC_SMALL ? S2T_TIP_SMALL : -1;
  if (k0 == SRC_CHERRY) return k1 == SRC_CHERRY ? S2T_CHERRY_CHERRY : -1;
  return -1;
}
// how the result of an op leaves the registers
enum S2TStore : int32_t {
  S2T_ST_NONE = 0,     // carried only
  S2T_ST_SMEM = 1,     // into a stack slot in shared memory (out_buf)
  S2T_ST_GLOBAL = 2,   // plain coalesced stores to the buffer tile (the tile is contiguous: nine 256-byte rows back to back)
  S2T_ST_STREAM = 4,   // ... with the streaming (evict-first) hint: nobody reads the partial back in this evaluation
  S2T_ST_BULK = 8      // through a tile buffer in shared memory (out_buf) and one bulk-async copy (CYBAYES_S2T_BULK=1)
};

constexpr int S2T_CODE_SLOTS = 4;  // per tile: tip codes of 4 consecutive ops (4 rows x 32 sites x 1 byte each), cp.async ring
constexpr int S2T_CODE_BYTES = S2T_CODE_SLOTS * 4 * S2T_W;

__host__ __device__ inline size_t s2t_smem_bytes(int n_bufs, int C, int minb) {
  return (size_t)s2t_ring_stages(minb) * S2T_RING_OPS * sizeof(S2TImage) + (size_t)S2T_WARPS * S2T_CODE_BYTES +
         (size_t)S2T_WARPS * n_bufs * s2t_tile_bytes(C) + 64;
}

// ---------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ unsigned s2t_smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void s2t_mbar_init(void* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s2t_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void s2t_mbar_expect_tx(void* bar, unsigned bytes) {
  asm volatile("{\n .reg .b64 st;\n mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}\n" ::"r"(s2t_smem_addr(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void s2t_mbar_wait(void* bar, unsigned parity) {
  const unsigned a = s2t_smem_addr(bar);
  asm volatile(
      "{\n"
      " .reg .pred p;\n"
      "S2T_WAIT_%=:\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra S2T_DONE_%=;\n"
      " bra S2T_WAIT_%=;\n"
      "S2T_DONE_%=:\n"
      "}\n" ::"r"(a), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void s2t_bulk_g2s(void* smem, const void* gmem, unsigned bytes, void* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(s2t_smem_addr(smem)),
               "l"(gmem), "r"(bytes), "r"(s2t_smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void s2t_bulk_s2g(void* gmem, const void* smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(gmem), "r"(s2t_smem_addr(smem)), "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
template <int N>
__device__ __forceinline__ void s2t_bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;\n" ::"n"(N) : "memory");
}
__device__ __forceinline__ void s2t_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory"); }
__device__ __forceinline__ void s2t_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }
// 4-byte asynchronous copy global -> shared (LDGSTS): no destination register, completion tracked per thread in groups
__device__ __forceinline__ void s2t_cp_async4(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s2t_smem_addr(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void s2t_cp_async8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s2t_smem_addr(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void s2t_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void s2t_cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s2t_smem_addr(smem)), "l"(gmem) : "memory");
}
template <int N>
__device__ __forceinline__ void s2t_cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------ pre-pass
// One block (32 threads) per op: descriptor + per-child tables.  Exactly the arithmetic prune_s2_kernel does
// while staging a chunk, so both kernels see the same table entries bit for bit.
template <int C>
__global__ void __launch_bounds__(32) s2t_image_kernel(const LaunchConst k, int n_ops, S2TImage* __restrict__ images) {
  constexpr int CS = s2_child_stage(CB_S2_MAX_CATS);
  const int o = blockIdx.x;
  if (o >= n_ops) return;
  const OpDesc* __restrict__ op = k.ops + o;
  S2TImage* im = images + o;
  const int t = threadIdx.x;
  if (t == 0) {
    im->dst = reinterpret_cast<char*>(op->dst);
    im->src[0] = static_cast<const char*>(op->src[0]);
    im->src[1] = static_cast<const char*>(op->src[1]);
    for (int ch = 0; ch < 2; ++ch) {
      const int kind = op->kind[ch];
      im->rows[2 * ch] = kind == SRC_TIP ? op->src[ch] : kind == SRC_CHERRY ? op->ctip[ch][0] : k.codes;
      im->rows[2 * ch + 1] = kind == SRC_CHERRY ? op->ctip[ch][1] : k.codes;
    }
    if (op->kind[1] == SRC_SMALL) {   // the subtree's own descriptor holds its children in canonical order: (tip, cherry)
      const OpDesc* sub = k.ops + op->in_buf[1];
      im->rows[1] = sub->src[0];
      im->rows[2] = sub->ctip[1][0];
      im->rows[3] = sub->ctip[1][1];
    }
    im->kind[0] = op->kind[0]; im->kind[1] = op->kind[1];
    im->is_root = op->is_root;
    im->combo = s2t_combo(op->kind[0], op->kind[1]);
    im->out_buf = op->out_buf;
    im->in_buf[0] = op->in_buf[0]; im->in_buf[1] = op->in_buf[1];
    // out_buf names a stack slot (the op is pushed) or a staging buffer of the bulk-store path
    const bool stored = op->dst != nullptr, pushed = (op->spill & 2) != 0, staged = op->out_buf >= 0 && !pushed;
    const bool spill = (op->spill & 1) != 0;
    int mode = pushed ? S2T_ST_SMEM : S2T_ST_NONE;
    if (stored) {
      if (staged || (pushed && k.s2t_bulk && !spill)) mode |= S2T_ST_BULK;
      else mode |= S2T_ST_GLOBAL | (op->pad_ ? S2T_ST_STREAM : 0);
    }
    im->store_mode = mode;
    im->pf_buf = op->pf_buf;
    im->pad_ = 0;
  }
  // a small subtree that stays in the returned cache as a record (never stored) keeps copies of its two edges' P
  if (op->frec_out >= 0)
    for (int idx = t; idx < 2 * C * 4; idx += 32) {
      const int e = idx & 3, c = (idx >> 2) % C, ch = idx / (4 * C);
      k.pmats_lib[((int64_t)op->frec_out * 2 * C + ch * C + c) * 4 + e] = __ldg(s2_pmat(k, op->pslot[ch][c]) + e);
    }
  // P matrices of internal and tip children (one thread per child, category and row); an inlined subtree's rows go
  // to tab[0] behind child 0's, followed by the rows of the subtree's edge to its tip
  for (int idx = t; idx < 6 * C; idx += 32) {
    const int i = idx & 1, c = (idx >> 1) % C, ch = min(idx / (2 * C), 1);
    const int kind = op->kind[ch];
    if (kind == SRC_CHERRY || (idx >= 4 * C && kind != SRC_SMALL)) continue;
    const int32_t slot = idx >= 4 * C ? k.ops[op->in_buf[1]].pslot[0][c] : op->pslot[ch][c];
    const double2 pr = __ldg(reinterpret_cast<const double2*>(s2_pmat(k, slot)) + i);
    if (kind == SRC_SMALL) reinterpret_cast<double2*>(&im->tab[0][0])[(idx >= 4 * C ? 4 * C : 2 * C) + c * 2 + i] = pr;
    else reinterpret_cast<double2*>(&im->tab[ch][0])[c * 2 + i] = pr;   // tips use the same rows (see s2t_child)
  }
  // lookup tables of folded cherries (one thread per child and pair of tip codes); an inlined subtree's cherry is
  // child 1 of the subtree's descriptor
  for (int idx = t; idx < 18; idx += 32) {
    const int q = idx % 9, ch = idx / 9;
    if (op->kind[ch] != SRC_CHERRY && op->kind[ch] != SRC_SMALL) continue;
    const OpDesc* cd = op->kind[ch] == SRC_SMALL ? k.ops + op->in_buf[ch] : op;
    const int cc = op->kind[ch] == SRC_SMALL ? 1 : ch;
    const int ca = q / 3, cb_ = q - 3 * ca;
    double L[C][2];
    int mh = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const double2* pa = reinterpret_cast<const double2*>(s2_pmat(k, cd->cslot[cc][0][c]));
      const double2* pb = reinterpret_cast<const double2*>(s2_pmat(k, cd->cslot[cc][1][c]));
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        L[c][j] = s2_tip_term(__ldg(pa + j), ca) * s2_tip_term(__ldg(pb + j), cb_);
        mh = max(mh, __double2hiint(L[c][j]));
      }
    }
    const int be = (mh >> 20) & 0x7ff;
    const int x = (be == 0 || be == 0x7ff) ? 0 : be - 1023;
    const double f = pow2_neg(x);
    double* tab = &im->tab[ch][0] + q * (2 * C + 1);
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const double l0 = L[c][0] * f, l1 = L[c][1] * f;
      const double2* pp = reinterpret_cast<const double2*>(s2_pmat(k, cd->pslot[cc][c]));
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double2 pr = __ldg(pp + i);
        tab[c * 2 + i] = fma(pr.y, l1, pr.x * l0);
      }
    }
    tab[2 * C] = (double)x;
    // a cherry that stays in the returned cache keeps its own copy of its two edges' P matrices (an inlined subtree's
    // descriptor gets an image of its own, which writes its records' copies)
    if (q == 0 && cd == op && op->crec_out[ch] >= 0) {
      double* out = k.pmats_lib + (int64_t)op->crec_out[ch] * 2 * C * 4;
#pragma unroll
      for (int tt = 0; tt < 2; ++tt)
#pragma unroll
        for (int c = 0; c < C; ++c) {
          const double* src = s2_pmat(k, op->cslot[ch][tt][c]);
#pragma unroll
          for (int e = 0; e < 4; ++e) out[(tt * C + c) * 4 + e] = __ldg(src + e);
        }
    }
  }
  (void)CS;
}

// ---------------------------------------------------------------------------------------- main kernel
// A warp owns V consecutive tiles (V = 2 by default: lane l handles site l of either tile).  Everything that does not
// depend on the site -- the op image, the jump to the op body, the broadcast loads of the P rows, pointer arithmetic,
// the ring and code pipelines -- is done once for both tiles, and the two sites' dependency chains interleave.
//
// contribution of one child to the op's product: FIRST initialises acc, the second child multiplies into it.
// codes: this op's slot of the warp's code ring, [row q][V * 32 sites]: child 0 uses rows 0, 1, child 1 rows 2, 3.
template <int C, int V, int KIND, int CH, bool FIRST>
__device__ __forceinline__ void s2t_child(const S2TImage& im, const double (&cur)[V][C][2], const int (&cur_e)[V],
                                          const unsigned char* codes, const unsigned char* mybufs, size_t tile_off, int lane,
                                          double (&acc)[V][C][2], int (&e_in)[V]) {
  constexpr int TB = s2t_tile_bytes(C);
  const double* pbase = &im.tab[CH][0];
  if constexpr (KIND == SRC_CARRIED || KIND == SRC_STACK || KIND == SRC_BUFFER) {
    double L[V][C][2];
    int se[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      if constexpr (KIND == SRC_CARRIED) {
#pragma unroll
        for (int c = 0; c < C; ++c) { L[v][c][0] = cur[v][c][0]; L[v][c][1] = cur[v][c][1]; }
        se[v] = cur_e[v];
      } else if constexpr (KIND == SRC_STACK) {
        const double* sb = reinterpret_cast<const double*>(mybufs + ((size_t)im.in_buf[CH] * V + v) * TB);
#pragma unroll
        for (int c = 0; c < C; ++c) {
          L[v][c][0] = sb[(2 * c) * S2T_W + lane];
          L[v][c][1] = sb[(2 * c + 1) * S2T_W + lane];
        }
        se[v] = reinterpret_cast<const int*>(sb + 2 * C * S2T_W)[lane];
      } else {
        const double* gb = reinterpret_cast<const double*>(im.src[CH] + tile_off + (size_t)v * TB);
#pragma unroll
        for (int c = 0; c < C; ++c) {
          L[v][c][0] = __ldcg(gb + (2 * c) * S2T_W + lane);
          L[v][c][1] = __ldcg(gb + (2 * c + 1) * S2T_W + lane);
        }
        se[v] = __ldcg(reinterpret_cast<const int*>(gb + 2 * C * S2T_W) + lane);
      }
    }
    const double2* pm = reinterpret_cast<const double2*>(pbase);   // (P[i][0], P[i][1]) broadcasts, shared by the V sites
#pragma unroll
    for (int c = 0; c < C; ++c) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double2 pr = pm[c * 2 + i];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const double x = fma(pr.y, L[v][c][1], pr.x * L[v][c][0]);      // v[i] = P[i][0] L[0] + P[i][1] L[1]
          if (FIRST) acc[v][c][i] = x; else acc[v][c][i] *= x;
        }
      }
    }
#pragma unroll
    for (int v = 0; v < V; ++v) { if (FIRST) e_in[v] = se[v]; else e_in[v] += se[v]; }
  } else if constexpr (KIND == SRC_TIP) {
    // A tip is its 0/1 indicator column (utils.pyx:99-111): state code 0 -> (1, 0), 1 -> (0, 1), missing -> (1, 1), run
    // through the same FMA chain as an internal child -- P[i][0], P[i][1] or fma(P[i][1], 1, P[i][0]) bit for bit.  The
    // P rows are broadcast loads shared by the V sites: 8 shared-memory wavefronts instead of 16 per site for a
    // per-lane table look-up (the kernel is bound by the shared-memory data pipe, not by FP64 issue).
    double m0[V], m1[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const unsigned cd = codes[(2 * CH) * (S2T_W * V) + v * S2T_W + lane];
      m0[v] = cd == 1u ? 0.0 : 1.0;
      m1[v] = cd == 0u ? 0.0 : 1.0;
    }
    const double2* pm = reinterpret_cast<const double2*>(pbase);
#pragma unroll
    for (int c = 0; c < C; ++c) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double2 pr = pm[c * 2 + i];
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const double x = fma(pr.y, m1[v], pr.x * m0[v]);
          if (FIRST) acc[v][c][i] = x; else acc[v][c][i] *= x;
        }
      }
    }
#pragma unroll
    for (int v = 0; v < V; ++v) if (FIRST) e_in[v] = 0;
  } else if constexpr (KIND == SRC_SMALL) {
    // A (tip, cherry) subtree, computed exactly as its own TIP_CHERRY op would (tip rows, times the cherry's row, then
    // the same power-of-two rescale) and then fed through the parent's P rows like a carried child.
    static_assert(CH == 1 && !FIRST, "an inlined subtree is child 1");
    const double2* pt = reinterpret_cast<const double2*>(&im.tab[0][0]) + 4 * C;   // subtree -> its tip
    const double2* pm = reinterpret_cast<const double2*>(&im.tab[0][0]) + 2 * C;   // parent -> subtree
    double L[V][C][2];
    int se[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const unsigned cd = codes[1 * (S2T_W * V) + v * S2T_W + lane];
      const double m0 = cd == 1u ? 0.0 : 1.0, m1 = cd == 0u ? 0.0 : 1.0;
#pragma unroll
      for (int c = 0; c < C; ++c)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const double2 pr = pt[c * 2 + i];
          L[v][c][i] = fma(pr.y, m1, pr.x * m0);
        }
      const unsigned ca = min((unsigned)codes[2 * (S2T_W * V) + v * S2T_W + lane], 2u);
      const unsigned cb_ = min((unsigned)codes[3 * (S2T_W * V) + v * S2T_W + lane], 2u);
      const double* tab = pbase + (ca * 3 + cb_) * (2 * C + 1);
      int mh = 0;
#pragma unroll
      for (int c = 0; c < C; ++c)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          L[v][c][i] *= tab[c * 2 + i];
          mh = c == 0 && i == 0 ? __double2hiint(L[v][0][0]) : max(mh, __double2hiint(L[v][c][i]));
        }
      const int be = (mh >> 20) & 0x7ff;
      const int x = (be == 0 || be == 0x7ff) ? 0 : be - 1023;
      const double f = pow2_neg(x);
#pragma unroll
      for (int c = 0; c < C; ++c) { L[v][c][0] *= f; L[v][c][1] *= f; }
      se[v] = (int)tab[2 * C] + x;
    }
#pragma unroll
    for (int c = 0; c < C; ++c) {
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double2 pr = pm[c * 2 + i];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v][c][i] *= fma(pr.y, L[v][c][1], pr.x * L[v][c][0]);
      }
    }
#pragma unroll
    for (int v = 0; v < V; ++v) e_in[v] += se[v];
  } else {  // folded cherry: the pair of tip codes selects a precomputed row
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const unsigned ca = min((unsigned)codes[(2 * CH) * (S2T_W * V) + v * S2T_W + lane], 2u);
      const unsigned cb_ = min((unsigned)codes[(2 * CH + 1) * (S2T_W * V) + v * S2T_W + lane], 2u);
      const double* tab = pbase + (ca * 3 + cb_) * (2 * C + 1);
#pragma unroll
      for (int c = 0; c < C; ++c) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const double x = tab[c * 2 + i];
          if (FIRST) acc[v][c][i] = x; else acc[v][c][i] *= x;
        }
      }
      if (FIRST) e_in[v] = (int)tab[2 * C]; else e_in[v] += (int)tab[2 * C];
    }
  }
}

template <int C, int V, int K0, int K1>
__device__ __forceinline__ void s2t_pair(const S2TImage& im, const double (&cur)[V][C][2], const int (&cur_e)[V],
                                         const unsigned char* codes, const unsigned char* mybufs, size_t tile_off, int lane,
                                         double (&out)[V][C][2], int (&e_in)[V]) {
  s2t_child<C, V, K0, 0, true>(im, cur, cur_e, codes, mybufs, tile_off, lane, out, e_in);
  s2t_child<C, V, K1, 1, false>(im, cur, cur_e, codes, mybufs, tile_off, lane, out, e_in);
}

// MINB: resident blocks per SM the kernel is compiled for; V: tiles per warp (block = 8 / V warps)
template <int C, int MINB, int V>
__global__ void __launch_bounds__(S2T_THREADS / V, MINB) prune_s2t_kernel(const LaunchConst k, const S2TImage* __restrict__ images,
                                                                           int n_bufs) {
  static_assert(C <= CB_S2_MAX_CATS, "2-state kernel supports at most CB_S2_MAX_CATS categories");
  static_assert(V == 1 || V == 2, "one or two tiles per warp");
  constexpr int TB = s2t_tile_bytes(C);
  constexpr int WARPS = S2T_WARPS / V;
  constexpr int S2T_RING_STAGES = s2t_ring_stages(MINB);
  constexpr int RING = S2T_RING_OPS * S2T_RING_STAGES;
  extern __shared__ __align__(128) unsigned char s2t_smem[];
  __shared__ double red[32];
  __shared__ int last_flag;
  __shared__ int done_cnt[S2T_RING_STAGES];
  __shared__ __align__(8) unsigned long long full_bar[S2T_RING_STAGES];

  const RangeDesc rg = k.ranges[blockIdx.y];
  const int nops = rg.end - rg.begin;
  const int n_chunks = (nops + S2T_RING_OPS - 1) / S2T_RING_OPS;
  const S2TImage* __restrict__ gimg = images + rg.begin;
  S2TImage* ring = reinterpret_cast<S2TImage*>(s2t_smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* mycodes = s2t_smem + (size_t)RING * sizeof(S2TImage) + (size_t)warp * V * S2T_CODE_BYTES;
  unsigned char* mybufs = s2t_smem + (size_t)RING * sizeof(S2TImage) + (size_t)S2T_WARPS * S2T_CODE_BYTES +
                          (size_t)warp * V * n_bufs * TB;

  const int64_t n_tiles = k.n_sites / S2T_W;                      // a multiple of 2 (sites are padded to 64)
  const int64_t tile = ((int64_t)blockIdx.x * WARPS + warp) * V;   // first of this warp's V tiles
  const int64_t tiles_left = n_tiles - (int64_t)blockIdx.x * S2T_WARPS;
  const int n_active = tiles_left < S2T_WARPS ? (int)((tiles_left + V - 1) / V) : WARPS;   // warps of this block that own tiles
  const bool active = warp < n_active;
  const int64_t site = tile * S2T_W + lane;
  const size_t tile_off = (size_t)tile * TB;

  auto issue_chunk = [&](int c) {  // one thread: bulk-load the images of chunk c into its ring stage
    const int b = c % S2T_RING_STAGES;
    const int n = min(S2T_RING_OPS, nops - c * S2T_RING_OPS);
    const unsigned bytes = (unsigned)n * (unsigned)sizeof(S2TImage);
    s2t_mbar_expect_tx(&full_bar[b], bytes);
    s2t_bulk_g2s(ring + (size_t)b * S2T_RING_OPS, gimg + (size_t)c * S2T_RING_OPS, bytes, &full_bar[b]);
  };
  // the warp's tip codes of op o: lane = 8 q + j copies bytes [4 V j, 4 V (j + 1)) of the 32 V codes of row q
  const int64_t code_off = tile * S2T_W + 4 * V * (lane & 7);
  auto issue_codes = [&](int o) {
    const S2TImage& im = ring[o % RING];
    unsigned char* dst = mycodes + (o % S2T_CODE_SLOTS) * (4 * S2T_W * V) + 4 * V * lane;
    const char* src = static_cast<const char*>(im.rows[lane >> 3]) + code_off;
    if constexpr (V == 1) s2t_cp_async4(dst, src); else s2t_cp_async8(dst, src);
  };
  // a stored partial that op o reads as its second child: the warp's V tiles (V * TB bytes, contiguous) in 16-byte pieces
  auto issue_prefetch = [&](int o) {
    const S2TImage& im = ring[o % RING];
    if (im.pf_buf >= 0) {
      const char* src = im.src[1] + tile_off;
      unsigned char* dst = mybufs + (size_t)im.pf_buf * V * TB;
#pragma unroll
      for (int j = 0; j < (V * TB / 16 + 31) / 32; ++j) {
        const int idx = lane + 32 * j;
        if (idx < V * TB / 16) s2t_cp_async16(dst + 16 * idx, src + 16 * idx);
      }
    }
  };
  auto wait_chunk_of = [&](int o) {  // the image of op o is in the ring (o is the first op of its chunk)
    const int c1 = o / S2T_RING_OPS;
    s2t_mbar_wait(&full_bar[c1 % S2T_RING_STAGES], (unsigned)(c1 / S2T_RING_STAGES) & 1u);
  };

  if (threadIdx.x == 0) {
#pragma unroll
    for (int b = 0; b < S2T_RING_STAGES; ++b) {
      s2t_mbar_init(&full_bar[b], 1);
      done_cnt[b] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    for (int c = 0; c < S2T_RING_STAGES && c < n_chunks; ++c) issue_chunk(c);
  }
  __syncthreads();

  double lnl = 0.0;
  if (active) {
    double cur[V][C][2];  // carried partial
    int cur_e[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      cur_e[v] = 0;
#pragma unroll
      for (int c = 0; c < C; ++c) cur[v][c][0] = cur[v][c][1] = 0.0;
    }
    bool groups_pending = false;

    // code pipeline: the copies of op o + 2 are issued at the end of op o; one commit group per op
    wait_chunk_of(0);
    issue_codes(0);
    issue_prefetch(0);
    s2t_cp_async_commit();
    if (nops > 1) {
      if (S2T_RING_OPS == 1) wait_chunk_of(1);
      issue_codes(1);
      issue_prefetch(1);
    }
    s2t_cp_async_commit();

#pragma unroll 1
    for (int o = 0; o < nops; ++o) {
      const S2TImage& im = ring[o % RING];
      s2t_cp_async_wait<1>();   // this op's codes have landed (the group of op o + 1 may still be in flight)
      __syncwarp();
      const unsigned char* codes = mycodes + (o % S2T_CODE_SLOTS) * (4 * S2T_W * V);

      double out[V][C][2];
      int e_in[V];
      switch (im.combo) {
#define CB_S2T_CASE(NAME, K0, K1) \
  case NAME: s2t_pair<C, V, K0, K1>(im, cur, cur_e, codes, mybufs, tile_off, lane, out, e_in); break;
        CB_S2T_CASE(S2T_CARRIED_STACK, SRC_CARRIED, SRC_STACK)
        CB_S2T_CASE(S2T_CARRIED_BUFFER, SRC_CARRIED, SRC_BUFFER)
        CB_S2T_CASE(S2T_CARRIED_TIP, SRC_CARRIED, SRC_TIP)
        CB_S2T_CASE(S2T_CARRIED_CHERRY, SRC_CARRIED, SRC_CHERRY)
        CB_S2T_CASE(S2T_BUFFER_BUFFER, SRC_BUFFER, SRC_BUFFER)
        CB_S2T_CASE(S2T_BUFFER_TIP, SRC_BUFFER, SRC_TIP)
        CB_S2T_CASE(S2T_BUFFER_CHERRY, SRC_BUFFER, SRC_CHERRY)
        CB_S2T_CASE(S2T_TIP_TIP, SRC_TIP, SRC_TIP)
        CB_S2T_CASE(S2T_TIP_CHERRY, SRC_TIP, SRC_CHERRY)
        CB_S2T_CASE(S2T_CARRIED_SMALL, SRC_CARRIED, SRC_SMALL)
        CB_S2T_CASE(S2T_TIP_SMALL, SRC_TIP, SRC_SMALL)
        default:
          s2t_pair<C, V, SRC_CHERRY, SRC_CHERRY>(im, cur, cur_e, codes, mybufs, tile_off, lane, out, e_in);
          break;
#undef CB_S2T_CASE
      }

      if (!im.is_root) {
        // exact power-of-two rescale: all entries are >= 0, so the max of the high words carries the exponent of the max
#pragma unroll
        for (int v = 0; v < V; ++v) {
          int mh = __double2hiint(out[v][0][0]);
#pragma unroll
          for (int c = 0; c < C; ++c) mh = max(mh, max(__double2hiint(out[v][c][0]), __double2hiint(out[v][c][1])));
          const int be = (mh >> 20) & 0x7ff;
          const int x = (be == 0 || be == 0x7ff) ? 0 : be - 1023;
          const double f = pow2_neg(x);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            cur[v][c][0] = out[v][c][0] * f;
            cur[v][c][1] = out[v][c][1] * f;
          }
          cur_e[v] = e_in[v] + x;
        }
      } else {
        // ll_p = sum_c (pi . L_c) / n_cats ; lnL += w_p * log(ll_p)      ML_gamma.pyx:38,40
        const double pi0 = __ldg(k.pi), pi1 = __ldg(k.pi + 1);
        const double ln2 = 0.693147180559945309417232121458;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const double w = __ldg(k.weights + site + v * S2T_W);
          double s = 0.0;
#pragma unroll
          for (int c = 0; c < C; ++c) s += fma(pi1, out[v][c][1], pi0 * out[v][c][0]) / k.cats;
          if (w != 0.0) lnl += w * (log(s) + (double)e_in[v] * ln2);
#pragma unroll
          for (int c = 0; c < C; ++c) {   // an (optionally) stored root partial is kept as computed, exponent e_in
            cur[v][c][0] = out[v][c][0];
            cur[v][c][1] = out[v][c][1];
          }
          cur_e[v] = e_in[v];
        }
      }

      const int mode = im.store_mode;
      if (mode != S2T_ST_NONE) {
        if (mode & S2T_ST_GLOBAL) {  // plain coalesced stores: a tile is one contiguous 2 KB piece of the buffer
#pragma unroll
          for (int v = 0; v < V; ++v) {
            double* gb = reinterpret_cast<double*>(im.dst + tile_off + (size_t)v * TB);
            if (mode & S2T_ST_STREAM) {
#pragma unroll
              for (int c = 0; c < C; ++c) {
                __stcs(gb + (2 * c) * S2T_W + lane, cur[v][c][0]);
                __stcs(gb + (2 * c + 1) * S2T_W + lane, cur[v][c][1]);
              }
              __stcs(reinterpret_cast<int*>(gb + 2 * C * S2T_W) + lane, cur_e[v]);
            } else {
#pragma unroll
              for (int c = 0; c < C; ++c) {
                __stcg(gb + (2 * c) * S2T_W + lane, cur[v][c][0]);
                __stcg(gb + (2 * c + 1) * S2T_W + lane, cur[v][c][1]);
              }
              __stcg(reinterpret_cast<int*>(gb + 2 * C * S2T_W) + lane, cur_e[v]);
            }
          }
        }
        if (mode & (S2T_ST_SMEM | S2T_ST_BULK)) {
          if (groups_pending) {
            // a staging buffer was last read by the bulk copy two groups ago; a stack slot may have been read by the
            // latest group, so wait for all of them there
            if (mode & S2T_ST_SMEM) s2t_bulk_wait_read<0>(); else s2t_bulk_wait_read<1>();
            __syncwarp();
          }
          unsigned char* sb0 = mybufs + (size_t)im.out_buf * V * TB;
#pragma unroll
          for (int v = 0; v < V; ++v) {
            double* sb = reinterpret_cast<double*>(sb0 + (size_t)v * TB);
#pragma unroll
            for (int c = 0; c < C; ++c) {
              sb[(2 * c) * S2T_W + lane] = cur[v][c][0];
              sb[(2 * c + 1) * S2T_W + lane] = cur[v][c][1];
            }
            reinterpret_cast<int*>(sb + 2 * C * S2T_W)[lane] = cur_e[v];
          }
          if (mode & S2T_ST_BULK) {
            s2t_fence_async_smem();
            __syncwarp();
            if (lane == 0) s2t_bulk_s2g(im.dst + tile_off, sb0, V * TB);
            groups_pending = true;
          }  // (a pushed tile is popped by the lanes that wrote it: columns are lane-private, no barrier needed)
        }
      }

      // codes of op o + 2 (its image must be in the ring: entering a chunk also pulls the tips two chunks ahead to L2)
      if (o + 2 < nops) {
        if ((o + 2) % S2T_RING_OPS == 0) {
          wait_chunk_of(o + 2);
          const int c1 = (o + 2) / S2T_RING_OPS;
          const int e = (c1 + 2) * S2T_RING_OPS + (lane >> 2);
          if (lane < 4 * S2T_RING_OPS && e < nops && warp == c1 % n_active) {  // one warp per block and chunk does it
            const S2TImage& ie = gimg[e];   // (the image kernel ran before this launch)
            const int q = lane & 3;
            if (s2t_row_used(ie.kind[0], ie.kind[1], q)) {
              const void* row = ie.rows[q];
              const char* a = static_cast<const char*>(row) + (int64_t)blockIdx.x * S2T_WARPS * S2T_W;   // the block's 256 sites
              asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
              asm volatile("prefetch.global.L2 [%0];" ::"l"(a + 128));
            }
          }
        }
        issue_codes(o + 2);
        issue_prefetch(o + 2);
      }
      s2t_cp_async_commit();

      // leaving a chunk: the warp that finishes it last refills its ring stage with the chunk STAGES ahead
      if ((o + 1) % S2T_RING_OPS == 0) {
        const int chunk = o / S2T_RING_OPS;
        if (chunk + S2T_RING_STAGES < n_chunks) {
          __syncwarp();
          if (lane == 0) {
            const int b = chunk % S2T_RING_STAGES;
            if (atomicAdd(&done_cnt[b], 1) == n_active - 1) {
              done_cnt[b] = 0;
              s2t_fence_async_smem();  // the warps' reads of this ring stage before the async writes
              issue_chunk(chunk + S2T_RING_STAGES);
            }
          }
        }
      }
    }
    if (groups_pending && lane == 0) s2t_bulk_wait_all();
  }
  if (rg.out_index >= 0) block_reduce_to_result(lnl, k, rg.out_index, red, &last_flag);
}

}  // namespace cb

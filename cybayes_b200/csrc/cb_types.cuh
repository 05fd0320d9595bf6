// Device-visible descriptors shared by the host scheduler and the pruning kernels.  Also compiled by the host compiler
// alone (plan.cpp), so nothing here needs CUDA headers.
#pragma once
#include <stdint.h>
#include "../../include/cybayes_b200.h"

#ifdef __CUDACC__
#define CB_HD __host__ __device__
#else
#define CB_HD
#endif

namespace cb {

// SRC_CHERRY (2-state family only): the child is a "cherry" -- an internal node whose two children are
// tips.  Its partial has only 3 x 3 possible values per rate category (state code of either tip: 0, 1,
// missing), so it is never computed per site, stored or read: the parent looks its contribution up.
// SRC_STACK (tiled 2-state kernel only): the child was pushed into a shared-memory tile buffer by an earlier op of the walk.
// SRC_SMALL (tiled 2-state kernel only): the child is a (tip, cherry) subtree that the parent's op computes itself, so it
// costs no op of its own and no stack slot.  Its descriptor is not in any range; in_buf names it (an index into ops).
enum SrcKind : int32_t { SRC_TIP = 0, SRC_BUFFER = 1, SRC_CARRIED = 2, SRC_CHERRY = 3, SRC_STACK = 4, SRC_SMALL = 5 };

constexpr int CB_S2_MAX_CATS = 4;            // rate categories of the 2-state kernels (1 or 4)
constexpr int32_t CB_LIB_SLOT = 1 << 30;     // P-slot ids with this bit address the library's own pool

// One node operation: L_node = (P_a . L_a) * (P_b . L_b), ML_gamma.pyx:24-36.
// 256 bytes, read by every block of a launch through the read-only path.
struct OpDesc {
  double* dst;                  // [C][S][P] or nullptr (not stored)
  int32_t* dst_scale;           // [P] (2-state family) or [C][P] (general family)
  const void* src[2];           // tip code row, partial buffer, or nullptr when carried / cherry
  const int32_t* src_scale[2];  // nullptr for tips
  int32_t kind[2];              // SrcKind
  int32_t pslot[2][CB_MAX_CATS];
  int32_t is_root;
  int32_t pad_;
  // folded cherry children (kind == SRC_CHERRY)
  const void* ctip[2][2];                  // code rows of the cherry's two tips
  int32_t cslot[2][2][CB_S2_MAX_CATS];     // P slots of the cherry's two tip edges, per category
  int32_t crec_out[2];                     // library record that must keep a copy of those P, or -1
  // tiled 2-state kernel (kernels_s2t.cuh)
  int32_t out_buf;                         // shared-memory tile buffer receiving the result, or -1
  int32_t in_buf[2];                       // kind == SRC_STACK: tile buffer holding the child; SRC_SMALL: its op index
  int32_t spill;                           // bit 0: stored AND read back inside the same launch (plain stores);
                                           // bit 1: out_buf is a stack slot (the result is popped by a later op)
  int32_t frec_out;                        // library record that must keep a copy of THIS op's two edges' P, or -1
  int32_t pf_buf;                          // >= 0: child 1 (SRC_STACK, src[1] = its stored partial) is prefetched into this tile buffer
};
static_assert(sizeof(OpDesc) == 256, "OpDesc must stay 256 bytes");

// A block walks ops [begin, end) in order for its site tile; results of a root op go to
// results[out_index].
struct RangeDesc {
  int32_t begin, end, out_index, pad_;
};

struct LaunchConst {
  const OpDesc* ops;
  const RangeDesc* ranges;
  const double* pmats;     // slot pool, S*S doubles per slot
  double* pmats_lib;       // library-owned slots (copies of the P matrices of folded cherries)
  const double* staged;    // register-carried DMMA kernel: P matrices re-laid out in consumption order (rc_restage_kernel)
  const double* weights;   // [P]
  const double* pi;        // [S]
  const double* amb;       // [n_amb][S] 0/1
  double* block_sums;      // [n_out][max_blocks]
  unsigned int* tickets;   // [n_out]
  double* results;         // [n_out]
  double* root_dot;        // general family: [n_out][C][P] per-category pi.L_root
  int32_t* root_exp;       // general family: [n_out][C][P]
  int64_t n_sites;         // padded pattern count P (multiple of 64)
  int32_t n_states, n_cats, code_bytes, max_blocks;
  double cats;            // n_cats as a double (the reference divides, ML_gamma.pyx:38)
  int32_t rc_stagger;     // register-carried DMMA kernel: anti-lockstep barriers between the warps of a sub-partition
  int32_t n_amb;          // rows of `amb`
  const void* codes;      // tip state codes [n_taxa][n_sites]
  int32_t s2t_bulk;       // tiled 2-state kernel: stored partials leave through shared memory + bulk-async copies
  // Site-sharded multi-GPU: the scalar all-reduce fused into the root kernel over NVLink peer memory (kernels_s2.cuh,
  // block_reduce_to_result).  n_ranks <= 1: single GPU.
  int32_t n_ranks, my_rank;
  unsigned long long epoch;            // evaluation counter, identical on every rank
  struct Mail* mailbox;                // this rank's mailbox [2][CB_MB_OUTS][n_ranks]
  struct Mail* const* peer_mailbox;    // device array: every rank's mailbox (peer pointers opened through CUDA IPC)
  int32_t* comm_error;                 // set when a peer never delivered (timeout)
  // Per-site output of the root epilogues (cb_eval_sites); both null in every other evaluation.
  double* site_lnl;                    // [P]: log(sum_c pi.L_c,p / n_cats) + e_p ln 2, the term the reduction sums
  double* site_post;                   // [C][P] or null: the category terms pi.L_c,p / n_cats the epilogue adds into s_p
};

// ---- tiled 2-state kernel (kernels_s2t.cuh): tile geometry and the child kinds its op bodies take
constexpr int S2T_W = 32;          // sites per tile
constexpr int S2T_WARPS = 8;       // tiles per block (a warp owns V consecutive tiles: 8 / V warps per block)
constexpr int S2T_THREADS = S2T_W * S2T_WARPS;
constexpr int S2T_STAGING = 2;     // bulk-store path only: tile buffers 0..1 per warp rotate as store staging, stack slots follow

// Children of an op are kept in a canonical order (products and exponent sums commute exactly), which leaves twelve
// possible pairs of child kinds; each has its own straight-line op body in the kernel.
//
// An inlined (tip, cherry) subtree (SRC_SMALL) is always child 1, beside a carried child or a tip.  Its op image holds
// three children's worth of tables: tab[0] = child 0's P rows (4C doubles), the parent's P rows for the subtree (4C),
// the subtree's P rows for its tip (4C); tab[1] = the subtree's cherry table.  Code rows: [0] child 0's tip, [1] the
// subtree's tip, [2] and [3] the tips of its cherry.
CB_HD constexpr int s2t_rank(int kind) {
  return kind == SRC_CARRIED ? 0 : kind == SRC_STACK ? 1 : kind == SRC_BUFFER ? 2 : kind == SRC_TIP ? 3 : kind == SRC_CHERRY ? 4 : 5;
}
enum S2TCombo : int32_t {
  S2T_CARRIED_STACK = 0, S2T_CARRIED_BUFFER, S2T_CARRIED_TIP, S2T_CARRIED_CHERRY, S2T_BUFFER_BUFFER, S2T_BUFFER_TIP,
  S2T_BUFFER_CHERRY, S2T_TIP_TIP, S2T_TIP_CHERRY, S2T_CHERRY_CHERRY, S2T_CARRIED_SMALL, S2T_TIP_SMALL, S2T_N_COMBOS
};
CB_HD inline int s2t_combo(int k0, int k1) {   // kinds in canonical order; -1: not a pair the walk produces
  if (k0 == SRC_CARRIED) return k1 == SRC_STACK ? S2T_CARRIED_STACK : k1 == SRC_BUFFER ? S2T_CARRIED_BUFFER : k1 == SRC_TIP ? S2T_CARRIED_TIP : k1 == SRC_CHERRY ? S2T_CARRIED_CHERRY : k1 == SRC_SMALL ? S2T_CARRIED_SMALL : -1;
  if (k0 == SRC_BUFFER) return k1 == SRC_BUFFER ? S2T_BUFFER_BUFFER : k1 == SRC_TIP ? S2T_BUFFER_TIP : k1 == SRC_CHERRY ? S2T_BUFFER_CHERRY : -1;
  if (k0 == SRC_TIP) return k1 == SRC_TIP ? S2T_TIP_TIP : k1 == SRC_CHERRY ? S2T_TIP_CHERRY : k1 == SRC_SMALL ? S2T_TIP_SMALL : -1;
  if (k0 == SRC_CHERRY) return k1 == SRC_CHERRY ? S2T_CHERRY_CHERRY : -1;
  return -1;
}

constexpr int CB_MB_OUTS = 64;          // results per evaluation the fused all-reduce handles (larger batches use NCCL)
struct Mail {
  double v;
  unsigned long long e;
};

}  // namespace cb

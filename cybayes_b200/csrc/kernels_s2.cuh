// Two-state (binary alignment) pruning kernel for sm_100a -- HBM-bandwidth bound.
//
// Restates ML_gamma.pyx:24-38 for S = 2: per node, per rate category, per site
//     v_k[i]  = P_k[i][0] * L_k[0] + P_k[i][1] * L_k[1]        (k = the two child edges)
//     L[i]    = v_a[i] * v_b[i]
// plus what the reference lacks: an exact power-of-two per-site rescale (one int32 exponent
// per site and node, shared by all categories) so deep trees do not underflow.
//
// Mapping: one thread owns two adjacent sites for ALL categories, so every global access is
// a fully coalesced 16-byte (double2) access and the cross-category max needs no
// communication.  A block walks a *range* of ops for its site tile: in level mode a range
// is one node (grid.y = nodes of the level); in path mode the range is a whole dirty path
// (ML_gamma.pyx:99-114) and the on-path partial never leaves registers.  The P matrices of
// the range are staged once per block in shared memory and read back as broadcasts.
// A root op does not store anything: it folds pi, the category mean, log, the site-pattern
// weight and the accumulated exponent into a per-block sum; the last block to finish adds the
// block sums in a fixed order (bit-reproducible, no floating-point atomics).
#pragma once
#include "cb_types.cuh"

namespace cb {

// A stored partial is read back at most once per evaluation: "last use" loads let L2 drop the line afterwards.
#ifndef CB_LD_BUFFER
#define CB_LD_BUFFER __ldlu
#endif
__device__ __forceinline__ double2 ld_cg2(const double* p) {
  return CB_LD_BUFFER(reinterpret_cast<const double2*>(p));
}
__device__ __forceinline__ void st_cg2(double* p, double2 v) {
  __stcg(reinterpret_cast<double2*>(p), v);
}

// exponent e with 2^e <= m < 2^(e+1) for normal m > 0; 0 otherwise
__device__ __forceinline__ int exponent_of(double m) {
  int hi = __double2hiint(m);
  int be = (hi >> 20) & 0x7ff;
  return (be == 0 || be == 0x7ff) ? 0 : be - 1023;
}
__device__ __forceinline__ double pow2_neg(int e) {  // 2^-e, |e| <= 1022
  return __hiloint2double((1023 - e) << 20, 0);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// Scalar all-reduce over the GPUs of a site-sharded evaluation, fused into the kernel that produces the shard's sum
// (one warp of its last block): lane r stores (sum, epoch) into rank r's mailbox through NVLink peer memory, then waits
// for rank r's entry in the local mailbox; the total is added in rank order, so every rank gets the same bits.  Mailboxes
// are double-buffered by epoch parity: a rank can be at most one evaluation ahead of the slowest one (to finish
// evaluation e it needs everybody's entry of e).  Replaces a separate ncclAllReduce launch + device -> host copy.
__device__ __forceinline__ double fused_allreduce(double s, const LaunchConst& k, int out_index, int lane) {
  s = __shfl_sync(0xffffffffu, s, 0);
  const int n = k.n_ranks;
  const size_t slot = ((size_t)(k.epoch & 1ull) * CB_MB_OUTS + out_index) * n;
  double v = 0.0;
  if (lane < n) {
    Mail* dst = k.peer_mailbox[lane] + slot + k.my_rank;
    *reinterpret_cast<volatile double*>(&dst->v) = s;
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long*>(&dst->e) = k.epoch;
    const Mail* src = k.mailbox + slot + lane;
    const long long t0 = clock64();
    bool ok = true;
    while (*reinterpret_cast<const volatile unsigned long long*>(&src->e) != k.epoch) {
      if (clock64() - t0 > 20000000000ll) { ok = false; break; }   // ~10 s: a peer died; report instead of hanging
    }
    __threadfence_system();
    v = *reinterpret_cast<const volatile double*>(&src->v);
    if (!ok) { *k.comm_error = 1; v = __longlong_as_double(0x7ff8000000000000ll); }
  }
  double total = 0.0;
  for (int r = 0; r < n; ++r) total += __shfl_sync(0xffffffffu, v, r);   // rank order: identical bits on every rank
  return total;
}

// Deterministic block -> grid reduction of one double per thread.
// red must hold 32 doubles; every thread of the block must call this.
__device__ __forceinline__ void block_reduce_to_result(double v, const LaunchConst& k, int out_index,
                                                       double* red, int* last_flag) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    double s = (lane < nwarp) ? red[lane] : 0.0;
    s = warp_sum(s);
    if (lane == 0) {
      __stcg(&k.block_sums[(int64_t)out_index * k.max_blocks + blockIdx.x], s);
      __threadfence();
      unsigned t = atomicAdd(&k.tickets[out_index], 1u);
      *last_flag = (t == gridDim.x - 1);
    }
  }
  __syncthreads();
  if (*last_flag && warp == 0) {
    __threadfence();
    const double* bs = k.block_sums + (int64_t)out_index * k.max_blocks;
    double s = 0.0;
    for (unsigned i = lane; i < gridDim.x; i += 32) s += __ldcg(bs + i);
    s = warp_sum(s);
    if (k.n_ranks > 1) s = fused_allreduce(s, k, out_index, lane);
    if (lane == 0) {
      k.results[out_index] = s;
      k.tickets[out_index] = 0u;
    }
  }
}

constexpr int S2_STAGE_OPS = 32;  // ops whose descriptors + P matrices / lookup tables are staged at a time

// Vector of V doubles / ints per thread (V sites), with 8*V-byte global accesses.
template <int V> struct VecD;
template <> struct VecD<1> {
  double v[1];
  __device__ __forceinline__ void load(const double* p) { v[0] = CB_LD_BUFFER(p); }
  __device__ __forceinline__ void load_ca(const double* p) { v[0] = __ldca(p); }
  __device__ __forceinline__ void store(double* p) const { __stcg(p, v[0]); }
  __device__ __forceinline__ void store_cs(double* p) const { __stcs(p, v[0]); }
};
template <> struct VecD<2> {
  double v[2];
  __device__ __forceinline__ void load(const double* p) { const double2 t = ld_cg2(p); v[0] = t.x; v[1] = t.y; }
  __device__ __forceinline__ void load_ca(const double* p) {
    const double2 t = __ldca(reinterpret_cast<const double2*>(p)); v[0] = t.x; v[1] = t.y;
  }
  __device__ __forceinline__ void store(double* p) const { st_cg2(p, make_double2(v[0], v[1])); }
  __device__ __forceinline__ void store_cs(double* p) const { __stcs(reinterpret_cast<double2*>(p), make_double2(v[0], v[1])); }
};
template <int V> __device__ __forceinline__ void load_ints(const int32_t* p, int (&e)[V]);
template <> __device__ __forceinline__ void load_ints<1>(const int32_t* p, int (&e)[1]) { e[0] = CB_LD_BUFFER(p); }
template <> __device__ __forceinline__ void load_ints<2>(const int32_t* p, int (&e)[2]) {
  const int2 t = __ldcg(reinterpret_cast<const int2*>(p)); e[0] = t.x; e[1] = t.y;
}
template <int V> __device__ __forceinline__ void store_ints(int32_t* p, const int (&e)[V]);
template <> __device__ __forceinline__ void store_ints<1>(int32_t* p, const int (&e)[1]) { __stcg(p, e[0]); }
template <> __device__ __forceinline__ void store_ints<2>(int32_t* p, const int (&e)[2]) {
  __stcg(reinterpret_cast<int2*>(p), make_int2(e[0], e[1]));
}
template <int V> __device__ __forceinline__ void load_codes(const void* row, int code_bytes, int64_t site, unsigned (&c)[V]);
template <> __device__ __forceinline__ void load_codes<1>(const void* row, int code_bytes, int64_t site, unsigned (&c)[1]) {
  c[0] = (code_bytes == 1) ? (unsigned)__ldg(static_cast<const uint8_t*>(row) + site)
                           : (unsigned)__ldg(static_cast<const uint16_t*>(row) + site);
}
template <> __device__ __forceinline__ void load_codes<2>(const void* row, int code_bytes, int64_t site, unsigned (&c)[2]) {
  if (code_bytes == 1) {
    const uchar2 t = __ldg(reinterpret_cast<const uchar2*>(static_cast<const uint8_t*>(row) + site));
    c[0] = t.x; c[1] = t.y;
  } else {
    const ushort2 t = __ldg(reinterpret_cast<const ushort2*>(static_cast<const uint16_t*>(row) + site));
    c[0] = t.x; c[1] = t.y;
  }
}

// per-op record staged in shared memory (96 B)
struct S2Stage {
  double* dst;
  int32_t* dst_scale;
  const void* src[2];
  const int32_t* src_scale[2];
  const void* ctip[2][2];
  int32_t kind[2];
  int32_t is_root, pad_;
};
static_assert(sizeof(S2Stage) == 96, "S2Stage is 96 bytes");

// Shared-memory stage per (op, child), in doubles:
//   internal child  [C][row] pairs (Pi0, Pi1)                                   2*2*C
//   tip child       [C][row][4] = (Pi0, Pi1, Pi0 + Pi1, -)                      8*C
//   cherry child    [9 code pairs][2*C + 1]: this edge's contribution v[c][i] for every pair of tip
//                   codes of the folded cherry, and the cherry's rescale exponent            9*(2C+1)
__host__ __device__ constexpr int s2_child_stage(int C) { return 9 * (2 * C + 1) + 1; }  // (+1: keeps 16-byte alignment)

__host__ __device__ inline size_t s2_smem_bytes(int ops, int C) {
  const int n = ops < S2_STAGE_OPS ? ops : S2_STAGE_OPS;
  return (size_t)n * (sizeof(S2Stage) + (size_t)2 * s2_child_stage(C) * sizeof(double));
}

// codes of the tips an op reads: child ch, tip t (t = 1 only for a cherry child)
template <int V>
__device__ __forceinline__ void fetch_codes(const S2Stage& op, int code_bytes, int64_t site, unsigned (&code)[2][2][V]) {
#pragma unroll
  for (int ch = 0; ch < 2; ++ch) {
    if (op.kind[ch] == SRC_TIP) {
      load_codes<V>(op.src[ch], code_bytes, site, code[ch][0]);
    } else if (op.kind[ch] == SRC_CHERRY) {
      load_codes<V>(op.ctip[ch][0], code_bytes, site, code[ch][0]);
      load_codes<V>(op.ctip[ch][1], code_bytes, site, code[ch][1]);
    }
  }
}

__device__ __forceinline__ const double* s2_pmat(const LaunchConst& k, int slot) {
  return (slot & CB_LIB_SLOT) ? k.pmats_lib + (int64_t)(slot & ~CB_LIB_SLOT) * 4 : k.pmats + (int64_t)slot * 4;
}
// contribution of a tip with state code `cd` through edge row (Pi0, Pi1): the FMA chain over the 0/1
// indicator column (utils.pyx:99-111): Pi0, Pi1, or Pi0 + Pi1 for '?', '-', '0/1'
__device__ __forceinline__ double s2_tip_term(double2 pr, int cd) {
  return cd == 0 ? pr.x : (cd == 1 ? pr.y : fma(pr.y, 1.0, pr.x * 1.0));
}

template <int C, int V, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) prune_s2_kernel(const LaunchConst k) {
  static_assert(C <= CB_S2_MAX_CATS, "2-state kernel supports at most CB_S2_MAX_CATS categories");
  constexpr int CS = s2_child_stage(C);
  extern __shared__ __align__(16) unsigned char s2_smem[];
  __shared__ double red[32];
  __shared__ int last_flag;

  const RangeDesc rg = k.ranges[blockIdx.y];
  const int nops = rg.end - rg.begin;
  const int n_stage = min(nops, S2_STAGE_OPS);
  S2Stage* st = reinterpret_cast<S2Stage*>(s2_smem);
  double* p_stage = reinterpret_cast<double*>(s2_smem + (size_t)n_stage * sizeof(S2Stage));

  const int64_t P = k.n_sites;
  const int64_t tile0 = (int64_t)blockIdx.x * (THREADS * V);
  const int64_t site = tile0 + (int64_t)threadIdx.x * V;
  const bool active = site < P;
  double lnl = 0.0;
  VecD<V> cur[C][2];  // carried partial: [category][state] x V sites
  int cur_e[V];
#pragma unroll
  for (int v = 0; v < V; ++v) cur_e[v] = 0;
#pragma unroll
  for (int c = 0; c < C; ++c)
#pragma unroll
    for (int v = 0; v < V; ++v) cur[c][0].v[v] = cur[c][1].v[v] = 0.0;

#pragma unroll 1
  for (int o0 = 0; o0 < nops; o0 += S2_STAGE_OPS) {
    const int o1 = min(nops, o0 + S2_STAGE_OPS);
    if (o0 > 0) __syncthreads();  // everybody is done with the previous chunk
    // stage descriptors (one thread per op) ...
    for (int o = threadIdx.x; o < o1 - o0; o += THREADS) {
      const OpDesc* __restrict__ op = k.ops + rg.begin + o0 + o;
      S2Stage r;
      r.dst = op->dst; r.dst_scale = op->dst_scale;
      r.src[0] = op->src[0]; r.src[1] = op->src[1];
      r.src_scale[0] = op->src_scale[0]; r.src_scale[1] = op->src_scale[1];
      r.ctip[0][0] = op->ctip[0][0]; r.ctip[0][1] = op->ctip[0][1];
      r.ctip[1][0] = op->ctip[1][0]; r.ctip[1][1] = op->ctip[1][1];
      r.kind[0] = op->kind[0]; r.kind[1] = op->kind[1];
      r.is_root = op->is_root; r.pad_ = op->pad_;
      st[o] = r;
    }
    // ... the P matrices of internal and tip children (one thread per category and row) ...
    for (int idx = threadIdx.x; idx < (o1 - o0) * 4 * C; idx += THREADS) {
      const int i = idx & 1, c = (idx >> 1) % C, ch = (idx / (2 * C)) & 1, o = idx / (4 * C);
      const OpDesc* __restrict__ op = k.ops + rg.begin + o0 + o;
      const int kind = op->kind[ch];
      if (kind == SRC_CHERRY) continue;
      const double2 pr = __ldg(reinterpret_cast<const double2*>(s2_pmat(k, op->pslot[ch][c])) + i);
      double* base = p_stage + (size_t)(o * 2 + ch) * CS;
      if (kind == SRC_TIP) {
        double* t = base + (c * 2 + i) * 4;
        t[0] = pr.x;
        t[1] = pr.y;
        t[2] = s2_tip_term(pr, 2);
        t[3] = 0.0;
      } else {
        reinterpret_cast<double2*>(base)[c * 2 + i] = pr;
      }
    }
    // ... and the lookup tables of folded cherries (one thread per pair of tip codes): exactly the
    // arithmetic the cherry's own op and the parent's carried-child step would do per site
    for (int idx = threadIdx.x; idx < (o1 - o0) * 2 * 9; idx += THREADS) {
      const int q = idx % 9, ch = (idx / 9) & 1, o = idx / 18;
      const OpDesc* __restrict__ op = k.ops + rg.begin + o0 + o;
      if (op->kind[ch] != SRC_CHERRY) continue;
      const int ca = q / 3, cb = q - 3 * ca;
      double L[C][2];
      int mh = 0;
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const double2* pa = reinterpret_cast<const double2*>(s2_pmat(k, op->cslot[ch][0][c]));
        const double2* pb = reinterpret_cast<const double2*>(s2_pmat(k, op->cslot[ch][1][c]));
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          L[c][j] = s2_tip_term(__ldg(pa + j), ca) * s2_tip_term(__ldg(pb + j), cb);
          mh = max(mh, __double2hiint(L[c][j]));
        }
      }
      const int be = (mh >> 20) & 0x7ff;
      const int x = (be == 0 || be == 0x7ff) ? 0 : be - 1023;
      const double f = pow2_neg(x);
      double* tab = p_stage + (size_t)(o * 2 + ch) * CS + q * (2 * C + 1);
#pragma unroll
      for (int c = 0; c < C; ++c) {
        const double l0 = L[c][0] * f, l1 = L[c][1] * f;
        const double2* pp = reinterpret_cast<const double2*>(s2_pmat(k, op->pslot[ch][c]));
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const double2 pr = __ldg(pp + i);
          tab[c * 2 + i] = fma(pr.y, l1, pr.x * l0);
        }
      }
      tab[2 * C] = (double)x;
      // a cherry that stays in the returned cache keeps its own copy of its two edges' P matrices
      if (q == 0 && blockIdx.x == 0 && op->crec_out[ch] >= 0) {
        double* out = k.pmats_lib + (int64_t)op->crec_out[ch] * 2 * C * 4;
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const double* src = s2_pmat(k, op->cslot[ch][t][c]);
#pragma unroll
            for (int e = 0; e < 4; ++e) out[(t * C + c) * 4 + e] = __ldg(src + e);
          }
      }
    }
    // ... and pull this tile's tip codes of the NEXT chunk towards L2 while this chunk computes
    {
      const int nxt = min(nops, o1 + S2_STAGE_OPS) - o1;
      const int tile_bytes = THREADS * V * k.code_bytes;
      const int lines = (tile_bytes + 127) / 128;
      for (int idx = threadIdx.x; idx < nxt * 4 * lines; idx += THREADS) {
        const int ln = idx % lines, oc = idx / lines;  // oc: op (2 bits below: child, tip)
        const OpDesc* __restrict__ op = k.ops + rg.begin + o1 + (oc >> 2);
        const int ch = (oc >> 1) & 1, t = oc & 1;
        const int kind = op->kind[ch];
        const void* row = kind == SRC_TIP ? (t == 0 ? op->src[ch] : nullptr) : (kind == SRC_CHERRY ? op->ctip[ch][t] : nullptr);
        if (row != nullptr) {
          const char* a = static_cast<const char*>(row) + tile0 * k.code_bytes + ln * 128;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
        }
      }
    }
    __syncthreads();
    if (!active) continue;
    // tip codes are fetched one op ahead (register prefetch): by the time an op starts, its codes
    // have had a whole op of compute to arrive from L2
    unsigned code_next[2][2][V];
    fetch_codes<V>(st[0], k.code_bytes, site, code_next);
#pragma unroll 1
    for (int o = o0; o < o1; ++o) {
      const S2Stage& op = st[o - o0];
      unsigned code[2][2][V];
#pragma unroll
      for (int ch = 0; ch < 2; ++ch)
#pragma unroll
        for (int t = 0; t < 2; ++t)
#pragma unroll
          for (int v = 0; v < V; ++v) code[ch][t][v] = code_next[ch][t][v];
      if (o + 1 < o1) fetch_codes<V>(st[o + 1 - o0], k.code_bytes, site, code_next);

      VecD<V> out[C][2];
      int e_in[V];
#pragma unroll
      for (int v = 0; v < V; ++v) e_in[v] = 0;
#pragma unroll
      for (int ch = 0; ch < 2; ++ch) {
        const int kind = op.kind[ch];
        const double* pbase = p_stage + (size_t)((o - o0) * 2 + ch) * CS;
        const double2* pm = reinterpret_cast<const double2*>(pbase);  // (P[i][0], P[i][1]) broadcasts
        // v[i] = P[i][0] L[0] + P[i][1] L[1]; first child initialises `out`, second multiplies into it
#define CB_S2_APPLY(L0, L1)                                                   \
  _Pragma("unroll") for (int c = 0; c < C; ++c) {                            \
    _Pragma("unroll") for (int i = 0; i < 2; ++i) {                          \
      const double2 pr = pm[c * 2 + i];                                       \
      _Pragma("unroll") for (int v = 0; v < V; ++v) {                        \
        const double x = fma(pr.y, (L1), pr.x * (L0));                        \
        if (ch == 0) out[c][i].v[v] = x; else out[c][i].v[v] *= x;            \
      }                                                                       \
    }                                                                         \
  }
        if (kind == SRC_CARRIED) {
          CB_S2_APPLY(cur[c][0].v[v], cur[c][1].v[v])
#pragma unroll
          for (int v = 0; v < V; ++v) e_in[v] += cur_e[v];
        } else if (kind == SRC_BUFFER) {
          const double* src = static_cast<const double*>(op.src[ch]) + site;
          VecD<V> L[C][2];
#pragma unroll
          for (int c = 0; c < C; ++c) {
            L[c][0].load(src + (int64_t)(2 * c) * P);
            L[c][1].load(src + (int64_t)(2 * c + 1) * P);
          }
          int se[V];
          load_ints<V>(op.src_scale[ch] + site, se);
          CB_S2_APPLY(L[c][0].v[v], L[c][1].v[v])
#pragma unroll
          for (int v = 0; v < V; ++v) e_in[v] += se[v];
        } else if (kind == SRC_TIP) {
          // state code 0 / 1 / 2 ('?', '-', '0/1') selects the staged contribution of this edge
          // (= the FMA chain over the 0/1 indicator column of utils.pyx:99-111, bit for bit)
#pragma unroll
          for (int c = 0; c < C; ++c) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
#pragma unroll
              for (int v = 0; v < V; ++v) {
                const double x = pbase[(c * 2 + i) * 4 + min(code[ch][0][v], 2u)];
                if (ch == 0) out[c][i].v[v] = x; else out[c][i].v[v] *= x;
              }
            }
          }
        } else {  // folded cherry: the pair of tip codes selects a precomputed row
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const double* tab = pbase + (min(code[ch][0][v], 2u) * 3 + min(code[ch][1][v], 2u)) * (2 * C + 1);
#pragma unroll
            for (int c = 0; c < C; ++c) {
#pragma unroll
              for (int i = 0; i < 2; ++i) {
                const double x = tab[c * 2 + i];
                if (ch == 0) out[c][i].v[v] = x; else out[c][i].v[v] *= x;
              }
            }
            e_in[v] += (int)tab[2 * C];
          }
        }
#undef CB_S2_APPLY
      }
      if (!op.is_root) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          // all entries are >= 0, so the max of the high words carries the exponent of the max
          int mh = __double2hiint(out[0][0].v[v]);
#pragma unroll
          for (int c = 0; c < C; ++c) mh = max(mh, max(__double2hiint(out[c][0].v[v]), __double2hiint(out[c][1].v[v])));
          const int be = (mh >> 20) & 0x7ff;
          const int x = (be == 0 || be == 0x7ff) ? 0 : be - 1023;
          const double f = pow2_neg(x);
#pragma unroll
          for (int c = 0; c < C; ++c) {
            cur[c][0].v[v] = out[c][0].v[v] * f;
            cur[c][1].v[v] = out[c][1].v[v] * f;
          }
          cur_e[v] = e_in[v] + x;
        }
        if (op.dst != nullptr) {
          double* dst = op.dst + site;
          if (op.pad_) {  // kept for the cache only: streaming stores leave L2 to the partials this walk reads back
#pragma unroll
            for (int c = 0; c < C; ++c) {
              cur[c][0].store_cs(dst + (int64_t)(2 * c) * P);
              cur[c][1].store_cs(dst + (int64_t)(2 * c + 1) * P);
            }
          } else {
#pragma unroll
            for (int c = 0; c < C; ++c) {
              cur[c][0].store(dst + (int64_t)(2 * c) * P);
              cur[c][1].store(dst + (int64_t)(2 * c + 1) * P);
            }
          }
          store_ints<V>(op.dst_scale + site, cur_e);
        }
      } else {
        // ll_p = sum_c (pi . L_c) / n_cats ; lnL += w_p * log(ll_p)      ML_gamma.pyx:38,40
        const double pi0 = __ldg(k.pi), pi1 = __ldg(k.pi + 1);
        if (op.dst != nullptr) {  // optional store of the (unscaled-at-this-node) root partial
          double* dst = op.dst + site;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            out[c][0].store(dst + (int64_t)(2 * c) * P);
            out[c][1].store(dst + (int64_t)(2 * c + 1) * P);
          }
          store_ints<V>(op.dst_scale + site, e_in);
        }
        VecD<V> w;
        w.load(k.weights + site);
        const double ln2 = 0.693147180559945309417232121458;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          double s = 0.0;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const double t = fma(pi1, out[c][1].v[v], pi0 * out[c][0].v[v]) / k.cats;
            s += t;
            if (k.site_post != nullptr) k.site_post[c * P + site + v] = t;   // cb_eval_sites (the library divides by s)
          }
          const double ell = log(s) + (double)e_in[v] * ln2;
          if (w.v[v] != 0.0) lnl += w.v[v] * ell;
          if (k.site_lnl != nullptr) k.site_lnl[site + v] = ell;   // cb_eval_sites: every padded site, pads included
        }
      }
    }
  }
  if (rg.out_index >= 0) block_reduce_to_result(lnl, k, rg.out_index, red, &last_flag);
}

}  // namespace cb

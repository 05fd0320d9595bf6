// General-S (multistate) pruning kernel and the root combine, sm_100a.
//
// Same recursion as kernels_s2.cuh (ML_gamma.pyx:24-38) for any number of states.  One
// block = one site tile (32 sites, lane = site) x one op range x ONE rate category, so the
// rescale exponent is per (node, category, site) and categories never communicate until the
// root combine.  Partials of the on-path child stay in shared memory while a block walks a
// dirty path (ML_gamma.pyx:99-114); child tiles are staged in shared memory; the two P
// matrices of the op are staged transposed, a chunk of rows at a time, and each thread
// keeps a 4-row register tile so a P broadcast (LDS.128) feeds two DFMAs.
// The contraction over child states runs j = 0..S-1 through one FMA chain per output, the
// order of a BLAS dot (ML_gamma.pyx:27 `p_t[parent,child].dot(...)`).
// Tip children are not multiplied at all: a one-hot column gathers column `code` of P, the
// all-ones '?'/'-' column (utils.pyx:99-100) takes the row sums, other 'a/b' sets take the
// dense chain.
#pragma once
#include "cb_types.cuh"
#include "kernels_s2.cuh"

namespace cb {

constexpr int GEN_T = 32;        // sites per tile
constexpr int GEN_THREADS = 128; // 4 warps
constexpr int GEN_RT = 4;        // rows per thread

// dynamic shared memory: 3 tiles [S][32] | Pt [2][S][R+2] | rowsum [2][R] | colmax [4][32]
__host__ __device__ inline size_t gen_smem_bytes(int S, int R) {
  return sizeof(double) * ((size_t)3 * S * GEN_T + (size_t)2 * S * (R + 2) + 2 * R + 4 * GEN_T);
}

__global__ void __launch_bounds__(GEN_THREADS) prune_general_kernel(const LaunchConst k, const int R) {
  extern __shared__ __align__(16) double sm[];
  const int S = k.n_states;
  const int Rp = R + 2;
  double* tiles = sm;
  double* Pt = tiles + 3 * S * GEN_T;
  double* rowsum = Pt + 2 * S * Rp;
  double* colmax = rowsum + 2 * R;

  const RangeDesc rg = k.ranges[blockIdx.y];
  const int c = blockIdx.z;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t P = k.n_sites;
  const int64_t site = (int64_t)blockIdx.x * GEN_T + lane;  // P is a multiple of 64: always valid

  int cur_tile = -1;  // which of the 3 tiles holds the carried partial
  int cur_e = 0;

#pragma unroll 1
  for (int o = rg.begin; o < rg.end; ++o) {
    const OpDesc* __restrict__ op = k.ops + o;
    int tile_of[2] = {-1, -1};
    int e_in[2] = {0, 0};
    unsigned code[2] = {0, 0};
    const bool has_carried = op->kind[0] == SRC_CARRIED || op->kind[1] == SRC_CARRIED;
    int used = (has_carried && cur_tile >= 0) ? (1 << cur_tile) : 0;
    __syncthreads();  // previous op finished reading its tiles
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
      const int kind = op->kind[ch];
      if (kind == SRC_CARRIED) {
        tile_of[ch] = cur_tile;
        e_in[ch] = cur_e;
      } else if (kind == SRC_BUFFER) {
        int t = (used & 1) ? ((used & 2) ? 2 : 1) : 0;
        used |= 1 << t;
        tile_of[ch] = t;
        const double* src = static_cast<const double*>(op->src[ch]) + (int64_t)c * S * P + site;
        double* dstt = tiles + t * S * GEN_T + lane;
        for (int j = w; j < S; j += 4) dstt[j * GEN_T] = __ldcg(src + (int64_t)j * P);
        e_in[ch] = __ldcg(op->src_scale[ch] + (int64_t)c * P + site);
      } else {
        code[ch] = (k.code_bytes == 1) ? (unsigned)__ldg(static_cast<const uint8_t*>(op->src[ch]) + site)
                                       : (unsigned)__ldg(static_cast<const uint16_t*>(op->src[ch]) + site);
      }
    }
    const int nxt_tile = (used & 1) ? ((used & 2) ? 2 : 1) : 0;
    double* nxt = tiles + nxt_tile * S * GEN_T;
    const double* pm0 = k.pmats + (int64_t)op->pslot[0][c] * S * S;
    const double* pm1 = k.pmats + (int64_t)op->pslot[1][c] * S * S;

    for (int r0 = 0; r0 < S; r0 += R) {
      __syncthreads();  // Pt of the previous chunk consumed; child tiles complete
      for (int idx = threadIdx.x; idx < R * S; idx += GEN_THREADS) {
        const int r = idx / S, j = idx - r * S;
        const int row = r0 + r;
        double a = 0.0, b = 0.0;
        if (row < S) {
          a = __ldg(pm0 + row * S + j);
          b = __ldg(pm1 + row * S + j);
        }
        Pt[j * Rp + r] = a;
        Pt[S * Rp + j * Rp + r] = b;
      }
      __syncthreads();
      if (op->kind[0] == SRC_TIP || op->kind[1] == SRC_TIP) {
        for (int idx = threadIdx.x; idx < 2 * R; idx += GEN_THREADS) {
          const int ch = idx / R, r = idx - ch * R;
          const double* col = Pt + ch * S * Rp + r;
          double s = 0.0;
          for (int j = 0; j < S; ++j) s += col[j * Rp];  // == fma(P, 1.0, s)
          rowsum[idx] = s;
        }
        __syncthreads();
      }
      for (int g = w; g * GEN_RT < R; g += 4) {
        const int r = g * GEN_RT;
        if (r0 + r >= S) break;
        double acc[2][GEN_RT];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
          const double* ptc = Pt + ch * S * Rp + r;
          if (op->kind[ch] != SRC_TIP) {
            const double* lt = tiles + tile_of[ch] * S * GEN_T + lane;
            double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 4
            for (int j = 0; j < S; ++j) {
              const double l = lt[j * GEN_T];
              const double2 p01 = *reinterpret_cast<const double2*>(ptc + j * Rp);
              const double2 p23 = *reinterpret_cast<const double2*>(ptc + j * Rp + 2);
              a0 = fma(p01.x, l, a0);
              a1 = fma(p01.y, l, a1);
              a2 = fma(p23.x, l, a2);
              a3 = fma(p23.y, l, a3);
            }
            acc[ch][0] = a0; acc[ch][1] = a1; acc[ch][2] = a2; acc[ch][3] = a3;
          } else {
            const unsigned cd = code[ch];
            if (cd < (unsigned)S) {
#pragma unroll
              for (int q = 0; q < GEN_RT; ++q) acc[ch][q] = ptc[cd * Rp + q];
            } else if (cd == (unsigned)S) {
#pragma unroll
              for (int q = 0; q < GEN_RT; ++q) acc[ch][q] = rowsum[ch * R + r + q];
            } else {
              const double* am = k.amb + (int64_t)(cd - S) * S;
              double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
              for (int j = 0; j < S; ++j) {
                const double l = __ldg(am + j);
                a0 = fma(ptc[j * Rp], l, a0);
                a1 = fma(ptc[j * Rp + 1], l, a1);
                a2 = fma(ptc[j * Rp + 2], l, a2);
                a3 = fma(ptc[j * Rp + 3], l, a3);
              }
              acc[ch][0] = a0; acc[ch][1] = a1; acc[ch][2] = a2; acc[ch][3] = a3;
            }
          }
        }
#pragma unroll
        for (int q = 0; q < GEN_RT; ++q)
          if (r0 + r + q < S) nxt[(r0 + r + q) * GEN_T + lane] = acc[0][q] * acc[1][q];
      }
    }
    __syncthreads();
    const int e_sum = e_in[0] + e_in[1];
    if (!op->is_root) {
      double m = 0.0;
      for (int j = w; j < S; j += 4) m = fmax(m, nxt[j * GEN_T + lane]);
      colmax[w * GEN_T + lane] = m;
      __syncthreads();
      m = fmax(fmax(colmax[lane], colmax[GEN_T + lane]), fmax(colmax[2 * GEN_T + lane], colmax[3 * GEN_T + lane]));
      const int x = exponent_of(m);
      const double f = pow2_neg(x);
      double* dst = op->dst ? op->dst + (int64_t)c * S * P + site : nullptr;
      for (int j = w; j < S; j += 4) {
        const double v = nxt[j * GEN_T + lane] * f;
        nxt[j * GEN_T + lane] = v;
        if (dst) __stcg(dst + (int64_t)j * P, v);
      }
      cur_e = e_sum + x;
      cur_tile = nxt_tile;
      if (dst && w == 0) __stcg(op->dst_scale + (int64_t)c * P + site, cur_e);
    } else {
      if (op->dst != nullptr) {
        double* dst = op->dst + (int64_t)c * S * P + site;
        for (int j = w; j < S; j += 4) __stcg(dst + (int64_t)j * P, nxt[j * GEN_T + lane]);
        if (w == 0) __stcg(op->dst_scale + (int64_t)c * P + site, e_sum);
      }
      if (w == 0) {
        double dot = 0.0;
        for (int j = 0; j < S; ++j) dot = fma(__ldg(k.pi + j), nxt[j * GEN_T + lane], dot);
        const int64_t at = ((int64_t)rg.out_index * k.n_cats + c) * P + site;
        __stcg(k.root_dot + at, dot);
        __stcg(k.root_exp + at, e_sum);
      }
    }
  }
}

// lnL = sum_p w_p * log( sum_c pi.L_root,c / n_cats ), categories brought to a common exponent.
// With k.site_lnl (cb_eval_sites, single evaluation) every padded site also writes its term, and with k.site_post the
// category terms added into s (the library divides them by s).
__global__ void __launch_bounds__(256) root_combine_kernel(const LaunchConst k) {
  __shared__ double red[32];
  __shared__ int last_flag;
  const int out = blockIdx.y;
  const int64_t P = k.n_sites;
  const int64_t site = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double lnl = 0.0;
  if (site < P) {
    const double w = __ldcg(k.weights + site);
    if (w != 0.0 || k.site_lnl != nullptr) {
      const int64_t base = (int64_t)out * k.n_cats * P + site;
      int emax = INT_MIN;
      for (int c = 0; c < k.n_cats; ++c) emax = max(emax, __ldcg(k.root_exp + base + (int64_t)c * P));
      double s = 0.0;
      for (int c = 0; c < k.n_cats; ++c) {
        const double d = __ldcg(k.root_dot + base + (int64_t)c * P);
        const int e = __ldcg(k.root_exp + base + (int64_t)c * P);
        s += ldexp(d, e - emax) / k.cats;
      }
      const double ell = log(s) + (double)emax * 0.693147180559945309417232121458;
      if (w != 0.0) lnl = w * ell;
      if (k.site_lnl != nullptr) {
        k.site_lnl[site] = ell;
        for (int c = 0; k.site_post != nullptr && c < k.n_cats; ++c) {
          const double d = __ldcg(k.root_dot + base + (int64_t)c * P);
          const int e = __ldcg(k.root_exp + base + (int64_t)c * P);
          k.site_post[(int64_t)c * P + site] = ldexp(d, e - emax) / k.cats;
        }
      }
    }
  }
  block_reduce_to_result(lnl, k, out, red, &last_flag);
}

}  // namespace cb

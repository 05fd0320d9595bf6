// Posterior predictive replicates (cb_simulate): simulate_kernel<T> overwrites, in place, every state cell of the
// context's alignment with a draw from the model.  One thread per alignment column.
//
// Mask rule: a cell that holds a state (code < S) receives a simulated state; ambiguity cells (code >= S: '?', '-',
// 'a/b') and padding columns are never written.  A replicate therefore keeps the observed alignment's missing-data and
// polymorphism layout, and simulating again into the same codes keeps it too.
//
// Random numbers are counter-based, so a column's replicate depends on (seed, replicate, global column) alone -- not on
// the launch shape or on the order of the edge list:
//   Philox4x32-10 (Salmon, Moraes, Dror & Shaw 2011), key = (seed lo32, seed hi32),
//   counter = (k / 4, column lo32, column hi32, replicate), draw k = output word k % 4;
//   k = 0: rate category, c = (x * C) >> 32;  k = 1: root state from pi;  k = 1 + child node id: the child's state from
//   row P[c][edge][parent state];  a draw x becomes u = (x + 0.5) 2^-32 (exact in fp64), and the state is the first j
//   with u < (row[0] + ... + row[j]) summed left to right in fp64, or S - 1 if there is none.
//
// Internal-node states (node n_taxa + 1 + i at index i) live in shared memory, [i][blockDim] of T, when 128 columns'
// worth fits the block; otherwise in a global scratch [n_taxa - 1][n_sites] (any tree size).  States fit T because
// codes do.
#pragma once
#include <stdint.h>

namespace cb {

constexpr int SIM_THREADS = 128;
constexpr int SIM_SMEM_MAX = 96 * 1024;  // two blocks per SM

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ uint32_t philox_word(const uint4& r, uint32_t w) {
  return w == 0 ? r.x : w == 1 ? r.y : w == 2 ? r.z : r.w;
}

// inverse CDF of one probability row
__device__ __forceinline__ int sim_pick(const double* __restrict__ row, int S, uint32_t x) {
  const double u = ((double)x + 0.5) * 0x1p-32;
  double acc = 0.0;
  for (int j = 0; j < S - 1; ++j) {
    acc += row[j];
    if (u < acc) return j;
  }
  return S - 1;
}

// inner[n_inner][2 + C]: (parent, child, P slot per category) of the edges whose child is internal, parents first.
// tips[n_taxa][1 + C]: (parent, P slot per category) of tip t's edge at row t - 1.
template <typename T>
__global__ void __launch_bounds__(SIM_THREADS) simulate_kernel(T* __restrict__ codes, int64_t row_stride, int64_t n_sites,
                                                       int n_taxa, int S, int C, int n_inner,
                                                       const int32_t* __restrict__ inner, const int32_t* __restrict__ tips,
                                                       const double* __restrict__ pmats, const double* __restrict__ pi,
                                                       int root, unsigned long long seed, uint32_t replicate,
                                                       long long column_offset, T* scratch) {
  extern __shared__ unsigned char sim_smem[];
  const int64_t site = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (site >= n_sites) return;
  T* st;
  int64_t stride;
  if (scratch) {
    st = scratch + site;
    stride = n_sites;
  } else {
    st = reinterpret_cast<T*>(sim_smem) + threadIdx.x;
    stride = blockDim.x;
  }
  const uint64_t col = (uint64_t)column_offset + (uint64_t)site;
  const uint32_t clo = (uint32_t)col, chi = (uint32_t)(col >> 32);
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const int64_t SS = (int64_t)S * S;

  const uint4 r0 = philox4x32_10(make_uint4(0u, clo, chi, replicate), k0, k1);
  const int c = (int)(((uint64_t)r0.x * (uint32_t)C) >> 32);
  st[(int64_t)(root - n_taxa - 1) * stride] = (T)sim_pick(pi, S, r0.y);

  const int w = 2 + C;
  for (int e = 0; e < n_inner; ++e) {
    const int32_t* ed = inner + (int64_t)e * w;
    const int parent = ed[0], child = ed[1];
    const uint32_t k = 1u + (uint32_t)child;
    const uint4 r = philox4x32_10(make_uint4(k >> 2, clo, chi, replicate), k0, k1);
    const int ps = st[(int64_t)(parent - n_taxa - 1) * stride];
    st[(int64_t)(child - n_taxa - 1) * stride] = (T)sim_pick(pmats + ed[2 + c] * SS + (int64_t)ps * S, S, philox_word(r, k & 3));
  }

  // tips in id order: four consecutive draw indices share one Philox block
  uint32_t have = 0;
  uint4 r = r0;
#pragma unroll 4
  for (int t = 1; t <= n_taxa; ++t) {
    T* cell = codes + (int64_t)(t - 1) * row_stride + site;
    const T code = *cell;
    if ((int)code >= S) continue;
    const int32_t* tp = tips + (int64_t)(t - 1) * (1 + C);
    const uint32_t k = 1u + (uint32_t)t;
    if ((k >> 2) != have) {
      have = k >> 2;
      r = philox4x32_10(make_uint4(have, clo, chi, replicate), k0, k1);
    }
    const int ps = st[(int64_t)(tp[0] - n_taxa - 1) * stride];
    *cell = (T)sim_pick(pmats + tp[1 + c] * SS + (int64_t)ps * S, S, philox_word(r, k & 3));
  }
}

}  // namespace cb

// hodlr_kernels.cuh — device kernels of the HODLR solver (K4..K7 of SURVEY.md §2.2).
//
// Reference semantics: src/george/include/george/hodlr.h (Node ctor :29-66, low_rank_approx :136-221, compute :75-103,
// factorize :223-235, apply_inverse :237-254, solve :107-114).  Design (see DESIGN.md):
//   * the tree is processed LEVEL-BATCHED instead of recursively: all leaves in one launch, all ACAs in one launch,
//     then one (gram -> small LU/solve -> update) triple per internal level, bottom-up;
//   * the low-rank factors of level l live in one column-major "panel" with N rows: rows [start, start+half) of a node
//     hold V_[0] (= initial U_[0]) and rows [start+half, start+size) hold U_[1] (= V_[1]) — hodlr.h:53-55 makes
//     the two panels identical before the up-sweep, so the ACA writes one panel (V) and the up-sweep works on a copy (U);
//   * ranks are padded with zero columns to the per-level maximum so every node of a level has the same shape.
#pragma once

#include <cooperative_groups.h>

#include "common.cuh"
#include "kernel_eval.cuh"

namespace bgp {

namespace cg = cooperative_groups;

// ---------------------------------------------------------------------------------------------------------------
// mt19937 + libstdc++'s uniform_int_distribution<int> (GCC >= 11: Lemire's multiply-shift with rejection,
// bits/uniform_int_dist.h) — the stream hodlr.h:179-180 consumes.  Driven by ONE thread.
// ---------------------------------------------------------------------------------------------------------------
struct MT19937 {
  uint32_t mt[624];
  int idx;
};
__device__ inline void mt_seed(MT19937& g, uint32_t s) {
  g.mt[0] = s;
  for (int i = 1; i < 624; ++i) g.mt[i] = 1812433253u * (g.mt[i - 1] ^ (g.mt[i - 1] >> 30)) + (uint32_t)i;
  g.idx = 624;
}
__device__ inline uint32_t mt_next(MT19937& g) {
  if (g.idx >= 624) {
    for (int i = 0; i < 624; ++i) {
      const uint32_t y = (g.mt[i] & 0x80000000u) | (g.mt[(i + 1) % 624] & 0x7fffffffu);
      g.mt[i] = g.mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    g.idx = 0;
  }
  uint32_t y = g.mt[g.idx++];
  y ^= (y >> 11);
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= (y >> 18);
  return y;
}
// uniform_int_distribution<int>(0, s-1)(mt19937): returns the draw, counts consumed words in *words
__device__ inline int mt_uniform(MT19937& g, uint32_t s, int* words) {
  uint64_t prod = (uint64_t)mt_next(g) * (uint64_t)s;
  uint32_t low = (uint32_t)prod;
  int w = 1;
  if (low < s) {
    const uint32_t thr = (0u - s) % s;
    while (low < thr) {
      prod = (uint64_t)mt_next(g) * (uint64_t)s;
      low = (uint32_t)prod;
      ++w;
    }
  }
  *words += w;
  return (int)(prod >> 32);
}
__host__ __device__ inline uint32_t node_seed(uint32_t seed, int pre_id) { return seed + 0x9E3779B9u * (uint32_t)pre_id; }

// ---------------------------------------------------------------------------------------------------------------
// K4: leaf build + LDL^T factorisation (hodlr.h:122-133 get_exact_matrix, :225-227 ldlt_.compute, :87-89 log-det)
// One CTA per leaf.  The m x m block is generated straight from the coordinates into its final location (column-major,
// leading dimension m) and factorised in place: unit-lower L below the diagonal, D on the diagonal.  Un-pivoted LDL^T
// keeps the reference's "never raises on an indefinite leaf, log|D|" behaviour (hodlr.h:89).
// ---------------------------------------------------------------------------------------------------------------
struct LeafDesc {
  int start, size, depth, _pad;
  int64_t off;  // offset of the leaf's block in the leaf-factor buffer
};

constexpr int LEAF_THREADS = 256;
constexpr int LEAF_NB = 32;  // panel width of the blocked factorisation

__global__ void __launch_bounds__(LEAF_THREADS) leaf_build_factor_kernel(const DevProgram* __restrict__ gprog,
                                                                         const double* __restrict__ x,
                                                                         const double* __restrict__ diag,
                                                                         const LeafDesc* __restrict__ leaves,
                                                                         double* __restrict__ Lbuf,
                                                                         double* __restrict__ leaf_logdet) {
  __shared__ DevProgram P;
  __shared__ double red[32];
  __shared__ double panel[LEAF_NB][LEAF_NB + 1];  // factorised diagonal block (L unit-lower, D on the diagonal)
  __shared__ double dinv[LEAF_NB];
  stage_program(&P, gprog);
  __syncthreads();
  const LeafDesc lf = leaves[blockIdx.x];
  const int m = lf.size, nd = P.ndim;
  double* A = Lbuf + lf.off;
  const double* xs = x + (int64_t)lf.start * nd;

  // build the lower triangle (i >= j); column-major so that consecutive threads write consecutive rows
  for (int j = 0; j < m; ++j) {
    for (int i = j + threadIdx.x; i < m; i += LEAF_THREADS) {
      double v = kernel_value(P, xs + (int64_t)i * nd, xs + (int64_t)j * nd);
      if (i == j) v += diag[lf.start + i];
      A[(int64_t)j * m + i] = v;
    }
  }
  __syncthreads();

  double logdet = 0.0;
  for (int k0 = 0; k0 < m; k0 += LEAF_NB) {
    const int nb = min(LEAF_NB, m - k0);
    // (1) diagonal block -> shared, factorise with one warp-synchronous loop over its columns
    for (int t = threadIdx.x; t < nb * nb; t += LEAF_THREADS) {
      const int i = t % nb, j = t / nb;
      panel[i][j] = (i >= j) ? A[(int64_t)(k0 + j) * m + k0 + i] : 0.0;
    }
    __syncthreads();
    for (int k = 0; k < nb; ++k) {
      const double d = panel[k][k];
      const double inv = 1.0 / d;
      __syncthreads();
      for (int i = k + 1 + threadIdx.x; i < nb; i += LEAF_THREADS) panel[i][k] *= inv;
      __syncthreads();
      // trailing update inside the block: A_ij -= l_ik d l_jk
      for (int t = threadIdx.x; t < (nb - k - 1) * (nb - k - 1); t += LEAF_THREADS) {
        const int i = k + 1 + t % (nb - k - 1), j = k + 1 + t / (nb - k - 1);
        if (i >= j) panel[i][j] -= panel[i][k] * d * panel[j][k];
      }
      __syncthreads();
    }
    if (threadIdx.x < nb) {
      const double d = panel[threadIdx.x][threadIdx.x];
      dinv[threadIdx.x] = 1.0 / d;
      logdet += log(fabs(d));
    }
    for (int t = threadIdx.x; t < nb * nb; t += LEAF_THREADS) {
      const int i = t % nb, j = t / nb;
      if (i >= j) A[(int64_t)(k0 + j) * m + k0 + i] = panel[i][j];
    }
    __syncthreads();
    const int rem = m - k0 - nb;
    if (rem <= 0) break;
    // (2) panel solve: rows below the block.  L21 = A21 * L11^-T * D^-1, one row per thread (row-wise forward subst.)
    for (int i = threadIdx.x; i < rem; i += LEAF_THREADS) {
      double* row = A + k0 + nb + i;  // element (k0+nb+i, k0+j) at row[(k0+j)*m]
      double w[LEAF_NB];
#pragma unroll
      for (int j = 0; j < LEAF_NB; ++j) w[j] = (j < nb) ? row[(int64_t)(k0 + j) * m] : 0.0;
      // solve w = y * L11^T for y (y_j = w_j - sum_{q<j} y_q L11[j][q]); y = L21 * D
#pragma unroll
      for (int j = 0; j < LEAF_NB; ++j) {
        if (j < nb) {
          double s = w[j];
#pragma unroll
          for (int q = 0; q < j; ++q) s -= w[q] * panel[j][q];
          w[j] = s;
        }
      }
#pragma unroll
      for (int j = 0; j < LEAF_NB; ++j)
        if (j < nb) row[(int64_t)(k0 + j) * m] = w[j] * dinv[j];
    }
    __syncthreads();
    // (3) trailing update: A22 -= L21 * D * L21^T (lower triangle), 4x4 register tiles
    {
      const int tiles = (rem + 3) / 4;
      const double* Lp = A + (int64_t)k0 * m + k0 + nb;  // L21(i, j) = Lp[j*m + i]
      for (int t = threadIdx.x; t < tiles * tiles; t += LEAF_THREADS) {
        const int ti = t % tiles, tj = t / tiles;
        if (ti < tj) continue;
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
        for (int q = 0; q < nb; ++q) {
          const double dq = panel[q][q];
          double li[4], lj[4];
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const int i = ti * 4 + a, j = tj * 4 + a;
            li[a] = (i < rem) ? Lp[(int64_t)q * m + i] : 0.0;
            lj[a] = (j < rem) ? Lp[(int64_t)q * m + j] * dq : 0.0;
          }
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] += li[a] * lj[b];
        }
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const int i = ti * 4 + a, j = tj * 4 + b;
            if (i < rem && j < rem && i >= j) A[(int64_t)(k0 + nb + j) * m + k0 + nb + i] -= acc[a][b];
          }
      }
    }
    __syncthreads();
  }
  logdet = block_sum(logdet, red);
  if (threadIdx.x == 0) leaf_logdet[blockIdx.x] = logdet;
}

// ---------------------------------------------------------------------------------------------------------------
// Leaf solve: X <- A^-1 X for the rows of each leaf and `ncols(depth)` columns of a column-major matrix
// (hodlr.h:242 ldlt_.solve, applied to the ancestors' U in the up-sweep :95-102 and to the right-hand side in
// solve :107-114).  grid = (leaf, column chunk); each thread owns one column of the chunk... the chunk of columns is
// staged in shared memory and all threads cooperate on the substitutions.
// ---------------------------------------------------------------------------------------------------------------
constexpr int LS_THREADS = 256;
constexpr int LS_COLS = 8;        // right-hand sides per CTA (32 measured slower for the up-sweep: DESIGN.md §8.3)
constexpr int LS_NB = 32;         // diagonal block

// Blocked substitution: per 32-column block of L, (a) the 32 x 32 diagonal block is staged in shared memory and each
// warp solves it for its right-hand sides (columns w, w + 8, ...) with shuffles (no block barrier inside), (b) the rows
// below (forward) / the columns of the block against the rows below (backward) are updated by the whole CTA with
// coalesced, independent loads.  m / 32 block steps with two barriers each instead of m dependent steps.
template <int COLS>
__global__ void __launch_bounds__(LS_THREADS) leaf_solve_kernel(const LeafDesc* __restrict__ leaves,
                                                                const double* __restrict__ Lbuf,
                                                                double* __restrict__ X, int64_t ldx,
                                                                const int* __restrict__ ncols_by_depth, int ncols_fixed,
                                                                int max_m) {
  extern __shared__ double xs[];  // max_m x COLS, column-major with leading dimension max_m
  __shared__ double sL[LS_NB][LS_NB + 1];
  const LeafDesc lf = leaves[blockIdx.x];
  const int ncols = ncols_by_depth ? ncols_by_depth[lf.depth] : ncols_fixed;
  const int c0 = blockIdx.y * COLS;
  if (c0 >= ncols) return;
  const int nc = min(COLS, ncols - c0);
  const int m = lf.size;
  const double* A = Lbuf + lf.off;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int NW = LS_THREADS / 32;
  for (int t = threadIdx.x; t < m * COLS; t += LS_THREADS) {  // (columns >= nc: zeros, so that they stay finite)
    const int i = t % m, c = t / m;
    xs[c * max_m + i] = (c < nc) ? X[(int64_t)(c0 + c) * ldx + lf.start + i] : 0.0;
  }
  // ---- forward: L y = b (unit lower) ----
  for (int kb = 0; kb < m; kb += LS_NB) {
    const int nb = min(LS_NB, m - kb);
    __syncthreads();  // xs updates of the previous block step (and the initial load) are visible; sL is free
    for (int t = threadIdx.x; t < LS_NB * LS_NB; t += LS_THREADS) {
      const int i = t % LS_NB, k = t / LS_NB;
      sL[i][k] = (i < nb && k < nb && i > k) ? A[(int64_t)(kb + k) * m + kb + i] : 0.0;
    }
    __syncthreads();
    for (int c = warp; c < nc; c += NW) {
      double y = (lane < nb) ? xs[c * max_m + kb + lane] : 0.0;
      for (int k = 0; k < nb; ++k) {
        const double yk = __shfl_sync(0xffffffffu, y, k);
        if (lane > k) y -= sL[lane][k] * yk;
      }
      if (lane < nb) xs[c * max_m + kb + lane] = y;
    }
    __syncthreads();
    const int r0 = kb + nb;
    for (int i = r0 + threadIdx.x; i < m; i += LS_THREADS) {
      double acc[COLS];
#pragma unroll
      for (int c = 0; c < COLS; ++c) acc[c] = 0.0;
      const double* Li = A + (int64_t)kb * m + i;
#pragma unroll 4
      for (int k = 0; k < nb; ++k) {
        const double l = Li[(int64_t)k * m];
#pragma unroll
        for (int c = 0; c < COLS; ++c) acc[c] += l * xs[c * max_m + kb + k];
      }
#pragma unroll
      for (int c = 0; c < COLS; ++c) if (c < nc) xs[c * max_m + i] -= acc[c];
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < m * nc; t += LS_THREADS) {
    const int i = t % m, c = t / m;
    xs[c * max_m + i] /= A[(int64_t)i * m + i];
  }
  // ---- backward: L^T z = y ----
  const int nblk = (m + LS_NB - 1) / LS_NB;
  for (int b = nblk - 1; b >= 0; --b) {
    const int kb = b * LS_NB;
    const int nb = min(LS_NB, m - kb);
    const int r0 = kb + nb;
    __syncthreads();
    for (int t = threadIdx.x; t < LS_NB * LS_NB; t += LS_THREADS) {
      const int i = t % LS_NB, k = t / LS_NB;
      sL[i][k] = (i < nb && k < nb && i > k) ? A[(int64_t)(kb + k) * m + kb + i] : 0.0;
    }
    // y_k -= sum_{i >= r0} L[i][k] z_i for the columns k of this block: warp w takes k = w, w + 8, ...
    for (int k = warp; k < nb; k += NW) {
      double acc[COLS];
#pragma unroll
      for (int c = 0; c < COLS; ++c) acc[c] = 0.0;
      const double* Lk = A + (int64_t)(kb + k) * m;
      for (int i = r0 + lane; i < m; i += 32) {
        const double l = Lk[i];
#pragma unroll
        for (int c = 0; c < COLS; ++c) acc[c] += l * xs[c * max_m + i];
      }
#pragma unroll
      for (int c = 0; c < COLS; ++c) {
        const double sres = warp_sum(acc[c]);
        if (lane == 0 && c < nc) xs[c * max_m + kb + k] -= sres;
      }
    }
    __syncthreads();
    for (int c = warp; c < nc; c += NW) {
      double y = (lane < nb) ? xs[c * max_m + kb + lane] : 0.0;
      for (int k = nb - 1; k >= 0; --k) {
        const double zk = __shfl_sync(0xffffffffu, y, k);
        if (lane < k) y -= sL[k][lane] * zk;
      }
      if (lane < nb) xs[c * max_m + kb + lane] = y;
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < m * nc; t += LS_THREADS) {
    const int i = t % m, c = t / m;
    X[(int64_t)(c0 + c) * ldx + lf.start + i] = xs[c * max_m + i];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K5: ACA — randomised-row / max-residual-column cross approximation of the block
//     rows [row0, row0+n_rows) x cols [col0, col0+n_cols)        (hodlr.h:136-221)
// One CTA per node (all nodes of the tree in one launch).  Factors are written into panel columns
// [vcol, vcol+cap): panel rows col0.. hold V (normalised row residuals), panel rows row0.. hold U (column residuals).
// ---------------------------------------------------------------------------------------------------------------
struct AcaDesc {
  int row0, n_rows, col0, n_cols;
  int vcol, cap, pre_id, node;  // node = index into the per-node output arrays
  int64_t idx_off;              // offset into the row-index workspace (n_rows ints)
  int64_t piv_off;              // offset into the pivot arrays (cap entries)
};
struct AcaOut {
  int rank, draws, fallback, status;  // status 1 = rank capacity exceeded
};

constexpr int ACA_THREADS = 512;
constexpr int ACA_MAX_NDIM = 32;

struct AcaShared {
  DevProgram P;
  MT19937 rng;
  double red[32];
  int redi[32];
  double xpiv[ACA_MAX_NDIM];
  double bc[4];
  int ibc[4];
};

__device__ __forceinline__ void block_argmax(double& v, int& i, double* red, int* redi) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  warp_argmax(v, i);
  __syncthreads();
  if (lane == 0) { red[w] = v; redi[w] = i; }
  __syncthreads();
  double tv = (lane < nw) ? red[lane] : -1.0;
  int ti = (lane < nw) ? redi[lane] : 0x7fffffff;
  warp_argmax(tv, ti);
  v = tv; i = ti;
}
__device__ __forceinline__ double block_max(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double t = (lane < nw) ? red[lane] : 0.0;
  return warp_max(t);
}

__device__ __forceinline__ double block_max_signed(double v, double* red) {  // any sign (block_max pads with 0)
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double t = (lane < nw) ? red[lane] : -__longlong_as_double(0x7ff0000000000000ll);
  return warp_max(t);
}

// rng_mode = reference: CTAs take tickets in pre-order and chain the single mt19937 through `chain_state`
// (624 words + index) guarded by `chain_done[k]` flags — the pre-order dependence of hodlr.h:35,58-61 made explicit.
__global__ void __launch_bounds__(ACA_THREADS) aca_kernel(const DevProgram* __restrict__ gprog,
                                                          const double* __restrict__ x,
                                                          const AcaDesc* __restrict__ descs, int n_desc,
                                                          double* __restrict__ Vp, int64_t ld, double tol,
                                                          uint32_t seed, int* __restrict__ idx_ws,
                                                          int* __restrict__ piv_rows, int* __restrict__ piv_cols,
                                                          AcaOut* __restrict__ outs, int* __restrict__ ticket,
                                                          uint32_t* chain_state, volatile int* chain_done,
                                                          int exhaust_mode) {
  extern __shared__ __align__(16) unsigned char aca_smem_raw[];
  AcaShared* S = reinterpret_cast<AcaShared*>(aca_smem_raw);
  double* rowbuf = reinterpret_cast<double*>(aca_smem_raw + ((sizeof(AcaShared) + 15) & ~size_t(15)));  // cap doubles
  __shared__ int s_ticket;

  stage_program(&S->P, gprog);
  if (threadIdx.x == 0) s_ticket = atomicAdd(ticket, 1);
  __syncthreads();
  const int tk = s_ticket;
  if (tk >= n_desc) return;
  const AcaDesc d = descs[tk];
  const int nd = S->P.ndim;
  const int n_rows = d.n_rows, n_cols = d.n_cols;
  const int max_rank = min(n_rows, n_cols);
  int* index = idx_ws + d.idx_off;
  double* Vcols = Vp + (int64_t)d.vcol * ld;  // column k at Vcols + k*ld
  const double* xr = x + (int64_t)d.row0 * nd;
  const double* xc = x + (int64_t)d.col0 * nd;

  for (int n = threadIdx.x; n < n_rows; n += blockDim.x) index[n] = n;
  if (threadIdx.x == 0) {
    if (tk > 0) {
      while (chain_done[tk - 1] == 0) __nanosleep(200);
      __threadfence();
      for (int i = 0; i < 624; ++i) S->rng.mt[i] = chain_state[i];
      S->rng.idx = (int)chain_state[624];
    } else {
      mt_seed(S->rng, seed);
    }
  }
  __syncthreads();

  int rank = 0, draws = 0, n_index = n_rows, fallback = 0, status = 0;
  double norm = 0.0;
  const double tol2 = tol * tol;

  while (true) {
    int i = 0, j = 0;
    double pivot = 0.0;
    bool exhausted = false;
    if (rank >= d.cap) { status = 1; break; }  // no room for another column (only possible when cap < max_rank)
    // ---- choose a row whose residual has a usable pivot (hodlr.h:159-191) ----
    while (true) {
      if (n_index == 0) { exhausted = true; break; }
      if (threadIdx.x == 0) {
        int w = 0;
        const int k = mt_uniform(S->rng, (uint32_t)n_index, &w);
        const int ii = index[k];
        index[k] = index[n_index - 1];
        S->ibc[0] = ii;
        S->ibc[1] = w;
      }
      __syncthreads();
      i = S->ibc[0];
      draws += S->ibc[1];
      n_index--;
      // gather U(i, 0:rank) and the pivot row's coordinates
      for (int k = threadIdx.x; k < rank; k += blockDim.x) rowbuf[k] = __ldcg(Vcols + (int64_t)k * ld + d.row0 + i);
      for (int q = threadIdx.x; q < nd; q += blockDim.x) S->xpiv[q] = xr[(int64_t)i * nd + q];
      __syncthreads();
      // residual of row i over all columns; running arg-max of |.|
      double best = -1.0;
      int bidx = 0x7fffffff;
      double* vnew = Vcols + (int64_t)rank * ld + d.col0;
      for (int n = threadIdx.x; n < n_cols; n += blockDim.x) {
        double val = kernel_value(S->P, S->xpiv, xc + (int64_t)n * nd);
        const double* vk = Vcols + d.col0 + n;
        int k = 0;
        for (; k + 4 <= rank; k += 4) {
          const double a0 = vk[(int64_t)(k + 0) * ld], a1 = vk[(int64_t)(k + 1) * ld];
          const double a2 = vk[(int64_t)(k + 2) * ld], a3 = vk[(int64_t)(k + 3) * ld];
          val -= rowbuf[k] * a0;
          val -= rowbuf[k + 1] * a1;
          val -= rowbuf[k + 2] * a2;
          val -= rowbuf[k + 3] * a3;
        }
        for (; k < rank; ++k) val -= rowbuf[k] * vk[(int64_t)k * ld];
        vnew[n] = val;
        const double a = fabs(val);
        if (a > best) { best = a; bidx = n; }
      }
      block_argmax(best, bidx, S->red, S->redi);
      j = bidx;
      __syncthreads();  // vnew visible to the whole CTA
      pivot = vnew[j];
      if (!(fabs(pivot) < 1e-14)) break;
    }
    if (exhausted) {
      // dense fallback (hodlr.h:161-176); n_cols <= n_rows always holds because half = size/2
      fallback = 1;
      if (exhaust_mode == BGP_EXHAUST_LOWRANK) break;  // every row was tested: |residual| < 1e-14 everywhere
      if (max_rank > d.cap) { status = 1; rank = 0; break; }
      for (int mcol = 0; mcol < n_cols; ++mcol) {
        double* vc = Vcols + (int64_t)mcol * ld;
        for (int n = threadIdx.x; n < n_cols; n += blockDim.x) vc[d.col0 + n] = (n == mcol) ? 1.0 : 0.0;
        for (int n = threadIdx.x; n < n_rows; n += blockDim.x)
          vc[d.row0 + n] = kernel_value(S->P, xr + (int64_t)n * nd, xc + (int64_t)mcol * nd);
      }
      rank = max_rank;
      break;
    }
    // ---- normalise the row residual (hodlr.h:194), its squared norm and max |V_prev^T v| ----
    double* vnew = Vcols + (int64_t)rank * ld + d.col0;
    double vn2 = 0.0;
    for (int n = threadIdx.x; n < n_cols; n += blockDim.x) {
      const double v = vnew[n] / pivot;
      vnew[n] = v;
      vn2 += v * v;
    }
    vn2 = block_sum(vn2, S->red);  // contains __syncthreads: normalised column visible
    double vdot = 0.0;
    {
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
      for (int k = warp; k < rank; k += nw) {
        const double* vk = Vcols + (int64_t)k * ld + d.col0;
        double s = 0.0;
        for (int n = lane; n < n_cols; n += 32) s += vk[n] * vnew[n];
        s = warp_sum(s);
        vdot = fmax(vdot, fabs(s));
      }
      vdot = block_max(vdot, S->red);
    }
    // ---- column residual (hodlr.h:197-199) ----
    for (int k = threadIdx.x; k < rank; k += blockDim.x) rowbuf[k] = __ldcg(Vcols + (int64_t)k * ld + d.col0 + j);
    for (int q = threadIdx.x; q < nd; q += blockDim.x) S->xpiv[q] = xc[(int64_t)j * nd + q];
    __syncthreads();
    double* unew = Vcols + (int64_t)rank * ld + d.row0;
    double un2 = 0.0;
    for (int n = threadIdx.x; n < n_rows; n += blockDim.x) {
      double val = kernel_value(S->P, xr + (int64_t)n * nd, S->xpiv);
      const double* uk = Vcols + d.row0 + n;
      int k = 0;
      for (; k + 4 <= rank; k += 4) {
        const double a0 = uk[(int64_t)(k + 0) * ld], a1 = uk[(int64_t)(k + 1) * ld];
        const double a2 = uk[(int64_t)(k + 2) * ld], a3 = uk[(int64_t)(k + 3) * ld];
        val -= rowbuf[k] * a0;
        val -= rowbuf[k + 1] * a1;
        val -= rowbuf[k + 2] * a2;
        val -= rowbuf[k + 3] * a3;
      }
      for (; k < rank; ++k) val -= rowbuf[k] * uk[(int64_t)k * ld];
      unew[n] = val;
      un2 += val * val;
    }
    un2 = block_sum(un2, S->red);
    double udot = 0.0;
    {
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
      for (int k = warp; k < rank; k += nw) {
        const double* uk = Vcols + (int64_t)k * ld + d.row0;
        double s = 0.0;
        for (int n = lane; n < n_rows; n += 32) s += uk[n] * unew[n];
        s = warp_sum(s);
        udot = fmax(udot, fabs(s));
      }
      udot = block_max(udot, S->red);
    }
    if (threadIdx.x == 0) { piv_rows[d.piv_off + rank] = i; piv_cols[d.piv_off + rank] = j; }
    rank++;
    if (rank >= max_rank) break;                   // hodlr.h:203
    const double rowcol = un2 * vn2;               // hodlr.h:206
    if (rowcol < tol2 * norm) break;               // hodlr.h:207
    norm += rowcol;                                // hodlr.h:210
    if (rank > 1) norm += 2.0 * udot + 2.0 * vdot; // hodlr.h:211-214
  }

  __syncthreads();
  if (threadIdx.x == 0) {
    AcaOut o;
    o.rank = rank; o.draws = draws; o.fallback = fallback; o.status = status;
    outs[d.node] = o;
    for (int q = 0; q < 624; ++q) chain_state[q] = S->rng.mt[q];
    chain_state[624] = (uint32_t)S->rng.idx;
    __threadfence();
    chain_done[tk] = 1;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Panel finalisation: U <- V for the used columns, zero padding up to the level's common rank (both panels).
// One CTA per (node, column): rows of the node only.
// ---------------------------------------------------------------------------------------------------------------
struct NodeDesc {
  int start, size, half, depth;
  int vcol;   // first panel column of the node's level in the V panel
  int ucol;   // first panel column of the node's level in the (packed) U panel
  int r;      // common (padded) rank of the level
  int rank;   // the node's own rank
  int64_t s_off;  // offset of the node's (2r x 2r LU | 2r pivots) block in the S buffer
};

__global__ void finalize_panels_kernel(const NodeDesc* __restrict__ nodes, double* __restrict__ Vp, int64_t ldv,
                                       double* __restrict__ Up, int64_t ldu) {
  const NodeDesc nd = nodes[blockIdx.x];
  const int k = blockIdx.y;
  if (k >= nd.r) return;
  double* v = Vp + (int64_t)(nd.vcol + k) * ldv + nd.start;
  double* u = Up + (int64_t)(nd.ucol + k) * ldu + nd.start;
  const bool used = k < nd.rank;
  for (int i = threadIdx.x; i < nd.size; i += blockDim.x) {
    double val = 0.0;
    if (used) val = v[i]; else v[i] = 0.0;
    u[i] = val;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K6a: batched tall-skinny "TN" product   W_h = V_h^T * X_h   for both halves h of every node of a level
//   V_h : rows of half h, the level's r columns of the V panel            (n_h x r)
//   X_h : rows of half h, columns [0, ncols) of X (the U panel or a RHS)  (n_h x ncols)
//   W_h : r x ncols, accumulated with atomics over row chunks.  The two halves of a node share one (2r x ncols)
//         column-major block (ld 2r): rows [0, r) = W_1 = V_1^T X_2, rows [r, 2r) = W_0 = V_0^T X_1 — the right-hand
//         side [W_1; W_0] of the node's Woodbury system, stored the way the LU solve wants it.
// hodlr.h:231-232 (Gram blocks of S) and :248-249 (V^T x) in one pass.
// grid = (row chunk, node*2 + h, column tile)
// ---------------------------------------------------------------------------------------------------------------
constexpr int GT_THREADS = 256;
constexpr int GT_ROWS = 64;   // rows per shared-memory slab
constexpr int GT_TQ = 32;     // W rows (V columns) per CTA pass
constexpr int GT_TC = 32;     // W cols (X columns) per CTA
constexpr int GT_CHUNK = 512;   // rows per CTA (8 slabs: the top levels get enough CTAs to hide the slab latency)

__global__ void __launch_bounds__(GT_THREADS) gram_tn_kernel(const NodeDesc* __restrict__ nodes,
                                                             const double* __restrict__ Vp, int64_t ldv,
                                                             const double* __restrict__ X, int64_t ldx, int ncols,
                                                             double* __restrict__ W, int64_t w_stride_node) {
  __shared__ double sv[GT_ROWS][GT_TQ + 1];
  __shared__ double sx[GT_ROWS][GT_TC + 1];
  const NodeDesc nd = nodes[blockIdx.y >> 1];
  const int h = blockIdx.y & 1;
  const int rs = nd.start + (h ? nd.half : 0), nh = h ? (nd.size - nd.half) : nd.half;
  const int row_lo = blockIdx.x * GT_CHUNK;
  if (row_lo >= nh) return;
  const int row_hi = min(nh, row_lo + GT_CHUNK);
  const int c0 = blockIdx.z * GT_TC;
  if (c0 >= ncols) return;
  const int nc = min(GT_TC, ncols - c0);
  const int r = nd.r;
  double* Wh = W + (int64_t)(blockIdx.y >> 1) * w_stride_node + (h ? 0 : r);  // rows of half h in the node's 2r x ncols block
  const int ldw = 2 * r;

  const int tq = threadIdx.x & 31, tc = threadIdx.x >> 5;  // thread -> (q = tq, c = tc + 8*e), e = 0..3
  for (int q0 = 0; q0 < r; q0 += GT_TQ) {
    const int nq = min(GT_TQ, r - q0);
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    for (int i0 = row_lo; i0 < row_hi; i0 += GT_ROWS) {
      const int ni = min(GT_ROWS, row_hi - i0);
      __syncthreads();
      for (int t = threadIdx.x; t < GT_ROWS * GT_TQ; t += GT_THREADS) {
        const int i = t % GT_ROWS, q = t / GT_ROWS;
        sv[i][q] = (i < ni && q < nq) ? Vp[(int64_t)(nd.vcol + q0 + q) * ldv + rs + i0 + i] : 0.0;
      }
      for (int t = threadIdx.x; t < GT_ROWS * GT_TC; t += GT_THREADS) {
        const int i = t % GT_ROWS, c = t / GT_ROWS;
        sx[i][c] = (i < ni && c < nc) ? X[(int64_t)(c0 + c) * ldx + rs + i0 + i] : 0.0;
      }
      __syncthreads();
#pragma unroll 8
      for (int i = 0; i < GT_ROWS; ++i) {
        const double a = sv[i][tq];
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[e] += a * sx[i][tc + 8 * e];
      }
    }
    if (tq < nq) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = tc + 8 * e;
        if (c < nc) atomicAdd(Wh + (int64_t)(c0 + c) * ldw + q0 + tq, acc[e]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K6b: per-node small dense step (hodlr.h:228-234 factorize, :90-93 log-det, :250 lu_.solve)
//   factor != 0: S = [[I, W_1[:, own]], [W_0[:, own], I]] (2r x 2r), LU with COMPLETE pivoting and the rank-revealing
//                solve of Eigen::FullPivLU (what the reference calls), log|det| -> node_logdet, LU stored.
//   then T = S^-1 [W_1[:, cols] ; W_0[:, cols]] for the `ncols - own` target columns, written back over W
//   (T_top -> W_1, T_bot -> W_0 so the update kernel reads half h's coefficients from W_{1-h}... see update_nn_kernel).
// One CTA per node, S in shared memory: the path for 2r <= SS_MAX_N; larger ranks go through hodlr_lu.cuh.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SS_THREADS = 256;
constexpr int SS_MAX_N = 142;  // 142^2 doubles = 157.5 KB of dynamic shared memory

__global__ void __launch_bounds__(SS_THREADS) small_solve_kernel(const NodeDesc* __restrict__ nodes,
                                                                 double* __restrict__ W, int64_t w_stride_node,
                                                                 int ncols, int own_off, int factor,
                                                                 double* __restrict__ Sbuf,
                                                                 double* __restrict__ node_logdet, int node_base) {
  extern __shared__ double ss_smem[];
  __shared__ double red[32];
  __shared__ int redi[32];
  __shared__ int s_piv;
  const NodeDesc nd = nodes[blockIdx.x];
  const int r = nd.r, n2 = 2 * r;
  if (r == 0) { if (factor && threadIdx.x == 0) node_logdet[node_base + blockIdx.x] = 0.0; return; }
  double* W1 = W + (int64_t)blockIdx.x * w_stride_node;  // half 1: V1^T X2  (rows [0, r) of the 2r x ncols block)
  double* W0 = W1 + r;                                    // half 0: V0^T X1  (rows [r, 2r))
  double* Sg = Sbuf + nd.s_off;                // n2 x n2 LU, column-major
  int* piv = reinterpret_cast<int*>(Sg + (int64_t)n2 * n2);
  double* S = ss_smem;

  // Eigen::FullPivLU semantics (hodlr.h:24,233,250): complete pivoting, P S Q = L U; solve() treats the pivots below
  // eps * n * |max pivot| as zero (rank-revealing pseudo-solve); log|det| sums log|u_kk| over ALL pivots (hodlr.h:90-93).
  int* rowt = piv;          // row transpositions
  int* colt = piv + n2;     // column transpositions
  int* meta = piv + 2 * n2; // [0] numerical rank used by solve()
  if (factor) {
    for (int t = threadIdx.x; t < n2 * n2; t += SS_THREADS) {
      const int i = t % n2, j = t / n2;
      double v = (i == j) ? 1.0 : 0.0;
      if (i < r && j >= r) v = W1[(int64_t)(own_off + j - r) * n2 + i];        // S(0:r, r:2r) = V1^T U1
      else if (i >= r && j < r) v = W0[(int64_t)(own_off + j) * n2 + (i - r)];  // S(r:2r, 0:r) = V0^T U0
      S[(int64_t)j * n2 + i] = v;
    }
    __syncthreads();
    double logdet = 0.0, maxpivot = 0.0;
    int nonzero = n2;
    for (int k = 0; k < n2; ++k) {
      // pivot search over the trailing block, first maximum in column-major order (Eigen's maxCoeff visitor)
      double best = -1.0;
      int bi = 0x7fffffff;
      const int rem0 = n2 - k;
      for (int t = threadIdx.x; t < rem0 * rem0; t += SS_THREADS) {
        const int i = k + t % rem0, j = k + t / rem0;
        const double a = fabs(S[(int64_t)j * n2 + i]);
        const int lin = j * n2 + i;
        if (a > best || (a == best && lin < bi)) { best = a; bi = lin; }
      }
      block_argmax(best, bi, red, redi);
      if (threadIdx.x == 0) s_piv = bi;
      __syncthreads();
      const int lin = s_piv;
      const bool no_pivot = lin == 0x7fffffff;  // nothing comparable in the trailing block (all NaN): stop, log|det| = NaN
      const int pr = no_pivot ? k : lin % n2, pc = no_pivot ? k : lin / n2;
      // |pivot| = the maximum block_argmax returned to EVERY thread: do not re-read S here, the swaps below start as soon
      // as a thread gets there (a thread that read the entry after a neighbour's swap would take a different branch)
      const double pv = best;
      if (pv == 0.0 || no_pivot) {  // the rest of the matrix is exactly zero: FullPivLU stops here (m_nonzero_pivots = k)
        nonzero = k;
        for (int q = k + threadIdx.x; q < n2; q += SS_THREADS) { rowt[q] = q; colt[q] = q; }
        break;
      }
      maxpivot = fmax(maxpivot, pv);
      if (threadIdx.x == 0) { rowt[k] = pr; colt[k] = pc; }
      if (pr != k) {
        for (int jj = threadIdx.x; jj < n2; jj += SS_THREADS) {
          const double a = S[(int64_t)jj * n2 + k];
          S[(int64_t)jj * n2 + k] = S[(int64_t)jj * n2 + pr];
          S[(int64_t)jj * n2 + pr] = a;
        }
      }
      __syncthreads();
      if (pc != k) {
        for (int ii = threadIdx.x; ii < n2; ii += SS_THREADS) {
          const double a = S[(int64_t)k * n2 + ii];
          S[(int64_t)k * n2 + ii] = S[(int64_t)pc * n2 + ii];
          S[(int64_t)pc * n2 + ii] = a;
        }
      }
      __syncthreads();
      const double dkk = S[(int64_t)k * n2 + k];
      const double inv = 1.0 / dkk;
      __syncthreads();
      for (int i = k + 1 + threadIdx.x; i < n2; i += SS_THREADS) S[(int64_t)k * n2 + i] *= inv;
      __syncthreads();
      const int rem = n2 - k - 1;
      for (int t = threadIdx.x; t < rem * rem; t += SS_THREADS) {
        const int i = k + 1 + t % rem, j = k + 1 + t / rem;
        S[(int64_t)j * n2 + i] -= S[(int64_t)k * n2 + i] * S[(int64_t)j * n2 + k];
      }
      __syncthreads();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 0; k < n2; ++k) logdet += log(fabs(S[(int64_t)k * n2 + k]));  // -inf for an exactly singular S, as the reference
      const double thr = maxpivot * 2.220446049250313e-16 * (double)n2;           // FullPivLU::threshold() * |maxPivot|
      int rk = 0;
      for (int k = 0; k < nonzero; ++k) rk += (fabs(S[(int64_t)k * n2 + k]) > thr) ? 1 : 0;
      meta[0] = rk;
      node_logdet[node_base + blockIdx.x] = logdet;
    }
    for (int t = threadIdx.x; t < n2 * n2; t += SS_THREADS) Sg[t] = S[t];
    __syncthreads();
  } else {
    for (int t = threadIdx.x; t < n2 * n2; t += SS_THREADS) S[t] = Sg[t];
    __syncthreads();
  }

  // solve for the target columns: one thread per column; rhs = [W1[:, c]; W0[:, c]] (hodlr.h:248-250)
  const int rk = meta[0];
  for (int c = threadIdx.x; c < ncols; c += SS_THREADS) {
    if (factor && c >= own_off && c < own_off + r) continue;  // own columns only feed S
    double* tc = W1 + (int64_t)c * n2;  // the column's 2r entries are contiguous: [W_1(:, c); W_0(:, c)]
    for (int k = 0; k < n2; ++k) {
      const int p = rowt[k];
      if (p != k) { const double a = tc[k]; tc[k] = tc[p]; tc[p] = a; }
    }
    for (int k = 0; k < n2; ++k) {
      const double bk = tc[k];
      for (int i = k + 1; i < n2; ++i) tc[i] -= S[(int64_t)k * n2 + i] * bk;
    }
    for (int k = rk - 1; k >= 0; --k) {
      const double bk = tc[k] / S[(int64_t)k * n2 + k];
      tc[k] = bk;
      for (int i = 0; i < k; ++i) tc[i] -= S[(int64_t)k * n2 + i] * bk;
    }
    for (int k = rk; k < n2; ++k) tc[k] = 0.0;
    for (int k = n2 - 1; k >= 0; --k) {
      const int p = colt[k];
      if (p != k) { const double a = tc[k]; tc[k] = tc[p]; tc[p] = a; }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// K6c: batched "NN" update   X_1 -= U_0 * T[0:r],  X_2 -= U_1 * T[r:2r]      (hodlr.h:252-253)
// After the solve, T[0:r] sits in rows [0, r) of the node's block and T[r:2r] in rows [r, 2r): half h reads rows h*r...
// Columns [col_lo, col_hi) of X are updated (ancestor columns in the up-sweep, all RHS columns in the solve).
// grid = (row chunk, node*2 + h, column tile)
// ---------------------------------------------------------------------------------------------------------------
constexpr int UP_THREADS = 256;
constexpr int UP_ROWS = 256;  // rows per CTA (one per thread)
constexpr int UP_TC = 16;     // columns per CTA
constexpr int UP_QC = 128;    // factor columns staged per pass

__global__ void __launch_bounds__(UP_THREADS) update_nn_kernel(const NodeDesc* __restrict__ nodes,
                                                               const double* __restrict__ Up, int64_t ldu,
                                                               double* __restrict__ X, int64_t ldx, int col_lo,
                                                               int col_hi, const double* __restrict__ W,
                                                               int64_t w_stride_node, int w_col_off) {
  __shared__ double st[UP_TC][UP_QC + 1];  // coefficient slab: UP_QC factor columns x UP_TC target columns
  const NodeDesc nd = nodes[blockIdx.y >> 1];
  const int h = blockIdx.y & 1;
  const int rs = nd.start + (h ? nd.half : 0), nh = h ? (nd.size - nd.half) : nd.half;
  const int row0 = blockIdx.x * UP_ROWS;
  if (row0 >= nh) return;
  const int c0 = col_lo + blockIdx.z * UP_TC;
  if (c0 >= col_hi) return;
  const int nc = min(UP_TC, col_hi - c0);
  const int r = nd.r;
  const double* T = W + (int64_t)(blockIdx.y >> 1) * w_stride_node + (h ? r : 0);  // T(:, c) for X column c at c + w_col_off
  const int ldw = 2 * r;
  const int i = row0 + threadIdx.x;
  const bool active = i < nh;
  double acc[UP_TC];
#pragma unroll
  for (int c = 0; c < UP_TC; ++c) acc[c] = 0.0;
  const double* u = Up + (int64_t)nd.ucol * ldu + rs + (active ? i : 0);
  for (int q0 = 0; q0 < r; q0 += UP_QC) {
    const int nq = min(UP_QC, r - q0);
    __syncthreads();
    for (int t = threadIdx.x; t < UP_QC * UP_TC; t += UP_THREADS) {
      const int q = t % UP_QC, c = t / UP_QC;
      st[c][q] = (q < nq && c < nc) ? T[(int64_t)(c0 + c + w_col_off) * ldw + q0 + q] : 0.0;
    }
    __syncthreads();
    if (active) {
      for (int q = 0; q < nq; ++q) {
        const double a = u[(int64_t)(q0 + q) * ldu];
#pragma unroll
        for (int c = 0; c < UP_TC; ++c) acc[c] += a * st[c][q];
      }
    }
  }
  if (!active) return;
#pragma unroll
  for (int c = 0; c < UP_TC; ++c)
    if (c < nc) X[(int64_t)(c0 + c) * ldx + rs + i] -= acc[c];
}

// small helpers -----------------------------------------------------------------------------------------------------
// pack / unpack of a row range of the (column-major) top panel for the multi-GPU exchange
__global__ void pack_rows_kernel(const double* __restrict__ P, int64_t ld, int64_t row0, int64_t rows, int64_t cols,
                                 double* __restrict__ buf, int64_t rows_pad) {
  const int64_t total = rows * cols;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t % rows, c = t / rows;
    buf[c * rows_pad + i] = P[c * ld + row0 + i];
  }
}
__global__ void unpack_rows_kernel(double* __restrict__ P, int64_t ld, int64_t row0, int64_t rows, int64_t cols,
                                   const double* __restrict__ buf, int64_t rows_pad) {
  const int64_t total = rows * cols;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t % rows, c = t / rows;
    P[c * ld + row0 + i] = buf[c * rows_pad + i];
  }
}
__global__ void square_kernel(const double* __restrict__ yerr, double* __restrict__ diag, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    diag[i] = yerr[i] * yerr[i];
}
__global__ void dot_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t n, double* out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    s += a[i] * b[i];
  s = block_sum(s, red);
  if (threadIdx.x == 0) atomicAdd(out, s);
}

}  // namespace bgp

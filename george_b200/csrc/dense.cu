// dense.cu — K3: dense solver behind BasicSolver (replaces src/george/solvers/basic.py:51-121, i.e.
// kernel.get_value + scipy.linalg.cholesky / cho_solve, LAPACK dpotrf/dpotrs).
//
// The covariance matrix is generated on the device by the fused kernel-matrix build (kmat.cu) with yerr^2 already on
// the diagonal, factorised in place (blocked right-looking Cholesky, lower factor L with K = L L^T; the reference keeps
// the upper factor U = L^T, basic.py:68) and never leaves HBM.  log-det = 2 sum log L_ii (basic.py:69).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "gemm_dmma.cuh"
#include "kernel_eval.cuh"

namespace bgp {
int upload_program(const DevProgram& P, DevBuf<DevProgram>& buf, cudaStream_t s);
int kmat_symmetric_launch(const DevProgram* dprog, int nd, const double* x, int64_t n, const double* diag_add,
                          double* out, int64_t ld, cudaStream_t s);
int kmat_symmetric_launch_auto(const DevProgram& P, const DevProgram* dprog, const double* x, int64_t n,
                               const double* diag_add, double* out, int64_t ld, cudaStream_t s);
int kmat_grad_contract_launch(const DevProgram* dprog, int nd, int np, const unsigned* which_dev, const double* x,
                              int64_t n, const double* M, int64_t ldm, const double* alpha, double ca, double cm,
                              double* g_dev, double* diag_dev, DevBuf<double>& scratch, cudaStream_t s);
int fill_identity_launch(double* A, int64_t n, cudaStream_t s);

constexpr int DN_NB = 64;   // inner panel width (diagonal block in shared memory)
constexpr int DN_MB = 256;  // middle block of the delayed-update hierarchy (see dense_potrf)
constexpr int DN_OB = 2048; // outer block: trailing updates beyond it run with K = 2048 on the tensor pipe.  Measured on
                            // config 4 (N = 32768): two levels 256 -> 556 ms, 512 -> 512 ms, 1024 -> 497 ms; three levels
                            // (64 | 256 | OB) with the slimmer GEMM loader: 1024 -> 419.7 ms, 2048 -> 412.9 ms
                            // (profiles/dense_cfg4_r01_v5_ob_sweep.txt, dense_cfg4_r01_v7.txt)

// ---- diagonal block Cholesky (NB x NB): one thread per ROW, the row lives in registers ------------------------------
// Right-looking, fully unrolled: at step k every thread scales its entry of column k and applies the rank-1 update to
// its own row; the only exchanges are the pivot and the scaled column, through (double-buffered) shared memory, two
// barriers per step.  info != 0 when a pivot is not positive (LAPACK dpotrf's info = k+1; scipy raises LinAlgError).
__global__ void __launch_bounds__(DN_NB) potf2_kernel(double* __restrict__ A, int64_t lda, int nb, int* info, int k0) {
  __shared__ double col[2][DN_NB];
  __shared__ double piv[2];
  const int i = threadIdx.x;
  double a[DN_NB];
#pragma unroll
  for (int j = 0; j < DN_NB; ++j) a[j] = (i < nb && j < nb) ? A[(int64_t)j * lda + i] : (i == j ? 1.0 : 0.0);
  if (i == 0) piv[0] = a[0];
  __syncthreads();
#pragma unroll
  for (int k = 0; k < DN_NB; ++k) {
    const double d = piv[k & 1];
    if (!(d > 0.0)) {  // also catches NaN; uniform: every thread reads the same pivot
      if (i == 0) atomicCAS(info, 0, k0 + k + 1);
      return;
    }
    // 1/sqrt(d) (one MUFU + Newton steps) instead of sqrt followed by a division: this scalar chain is the critical
    // path of the whole factorisation step; the factor entries differ from sqrt/divide by <= 2 ulp
    const double rinv = rsqrt(d);
    const double lik = (i == k) ? d * rinv : a[k] * rinv;
    a[k] = lik;
    col[k & 1][i] = lik;
    __syncthreads();
#pragma unroll
    for (int j = k + 1; j < DN_NB; ++j) a[j] = fma(-lik, col[k & 1][j], a[j]);  // entries above the diagonal are scratch
    if (k + 1 < DN_NB) {
      if (i == k + 1) piv[(k + 1) & 1] = a[k + 1];
      __syncthreads();
    }
  }
  if (i < nb) {
#pragma unroll
    for (int j = 0; j < DN_NB; ++j)
      if (j < nb) A[(int64_t)j * lda + i] = (j <= i) ? a[j] : 0.0;  // explicit zeros above the diagonal of the block
  }
}

// ---- panel solve: rows below the diagonal block, L21 = A21 * L11^-T; one row per thread ---------------------------
// Column-oriented substitution (x_j = w_j / l_jj, then w_q -= x_j l_qj for q > j): the 2016 updates of a row are
// independent FMAs instead of 64 dependent dot products; the 64 divisions are multiplications by reciprocals computed
// once per CTA.
__global__ void __launch_bounds__(128, 1) trsm_panel_kernel(double* __restrict__ A, int64_t lda, int64_t rows, int nb,
                                                         const int* info) {
  __shared__ double l[DN_NB][DN_NB + 1];
  __shared__ double rl[DN_NB];
  if (*info != 0) return;
  for (int t = threadIdx.x; t < DN_NB * DN_NB; t += blockDim.x) {
    const int i = t % DN_NB, j = t / DN_NB;
    l[i][j] = (i < nb && j < nb) ? A[(int64_t)j * lda + i] : (i == j ? 1.0 : 0.0);
  }
  __syncthreads();
  if (threadIdx.x < DN_NB) rl[threadIdx.x] = 1.0 / l[threadIdx.x][threadIdx.x];
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows) return;
  double* row = A + nb + i;  // element (nb + i, j) at row[j*lda]
  double w[DN_NB];
#pragma unroll
  for (int j = 0; j < DN_NB; ++j) w[j] = (j < nb) ? row[(int64_t)j * lda] : 0.0;
#pragma unroll
  for (int j = 0; j < DN_NB; ++j) {
    const double xj = w[j] * rl[j];
    w[j] = xj;
#pragma unroll
    for (int q = j + 1; q < DN_NB; ++q) w[q] = fma(-xj, l[q][j], w[q]);
  }
#pragma unroll
  for (int j = 0; j < DN_NB; ++j)
    if (j < nb) row[(int64_t)j * lda] = w[j];
}

// ---- generic column-major tile GEMM:  C (M x N) -= op(A) * op(B)   -------------------------------------------------
//   TA == 0: A is M x K (lda), element (i,k) = A[k*lda + i];   TA == 1: A is K x M, element (i,k) = A[i*lda + k]
//   TB == 0: B is K x N (ldb), element (k,j) = B[j*ldb + k];   TB == 1: B is N x K, element (k,j) = B[k*ldb + j]
//   lower != 0: only tiles with i-tile >= j-tile are computed (SYRK-style trailing update)
constexpr int GM_T = 64, GM_K = 16;
template <int TA, int TB>
__global__ void __launch_bounds__(256) gemm_sub_kernel(int64_t M, int64_t N, int K, const double* __restrict__ A,
                                                       int64_t lda, const double* __restrict__ B, int64_t ldb,
                                                       double* __restrict__ C, int64_t ldc, int lower,
                                                       const int* info) {
  if (info && *info != 0) return;
  if (lower && blockIdx.x < blockIdx.y) return;
  __shared__ double sa[GM_K][GM_T + 4];
  __shared__ double sb[GM_K][GM_T + 4];
  const int64_t i0 = (int64_t)blockIdx.x * GM_T, j0 = (int64_t)blockIdx.y * GM_T;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16 threads, 4x4 outputs each
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  for (int k0 = 0; k0 < K; k0 += GM_K) {
    for (int t = threadIdx.x; t < GM_T * GM_K; t += 256) {
      int i, k;
      if (TA == 0) { i = t % GM_T; k = t / GM_T; } else { k = t % GM_K; i = t / GM_K; }
      const int64_t gi = i0 + i;
      const int gk = k0 + k;
      double v = 0.0;
      if (gi < M && gk < K) v = (TA == 0) ? A[(int64_t)gk * lda + gi] : A[gi * lda + gk];
      sa[k][i] = v;
    }
    for (int t = threadIdx.x; t < GM_T * GM_K; t += 256) {
      int j, k;
      if (TB == 1) { j = t % GM_T; k = t / GM_T; } else { k = t % GM_K; j = t / GM_K; }
      const int64_t gj = j0 + j;
      const int gk = k0 + k;
      double v = 0.0;
      if (gj < N && gk < K) v = (TB == 1) ? B[(int64_t)gk * ldb + gj] : B[gj * ldb + gk];
      sb[k][j] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GM_K; ++k) {
      double a[4], b[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) { a[e] = sa[k][tx + 16 * e]; b[e] = sb[k][ty + 16 * e]; }
#pragma unroll
      for (int e = 0; e < 4; ++e)
#pragma unroll
        for (int f = 0; f < 4; ++f) acc[e][f] += a[e] * b[f];
    }
    __syncthreads();
  }
#pragma unroll
  for (int f = 0; f < 4; ++f)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t gi = i0 + tx + 16 * e, gj = j0 + ty + 16 * f;
      if (gi < M && gj < N && (!lower || gi >= gj)) C[gj * ldc + gi] -= acc[e][f];
    }
}

// ---- triangular solves with the diagonal block for a slab of right-hand sides --------------------------------------
// forward: X_k <- L_kk^-1 X_k ; backward: X_k <- L_kk^-T X_k.  One thread per RHS column; L_kk in shared memory.
__global__ void __launch_bounds__(128) trsv_block_kernel(const double* __restrict__ L, int64_t ldl, int nb,
                                                         double* __restrict__ X, int64_t ldx, int64_t nrhs,
                                                         int backward) {
  __shared__ double l[DN_NB][DN_NB + 1];
  for (int t = threadIdx.x; t < nb * nb; t += blockDim.x) {
    const int i = t % nb, j = t / nb;
    l[i][j] = L[(int64_t)j * ldl + i];
  }
  __syncthreads();
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nrhs) return;
  double* x = X + c * ldx;
  double w[DN_NB];
#pragma unroll
  for (int j = 0; j < DN_NB; ++j) w[j] = (j < nb) ? x[j] : 0.0;
  if (!backward) {
#pragma unroll
    for (int j = 0; j < DN_NB; ++j)
      if (j < nb) {
        double s = w[j];
#pragma unroll
        for (int q = 0; q < j; ++q) s -= l[j][q] * w[q];
        w[j] = s / l[j][j];
      }
  } else {
#pragma unroll
    for (int j = DN_NB - 1; j >= 0; --j)
      if (j < nb) {
        double s = w[j];
#pragma unroll
        for (int q = j + 1; q < DN_NB; ++q)
          if (q < nb) s -= l[q][j] * w[q];
        w[j] = s / l[j][j];
      }
  }
#pragma unroll
  for (int j = 0; j < DN_NB; ++j)
    if (j < nb) x[j] = w[j];
}

// ---- few right-hand sides (log_likelihood's single solve, predict's alpha): one launch per 64-column block ---------
// The generic path above spends ~30 us per block in a one-thread-per-RHS substitution; with 1..8 right-hand sides the
// solve is a chain of n/64 dependent steps whose useful work is reading L once (8 n^2 / 2 bytes per sweep), so every
// step is ONE launch: each CTA redundantly solves the 64 x 64 diagonal block with a warp per right-hand side (two
// entries per lane, pivots broadcast by shuffle) and then applies it to its own 256 rows (forward) or 256 columns
// (backward) of the panel.  The solved block goes to a second buffer so that no CTA reads entries another one is
// writing: forward reads B and writes Y, backward reads Y and writes the result back into B.
constexpr int DS_MAX_RHS = 8;
constexpr int DS_ROWS = 256;   // rows of the panel per CTA (forward)
constexpr int DS_COLS = 64;    // columns of the panel per CTA (backward)

// diagonal block (identity-padded to 64 x 64) and the reciprocals of its diagonal
__device__ __forceinline__ void load_diag_block(double (*l)[DN_NB + 1], double* rl, const double* __restrict__ Lkk,
                                                int64_t ld, int nb) {
  for (int t = threadIdx.x; t < DN_NB * DN_NB; t += blockDim.x) {
    const int i = t % DN_NB, j = t / DN_NB;
    l[i][j] = (i < nb && j < nb) ? Lkk[(int64_t)j * ld + i] : (i == j ? 1.0 : 0.0);
  }
  if (threadIdx.x < DN_NB) rl[threadIdx.x] = (threadIdx.x < nb) ? 1.0 / Lkk[(int64_t)threadIdx.x * ld + threadIdx.x] : 1.0;
}

// warp-level substitution with the 64 x 64 block in shared memory; entries (lane, lane + 32) of the vector per lane
__device__ __forceinline__ void warp_trsv_lower(const double (*l)[DN_NB + 1], const double* rl, int nb, int lane,
                                                double& w0, double& w1) {
  for (int j = 0; j < nb; ++j) {  // L x = b
    const double xj = __shfl_sync(0xffffffffu, (j < 32) ? w0 : w1, j & 31) * rl[j];
    if (j < 32) {
      if (lane == j) w0 = xj; else if (lane > j) w0 = fma(-l[lane][j], xj, w0);
      w1 = fma(-l[lane + 32][j], xj, w1);
    } else {
      const int jj = j - 32;
      if (lane == jj) w1 = xj; else if (lane > jj) w1 = fma(-l[lane + 32][j], xj, w1);
    }
  }
}
__device__ __forceinline__ void warp_trsv_lower_t(const double (*l)[DN_NB + 1], const double* rl, int nb, int lane,
                                                  double& w0, double& w1) {
  for (int j = nb - 1; j >= 0; --j) {  // L^T x = y
    const double xj = __shfl_sync(0xffffffffu, (j < 32) ? w0 : w1, j & 31) * rl[j];
    if (j >= 32) {
      const int jj = j - 32;
      if (lane == jj) w1 = xj; else if (lane < jj) w1 = fma(-l[j][lane + 32], xj, w1);
      w0 = fma(-l[j][lane], xj, w0);
    } else {
      if (lane == j) w0 = xj; else if (lane < j) w0 = fma(-l[j][lane], xj, w0);
    }
  }
}

// step k0 of  L y = b :  Y[k0:k0+nb] = L_kk^-1 B[k0:k0+nb] ;  B[k0+nb:] -= L[k0+nb:, k0:k0+nb] Y[k0:k0+nb]
template <int NR>
__global__ void __launch_bounds__(DS_ROWS) trsv_fwd_step_kernel(const double* __restrict__ L, int64_t ld, int64_t n,
                                                                int64_t k0, int nb, double* __restrict__ B, int64_t ldb,
                                                                double* __restrict__ Y, int64_t ldy, int nrhs) {
  __shared__ double l[DN_NB][DN_NB + 1];
  __shared__ double rl[DN_NB];
  __shared__ double xs[DS_MAX_RHS][DN_NB];
  // this thread's row of the panel: the 64 loads are issued first so that they are in flight during the substitution
  const int64_t row = k0 + nb + (int64_t)blockIdx.x * DS_ROWS + threadIdx.x;
  double v[DN_NB];
  {
    const double* a = L + k0 * ld + (row < n ? row : k0);
#pragma unroll
    for (int q = 0; q < DN_NB; ++q) v[q] = (q < nb && row < n) ? a[(int64_t)q * ld] : 0.0;
  }
  load_diag_block(l, rl, L + k0 * ld + k0, ld, nb);
  for (int t = threadIdx.x; t < DS_MAX_RHS * DN_NB; t += blockDim.x) xs[t / DN_NB][t % DN_NB] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (w < nrhs) {
    const double* b = B + (int64_t)w * ldb + k0;
    double w0 = (lane < nb) ? b[lane] : 0.0, w1 = (lane + 32 < nb) ? b[lane + 32] : 0.0;
    warp_trsv_lower(l, rl, nb, lane, w0, w1);
    xs[w][lane] = w0; xs[w][lane + 32] = w1;
  }
  __syncthreads();
  if (blockIdx.x == 0)
    for (int t = threadIdx.x; t < nrhs * nb; t += blockDim.x) Y[(int64_t)(t / nb) * ldy + k0 + t % nb] = xs[t / nb][t % nb];
  if (row >= n) return;
  double acc[NR];
#pragma unroll
  for (int c = 0; c < NR; ++c) acc[c] = 0.0;
#pragma unroll
  for (int q = 0; q < DN_NB; ++q) {
#pragma unroll
    for (int c = 0; c < NR; ++c) acc[c] = fma(v[q], xs[c][q], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < NR; ++c)
    if (c < nrhs) B[(int64_t)c * ldb + row] -= acc[c];
}

// step k0 of  L^T x = y :  X[k0:k0+nb] = L_kk^-T Y[k0:k0+nb] ;  Y[0:k0] -= L[k0:k0+nb, 0:k0]^T X[k0:k0+nb]
// The CTA's 64 columns of the panel (64 x 64, each column 512 contiguous bytes) are staged through shared memory with
// all loads in flight at once; then one thread per (column, right-hand side) takes the dot product.
template <int NR>
__global__ void __launch_bounds__(256) trsv_bwd_step_kernel(const double* __restrict__ L, int64_t ld, int64_t k0,
                                                            int nb, double* __restrict__ Y, int64_t ldy,
                                                            double* __restrict__ X, int64_t ldx, int nrhs) {
  extern __shared__ __align__(16) double bwd_smem[];  // 71 KB: above the 48 KB static limit, opted in by the launcher
  double (*l)[DN_NB + 1] = reinterpret_cast<double (*)[DN_NB + 1]>(bwd_smem);
  double (*tile)[DN_NB + 1] = reinterpret_cast<double (*)[DN_NB + 1]>(bwd_smem + DN_NB * (DN_NB + 1));  // tile[c][q] = L[k0 + q, c_begin + c]
  double* rl = bwd_smem + (DN_NB + DS_COLS) * (DN_NB + 1);
  double (*xs)[DN_NB] = reinterpret_cast<double (*)[DN_NB]>(rl + DN_NB);
  const int64_t c_begin = (int64_t)blockIdx.x * DS_COLS;
  const int nc = (int)max((int64_t)0, min((int64_t)DS_COLS, k0 - c_begin));
  for (int t = threadIdx.x; t < DS_COLS * DN_NB; t += blockDim.x) {
    const int q = t % DN_NB, c = t / DN_NB;
    tile[c][q] = (c < nc && q < nb) ? L[(c_begin + c) * ld + k0 + q] : 0.0;
  }
  load_diag_block(l, rl, L + k0 * ld + k0, ld, nb);
  for (int t = threadIdx.x; t < DS_MAX_RHS * DN_NB; t += blockDim.x) xs[t / DN_NB][t % DN_NB] = 0.0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (w < nrhs) {
    const double* y = Y + (int64_t)w * ldy + k0;
    double w0 = (lane < nb) ? y[lane] : 0.0, w1 = (lane + 32 < nb) ? y[lane + 32] : 0.0;
    warp_trsv_lower_t(l, rl, nb, lane, w0, w1);
    xs[w][lane] = w0; xs[w][lane + 32] = w1;
  }
  __syncthreads();
  if (blockIdx.x == 0)
    for (int t = threadIdx.x; t < nrhs * nb; t += blockDim.x) X[(int64_t)(t / nb) * ldx + k0 + t % nb] = xs[t / nb][t % nb];
  // thread (c, r0): column c of this CTA's slab, right-hand sides r0, r0 + 4, ...
  const int c = threadIdx.x % DS_COLS, r0 = threadIdx.x / DS_COLS;
  if (c >= nc) return;
#pragma unroll
  for (int rr = 0; rr < (NR + 3) / 4; ++rr) {
    const int r = r0 + 4 * rr;
    if (r < nrhs) {
      double s = 0.0;
#pragma unroll 16
      for (int q = 0; q < DN_NB; ++q) s = fma(tile[c][q], xs[r][q], s);
      Y[(int64_t)r * ldy + c_begin + c] -= s;
    }
  }
}

__global__ void logdet_diag_kernel(const double* __restrict__ A, int64_t lda, int64_t n, double* out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) s += log(A[i * lda + i]);
  s = block_sum(s, red);
  if (threadIdx.x == 0) *out = 2.0 * s;
}
__global__ void dot2_kernel(const double* __restrict__ a, const double* __restrict__ b, int64_t n, double* out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    s += a[i] * b[i];
  s = block_sum(s, red);
  if (threadIdx.x == 0) atomicAdd(out, s);
}
__global__ void square2_kernel(const double* __restrict__ yerr, double* __restrict__ diag, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    diag[i] = yerr[i] * yerr[i];
}
// out (nr x n, row-major) = r (nr x n, row-major) @ U with U = L^T:  out[a][j] = sum_{i<=j} r[a][i] L[j][i]
__global__ void apply_sqrt_kernel(const double* __restrict__ L, int64_t n, const double* __restrict__ r, int64_t nr,
                                  double* __restrict__ out) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t a = blockIdx.y;
  if (j >= n) return;
  double s = 0.0;
  for (int64_t i = 0; i <= j; ++i) s += r[a * n + i] * L[i * n + j];  // L[j][i] column-major = L[i*n + j]
  out[a * n + j] = s;
}

}  // namespace bgp

using namespace bgp;

struct bgp_dense {
  Stream s;  // declared before every DevBuf: streams outlive buffers
  Event ev[4];
  ~bgp_dense() { s.sync(); }
  int64_t n = 0;
  bool computed = false;
  double log_det = 0.0;
  DevBuf<DevProgram> d_prog;
  DevBuf<double> d_x, d_yerr, d_diag, d_A, d_rhs, d_scalar;
  DevBuf<double> d_tmp;              // second buffer of the few-RHS solve
  DevBuf<double> d_inv, d_gscratch;  // grad_terms: K^-1 (n x n) and the contraction partials
  DevBuf<unsigned> d_which;
  bool has_inputs = false;           // d_x / d_prog describe the factor in d_A (false after import_factor)
  int ndim = 0, n_params = 0;
  DevBuf<int> d_info;
  DevBuf<GemmDesc> d_gdesc;
  double t_ms[2] = {0, 0};
};

static int ensure_stream(bgp_dense* h) {
  BGP_TRY(h->s.create());
  for (Event& e : h->ev) BGP_TRY(e.create());
  return BGP_OK;
}

// Blocked right-looking Cholesky with DELAYED trailing updates on three nested block sizes (64 | DN_MB | DN_OB): after
// the panel ending at column e, the rank-64 update touches only the rest of the current DN_MB block; when e closes a
// DN_MB block its accumulated rank-DN_MB update touches the rest of the current DN_OB block; when e closes a DN_OB block
// the rank-DN_OB update touches everything to the right.  Almost all flops therefore run as GEMMs with K = DN_OB, whose
// read-modify-write epilogue of C is amortised over 16x more tensor work than at K = 64.
static_assert(DN_MB % DN_NB == 0 && DN_MB < DN_OB && DN_OB % DN_MB == 0, "the three block sizes nest");

static int dense_potrf(bgp_dense* h) {
  const int64_t n = h->n;
  double* A = h->d_A.p;
  cudaStream_t s = h->s;
  // all trailing-update descriptors of the factorisation, uploaded once
  std::vector<GemmDesc> descs;
  struct Step { int64_t k0; int nb; int64_t rem; int desc[3]; };
  std::vector<Step> steps;
  // C[e:n, e:cend) -= L[e:n, b:e) L[e:cend, b:e)^T   (lower part only)
  auto add_update = [&](int64_t b, int64_t e, int64_t cend) -> int {
    if (e >= n || cend <= e || e <= b) return -1;
    GemmDesc d;
    const double* P = A + b * n + e;          // rows e.., columns b..e of the factor
    d.A = P; d.lda = n; d.B = P; d.ldb = n;   // B' = P^T restricted to the first (cend - e) rows of P
    d.C = A + e * n + e; d.ldc = n;
    d.M = (int)(n - e); d.N = (int)(cend - e); d.K = (int)(e - b); d.mode = GD_SUB | GD_LOWER;
    descs.push_back(d);
    return (int)descs.size() - 1;
  };
  for (int64_t j0 = 0; j0 < n; j0 += DN_NB) {
    Step st;
    st.k0 = j0; st.nb = (int)std::min<int64_t>(DN_NB, n - j0); st.rem = n - j0 - st.nb;
    const int64_t e = j0 + st.nb;
    const int64_t mb0 = (j0 / DN_MB) * DN_MB, mb1 = std::min<int64_t>(n, mb0 + DN_MB);  // the DN_MB block holding this panel
    const int64_t ob0 = (j0 / DN_OB) * DN_OB, ob1 = std::min<int64_t>(n, ob0 + DN_OB);  // the DN_OB block holding it
    st.desc[0] = add_update(j0, e, mb1);
    st.desc[1] = (e == mb1) ? add_update(mb0, e, ob1) : -1;
    st.desc[2] = (e == ob1) ? add_update(ob0, e, n) : -1;
    steps.push_back(st);
  }
  BGP_TRY(h->d_gdesc.reserve(std::max<size_t>(descs.size(), 1), s));
  if (!descs.empty())
    BGP_CUDA(cudaMemcpyAsync(h->d_gdesc.p, descs.data(), sizeof(GemmDesc) * descs.size(), cudaMemcpyHostToDevice, s));
  for (const Step& st : steps) {
    double* Akk = A + st.k0 * n + st.k0;
    potf2_kernel<<<1, DN_NB, 0, s>>>(Akk, n, st.nb, h->d_info.p, (int)st.k0);
    BGP_LAUNCH_CHECK();
    if (st.rem <= 0) break;
    trsm_panel_kernel<<<(unsigned)((st.rem + 127) / 128), 128, 0, s>>>(Akk, n, st.rem, st.nb, h->d_info.p);
    BGP_LAUNCH_CHECK();
    for (int l = 0; l < 3; ++l)
      if (st.desc[l] >= 0)
        BGP_TRY((gemm_dmma_launch<false, false>(h->d_gdesc.p + st.desc[l], 1, descs[st.desc[l]].M, descs[st.desc[l]].N, h->d_info.p, s)));
  }
  return BGP_OK;
}

// X (n x nrhs, column-major ldx) <- K^-1 X on the device
constexpr size_t DS_BWD_SMEM = sizeof(double) * ((DN_NB + DS_COLS) * (DN_NB + 1) + DN_NB + DS_MAX_RHS * DN_NB);

static int dense_potrs_small(bgp_dense* h, double* X, int nrhs, int64_t ldx) {
  // (the attribute is per device / context: set it on every call, it is cheap)
  cudaFuncSetAttribute(trsv_bwd_step_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DS_BWD_SMEM);
    cudaFuncSetAttribute(trsv_bwd_step_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DS_BWD_SMEM);
    cudaFuncSetAttribute(trsv_bwd_step_kernel<DS_MAX_RHS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DS_BWD_SMEM);
  const int64_t n = h->n;
  const double* L = h->d_A.p;
  cudaStream_t s = h->s;
  BGP_TRY(h->d_tmp.reserve((size_t)n * DS_MAX_RHS, s));
  double* Y = h->d_tmp.p;
  for (int64_t k0 = 0; k0 < n; k0 += DN_NB) {
    const int nb = (int)std::min<int64_t>(DN_NB, n - k0);
    const int64_t rem = n - k0 - nb;
    const unsigned g = (unsigned)std::max<int64_t>(1, (rem + DS_ROWS - 1) / DS_ROWS);
    if (nrhs == 1) trsv_fwd_step_kernel<1><<<g, DS_ROWS, 0, s>>>(L, n, n, k0, nb, X, ldx, Y, n, nrhs);
    else if (nrhs <= 4) trsv_fwd_step_kernel<4><<<g, DS_ROWS, 0, s>>>(L, n, n, k0, nb, X, ldx, Y, n, nrhs);
    else trsv_fwd_step_kernel<DS_MAX_RHS><<<g, DS_ROWS, 0, s>>>(L, n, n, k0, nb, X, ldx, Y, n, nrhs);
    BGP_LAUNCH_CHECK();
  }
  for (int64_t k0 = ((n - 1) / DN_NB) * DN_NB; k0 >= 0; k0 -= DN_NB) {
    const int nb = (int)std::min<int64_t>(DN_NB, n - k0);
    const unsigned g = (unsigned)std::max<int64_t>(1, (k0 + DS_COLS - 1) / DS_COLS);
    if (nrhs == 1) trsv_bwd_step_kernel<1><<<g, 256, DS_BWD_SMEM, s>>>(L, n, k0, nb, Y, n, X, ldx, nrhs);
    else if (nrhs <= 4) trsv_bwd_step_kernel<4><<<g, 256, DS_BWD_SMEM, s>>>(L, n, k0, nb, Y, n, X, ldx, nrhs);
    else trsv_bwd_step_kernel<DS_MAX_RHS><<<g, 256, DS_BWD_SMEM, s>>>(L, n, k0, nb, Y, n, X, ldx, nrhs);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

static int dense_potrs_dev(bgp_dense* h, double* X, int64_t nrhs, int64_t ldx) {
  if (nrhs <= DS_MAX_RHS) return dense_potrs_small(h, X, (int)nrhs, ldx);
  const int64_t n = h->n;
  const double* L = h->d_A.p;
  cudaStream_t s = h->s;
  const unsigned cb = (unsigned)((nrhs + 127) / 128);
  for (int64_t k0 = 0; k0 < n; k0 += DN_NB) {  // forward: L y = b
    const int nb = (int)std::min<int64_t>(DN_NB, n - k0);
    trsv_block_kernel<<<cb, 128, 0, s>>>(L + k0 * n + k0, n, nb, X + k0, ldx, nrhs, 0);
    BGP_LAUNCH_CHECK();
    const int64_t rem = n - k0 - nb;
    if (rem <= 0) break;
    dim3 grid((unsigned)((rem + GM_T - 1) / GM_T), (unsigned)((nrhs + GM_T - 1) / GM_T));
    gemm_sub_kernel<0, 0><<<grid, 256, 0, s>>>(rem, nrhs, nb, L + k0 * n + k0 + nb, n, X + k0, ldx, X + k0 + nb, ldx, 0, nullptr);
    BGP_LAUNCH_CHECK();
  }
  const int64_t last = ((n - 1) / DN_NB) * DN_NB;
  for (int64_t k0 = last; k0 >= 0; k0 -= DN_NB) {  // backward: L^T x = y
    const int nb = (int)std::min<int64_t>(DN_NB, n - k0);
    trsv_block_kernel<<<cb, 128, 0, s>>>(L + k0 * n + k0, n, nb, X + k0, ldx, nrhs, 1);
    BGP_LAUNCH_CHECK();
    if (k0 == 0) break;
    // X[0:k0] -= L[k0:k0+nb, 0:k0]^T X[k0:k0+nb]
    dim3 grid((unsigned)((k0 + GM_T - 1) / GM_T), (unsigned)((nrhs + GM_T - 1) / GM_T));
    gemm_sub_kernel<1, 0><<<grid, 256, 0, s>>>(k0, nrhs, nb, L + k0, n, X + k0, ldx, X, ldx, 0, nullptr);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

extern "C" {

int bgp_dense_create(bgp_dense_t** out) {
  *out = new (std::nothrow) bgp_dense();
  if (!*out) { set_error("out of host memory"); return BGP_ERR_NOMEM; }
  return BGP_OK;
}

void bgp_dense_destroy(bgp_dense_t* h) {
  if (!h) return;
  delete h;
}

int bgp_dense_compute(bgp_dense_t* h, const bgp_kernel_spec_t* spec, const double* x, int64_t n, int32_t ndim,
                      const double* yerr) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  h->computed = false;
  BGP_TRY(require_device());
  BGP_TRY(ensure_stream(h));
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  if (P.ndim != ndim) { set_error("dimension mismatch: kernel ndim %d, input ndim %d", P.ndim, ndim); return BGP_ERR_DIM; }
  if (n <= 0) { set_error("invalid number of points"); return BGP_ERR_INVALID; }
  cudaStream_t s = h->s;
  h->n = n;
  h->has_inputs = false;
  h->ndim = ndim;
  h->n_params = P.n_params_total;
  BGP_TRY(upload_program(P, h->d_prog, s));
  BGP_TRY(h->d_x.reserve((size_t)n * ndim, s));
  BGP_TRY(h->d_yerr.reserve((size_t)n, s));
  BGP_TRY(h->d_diag.reserve((size_t)n, s));
  BGP_TRY(h->d_A.reserve((size_t)n * n, s));
  BGP_TRY(h->d_info.reserve(1, s));
  BGP_TRY(h->d_scalar.reserve(2, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_x.p, x, sizeof(double) * n * ndim, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_yerr.p, yerr, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemsetAsync(h->d_info.p, 0, sizeof(int), s));
  square2_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1184), 256, 0, s>>>(h->d_yerr.p, h->d_diag.p, n);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaEventRecord(h->ev[0], s));
  BGP_TRY(kmat_symmetric_launch_auto(P, h->d_prog.p, h->d_x.p, n, h->d_diag.p, h->d_A.p, n, s));
  BGP_CUDA(cudaEventRecord(h->ev[1], s));
  BGP_TRY(dense_potrf(h));
  logdet_diag_kernel<<<1, 1024, 0, s>>>(h->d_A.p, n, n, h->d_scalar.p);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaEventRecord(h->ev[2], s));
  int info = 0;
  double ld = 0.0;
  BGP_CUDA(cudaMemcpyAsync(&info, h->d_info.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaMemcpyAsync(&ld, h->d_scalar.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->t_ms[0] = ms;
  cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]); h->t_ms[1] = ms;
  if (info != 0) {
    set_error("%d-th leading minor of the array is not positive definite", info);
    return BGP_ERR_LINALG;
  }
  h->log_det = ld;
  h->computed = true;
  h->has_inputs = true;
  return BGP_OK;
}

int bgp_dense_log_determinant(const bgp_dense_t* h, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  *out = h->log_det;
  return BGP_OK;
}

int bgp_dense_apply_inverse(bgp_dense_t* h, double* b, int64_t nrhs, int64_t ldb) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  if (nrhs <= 0) return BGP_OK;
  if (ldb < h->n) { set_error("dimension mismatch: ldb < n"); return BGP_ERR_DIM; }
  const int64_t n = h->n;
  cudaStream_t s = h->s;
  const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(nrhs, (int64_t)(1ull << 28) / n));
  BGP_TRY(h->d_rhs.reserve((size_t)n * slab, s));
  for (int64_t c0 = 0; c0 < nrhs; c0 += slab) {
    const int64_t nc = std::min(slab, nrhs - c0);
    BGP_CUDA(cudaMemcpy2DAsync(h->d_rhs.p, sizeof(double) * n, b + c0 * ldb, sizeof(double) * ldb, sizeof(double) * n, nc, cudaMemcpyHostToDevice, s));
    BGP_TRY(dense_potrs_dev(h, h->d_rhs.p, nc, n));
    BGP_CUDA(cudaMemcpy2DAsync(b + c0 * ldb, sizeof(double) * ldb, h->d_rhs.p, sizeof(double) * n, sizeof(double) * n, nc, cudaMemcpyDeviceToHost, s));
    BGP_CUDA(cudaStreamSynchronize(s));
  }
  return BGP_OK;
}

int bgp_dense_dot_solve(bgp_dense_t* h, const double* y, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  cudaStream_t s = h->s;
  BGP_TRY(h->d_rhs.reserve((size_t)n * 2, s));
  double* yd = h->d_rhs.p;
  double* xd = h->d_rhs.p + n;
  BGP_CUDA(cudaMemcpyAsync(yd, y, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(xd, yd, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
  BGP_TRY(dense_potrs_dev(h, xd, 1, n));
  BGP_CUDA(cudaMemsetAsync(h->d_scalar.p + 1, 0, sizeof(double), s));
  dot2_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 592), 256, 0, s>>>(yd, xd, n, h->d_scalar.p + 1);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaMemcpyAsync(out, h->d_scalar.p + 1, sizeof(double), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_dense_apply_sqrt(bgp_dense_t* h, const double* r, int64_t nr, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  cudaStream_t s = h->s;
  if (nr <= 0) return BGP_OK;
  DevBuf<double> dr, dout;
  BGP_TRY(dr.alloc((size_t)nr * n, s));
  BGP_TRY(dout.alloc((size_t)nr * n, s));
  BGP_CUDA(cudaMemcpyAsync(dr.p, r, sizeof(double) * nr * n, cudaMemcpyHostToDevice, s));
  dim3 grid((unsigned)((n + 127) / 128), (unsigned)nr);
  apply_sqrt_kernel<<<grid, 128, 0, s>>>(h->d_A.p, n, dr.p, nr, dout.p);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * nr * n, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_dense_get_inverse(bgp_dense_t* h, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  for (int64_t j = 0; j < n; ++j) {
    double* c = out + j * n;
    memset(c, 0, sizeof(double) * n);
    c[j] = 1.0;
  }
  return bgp_dense_apply_inverse(h, out, n, n);
}

int bgp_dense_grad_terms(bgp_dense_t* h, const uint32_t* which, const double* r, double* alpha_out, double* g_out,
                         double* diag_out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  if (!h->has_inputs) { set_error("the factor was imported: the handle holds no kernel/coordinates"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  const int np = h->n_params;
  cudaStream_t s = h->s;
  BGP_TRY(h->d_rhs.reserve((size_t)n * 2 + 64, s));
  double* alpha = h->d_rhs.p;
  double* dg = h->d_rhs.p + n;       // np <= 64 entries
  double* ddiag = h->d_rhs.p + n + 64;
  BGP_CUDA(cudaMemcpyAsync(alpha, r, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  BGP_TRY(dense_potrs_dev(h, alpha, 1, n));
  if (alpha_out) BGP_CUDA(cudaMemcpyAsync(alpha_out, alpha, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  if (np > 64) { set_error("gradient supports at most 64 hyper-parameters"); return BGP_ERR_INVALID; }
  BGP_TRY(h->d_inv.reserve((size_t)n * n, s));
  BGP_TRY(fill_identity_launch(h->d_inv.p, n, s));
  BGP_TRY(dense_potrs_dev(h, h->d_inv.p, n, n));
  BGP_TRY(h->d_which.reserve(std::max(np, 1), s));
  if (np) BGP_CUDA(cudaMemcpyAsync(h->d_which.p, which, sizeof(unsigned) * np, cudaMemcpyHostToDevice, s));
  // kernel term of gp.py:457-466 and diag(alpha alpha^T - K^-1) for the white-noise term of gp.py:452-456
  BGP_TRY(kmat_grad_contract_launch(h->d_prog.p, h->ndim, np, h->d_which.p, h->d_x.p, n, h->d_inv.p, n, alpha, 1.0, -1.0, dg,
                                    diag_out ? ddiag : nullptr, h->d_gscratch, s));
  if (np && g_out) BGP_CUDA(cudaMemcpyAsync(g_out, dg, sizeof(double) * np, cudaMemcpyDeviceToHost, s));
  if (diag_out) BGP_CUDA(cudaMemcpyAsync(diag_out, ddiag, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_dense_export_factor(bgp_dense_t* h, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  BGP_CUDA(cudaMemcpyAsync(out, h->d_A.p, sizeof(double) * n * n, cudaMemcpyDeviceToHost, h->s));
  BGP_CUDA(cudaStreamSynchronize(h->s));
  for (int64_t j = 1; j < n; ++j)
    for (int64_t i = 0; i < j; ++i) out[j * n + i] = 0.0;  // column-major: element (i, j) with i < j
  return BGP_OK;
}

int bgp_dense_import_factor(bgp_dense_t* h, const double* factor, int64_t n, double log_det) {
  if (!h || n <= 0) { set_error("invalid argument"); return BGP_ERR_INVALID; }
  h->computed = false;
  BGP_TRY(require_device());
  BGP_TRY(ensure_stream(h));
  h->n = n;
  h->has_inputs = false;
  BGP_TRY(h->d_A.reserve((size_t)n * n, h->s));
  BGP_TRY(h->d_scalar.reserve(2, h->s));
  BGP_CUDA(cudaMemcpyAsync(h->d_A.p, factor, sizeof(double) * n * n, cudaMemcpyHostToDevice, h->s));
  BGP_CUDA(cudaStreamSynchronize(h->s));
  h->log_det = log_det;
  h->computed = true;
  return BGP_OK;
}

int bgp_dense_last_timing(const bgp_dense_t* h, double* ms2) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  ms2[0] = h->t_ms[0]; ms2[1] = h->t_ms[1];
  return BGP_OK;
}

}  // extern "C"

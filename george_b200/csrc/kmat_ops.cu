// kmat_ops.cu — matrix-free consumers of the covariance function: nothing here ever materialises a kernel matrix.
//
//   kmat_matvec_kernel       out = K(x1, x2) V   (+ diag . V)      -> GP.predict's mean  K(x*, x) alpha
//                            (reference: kernel.get_value(xs, x) then numpy dot, src/george/gp.py:524-528 over
//                             kernel_interface.cpp:47-60), and the full-size round-trip check  K (K^-1 y) == y.
//   kmat_grad_contract_kernel  g_p = sum_ij A_ij dK_ij/dtheta_p     -> GP.grad_log_likelihood's kernel term
//                            (reference: kernel.get_gradient(x) -> (n, n, P) tensor, then
//                             0.5 * einsum("ijk,ij", dK, alpha alpha^T - K^-1), src/george/gp.py:437-466 over
//                             kernel_interface.cpp:109-125).  A is read once (8 n^2 bytes); the (n, n, P) tensor is never
//                             formed.
//
// Roofline: matvec is FP64-ALU bound (one covariance evaluation per (i, j), no HBM traffic beyond x and V);
// the contraction reads A once -> HBM bound at 8 B per pair for cheap kernels, FP64 bound for the gradient of
// expensive ones.  Partial sums are written per CTA and reduced by a second tiny kernel in a fixed order, so results
// are run-to-run deterministic (no atomics).
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "kernel_eval.cuh"

namespace bgp {
int upload_program(const DevProgram& P, DevBuf<DevProgram>& buf, cudaStream_t s);

constexpr int MV_TI = 64;        // rows per CTA
constexpr int MV_TJ = 512;       // columns staged per iteration
constexpr int MV_THREADS = 256;  // 64 rows x 4 column lanes
constexpr int MV_NR = 4;         // right-hand sides per launch

struct MvSmem {
  DevProgram prog;
  uint64_t bar;
};

// partial[(split * n1 + i) * MV_NR + c] = sum_{j in split's chunks} k(x1_i, x2_j) V[j + c*ldv]
template <typename Fn>
__device__ __forceinline__ void matvec_tile(const Fn& fn, int nd, const double* sx1, const double* sx2,
                                            const double* sv, int ni, int nj, int row, int lane4, double (&acc)[MV_NR]) {
  if (row >= ni) return;
  const double* xi = sx1 + row * nd;
  for (int j = lane4; j < nj; j += MV_THREADS / MV_TI) {
    const double k = fn(xi, sx2 + j * nd);
#pragma unroll
    for (int c = 0; c < MV_NR; ++c) acc[c] = fma(k, sv[c * MV_TJ + j], acc[c]);
  }
}

__global__ void __launch_bounds__(MV_THREADS) kmat_matvec_kernel(const DevProgram* __restrict__ gprog,
                                                                 const double* __restrict__ x1, int64_t n1,
                                                                 const double* __restrict__ x2, int64_t n2,
                                                                 const double* __restrict__ V, int64_t ldv, int nrhs,
                                                                 double* __restrict__ partial, int chunks_per_split) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  MvSmem* S = reinterpret_cast<MvSmem*>(smem_raw);
  const int nd = gprog->ndim;
  double* sx1 = reinterpret_cast<double*>(smem_raw + ((sizeof(MvSmem) + 15) & ~size_t(15)));
  double* sx2 = sx1 + MV_TI * nd + ((MV_TI * nd) & 1);
  double* sv = sx2 + MV_TJ * nd;           // MV_NR x MV_TJ
  double* red = sv + MV_NR * MV_TJ;         // MV_THREADS x MV_NR

  stage_program(&S->prog, gprog);
  if (threadIdx.x == 0) { mbar_init(&S->bar, 1); mbar_fence_init(); }
  __syncthreads();
  uint32_t phase = 0;

  const int64_t i0 = (int64_t)blockIdx.x * MV_TI;
  const int ni = (int)min((int64_t)MV_TI, n1 - i0);
  load_coords(sx1, x1 + i0 * nd, ni * nd, &S->bar, phase);

  const int row = threadIdx.x & (MV_TI - 1), lane4 = threadIdx.x / MV_TI;
  double acc[MV_NR];
#pragma unroll
  for (int c = 0; c < MV_NR; ++c) acc[c] = 0.0;

  const int64_t nchunks = (n2 + MV_TJ - 1) / MV_TJ;
  const int64_t c_begin = (int64_t)blockIdx.y * chunks_per_split;
  const int64_t c_end = min(nchunks, c_begin + chunks_per_split);
  for (int64_t ch = c_begin; ch < c_end; ++ch) {
    const int64_t j0 = ch * MV_TJ;
    const int nj = (int)min((int64_t)MV_TJ, n2 - j0);
    __syncthreads();  // previous iteration's readers are done with sx2 / sv
    load_coords(sx2, x2 + j0 * nd, nj * nd, &S->bar, phase);
    for (int t = threadIdx.x; t < MV_NR * MV_TJ; t += MV_THREADS) {
      const int c = t / MV_TJ, j = t - c * MV_TJ;
      sv[t] = (c < nrhs && j < nj) ? V[(int64_t)c * ldv + j0 + j] : 0.0;
    }
    __syncthreads();
    BGP_DISPATCH_SHAPE(S->prog, matvec_tile(fn, nd, sx1, sx2, sv, ni, nj, row, lane4, acc));
  }
  // combine the 4 column lanes of each row (fixed order), one partial per (split, row, rhs)
#pragma unroll
  for (int c = 0; c < MV_NR; ++c) red[threadIdx.x * MV_NR + c] = acc[c];
  __syncthreads();
  if (lane4 == 0 && row < ni) {
#pragma unroll
    for (int c = 0; c < MV_NR; ++c) {
      double s = red[row * MV_NR + c];
      for (int q = 1; q < MV_THREADS / MV_TI; ++q) s += red[(q * MV_TI + row) * MV_NR + c];
      partial[((int64_t)blockIdx.y * n1 + i0 + row) * MV_NR + c] = s;
    }
  }
}

// out[i + c*ldo] = sum_s partial[(s*n1 + i)*MV_NR + c]  (+ diag[i] * V[i + c*ldv])
__global__ void kmat_matvec_reduce_kernel(const double* __restrict__ partial, int64_t n1, int nsplit, int nrhs,
                                          const double* __restrict__ diag, const double* __restrict__ V, int64_t ldv,
                                          double* __restrict__ out, int64_t ldo) {
  const int64_t total = n1 * nrhs;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = t / n1, i = t - c * n1;
    double s = 0.0;
    for (int sp = 0; sp < nsplit; ++sp) s += partial[((int64_t)sp * n1 + i) * MV_NR + c];
    if (diag) s = fma(diag[i], V[c * ldv + i], s);
    out[c * ldo + i] = s;
  }
}

static size_t matvec_smem(int nd) {
  return ((sizeof(MvSmem) + 15) & ~size_t(15)) +
         sizeof(double) * ((size_t)MV_TI * nd + 1 + (size_t)MV_TJ * nd + (size_t)MV_NR * MV_TJ + (size_t)MV_THREADS * MV_NR);
}

// out (n1 x nrhs, column-major ldo) = K(x1, x2) V (n2 x nrhs, column-major ldv) [+ diag .* V, only when n1 == n2]
int kmat_matvec_launch(const DevProgram* dprog, int nd, const double* x1, int64_t n1, const double* x2, int64_t n2,
                       const double* diag, const double* V, int64_t ldv, int64_t nrhs, double* out, int64_t ldo,
                       DevBuf<double>& scratch, cudaStream_t s) {
  if (n1 <= 0 || nrhs <= 0) return BGP_OK;
  if (n2 <= 0) {
    for (int64_t c = 0; c < nrhs; ++c) BGP_CUDA(cudaMemsetAsync(out + c * ldo, 0, sizeof(double) * n1, s));
    return BGP_OK;
  }
  // (the attribute is per device / context: set it on every call, it is cheap)
  cudaFuncSetAttribute(kmat_matvec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
  const size_t smem = matvec_smem(nd);
  const int64_t row_tiles = (n1 + MV_TI - 1) / MV_TI;
  const int64_t nchunks = (n2 + MV_TJ - 1) / MV_TJ;
  // enough CTAs for ~8 per SM; when there are few row tiles (predict at a handful of points) split the columns instead
  int64_t nsplit = std::max<int64_t>(1, std::min<int64_t>(nchunks, (8 * (int64_t)num_sms() + row_tiles - 1) / row_tiles));
  const int cps = (int)((nchunks + nsplit - 1) / nsplit);
  nsplit = (nchunks + cps - 1) / cps;
  if (row_tiles > 0x7fffffffLL || nsplit > 65535) { set_error("kmat_matvec: problem too large for one launch"); return BGP_ERR_INVALID; }
  BGP_TRY(scratch.reserve((size_t)nsplit * (size_t)n1 * MV_NR, s));
  for (int64_t c0 = 0; c0 < nrhs; c0 += MV_NR) {
    const int nc = (int)std::min<int64_t>(MV_NR, nrhs - c0);
    dim3 grid((unsigned)row_tiles, (unsigned)nsplit);
    kmat_matvec_kernel<<<grid, MV_THREADS, smem, s>>>(dprog, x1, n1, x2, n2, V + c0 * ldv, ldv, nc, scratch.p, cps);
    BGP_LAUNCH_CHECK();
    const int blocks = (int)std::min<int64_t>((n1 * nc + 255) / 256, 8 * (int64_t)num_sms());
    kmat_matvec_reduce_kernel<<<blocks, 256, 0, s>>>(scratch.p, n1, (int)nsplit, nc, diag, V + c0 * ldv, ldv,
                                                     out + c0 * ldo, ldo);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// gradient contraction.  Pairs (i, j) with i <= j are evaluated once, as the reference does (kernel_interface.cpp:
// 116-121 evaluates the upper triangle and mirrors), and weighted with A_ij + A_ji (A_ii on the diagonal), where
//     A_ij = ca * alpha_i * alpha_j + cm * M_ij          (grad_log_likelihood: ca = 1, cm = -1, M = K^-1).
// Tiles of 32 x 32 pairs; M's tile and its transposed partner are staged through shared memory so both reads are
// coalesced.  NPMAX is the register budget for the per-parameter accumulators.
// ---------------------------------------------------------------------------------------------------------------
constexpr int GC_T = 32;
constexpr int GC_THREADS = 256;

template <int NPMAX>
__global__ void __launch_bounds__(GC_THREADS) kmat_grad_contract_kernel(const DevProgram* __restrict__ gprog,
                                                                        const unsigned* __restrict__ which,
                                                                        const double* __restrict__ x, int64_t n,
                                                                        const double* __restrict__ M, int64_t ldm,
                                                                        const double* __restrict__ alpha, double ca,
                                                                        double cm, double* __restrict__ partial) {
  __shared__ DevProgram P;
  __shared__ unsigned sw[BGP_MAX_LEAVES * (4 + BGP_MAX_METRIC)];
  __shared__ double tA[GC_T][GC_T + 1], tB[GC_T][GC_T + 1];
  __shared__ double red[32];
  const int np = gprog->n_params_total;
  double acc[NPMAX];
#pragma unroll
  for (int q = 0; q < NPMAX; ++q) acc[q] = 0.0;
  const int64_t nt = (n + GC_T - 1) / GC_T;
  const int64_t bi = blockIdx.y, bj = blockIdx.x;
  const int64_t cta = bi * gridDim.x + bj;
  if (bi <= bj && bi < nt && bj < nt) {
    stage_program(&P, gprog);
    for (int q = threadIdx.x; q < np; q += blockDim.x) sw[q] = which[q];
    const int nd = gprog->ndim;
    const int64_t i0 = bi * GC_T, j0 = bj * GC_T;
    const int ni = (int)min((int64_t)GC_T, n - i0), nj = (int)min((int64_t)GC_T, n - j0);
    // tA[r][c] = M[i0+r][j0+c],  tB[c][r] = M[j0+c][i0+r]   (row-major M with leading dimension ldm; symmetric use)
    for (int t = threadIdx.x; t < GC_T * GC_T; t += GC_THREADS) {
      const int r = t / GC_T, c = t % GC_T;
      tA[r][c] = (r < ni && c < nj) ? M[(i0 + r) * ldm + j0 + c] : 0.0;
      tB[r][c] = (r < nj && c < ni) ? M[(j0 + r) * ldm + i0 + c] : 0.0;
    }
    __syncthreads();
    double g[NPMAX];
    for (int t = threadIdx.x; t < GC_T * GC_T; t += GC_THREADS) {
      const int r = t / GC_T, c = t % GC_T;
      if (r >= ni || c >= nj) continue;
      const int64_t i = i0 + r, j = j0 + c;
      if (i > j) continue;
      double w;
      if (i == j) w = cm * tA[r][c] + (alpha ? ca * alpha[i] * alpha[i] : 0.0);
      else w = cm * (tA[r][c] + tB[c][r]) + (alpha ? 2.0 * ca * alpha[i] * alpha[j] : 0.0);
      kernel_value_grad(P, x + i * nd, x + j * nd, sw, g);
#pragma unroll
      for (int q = 0; q < NPMAX; ++q)
        if (q < np) acc[q] = fma(w, g[q], acc[q]);
    }
  }
  // one partial per (CTA, parameter); CTAs below the diagonal write zeros so the reduction is a plain sum
#pragma unroll
  for (int q = 0; q < NPMAX; ++q) {
    if (q < np) {  // uniform across the CTA
      const double s = block_sum(acc[q], red);
      if (threadIdx.x == 0) partial[cta * np + q] = s;
    }
  }
}

__global__ void grad_contract_reduce_kernel(const double* __restrict__ partial, int64_t nctas, int np,
                                            double* __restrict__ out) {
  __shared__ double red[32];
  const int q = blockIdx.x;
  double s = 0.0;
  for (int64_t c = threadIdx.x; c < nctas; c += blockDim.x) s += partial[c * np + q];
  s = block_sum(s, red);
  if (threadIdx.x == 0) out[q] = s;
}

// diagA[i] = ca * alpha_i^2 + cm * M_ii
__global__ void grad_diag_kernel(const double* __restrict__ M, int64_t ldm, const double* __restrict__ alpha, double ca,
                                 double cm, int64_t n, double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = cm * M[i * ldm + i] + (alpha ? ca * alpha[i] * alpha[i] : 0.0);
}

// g_dev[np] = sum_ij (ca alpha_i alpha_j + cm M_ij) dK_ij/dtheta ; diag_dev[n] (may be null) = diag of that weight matrix
int kmat_grad_contract_launch(const DevProgram* dprog, int nd, int np, const unsigned* which_dev, const double* x,
                              int64_t n, const double* M, int64_t ldm, const double* alpha, double ca, double cm,
                              double* g_dev, double* diag_dev, DevBuf<double>& scratch, cudaStream_t s) {
  (void)nd;
  if (n <= 0) return BGP_OK;
  if (np > 64) { set_error("gradient supports at most 64 hyper-parameters"); return BGP_ERR_INVALID; }
  if (np > 0) {
    const int64_t nt = (n + GC_T - 1) / GC_T;
    if (nt > 65535) { set_error("kmat_grad_contract: n too large for one launch"); return BGP_ERR_INVALID; }
    const int64_t nctas = nt * nt;
    BGP_TRY(scratch.reserve((size_t)nctas * np, s));
    dim3 grid((unsigned)nt, (unsigned)nt);
    if (np <= 8) kmat_grad_contract_kernel<8><<<grid, GC_THREADS, 0, s>>>(dprog, which_dev, x, n, M, ldm, alpha, ca, cm, scratch.p);
    else kmat_grad_contract_kernel<64><<<grid, GC_THREADS, 0, s>>>(dprog, which_dev, x, n, M, ldm, alpha, ca, cm, scratch.p);
    BGP_LAUNCH_CHECK();
    grad_contract_reduce_kernel<<<np, 256, 0, s>>>(scratch.p, nctas, np, g_dev);
    BGP_LAUNCH_CHECK();
  }
  if (diag_dev) {
    grad_diag_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1184), 256, 0, s>>>(M, ldm, alpha, ca, cm, n, diag_dev);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

// I (n x n, column-major == row-major) on the device
__global__ void fill_identity_kernel(double* __restrict__ A, int64_t n) {
  const int64_t total = n * n;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x)
    A[t] = (t / n == t % n) ? 1.0 : 0.0;
}
int fill_identity_launch(double* A, int64_t n, cudaStream_t s) {
  fill_identity_kernel<<<(unsigned)std::min<int64_t>((n * n + 255) / 256, 16 * (int64_t)num_sms()), 256, 0, s>>>(A, n);
  BGP_LAUNCH_CHECK();
  return BGP_OK;
}

}  // namespace bgp

using namespace bgp;

extern "C" {

int bgp_kmat_matvec(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2, int64_t n2,
                    const double* diag, const double* v, int64_t nrhs, double* out) {
  BGP_TRY(require_device());
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  if (n1 < 0 || n2 < 0 || nrhs < 0) { set_error("negative size"); return BGP_ERR_INVALID; }
  if (diag && n1 != n2) { set_error("dimension mismatch: a diagonal term needs a square operator"); return BGP_ERR_DIM; }
  if (n1 == 0 || nrhs == 0) return BGP_OK;
  cudaStream_t s = 0;
  const int nd = P.ndim;
  const bool same = (x1 == x2 && n1 == n2);
  DevBuf<DevProgram> dprog;
  DevBuf<double> dx1, dx2, dv, dd, dout, scratch;
  BGP_TRY(upload_program(P, dprog, s));
  BGP_TRY(dx1.alloc((size_t)n1 * nd, s));
  BGP_CUDA(cudaMemcpyAsync(dx1.p, x1, sizeof(double) * n1 * nd, cudaMemcpyHostToDevice, s));
  const double* px2 = dx1.p;
  if (!same) {
    BGP_TRY(dx2.alloc((size_t)n2 * nd, s));
    if (n2) BGP_CUDA(cudaMemcpyAsync(dx2.p, x2, sizeof(double) * n2 * nd, cudaMemcpyHostToDevice, s));
    px2 = dx2.p;
  }
  BGP_TRY(dv.alloc((size_t)std::max<int64_t>(n2, 1) * nrhs, s));
  if (n2) BGP_CUDA(cudaMemcpyAsync(dv.p, v, sizeof(double) * n2 * nrhs, cudaMemcpyHostToDevice, s));
  if (diag) {
    BGP_TRY(dd.alloc((size_t)n1, s));
    BGP_CUDA(cudaMemcpyAsync(dd.p, diag, sizeof(double) * n1, cudaMemcpyHostToDevice, s));
  }
  BGP_TRY(dout.alloc((size_t)n1 * nrhs, s));
  BGP_TRY(kmat_matvec_launch(dprog.p, nd, dx1.p, n1, px2, n2, diag ? dd.p : nullptr, dv.p, n2, nrhs, dout.p, n1, scratch, s));
  BGP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * n1 * nrhs, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_kmat_gradient_contract(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x, int64_t n,
                               const double* A, double* out) {
  BGP_TRY(require_device());
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  const int np = P.n_params_total, nd = P.ndim;
  if (n < 0) { set_error("negative size"); return BGP_ERR_INVALID; }
  if (np > 64) { set_error("gradient supports at most 64 hyper-parameters"); return BGP_ERR_INVALID; }
  for (int q = 0; q < np; ++q) out[q] = 0.0;
  if (np == 0 || n == 0) return BGP_OK;
  cudaStream_t s = 0;
  DevBuf<DevProgram> dprog;
  DevBuf<double> dx, dA, dg, scratch;
  DevBuf<unsigned> dw;
  BGP_TRY(upload_program(P, dprog, s));
  BGP_TRY(dx.alloc((size_t)n * nd, s));
  BGP_CUDA(cudaMemcpyAsync(dx.p, x, sizeof(double) * n * nd, cudaMemcpyHostToDevice, s));
  BGP_TRY(dA.alloc((size_t)n * n, s));
  BGP_CUDA(cudaMemcpyAsync(dA.p, A, sizeof(double) * n * n, cudaMemcpyHostToDevice, s));
  BGP_TRY(dw.alloc(np, s));
  BGP_CUDA(cudaMemcpyAsync(dw.p, which, sizeof(unsigned) * np, cudaMemcpyHostToDevice, s));
  BGP_TRY(dg.alloc(np, s));
  BGP_TRY(kmat_grad_contract_launch(dprog.p, nd, np, dw.p, dx.p, n, dA.p, n, nullptr, 0.0, 1.0, dg.p, nullptr, scratch, s));
  BGP_CUDA(cudaMemcpyAsync(out, dg.p, sizeof(double) * np, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

}  // extern "C"

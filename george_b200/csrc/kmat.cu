// kmat.cu — K1/K2: fused pairwise-metric + covariance kernel-matrix build (value and hyper-parameter gradient).
//
// Replaces the serial double loops of KernelInterface::value_symmetric / value_general / value_diagonal /
// gradient_symmetric / gradient_general (reference src/george/kernel_interface.cpp:47-125).
//
// Roofline: HBM-write bound, 8 algorithmic bytes per entry (x reads are n*ndim*8 B, negligible).  Coordinates of a tile
// are staged into shared memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier; falls back to plain loads for
// unaligned tails); every thread owns two adjacent output columns so a warp writes 512 contiguous bytes per row
// (st.global.v2.f64).  The symmetric build evaluates only tiles on/above the diagonal and writes the mirrored tile
// through a shared-memory transpose so both stores stay coalesced.
#include <algorithm>
#include <cstdlib>
#include "common.cuh"
#include "kernel_eval.cuh"

namespace bgp {

constexpr int KM_TI = 64;    // tile rows
constexpr int KM_TJ = 128;   // tile cols (general build)
constexpr int KM_THREADS = 256;

struct KmatSmem {
  DevProgram prog;
  uint64_t bar;
};

// out[i*ld + j] = k(x1_i, x2_j)
__global__ void __launch_bounds__(KM_THREADS) kmat_general_kernel(const DevProgram* __restrict__ gprog,
                                                                  const double* __restrict__ x1, int64_t n1,
                                                                  const double* __restrict__ x2, int64_t n2,
                                                                  double* __restrict__ out, int64_t ld) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  KmatSmem* S = reinterpret_cast<KmatSmem*>(smem_raw);
  const int nd = gprog->ndim;
  double* sx1 = reinterpret_cast<double*>(smem_raw + ((sizeof(KmatSmem) + 15) & ~size_t(15)));
  double* sx2 = sx1 + KM_TI * nd + ((KM_TI * nd) & 1);

  stage_program(&S->prog, gprog);
  if (threadIdx.x == 0) { mbar_init(&S->bar, 1); mbar_fence_init(); }
  __syncthreads();
  uint32_t phase = 0;

  const int64_t i0 = (int64_t)blockIdx.y * KM_TI, j0 = (int64_t)blockIdx.x * KM_TJ;
  const int ni = (int)min((int64_t)KM_TI, n1 - i0), nj = (int)min((int64_t)KM_TJ, n2 - j0);
  load_coords(sx1, x1 + i0 * nd, ni * nd, &S->bar, phase);
  load_coords(sx2, x2 + j0 * nd, nj * nd, &S->bar, phase);
  __syncthreads();

  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const int ja = 2 * tx, jb = 2 * tx + 1;
  const bool vec = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) && ((j0 & 1) == 0);
  if (ja < nj) {
    const double* xa = sx2 + ja * nd;
    const double* xb = sx2 + (jb < nj ? jb : ja) * nd;
    for (int i = ty; i < ni; i += KM_THREADS / 64) {
      const double* xi = sx1 + i * nd;
      const double va = kernel_value(S->prog, xi, xa);
      const double vb = (jb < nj) ? kernel_value(S->prog, xi, xb) : 0.0;
      double* o = out + (i0 + i) * ld + j0 + ja;
      if (vec && jb < nj) {
        *reinterpret_cast<double2*>(o) = make_double2(va, vb);
      } else {
        o[0] = va;
        if (jb < nj) o[1] = vb;
      }
    }
  }
}

// symmetric build: out (n x n, leading dimension ld), optional diag_add on the diagonal (basic.py:64-65 fused)
constexpr int KS_T = 64;
__global__ void __launch_bounds__(KM_THREADS) kmat_symmetric_kernel(const DevProgram* __restrict__ gprog,
                                                                    const double* __restrict__ x, int64_t n,
                                                                    const double* __restrict__ diag_add,
                                                                    double* __restrict__ out, int64_t ld) {
  if (blockIdx.x < blockIdx.y) return;  // tiles below the diagonal are produced by the mirror store
  extern __shared__ __align__(16) unsigned char smem_raw[];
  KmatSmem* S = reinterpret_cast<KmatSmem*>(smem_raw);
  const int nd = gprog->ndim;
  double* sxi = reinterpret_cast<double*>(smem_raw + ((sizeof(KmatSmem) + 15) & ~size_t(15)));
  double* sxj = sxi + KS_T * nd + ((KS_T * nd) & 1);
  double* tile = sxj + KS_T * nd + ((KS_T * nd) & 1);  // KS_T x (KS_T+1)

  stage_program(&S->prog, gprog);
  if (threadIdx.x == 0) { mbar_init(&S->bar, 1); mbar_fence_init(); }
  __syncthreads();
  uint32_t phase = 0;

  const int64_t i0 = (int64_t)blockIdx.y * KS_T, j0 = (int64_t)blockIdx.x * KS_T;
  const int ni = (int)min((int64_t)KS_T, n - i0), nj = (int)min((int64_t)KS_T, n - j0);
  const bool on_diag = (blockIdx.x == blockIdx.y);
  load_coords(sxi, x + i0 * nd, ni * nd, &S->bar, phase);
  load_coords(sxj, x + j0 * nd, nj * nd, &S->bar, phase);
  __syncthreads();

  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // one column per thread, 16 rows
  if (on_diag) {
    // evaluate k(x_i, x_j) for j >= i only and mirror, exactly like the reference loop (kernel_interface.cpp:69-75):
    // FMA contraction makes k(a, b) and k(b, a) differ in the last bit for some kernels.
    if (tx < nj) {
      const double* xj = sxj + tx * nd;
      for (int i = ty; i < ni && i <= tx; i += KM_THREADS / 64) {
        double v = kernel_value(S->prog, sxi + i * nd, xj);
        if (i == tx && diag_add) v += diag_add[i0 + i];
        tile[i * (KS_T + 1) + tx] = v;
      }
    }
    __syncthreads();
    if (tx < nj) {
      for (int i = ty; i < ni; i += KM_THREADS / 64)
        out[(i0 + i) * ld + j0 + tx] = (i <= tx) ? tile[i * (KS_T + 1) + tx] : tile[tx * (KS_T + 1) + i];
    }
    return;
  }
  if (tx < nj) {
    const double* xj = sxj + tx * nd;
    for (int i = ty; i < ni; i += KM_THREADS / 64) {
      const double v = kernel_value(S->prog, sxi + i * nd, xj);
      out[(i0 + i) * ld + j0 + tx] = v;
      tile[i * (KS_T + 1) + tx] = v;
    }
  }
  __syncthreads();
  // mirrored tile: out[j0 + c][i0 + r] = tile[r][c], r fastest across threads for coalescing
  if (tx < ni) {
    for (int c = ty; c < nj; c += KM_THREADS / 64) out[(j0 + c) * ld + i0 + tx] = tile[tx * (KS_T + 1) + c];
  }
}

__global__ void kmat_diagonal_kernel(const DevProgram* __restrict__ gprog, const double* __restrict__ x1,
                                     const double* __restrict__ x2, int64_t n, double* __restrict__ out) {
  __shared__ DevProgram P;
  stage_program(&P, gprog);
  __syncthreads();
  const int nd = P.ndim;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = kernel_value(P, x1 + i * nd, x2 + i * nd);
}

// gradient: out[(i*n2 + j)*np + q].  One thread per pair; not on the log-likelihood path.
__global__ void __launch_bounds__(128) kmat_gradient_kernel(const DevProgram* __restrict__ gprog,
                                                            const unsigned* __restrict__ which,
                                                            const double* __restrict__ x1, int64_t n1,
                                                            const double* __restrict__ x2, int64_t n2,
                                                            double* __restrict__ out, int symmetric) {
  __shared__ DevProgram P;
  __shared__ unsigned sw[BGP_MAX_LEAVES * (4 + BGP_MAX_METRIC)];
  stage_program(&P, gprog);
  __syncthreads();
  const int np = P.n_params_total, nd = P.ndim;
  for (int q = threadIdx.x; q < np; q += blockDim.x) sw[q] = which[q];
  __syncthreads();
  const int64_t total = n1 * n2;
  double g[64];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / n2, j = t - i * n2;
    // the reference evaluates (i, j) with i <= j and mirrors (kernel_interface.cpp:116-121)
    const double* a = x1 + ((symmetric && j < i) ? j : i) * nd;
    const double* b = x2 + ((symmetric && j < i) ? i : j) * nd;
    kernel_value_grad(P, a, b, sw, g);
    double* o = out + t * np;
    for (int q = 0; q < np; ++q) o[q] = g[q];
  }
}

// input-coordinate gradient: out[(i*n2 + j)*ndim + q] = d k(x1_i, x2_j) / d x{side}_q  (kernel_interface.cpp:127-157)
__global__ void __launch_bounds__(128) kmat_x_gradient_kernel(const DevProgram* __restrict__ gprog, int side,
                                                              const double* __restrict__ x1, int64_t n1,
                                                              const double* __restrict__ x2, int64_t n2,
                                                              double* __restrict__ out) {
  __shared__ DevProgram P;
  stage_program(&P, gprog);
  __syncthreads();
  const int nd = P.ndim;
  const int64_t total = n1 * n2;
  double g[BGP_MAX_DIM];
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = t / n2, j = t - i * n2;
    kernel_x_gradient(P, side, x1 + i * nd, x2 + j * nd, g);
    double* o = out + t * nd;
    for (int q = 0; q < nd; ++q) o[q] = g[q];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Specialised builds for the commonest programs:  c * f(r2)  with f in {ExpSquared, Matern32, Matern52, Exp} and an
// isotropic or axis-aligned metric over ALL input axes (ndim <= 3, no block mask).  The postfix interpreter costs more
// instruction issue slots than the covariance itself (ncu on the generic kernel, Matern52 3-D: issue slots 83 % busy,
// FP64 pipe 18 %, 1.1 TB/s of stores); here the evaluator is a POD functor passed by value, the loops over axes are
// unrolled and nothing is staged but the coordinates.  Same tile geometry, same i <= j evaluation order on diagonal
// tiles, same arithmetic (metrics.h:76-85 | 108-117, kernels.h radial profiles) as the generic kernels above.
// ---------------------------------------------------------------------------------------------------------------
template <int SHAPE, int ND, bool AXIS>
struct ProfileND {
  double c;
  double m[ND];
  __device__ __forceinline__ double operator()(const double* x1, const double* x2) const {
    double r2 = 0.0;
#pragma unroll
    for (int i = 0; i < ND; ++i) {
      const double d = x1[i] - x2[i];
      if (AXIS) r2 += d * d * m[i];
      else r2 += d * d;
    }
    if (!AXIS) r2 = r2 * m[0];
    double f;
    if (SHAPE == BGP_SHAPE_EXPSQ) f = exp(-0.5 * r2);
    else if (SHAPE == BGP_SHAPE_M32) { const double r = sqrt(3.0 * r2); f = (1.0 + r) * exp(-r); }
    else if (SHAPE == BGP_SHAPE_M52) { const double r = sqrt(5.0 * r2); f = (1 + r + 5.0 * r2 / 3.0) * exp(-r); }
    else f = exp(-sqrt(r2));
    return c * f;
  }
};

template <class Fn, int ND>
__global__ void __launch_bounds__(KM_THREADS) kmat_general_fn_kernel(const Fn fn, const double* __restrict__ x1,
                                                                     int64_t n1, const double* __restrict__ x2,
                                                                     int64_t n2, double* __restrict__ out, int64_t ld) {
  __shared__ __align__(16) double sx1[KM_TI * ND];
  __shared__ __align__(16) double sx2[KM_TJ * ND];
  __shared__ uint64_t bar;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  __syncthreads();
  uint32_t phase = 0;
  const int64_t i0 = (int64_t)blockIdx.y * KM_TI, j0 = (int64_t)blockIdx.x * KM_TJ;
  const int ni = (int)min((int64_t)KM_TI, n1 - i0), nj = (int)min((int64_t)KM_TJ, n2 - j0);
  load_coords(sx1, x1 + i0 * ND, ni * ND, &bar, phase);
  load_coords(sx2, x2 + j0 * ND, nj * ND, &bar, phase);
  __syncthreads();
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const int ja = 2 * tx, jb = 2 * tx + 1;
  const bool vec = ((ld & 1) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15u) == 0) && ((j0 & 1) == 0);
  if (ja < nj) {
    double xa[ND], xb[ND];
#pragma unroll
    for (int q = 0; q < ND; ++q) { xa[q] = sx2[ja * ND + q]; xb[q] = sx2[(jb < nj ? jb : ja) * ND + q]; }
    for (int i = ty; i < ni; i += KM_THREADS / 64) {
      const double* xi = sx1 + i * ND;
      const double va = fn(xi, xa);
      const double vb = (jb < nj) ? fn(xi, xb) : 0.0;
      double* o = out + (i0 + i) * ld + j0 + ja;
      if (vec && jb < nj) {
        *reinterpret_cast<double2*>(o) = make_double2(va, vb);
      } else {
        o[0] = va;
        if (jb < nj) o[1] = vb;
      }
    }
  }
}

template <class Fn, int ND>
__global__ void __launch_bounds__(KM_THREADS) kmat_symmetric_fn_kernel(const Fn fn, const double* __restrict__ x, int64_t n,
                                                                       const double* __restrict__ diag_add,
                                                                       double* __restrict__ out, int64_t ld) {
  if (blockIdx.x < blockIdx.y) return;  // tiles below the diagonal are produced by the mirror store
  __shared__ __align__(16) double sxi[KS_T * ND];
  __shared__ __align__(16) double sxj[KS_T * ND];
  __shared__ double tile[KS_T * (KS_T + 1)];
  __shared__ uint64_t bar;
  if (threadIdx.x == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  __syncthreads();
  uint32_t phase = 0;
  const int64_t i0 = (int64_t)blockIdx.y * KS_T, j0 = (int64_t)blockIdx.x * KS_T;
  const int ni = (int)min((int64_t)KS_T, n - i0), nj = (int)min((int64_t)KS_T, n - j0);
  const bool on_diag = (blockIdx.x == blockIdx.y);
  load_coords(sxi, x + i0 * ND, ni * ND, &bar, phase);
  load_coords(sxj, x + j0 * ND, nj * ND, &bar, phase);
  __syncthreads();
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  double xj[ND];
#pragma unroll
  for (int q = 0; q < ND; ++q) xj[q] = sxj[(tx < nj ? tx : 0) * ND + q];
  if (on_diag) {
    if (tx < nj) {
      for (int i = ty; i < ni && i <= tx; i += KM_THREADS / 64) {
        double v = fn(sxi + i * ND, xj);
        if (i == tx && diag_add) v += diag_add[i0 + i];
        tile[i * (KS_T + 1) + tx] = v;
      }
    }
    __syncthreads();
    if (tx < nj) {
      for (int i = ty; i < ni; i += KM_THREADS / 64)
        out[(i0 + i) * ld + j0 + tx] = (i <= tx) ? tile[i * (KS_T + 1) + tx] : tile[tx * (KS_T + 1) + i];
    }
    return;
  }
  if (tx < nj) {
    for (int i = ty; i < ni; i += KM_THREADS / 64) {
      const double v = fn(sxi + i * ND, xj);
      out[(i0 + i) * ld + j0 + tx] = v;
      tile[i * (KS_T + 1) + tx] = v;
    }
  }
  __syncthreads();
  if (tx < ni) {
    for (int c = ty; c < nj; c += KM_THREADS / 64) out[(j0 + c) * ld + i0 + tx] = tile[tx * (KS_T + 1) + c];
  }
}

// host: does the digested program have the shape  [Constant *] f(metric over all axes) ?
struct FastShape {
  int shape = 0, nd = 0;
  bool axis = false;
  double c = 1.0, m[3] = {1.0, 1.0, 1.0};
};
static bool detect_fast_shape(const DevProgram& P, FastShape* out) {
  if (P.ndim < 1 || P.ndim > 3) return false;
  const DevLeaf* S = nullptr;
  const DevLeaf* C = nullptr;
  if (P.n_nodes == 1 && P.n_leaves == 1 && P.code[0] == 0) S = &P.leaf[0];
  else if (P.n_nodes == 3 && P.n_leaves == 2 && P.code[0] == 0 && P.code[1] == 1 && P.code[2] == -2) {
    if (P.leaf[0].kernel_type == BGP_K_CONSTANT) { C = &P.leaf[0]; S = &P.leaf[1]; }
    else if (P.leaf[1].kernel_type == BGP_K_CONSTANT) { C = &P.leaf[1]; S = &P.leaf[0]; }
    else return false;
  } else return false;
  switch (S->kernel_type) {
    case BGP_K_EXP_SQUARED: out->shape = BGP_SHAPE_EXPSQ; break;
    case BGP_K_MATERN32: out->shape = BGP_SHAPE_M32; break;
    case BGP_K_MATERN52: out->shape = BGP_SHAPE_M52; break;
    case BGP_K_EXP: out->shape = BGP_SHAPE_EXP; break;
    default: return false;
  }
  if (S->blocked || S->naxes != P.ndim) return false;
  for (int i = 0; i < S->naxes; ++i) if (S->axes[i] != i) return false;
  if (S->metric_type == BGP_METRIC_ISOTROPIC) { out->axis = false; out->m[0] = S->mvec[0]; }
  else if (S->metric_type == BGP_METRIC_AXIS_ALIGNED) { out->axis = true; for (int i = 0; i < S->naxes; ++i) out->m[i] = S->mvec[i]; }
  else return false;
  out->nd = P.ndim;
  out->c = 1.0;
  if (C) {  // the constant kernel is summed over its axes (kernels.h:1720-1732): reproduce the additions
    if (C->naxes < 1) return false;
    double v = 0.0;
    for (int a = 0; a < C->naxes; ++a) v += C->rp[0];
    out->c = v;
  }
  return true;
}

template <int SHAPE, int ND, bool AXIS>
static int launch_fast(const FastShape& F, bool symmetric, const double* x1, int64_t n1, const double* x2, int64_t n2,
                       const double* diag_add, double* out, int64_t ld, cudaStream_t s) {
  typedef ProfileND<SHAPE, ND, AXIS> Fn;
  Fn fn;
  fn.c = F.c;
  for (int i = 0; i < ND; ++i) fn.m[i] = F.m[i];
  if (symmetric) {
    const unsigned nt = (unsigned)((n1 + KS_T - 1) / KS_T);
    if (nt > 65535) { set_error("kmat_symmetric: n too large for one launch"); return BGP_ERR_INVALID; }
    kmat_symmetric_fn_kernel<Fn, ND><<<dim3(nt, nt), KM_THREADS, 0, s>>>(fn, x1, n1, diag_add, out, ld);
  } else {
    dim3 grid((unsigned)((n2 + KM_TJ - 1) / KM_TJ), (unsigned)((n1 + KM_TI - 1) / KM_TI));
    if (grid.y > 65535) { set_error("kmat_general: n1 too large for one launch"); return BGP_ERR_INVALID; }
    kmat_general_fn_kernel<Fn, ND><<<grid, KM_THREADS, 0, s>>>(fn, x1, n1, x2, n2, out, ld);
  }
  BGP_LAUNCH_CHECK();
  return BGP_OK;
}
template <int SHAPE, int ND>
static int launch_fast_axis(const FastShape& F, bool symmetric, const double* x1, int64_t n1, const double* x2, int64_t n2,
                            const double* diag_add, double* out, int64_t ld, cudaStream_t s) {
  return F.axis ? launch_fast<SHAPE, ND, true>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s)
                : launch_fast<SHAPE, ND, false>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
}
template <int SHAPE>
static int launch_fast_nd(const FastShape& F, bool symmetric, const double* x1, int64_t n1, const double* x2, int64_t n2,
                          const double* diag_add, double* out, int64_t ld, cudaStream_t s) {
  switch (F.nd) {
    case 1: return launch_fast_axis<SHAPE, 1>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
    case 2: return launch_fast_axis<SHAPE, 2>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
    default: return launch_fast_axis<SHAPE, 3>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
  }
}
// returns -1 when the program has no specialised build (the caller then launches the interpreter kernels)
static int try_launch_fast(const DevProgram& P, bool symmetric, const double* x1, int64_t n1, const double* x2, int64_t n2,
                           const double* diag_add, double* out, int64_t ld, cudaStream_t s) {
  FastShape F;
  if (!detect_fast_shape(P, &F)) return -1;
  switch (F.shape) {
    case BGP_SHAPE_EXPSQ: return launch_fast_nd<BGP_SHAPE_EXPSQ>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
    case BGP_SHAPE_M32: return launch_fast_nd<BGP_SHAPE_M32>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
    case BGP_SHAPE_M52: return launch_fast_nd<BGP_SHAPE_M52>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
    case BGP_SHAPE_EXP: return launch_fast_nd<BGP_SHAPE_EXP>(F, symmetric, x1, n1, x2, n2, diag_add, out, ld, s);
  }
  return -1;
}

static size_t kmat_smem_general(int nd) {
  return ((sizeof(KmatSmem) + 15) & ~size_t(15)) + sizeof(double) * ((size_t)KM_TI * nd + 1 + (size_t)KM_TJ * nd + 1);
}
static size_t kmat_smem_sym(int nd) {
  return ((sizeof(KmatSmem) + 15) & ~size_t(15)) +
         sizeof(double) * (2 * ((size_t)KS_T * nd + 1) + (size_t)KS_T * (KS_T + 1));
}

// ---- device-pointer launchers (used by the solvers) -------------------------------------------------------------
int kmat_general_launch(const DevProgram* dprog, int nd, const double* x1, int64_t n1, const double* x2, int64_t n2,
                        double* out, int64_t ld, cudaStream_t s) {
  if (n1 == 0 || n2 == 0) return BGP_OK;
  const size_t smem = kmat_smem_general(nd);
  // (the attribute is per device / context: set it on every call, it is cheap)
  cudaFuncSetAttribute(kmat_general_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  dim3 grid((unsigned)((n2 + KM_TJ - 1) / KM_TJ), (unsigned)((n1 + KM_TI - 1) / KM_TI));
  if (grid.y > 65535) { set_error("kmat_general: n1 too large for one launch"); return BGP_ERR_INVALID; }
  kmat_general_kernel<<<grid, KM_THREADS, smem, s>>>(dprog, x1, n1, x2, n2, out, ld);
  BGP_LAUNCH_CHECK();
  return BGP_OK;
}

int kmat_symmetric_launch(const DevProgram* dprog, int nd, const double* x, int64_t n, const double* diag_add,
                          double* out, int64_t ld, cudaStream_t s) {
  if (n == 0) return BGP_OK;
  const size_t smem = kmat_smem_sym(nd);
  // (the attribute is per device / context: set it on every call, it is cheap)
  cudaFuncSetAttribute(kmat_symmetric_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  const unsigned nt = (unsigned)((n + KS_T - 1) / KS_T);
  if (nt > 65535) { set_error("kmat_symmetric: n too large for one launch"); return BGP_ERR_INVALID; }
  dim3 grid(nt, nt);
  kmat_symmetric_kernel<<<grid, KM_THREADS, smem, s>>>(dprog, x, n, diag_add, out, ld);
  BGP_LAUNCH_CHECK();
  return BGP_OK;
}

// host program known: specialised build when the program has one, interpreter otherwise
int kmat_symmetric_launch_auto(const DevProgram& P, const DevProgram* dprog, const double* x, int64_t n,
                               const double* diag_add, double* out, int64_t ld, cudaStream_t s) {
  if (n == 0) return BGP_OK;
  const int r = try_launch_fast(P, true, x, n, x, n, diag_add, out, ld, s);
  return r >= 0 ? r : kmat_symmetric_launch(dprog, P.ndim, x, n, diag_add, out, ld, s);
}
int kmat_general_launch_auto(const DevProgram& P, const DevProgram* dprog, const double* x1, int64_t n1, const double* x2,
                             int64_t n2, double* out, int64_t ld, cudaStream_t s) {
  if (n1 == 0 || n2 == 0) return BGP_OK;
  const int r = try_launch_fast(P, false, x1, n1, x2, n2, nullptr, out, ld, s);
  return r >= 0 ? r : kmat_general_launch(dprog, P.ndim, x1, n1, x2, n2, out, ld, s);
}

// upload a digested program to a fresh device buffer
int upload_program(const DevProgram& P, DevBuf<DevProgram>& buf, cudaStream_t s) {
  BGP_TRY(buf.reserve(1, s));
  BGP_CUDA(cudaMemcpyAsync(buf.p, &P, sizeof(DevProgram), cudaMemcpyHostToDevice, s));
  return BGP_OK;
}

}  // namespace bgp

using namespace bgp;

// ---- host-pointer entry points --------------------------------------------------------------------------------
static int kmat_host(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2, int64_t n2,
                     double* out, int mode /*0 general,1 symmetric,2 diagonal*/) {
  BGP_TRY(require_device());
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  if (n1 < 0 || n2 < 0) { set_error("negative size"); return BGP_ERR_INVALID; }
  cudaStream_t s = 0;
  const int nd = P.ndim;
  DevBuf<DevProgram> dprog;
  DevBuf<double> dx1, dx2, dout;
  BGP_TRY(upload_program(P, dprog, s));
  BGP_TRY(dx1.alloc((size_t)n1 * nd, s));
  if (n1) BGP_CUDA(cudaMemcpyAsync(dx1.p, x1, sizeof(double) * n1 * nd, cudaMemcpyHostToDevice, s));
  const double* px2 = dx1.p;
  if (mode != 1) {
    BGP_TRY(dx2.alloc((size_t)n2 * nd, s));
    if (n2) BGP_CUDA(cudaMemcpyAsync(dx2.p, x2, sizeof(double) * n2 * nd, cudaMemcpyHostToDevice, s));
    px2 = dx2.p;
  }
  const size_t nout = mode == 2 ? (size_t)n1 : (size_t)n1 * (size_t)(mode == 1 ? n1 : n2);
  BGP_TRY(dout.alloc(nout, s));
  if (nout == 0) return BGP_OK;
  if (mode == 0) BGP_TRY(kmat_general_launch_auto(P, dprog.p, dx1.p, n1, px2, n2, dout.p, n2, s));
  else if (mode == 1) BGP_TRY(kmat_symmetric_launch_auto(P, dprog.p, dx1.p, n1, nullptr, dout.p, n1, s));
  else {
    const int blocks = (int)std::min<int64_t>((n1 + 255) / 256, 4 * num_sms());
    kmat_diagonal_kernel<<<blocks, 256, 0, s>>>(dprog.p, dx1.p, px2, n1, dout.p);
    BGP_LAUNCH_CHECK();
  }
  BGP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * nout, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

static int kmat_grad_host(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x1, int64_t n1,
                          const double* x2, int64_t n2, double* out, int symmetric) {
  BGP_TRY(require_device());
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  const int np = P.n_params_total, nd = P.ndim;
  if (np > 64) { set_error("gradient supports at most 64 hyper-parameters"); return BGP_ERR_INVALID; }
  if (np == 0 || n1 == 0 || n2 == 0) return BGP_OK;
  cudaStream_t s = 0;
  DevBuf<DevProgram> dprog;
  DevBuf<double> dx1, dx2, dout;
  DevBuf<unsigned> dw;
  BGP_TRY(upload_program(P, dprog, s));
  BGP_TRY(dx1.alloc((size_t)n1 * nd, s));
  BGP_CUDA(cudaMemcpyAsync(dx1.p, x1, sizeof(double) * n1 * nd, cudaMemcpyHostToDevice, s));
  const double* px2 = dx1.p;
  if (!symmetric) {
    BGP_TRY(dx2.alloc((size_t)n2 * nd, s));
    BGP_CUDA(cudaMemcpyAsync(dx2.p, x2, sizeof(double) * n2 * nd, cudaMemcpyHostToDevice, s));
    px2 = dx2.p;
  }
  BGP_TRY(dw.alloc(np, s));
  BGP_CUDA(cudaMemcpyAsync(dw.p, which, sizeof(unsigned) * np, cudaMemcpyHostToDevice, s));
  const size_t nout = (size_t)n1 * n2 * np;
  BGP_TRY(dout.alloc(nout, s));
  const int blocks = (int)std::min<int64_t>((n1 * n2 + 127) / 128, 16 * num_sms());
  kmat_gradient_kernel<<<blocks, 128, 0, s>>>(dprog.p, dw.p, dx1.p, n1, px2, n2, dout.p, symmetric);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * nout, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

static int kmat_xgrad_host(const bgp_kernel_spec_t* spec, int side, const double* x1, int64_t n1, const double* x2,
                           int64_t n2, double* out) {
  BGP_TRY(require_device());
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  const int nd = P.ndim;
  // kernel_x_gradient keeps one ndim-vector per stack level in fixed-size local arrays (BGP_MAX_DIM entries)
  if (nd > BGP_MAX_DIM) { set_error("input-coordinate gradients support at most %d dimensions (got %d)", BGP_MAX_DIM, nd); return BGP_ERR_INVALID; }
  if (n1 < 0 || n2 < 0) { set_error("negative size"); return BGP_ERR_INVALID; }
  if (n1 == 0 || n2 == 0) return BGP_OK;
  cudaStream_t s = 0;
  DevBuf<DevProgram> dprog;
  DevBuf<double> dx1, dx2, dout;
  BGP_TRY(upload_program(P, dprog, s));
  BGP_TRY(dx1.alloc((size_t)n1 * nd, s));
  BGP_CUDA(cudaMemcpyAsync(dx1.p, x1, sizeof(double) * n1 * nd, cudaMemcpyHostToDevice, s));
  BGP_TRY(dx2.alloc((size_t)n2 * nd, s));
  BGP_CUDA(cudaMemcpyAsync(dx2.p, x2, sizeof(double) * n2 * nd, cudaMemcpyHostToDevice, s));
  const size_t nout = (size_t)n1 * n2 * nd;
  BGP_TRY(dout.alloc(nout, s));
  const int blocks = (int)std::min<int64_t>((n1 * n2 + 127) / 128, 16 * num_sms());
  kmat_x_gradient_kernel<<<blocks, 128, 0, s>>>(dprog.p, side, dx1.p, n1, dx2.p, n2, dout.p);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaMemcpyAsync(out, dout.p, sizeof(double) * nout, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

extern "C" {

int bgp_kmat_x1_gradient_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2,
                                 int64_t n2, double* out) {
  return kmat_xgrad_host(spec, 1, x1, n1, x2, n2, out);
}
int bgp_kmat_x2_gradient_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2,
                                 int64_t n2, double* out) {
  return kmat_xgrad_host(spec, 2, x1, n1, x2, n2, out);
}

int bgp_kmat_symmetric(const bgp_kernel_spec_t* spec, const double* x, int64_t n, double* out) {
  return kmat_host(spec, x, n, x, n, out, 1);
}
int bgp_kmat_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2, int64_t n2,
                     double* out) {
  return kmat_host(spec, x1, n1, x2, n2, out, 0);
}
int bgp_kmat_diagonal(const bgp_kernel_spec_t* spec, const double* x1, const double* x2, int64_t n, double* out) {
  return kmat_host(spec, x1, n, x2, n, out, 2);
}
int bgp_kmat_gradient_symmetric(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x, int64_t n,
                                double* out) {
  return kmat_grad_host(spec, which, x, n, x, n, out, 1);
}
int bgp_kmat_gradient_general(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x1, int64_t n1,
                              const double* x2, int64_t n2, double* out) {
  return kmat_grad_host(spec, which, x1, n1, x2, n2, out, 0);
}

}  // extern "C"

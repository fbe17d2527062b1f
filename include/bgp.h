/*
 * bgp.h — C ABI of the B200-native GP covariance engine (libbgp_b200.so).
 *
 * This is the drop-in boundary for ONE path of dfm/george:
 *     gp.compute(x, yerr) + gp.log_likelihood(y) (+ gp.predict on the same factorisation)
 * i.e. kernel-matrix build -> factorisation (dense Cholesky | HODLR) -> log-det -> solve -> quadratic form.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes, returns an int status
 * (0 = BGP_OK) and never lets a C++ exception cross the boundary; the message for the last
 * failing call on the calling thread is available from bgp_last_error().
 *
 * Each function names the reference interface it replaces (paths relative to the dfm/george
 * checkout, commit b5023758).  Host pointers are borrowed for the duration of a call only
 * (the reference copies its inputs as well: src/george/solvers/_hodlr.cpp:71-81,156-164).
 * Pointers are HOST pointers unless the name ends in `_dev`.
 */
#ifndef BGP_B200_H_
#define BGP_B200_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Status codes.  The Python host maps them to the exception types the reference raises
 * (SURVEY.md §8b "Errors"): DIM -> RuntimeError (george::dimension_mismatch, exceptions.h:8-12),
 * NOT_COMPUTED -> RuntimeError (exceptions.h:14-18), INVALID -> ValueError (std::invalid_argument,
 * parser.h:16,33,505), INDEX -> IndexError (_hodlr.cpp:26), LINALG -> numpy.linalg.LinAlgError
 * (what scipy.linalg.cholesky raises, solvers/basic.py:68).
 * ------------------------------------------------------------------------------------------ */
enum {
  BGP_OK = 0,
  BGP_ERR_INVALID = 1,       /* malformed kernel program / argument                              */
  BGP_ERR_DIM = 2,           /* dimension mismatch between x and the kernel                      */
  BGP_ERR_NOT_COMPUTED = 3,  /* solve before compute                                             */
  BGP_ERR_LINALG = 4,        /* matrix not positive definite (dense path only)                   */
  BGP_ERR_CUDA = 5,          /* CUDA runtime failure; no CPU fallback exists                     */
  BGP_ERR_NO_DEVICE = 6,     /* no sm_100 device visible: the library refuses to run             */
  BGP_ERR_RANK_CAPACITY = 7, /* ACA rank exceeded the configured capacity (see bgp_hodlr_opts_t) */
  BGP_ERR_INDEX = 8,
  BGP_ERR_NOMEM = 9
};

const char* bgp_last_error(void);
/* Library/ABI version (major*1000+minor). */
int bgp_version(void);
/* Number of visible CUDA devices with compute capability 10.x; 0 if none (never an error). */
int bgp_device_count(void);
/* Select the CUDA device used by subsequently created handles of the calling thread. */
int bgp_set_device(int device);
/* Count of kernel launches issued by this library since process start (bench.py "gpu_launches"). */
uint64_t bgp_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Kernel program: the POD form of the Python kernel-spec tree that the reference walks with
 * pybind11 attribute reads (src/george/include/george/parser.h:14-509).  Nodes are in POSTFIX
 * order (operands before their operator), so the flattened hyper-parameter vector is the
 * concatenation over leaves in program order — the order Operator::set_parameter uses
 * (kernels.h:56-69) — with, inside a stationary leaf, the kernel's own parameters first and the
 * metric parameters after them (kernels.h:1870-1875, size() at kernels.h:2005).
 * ------------------------------------------------------------------------------------------ */
#define BGP_MAX_DIM 8      /* max axes a kernel leaf may act on                                  */
#define BGP_MAX_METRIC 36  /* BGP_MAX_DIM*(BGP_MAX_DIM+1)/2 packed-Cholesky entries (metrics.h:166-168) */
#define BGP_MAX_NODES 32   /* max nodes (leaves + operators) of one program                       */

enum { BGP_OP_KERNEL = 0, BGP_OP_SUM = 1, BGP_OP_PRODUCT = 2 }; /* kernels.py:234-247 operator_type+1 */

/* kernel_type ids are the reference's (kernels.py: kernel_type attributes; parser.h:40-505). */
enum {
  BGP_K_LINEAR = 0, BGP_K_RATIONAL_QUADRATIC = 1, BGP_K_EXP = 2, BGP_K_LOCAL_GAUSSIAN = 3,
  BGP_K_EMPTY = 4, BGP_K_COSINE = 5, BGP_K_MATERN52 = 6, BGP_K_EXP_SINE2 = 7, BGP_K_CONSTANT = 8,
  BGP_K_EXP_SQUARED = 9, BGP_K_MATERN32 = 10, BGP_K_POLYNOMIAL = 11, BGP_K_DOT_PRODUCT = 12,
  /* user kernels compiled in from kernels/*.yml by tools/generate_kernels.py (the reference's generate_kernels.py:10-42
   * / docs/tutorials/new-kernel.rst): entry i of the sorted file list has id BGP_K_USER0 + i */
  BGP_K_USER0 = 13
};
enum { BGP_METRIC_NONE = -1, BGP_METRIC_ISOTROPIC = 0, BGP_METRIC_AXIS_ALIGNED = 1, BGP_METRIC_GENERAL = 2 };

typedef struct bgp_kernel_node {
  int32_t op;           /* BGP_OP_*                                                              */
  int32_t kernel_type;  /* BGP_K_* (leaf only)                                                   */
  int32_t metric_type;  /* BGP_METRIC_* ; NONE for the non-stationary kernels                    */
  int32_t ndim;         /* dimension of the input space                                          */
  int32_t naxes;        /* number of axes the leaf acts on (subspace.h:10-25)                    */
  int32_t blocked;      /* stationary kernels: block mask active (kernels.h:1897-1905)           */
  int32_t n_params;     /* number of the kernel's own hyper-parameters (excl. metric)            */
  int32_t n_metric;     /* number of metric parameters (1 | naxes | naxes(naxes+1)/2)            */
  int32_t axes[BGP_MAX_DIM];
  /* raw Python-side values, exactly what parser.h passes to the constructors:
   *   Linear: {log_gamma2, order}   RationalQuadratic: {log_alpha}   LocalGaussian: {location, log_width}
   *   Cosine: {log_period}   ExpSine2: {gamma, log_period}   Constant: {log_constant}
   *   Polynomial: {log_sigma2, order}   (order is a constant, not a hyper-parameter)                  */
  double params[4];
  double metric[BGP_MAX_METRIC];    /* metric.get_parameter_vector(include_frozen=True) (parser.h:111-116) */
  double min_block[BGP_MAX_DIM];
  double max_block[BGP_MAX_DIM];
} bgp_kernel_node_t;

typedef struct bgp_kernel_spec {
  int32_t n_nodes;
  int32_t ndim;
  bgp_kernel_node_t nodes[BGP_MAX_NODES];
} bgp_kernel_spec_t;

/* Validate a program (stack discipline, ids, dimensions).  Replaces the checks in parser.h:16-37,505. */
int bgp_spec_validate(const bgp_kernel_spec_t* spec);
/* Total number of hyper-parameters = Kernel::size() (kernels.h:56, 2005). */
int bgp_spec_num_params(const bgp_kernel_spec_t* spec, int* n_params);

/* ------------------------------------------------------------------------------------------
 * Kernel-matrix build.  Replaces KernelInterface::value_symmetric / value_general / value_diagonal
 * (src/george/kernel_interface.cpp:62-77, 47-60, 79-90) and gradient_symmetric / gradient_general
 * (kernel_interface.cpp:109-125, 92-107).  x1: (n1, ndim) row-major f64; out row-major f64.
 * `which` (n_params uint32) selects the hyper-parameters to differentiate; unselected slices are 0.
 * ------------------------------------------------------------------------------------------ */
int bgp_kmat_symmetric(const bgp_kernel_spec_t* spec, const double* x, int64_t n, double* out /* n*n */);
int bgp_kmat_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2, int64_t n2,
                     double* out /* n1*n2 */);
int bgp_kmat_diagonal(const bgp_kernel_spec_t* spec, const double* x1, const double* x2, int64_t n,
                      double* out /* n */);
int bgp_kmat_gradient_symmetric(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x, int64_t n,
                                double* out /* n*n*n_params */);
int bgp_kmat_gradient_general(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x1, int64_t n1,
                              const double* x2, int64_t n2, double* out /* n1*n2*n_params */);
/* d k(x1_i, x2_j) / d x1_i  and  / d x2_j  — kernel_interface.cpp:127-141 (x1_gradient_general) and 143-157
 * (x2_gradient_general).  out[(i*n2 + j)*ndim + q]. */
int bgp_kmat_x1_gradient_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2,
                                 int64_t n2, double* out /* n1*n2*ndim */);
int bgp_kmat_x2_gradient_general(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2,
                                 int64_t n2, double* out /* n1*n2*ndim */);

/* ------------------------------------------------------------------------------------------
 * Matrix-free consumers of the covariance function (csrc/kmat_ops.cu): the kernel matrix is never formed.
 *
 * bgp_kmat_matvec: out (n1 x nrhs, column-major, ld n1) = K(x1, x2) v (n2 x nrhs, column-major, ld n2) [+ diag .* v].
 *   Replaces `np.dot(kernel.get_value(xs, x), alpha)` of GP.predict (src/george/gp.py:524-528, i.e.
 *   KernelInterface::value_general kernel_interface.cpp:47-60 followed by a host GEMV) without the (n1, n2) matrix;
 *   with x1 == x2 and diag = yerr^2 it applies the GP covariance itself (K (K^-1 y) == y round-trip checks at sizes
 *   where K cannot be stored).  `diag` may be NULL; it requires n1 == n2.
 * bgp_kmat_gradient_contract: out[p] = sum_ij A_ij dK_ij/dtheta_p for the symmetric gradient
 *   (kernel_interface.cpp:109-125) and a host matrix A (n, n) row-major: the `einsum("ijk,ij", dK, A)` of
 *   GP.grad_log_likelihood (gp.py:465-466) without the (n, n, P) tensor.  Unselected parameters (which[p] == 0) give 0.
 * ------------------------------------------------------------------------------------------ */
int bgp_kmat_matvec(const bgp_kernel_spec_t* spec, const double* x1, int64_t n1, const double* x2, int64_t n2,
                    const double* diag, const double* v, int64_t nrhs, double* out);
int bgp_kmat_gradient_contract(const bgp_kernel_spec_t* spec, const uint32_t* which, const double* x, int64_t n,
                               const double* A, double* out /* n_params */);

/* ------------------------------------------------------------------------------------------
 * Dense solver.  Replaces BasicSolver (src/george/solvers/basic.py:51-121): kernel matrix +
 * yerr^2 on the diagonal, Cholesky, log-det = 2 sum log diag, cho_solve, r @ U, dense inverse.
 * ------------------------------------------------------------------------------------------ */
typedef struct bgp_dense bgp_dense_t;
int bgp_dense_create(bgp_dense_t** out);
void bgp_dense_destroy(bgp_dense_t* h);
/* basic.py:51-70.  yerr is the standard deviation; yerr^2 is added on the diagonal. */
int bgp_dense_compute(bgp_dense_t* h, const bgp_kernel_spec_t* spec, const double* x, int64_t n, int32_t ndim,
                      const double* yerr);
int bgp_dense_log_determinant(const bgp_dense_t* h, double* out);
/* basic.py:72-87.  b: (n, nrhs) column-major with leading dimension ldb (a plain vector has nrhs=1); in place. */
int bgp_dense_apply_inverse(bgp_dense_t* h, double* b, int64_t nrhs, int64_t ldb);
/* basic.py:89-102 */
int bgp_dense_dot_solve(bgp_dense_t* h, const double* y, double* out);
/* basic.py:104-114: out = r @ U with r (nr, n) row-major, out (nr, n) row-major, U the upper factor. */
int bgp_dense_apply_sqrt(bgp_dense_t* h, const double* r, int64_t nr, double* out);
/* basic.py:116-121: out (n, n); symmetric so the order does not matter. */
int bgp_dense_get_inverse(bgp_dense_t* h, double* out);
/* Pickle support (the reference pickles its numpy factor, tests/test_pickle.py:21-36): copy the lower Cholesky
 * factor out (n*n, column-major, strictly-upper part zeroed) and load it back into a fresh handle. */
int bgp_dense_export_factor(bgp_dense_t* h, double* out);
int bgp_dense_import_factor(bgp_dense_t* h, const double* factor, int64_t n, double log_det);
/* Everything GP.grad_log_likelihood (gp.py:406-468) needs from the solver, computed on the device from the stored
 * factor, kernel and coordinates: alpha = K^-1 r (n), g[p] = sum_ij (alpha alpha^T - K^-1)_ij dK_ij/dtheta_p (n_params;
 * the caller multiplies by 0.5 and selects the unfrozen entries) and diag(alpha alpha^T - K^-1) (n, for the white-noise
 * term gp.py:452-456).  Replaces solver.get_inverse() (basic.py:116-121) + kernel.get_gradient (N x N x P on the host)
 * + einsum.  Any output pointer may be NULL.  Returns BGP_ERR_NOT_COMPUTED on a handle restored by
 * bgp_dense_import_factor (it holds no kernel / coordinates). */
int bgp_dense_grad_terms(bgp_dense_t* h, const uint32_t* which, const double* r, double* alpha_out, double* g_out,
                         double* diag_out);
/* timing of the last compute: [0]=kernel-matrix build ms, [1]=potrf ms (device events). */
int bgp_dense_last_timing(const bgp_dense_t* h, double* ms2);

/* ------------------------------------------------------------------------------------------
 * HODLR solver.  Replaces _hodlr.HODLRSolver (src/george/solvers/_hodlr.cpp:115-204) and the
 * hodlr::Node tree behind it (src/george/include/george/hodlr.h:13-256).
 * ------------------------------------------------------------------------------------------ */
typedef struct bgp_hodlr bgp_hodlr_t;

enum {
  BGP_RNG_PER_NODE = 0, /* each tree node draws from its own mt19937 stream (level-parallel build)     */
  BGP_RNG_REFERENCE = 1 /* one mt19937 threaded through the pre-order recursion, as hodlr.h:35,58-61   */
};

typedef struct bgp_hodlr_opts {
  int32_t min_size;      /* default 100 (_hodlr.cpp:202)                                         */
  int32_t seed;          /* default 42                                                            */
  double  tol;           /* default 0.1                                                           */
  int32_t rng_mode;      /* BGP_RNG_*                                                             */
  int32_t rank_capacity; /* max columns kept per low-rank factor; 0 = automatic                   */
  /* multi-GPU sharding by top-level sub-tree (SURVEY.md §8e): this process owns sub-tree
   * `shard_rank` of `shard_count` (a power of two; 1 = whole tree).                             */
  int32_t shard_rank;
  int32_t shard_count;
  /* What to do when the ACA runs out of candidate rows (every remaining row's residual is < 1e-14):
   *   BGP_EXHAUST_DENSE   (0, default) return the dense factorisation, rank = min(rows, cols), as hodlr.h:161-176 does;
   *   BGP_EXHAUST_LOWRANK (1) keep the low-rank factors found so far: at that point EVERY row has been tested, so the
   *                        approximation is verified to 1e-14 per entry and differs from the dense answer by rounding.
   * Kernels that are exactly low rank on sorted 1-D inputs (Matern-3/2, Cosine, ...) hit this on most small nodes. */
  int32_t exhaust_mode;
} bgp_hodlr_opts_t;
enum { BGP_EXHAUST_DENSE = 0, BGP_EXHAUST_LOWRANK = 1 };

/* The reference's defaults (solvers/hodlr.py:43, _hodlr.cpp:202): min_size 100, tol 0.1, seed 42 — and, because at that
 * tolerance the result depends on the pivot order, rng_mode = BGP_RNG_REFERENCE and exhaust_mode = BGP_EXHAUST_DENSE: a
 * caller that changes nothing gets the reference's algorithm.  The level-parallel BGP_RNG_PER_NODE is the mode to choose
 * for tight tolerances (the Python plug-in does so automatically for tol <= 1e-6) and the only one that shards. */
void bgp_hodlr_default_opts(bgp_hodlr_opts_t* o);
int bgp_hodlr_create(bgp_hodlr_t** out);
void bgp_hodlr_destroy(bgp_hodlr_t* h);
/* _hodlr.cpp:55-94 (Solver::compute): snapshot kernel + x, diag = yerr^2, build and factor the tree. */
int bgp_hodlr_compute(bgp_hodlr_t* h, const bgp_kernel_spec_t* spec, const double* x, int64_t n, int32_t ndim,
                      const double* yerr, const bgp_hodlr_opts_t* opts);
/* same with x / yerr already resident on the device (bench "value" leg; inputs in HBM). */
int bgp_hodlr_compute_dev(bgp_hodlr_t* h, const bgp_kernel_spec_t* spec, const double* x_dev, int64_t n,
                          int32_t ndim, const double* yerr_dev, const bgp_hodlr_opts_t* opts);
int bgp_hodlr_computed(const bgp_hodlr_t* h);               /* _hodlr.cpp:123 */
int bgp_hodlr_log_determinant(const bgp_hodlr_t* h, double* out); /* _hodlr.cpp:124 */
/* _hodlr.cpp:156-164: b (n, nrhs) column-major, leading dimension ldb, solved in place. */
int bgp_hodlr_apply_inverse(bgp_hodlr_t* h, double* b, int64_t nrhs, int64_t ldb);
/* _hodlr.cpp:178-182 */
int bgp_hodlr_dot_solve(bgp_hodlr_t* h, const double* y, double* out);
int bgp_hodlr_dot_solve_dev(bgp_hodlr_t* h, const double* y_dev, double* out);
/* _hodlr.cpp:193-199: dense inverse (n, n). */
int bgp_hodlr_get_inverse(bgp_hodlr_t* h, double* out);

/* The HODLR counterpart of bgp_dense_grad_terms (K^-1 by solving against the identity on the device, as
 * _hodlr.cpp:193-199 does on the host).  Not available on a sharded factorisation. */
int bgp_hodlr_grad_terms(bgp_hodlr_t* h, const uint32_t* which, const double* r, double* alpha_out, double* g_out,
                         double* diag_out);

/* Tree / index structure introspection (bit-exact parity target; hodlr.h:48-61).
 * Nodes are listed in the reference's PRE-ORDER construction order. */
typedef struct bgp_hodlr_node_info {
  int32_t start, size, half; /* half = size/2 (hodlr.h:48); children are [start,half) and [start+half,size-half) */
  int32_t is_leaf;
  int32_t parent;            /* pre-order index of the parent, -1 for the root                     */
  int32_t direction;         /* 0 = left child, 1 = right child (hodlr.h:58-61)                    */
  int32_t depth;
  int32_t rank;              /* ACA rank of the node's off-diagonal block (0 for leaves)           */
  int32_t rng_draws;         /* number of mt19937 words the node's ACA consumed                    */
  int32_t dense_fallback;    /* 1 if the rows ran out and the dense factorisation was returned (hodlr.h:161-176) */
} bgp_hodlr_node_info_t;
int bgp_hodlr_num_nodes(const bgp_hodlr_t* h, int64_t* out);
int bgp_hodlr_node_info(const bgp_hodlr_t* h, bgp_hodlr_node_info_t* out /* num_nodes */);
/* ACA pivots of node `node` (pre-order index): rows[k], cols[k] for k < rank, block-relative. */
int bgp_hodlr_node_pivots(const bgp_hodlr_t* h, int64_t node, int32_t* rows, int32_t* cols);
/* Device-event timings of the last compute, ms: [0] leaves (build+factor; stream A, CONCURRENT with [1]),
 * [1] ACA (stream B, from the start of compute), [2] up-sweep (panel finalisation + leaf solves + level sweeps, from the
 * moment both streams have drained), [3] total compute, [4] last solve.  [3] ~ max([0], [1]) + host gap + [2]. */
int bgp_hodlr_last_timing(const bgp_hodlr_t* h, double* ms5);
/* Algorithmic work of the last compute (SURVEY.md §8d): [0] kernel evaluations, [1] bytes, [2] flops,
 * [3] sum of per-level max ranks R, [4] leaf size m, [5] number of levels. */
int bgp_hodlr_last_work(const bgp_hodlr_t* h, double* w6);
/* Optional per-kernel timing of the lock-step ACA loop: with profiling on, every launch is bracketed by CUDA events on
 * its stream.  p12 = [0] summed a2_eval launch time ms, [1] launches of each kernel (= lock-step iterations),
 * [2] candidate-row entries verified against the 1e-14 pivot threshold (hodlr.h:191), [3] residual-update FMAs,
 * [4] candidate rows examined, [5] entries of [2] that were actually evaluated (the others were bounded below the
 * threshold from the kernel's decay and the factor magnitudes, without evaluation; decisions are identical),
 * [6..11] summed launch times ms of a2_eval, a2_decide, a2_vrow, a2_pivot, a2_vnorm_ucol, a2_finish. */
int bgp_hodlr_set_profiling(bgp_hodlr_t* h, int on);
int bgp_hodlr_last_aca_profile(const bgp_hodlr_t* h, double* p12);

/* Diagnostics: the dense building blocks of the big-rank Woodbury step (csrc/hodlr_lu.cuh, csrc/gemm_dmma.cuh),
 * callable on their own with HOST pointers so the tests can check them against LAPACK.
 *   bgp_selftest_lu: S (n x n, column-major) is LU-factored with partial pivoting in blocks of 32, R (n x nrhs,
 *     column-major, ld n) is overwritten by S^-1 R, *logdet = log|det S|      (stands in for Eigen::FullPivLU,
 *     hodlr.h:228-234, :90-93, :250).
 *   bgp_selftest_gemm: C (m x n, column-major ldc) -= A' B' (or += with atomics); A' (m,k) = a_kcontig ? A[m*lda+k]
 *     : A[k*lda+m]; B' (k,n) = B[n*ldb+k] (b_kcontig must be 1). */
int bgp_selftest_lu(int32_t n, int32_t nrhs, const double* S_host, double* R_host, double* logdet);
int bgp_selftest_gemm(int32_t a_kcontig, int32_t b_kcontig, int32_t m, int32_t n, int32_t k, const double* A_host,
                      int64_t lda, const double* B_host, int64_t ldb, double* C_host, int64_t ldc, int32_t atomic_add);

/* Multi-GPU (SURVEY.md §8e).  A factorisation with opts.shard_count > 1 is COLLECTIVE: it needs the library's
 * communicator (bgp_comm_init) with world == opts.shard_count and rank == opts.shard_rank, and bgp_hodlr_compute[_dev]
 * fails with BGP_ERR_INVALID without one.  Each rank factors its local sub-tree, the ranks all-gather the rows each owns
 * of the top-level factor panel (pack kernel -> ncclAllGather -> unpack kernels on the solver's stream), every rank
 * finishes the nodes above the cut, and the log-det is all-reduced.  apply_inverse / dot_solve on such a handle are
 * collective too (replicated right-hand side, one all-gather of the locally solved slices).
 * The communicator is one per process.  Rank 0 makes a unique id (128 bytes), the host broadcasts it over whatever it
 * has (torch.distributed, MPI, a file), every rank calls bgp_comm_init.  `nccl_path` may be NULL: the library already
 * loaded in the process (torch's libnccl.so.2) is used, else libnccl.so.2 is dlopen'ed. */
int bgp_comm_unique_id(void* out128, const char* nccl_path);
int bgp_comm_init(const void* id128, int rank, int world, const char* nccl_path);
int bgp_comm_destroy(void);

/* ------------------------------------------------------------------------------------------
 * Device memory helpers so a host without torch can stage inputs (bench "value" leg).
 * ------------------------------------------------------------------------------------------ */
int bgp_dev_alloc(void** ptr_dev, size_t bytes);
int bgp_dev_free(void* ptr_dev);
int bgp_dev_upload(void* dst_dev, const void* src_host, size_t bytes);
int bgp_host_alloc_pinned(void** ptr, size_t bytes);
int bgp_host_free_pinned(void* ptr);

#ifdef __cplusplus
}
#endif
#endif /* BGP_B200_H_ */

// core.cu — library-wide host plumbing: error strings, device checks, stream-ordered memory, the host-side
// digestion of a kernel program (replacement for parse_kernel_spec, reference parser.h:14-509), and the small
// utility entry points of include/bgp.h.
#include <cmath>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "kernel_eval.cuh"

namespace bgp {

static thread_local char t_error[1024] = {0};
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_error, sizeof(t_error), fmt, ap);
  va_end(ap);
}

static int g_sm_count[64] = {0};

int require_device() {
  int dev = -1;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("no CUDA device available (%s): libbgp_b200 has no CPU fallback", cudaGetErrorString(e));
    return BGP_ERR_NO_DEVICE;
  }
  if (dev >= 0 && dev < 64 && g_sm_count[dev] > 0) return BGP_OK;
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaGetDeviceProperties failed: %s", cudaGetErrorString(e));
    return BGP_ERR_NO_DEVICE;
  }
  if (prop.major != 10) {
    set_error("device %d (%s, sm_%d%d) is not a Blackwell sm_100 GPU; this library ships sm_100a code only", dev,
              prop.name, prop.major, prop.minor);
    return BGP_ERR_NO_DEVICE;
  }
  // keep freed blocks cached in the default pool: compute() is called over and over with the same sizes
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  if (dev < 64) g_sm_count[dev] = prop.multiProcessorCount;
  return BGP_OK;
}

int num_sms() {
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && g_sm_count[dev] > 0) return g_sm_count[dev];
  return 148;
}

int dev_alloc(void** p, size_t bytes, cudaStream_t s) {
  *p = nullptr;
  if (bytes == 0) return BGP_OK;
  cudaError_t e = cudaMallocAsync(p, bytes, s);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? BGP_ERR_NOMEM : BGP_ERR_CUDA;
  }
  return BGP_OK;
}

void dev_free(void* p, cudaStream_t s) {
  if (p) cudaFreeAsync(p, s);
}

static inline bool is_user(int kt) { return kt >= BGP_K_USER0 && kt < BGP_K_USER0 + BGP_N_USER_KERNELS; }
static inline bool is_stationary(int kt) {
  if (is_user(kt)) return user::kInfo[kt - BGP_K_USER0].stationary != 0;
  return kt == BGP_K_RATIONAL_QUADRATIC || kt == BGP_K_EXP || kt == BGP_K_MATERN52 || kt == BGP_K_EXP_SQUARED ||
         kt == BGP_K_MATERN32;
}
static inline int own_params(int kt) {
  if (is_user(kt)) return user::kInfo[kt - BGP_K_USER0].n_params;
  switch (kt) {
    case BGP_K_LINEAR: case BGP_K_RATIONAL_QUADRATIC: case BGP_K_COSINE: case BGP_K_CONSTANT: case BGP_K_POLYNOMIAL: return 1;
    case BGP_K_LOCAL_GAUSSIAN: case BGP_K_EXP_SINE2: return 2;
    default: return 0;
  }
}
static inline bool general_diag_host(int i) {
  for (int j = 0, d = 2; j <= i; j += d, ++d)
    if (i == j) return true;
  return false;
}

int build_dev_program(const bgp_kernel_spec_t* s, DevProgram* P) {
  if (!s) { set_error("invalid kernel: null program"); return BGP_ERR_INVALID; }
  if (s->n_nodes <= 0 || s->n_nodes > BGP_MAX_NODES) { set_error("invalid kernel: %d nodes", s->n_nodes); return BGP_ERR_INVALID; }
  if (s->ndim <= 0) { set_error("invalid kernel: ndim = %d", s->ndim); return BGP_ERR_INVALID; }
  memset(P, 0, sizeof(*P));
  P->n_nodes = s->n_nodes;
  P->ndim = s->ndim;
  int depth = 0, max_depth = 0, nl = 0, off = 0;
  for (int n = 0; n < s->n_nodes; ++n) {
    const bgp_kernel_node_t& k = s->nodes[n];
    if (k.op == BGP_OP_SUM || k.op == BGP_OP_PRODUCT) {
      if (depth < 2) { set_error("invalid kernel: operator %d has fewer than two operands", n); return BGP_ERR_INVALID; }
      depth -= 1;
      P->code[n] = (k.op == BGP_OP_SUM) ? -1 : -2;
      continue;
    }
    if (k.op != BGP_OP_KERNEL) { set_error("unrecognized operator"); return BGP_ERR_INVALID; }
    if (k.kernel_type < 0 || (k.kernel_type > BGP_K_DOT_PRODUCT && !is_user(k.kernel_type))) {
      set_error("unrecognized kernel type %d (%d user kernel(s) compiled in: tools/generate_kernels.py)", k.kernel_type, BGP_N_USER_KERNELS);
      return BGP_ERR_INVALID;
    }
    if (nl >= BGP_MAX_LEAVES) { set_error("invalid kernel: more than %d leaves", BGP_MAX_LEAVES); return BGP_ERR_INVALID; }
    if (k.ndim != s->ndim) { set_error("dimension mismatch between kernel leaves (%d vs %d)", k.ndim, s->ndim); return BGP_ERR_DIM; }
    if (k.naxes < 0 || k.naxes > BGP_MAX_DIM) { set_error("invalid kernel: naxes = %d", k.naxes); return BGP_ERR_INVALID; }
    DevLeaf& L = P->leaf[nl];
    L.kernel_type = k.kernel_type;
    L.naxes = k.naxes;
    L.blocked = k.blocked;
    L.n_params = own_params(k.kernel_type);
    L.param_off = off;
    for (int i = 0; i < k.naxes; ++i) {
      if (k.axes[i] < 0 || k.axes[i] >= s->ndim) { set_error("invalid axis %d for %d dimensional input", k.axes[i], s->ndim); return BGP_ERR_INVALID; }
      L.axes[i] = k.axes[i];
      L.mn[i] = k.min_block[i];
      L.mx[i] = k.max_block[i];
    }
    for (int i = 0; i < 4; ++i) L.p[i] = k.params[i];
    switch (k.kernel_type) {  // update_reparams() of each generated class (kernels/*.yml "reparams")
      case BGP_K_LINEAR: L.rp[0] = exp(-L.p[0]); break;
      case BGP_K_RATIONAL_QUADRATIC: L.rp[0] = exp(L.p[0]); break;
      case BGP_K_LOCAL_GAUSSIAN: L.rp[0] = 0.5 * exp(-L.p[1]); break;
      case BGP_K_COSINE: L.rp[0] = 2 * 3.141592653589793238462643383279502884 * exp(-L.p[0]); break;
      case BGP_K_EXP_SINE2: L.rp[0] = 3.141592653589793238462643383279502884 * exp(-L.p[1]); break;
      case BGP_K_CONSTANT: L.rp[0] = exp(L.p[0]); break;
      case BGP_K_POLYNOMIAL: L.rp[0] = exp(L.p[0]); break;
      default: if (is_user(k.kernel_type)) user::reparams(k.kernel_type - BGP_K_USER0, L.p, L.rp); break;
    }
    if (is_stationary(k.kernel_type)) {
      if (k.metric_type < 0 || k.metric_type > 2) { set_error("unrecognized metric"); return BGP_ERR_INVALID; }
      const int expect = k.metric_type == 0 ? 1 : (k.metric_type == 1 ? k.naxes : k.naxes * (k.naxes + 1) / 2);
      if (k.n_metric != expect) { set_error("metric has %d parameters, expected %d", k.n_metric, expect); return BGP_ERR_INVALID; }
      L.metric_type = k.metric_type;
      L.n_metric = k.n_metric;
      for (int i = 0; i < k.n_metric; ++i) {
        if (k.metric_type == BGP_METRIC_GENERAL) L.mvec[i] = general_diag_host(i) ? exp(-k.metric[i]) : k.metric[i];
        else L.mvec[i] = exp(-k.metric[i]);  // metrics.h:46-49
      }
    } else {
      L.metric_type = BGP_METRIC_NONE;
      L.n_metric = 0;
    }
    off += L.n_params + L.n_metric;
    P->code[n] = (signed char)nl;
    nl++;
    depth++;
    if (depth > max_depth) max_depth = depth;
  }
  if (depth != 1) { set_error("invalid kernel: program leaves %d values on the stack", depth); return BGP_ERR_INVALID; }
  if (max_depth > BGP_STACK) { set_error("kernel expression too deep for the device interpreter (%d > %d)", max_depth, BGP_STACK); return BGP_ERR_INVALID; }
  P->n_leaves = nl;
  P->n_params_total = off;
  // fast 1-D path: every leaf is a function of d = x1 - x2 alone
  bool fast = (s->ndim == 1);
  for (int i = 0; i < nl && fast; ++i) {
    const DevLeaf& L = P->leaf[i];
    const int kt = L.kernel_type;
    if (L.naxes != 1 || L.axes[0] != 0 || is_user(kt)) fast = false;  // (user kernels run on the general interpreter path)
    else if (is_stationary(kt)) fast = (L.metric_type != BGP_METRIC_GENERAL) && !L.blocked;
    else fast = (kt == BGP_K_EXP_SINE2 || kt == BGP_K_COSINE || kt == BGP_K_CONSTANT);
  }
  P->flags = fast ? 1 : 0;
  // program shape.  One-term: [S] or [Constant, S, *] / [S, Constant, *] with S in {ExpSquared, Matern32, Matern52, Exp}.
  // Two-term (1-D quasi-periodic models), T = S | Constant S * | S Constant *  and  E = ExpSine2 | Constant E * | ...:
  //   T E +  (either order)          ->  c*S + c2*E
  //   T ExpSine2 *                   ->  (c*S) * E      (the association `c * S * E` produces; other groupings round
  //                                                      differently and stay on the interpreter)
  P->shape = BGP_SHAPE_GENERIC; P->sc = 1.0; P->sm = 1.0; P->sc2 = 1.0; P->sg = 0.0; P->sw = 0.0;
  if (fast) {
    auto shape_of = [](int kt) {
      switch (kt) {
        case BGP_K_EXP_SQUARED: return (int)BGP_SHAPE_EXPSQ;
        case BGP_K_MATERN32: return (int)BGP_SHAPE_M32;
        case BGP_K_MATERN52: return (int)BGP_SHAPE_M52;
        case BGP_K_EXP: return (int)BGP_SHAPE_EXP;
        default: return 0;
      }
    };
    // a "scaled leaf" starting at code position pos: returns the number of code entries it spans (0 = no match)
    struct Term { int leaf = -1; double c = 1.0; };
    auto parse_term = [&](int pos, Term* t) -> int {
      if (pos >= P->n_nodes || P->code[pos] < 0) return 0;
      const int l0 = P->code[pos];
      if (pos + 2 < P->n_nodes && P->code[pos + 1] >= 0 && P->code[pos + 2] == -2) {
        const int l1 = P->code[pos + 1];
        const bool c0 = P->leaf[l0].kernel_type == BGP_K_CONSTANT, c1 = P->leaf[l1].kernel_type == BGP_K_CONSTANT;
        if (c0 && !c1) { t->leaf = l1; t->c = P->leaf[l0].rp[0]; return 3; }
        if (c1 && !c0) { t->leaf = l0; t->c = P->leaf[l1].rp[0]; return 3; }
      }
      if (P->leaf[l0].kernel_type == BGP_K_CONSTANT) return 0;
      t->leaf = l0; t->c = 1.0;
      return 1;
    };
    Term t0, t1;
    const int n0 = parse_term(0, &t0);
    if (n0 && n0 == P->n_nodes && shape_of(P->leaf[t0.leaf].kernel_type)) {
      P->shape = shape_of(P->leaf[t0.leaf].kernel_type); P->sc = t0.c; P->sm = P->leaf[t0.leaf].mvec[0];
    } else if (n0) {
      const int n1 = parse_term(n0, &t1);
      const bool closes = n1 && n0 + n1 + 1 == P->n_nodes;
      if (closes) {
        const int op = P->code[n0 + n1];
        const DevLeaf& a = P->leaf[t0.leaf];
        const DevLeaf& b = P->leaf[t1.leaf];
        const int sa = shape_of(a.kernel_type), sb = shape_of(b.kernel_type);
        const bool ea = a.kernel_type == BGP_K_EXP_SINE2, eb = b.kernel_type == BGP_K_EXP_SINE2;
        auto two = [&](const Term& ts, const DevLeaf& S, int sshape, const Term& te, const DevLeaf& E, bool sum) {
          if (sshape != BGP_SHAPE_EXPSQ && sshape != BGP_SHAPE_M32) return;
          P->shape = sum ? (sshape == BGP_SHAPE_EXPSQ ? BGP_SHAPE_SUM_EXPSQ_ES2 : BGP_SHAPE_SUM_M32_ES2)
                         : (sshape == BGP_SHAPE_EXPSQ ? BGP_SHAPE_PROD_EXPSQ_ES2 : BGP_SHAPE_PROD_M32_ES2);
          P->sc = ts.c; P->sm = S.mvec[0]; P->sc2 = te.c; P->sg = E.p[0]; P->sw = E.rp[0];
        };
        if (op == -1) {  // sum: commutative, either order
          if (sa && eb) two(t0, a, sa, t1, b, true);
          else if (ea && sb) two(t1, b, sb, t0, a, true);
        } else if (op == -2 && n1 == 1) {  // (c*S) * E  or  (c*E) * S is NOT the same rounding: only the first form
          if (sa && eb) two(t0, a, sa, t1, b, false);
        }
      }
    }
  }
  return BGP_OK;
}

}  // namespace bgp

using namespace bgp;

extern "C" {

const char* bgp_last_error(void) { return t_error; }
int bgp_version(void) { return 1000; }

int bgp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  int ok = 0;
  for (int d = 0; d < n; ++d) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
  }
  return ok;
}

int bgp_set_device(int device) {
  BGP_CUDA(cudaSetDevice(device));
  return require_device();
}

uint64_t bgp_launch_count(void) { return g_launches.load(); }

int bgp_spec_validate(const bgp_kernel_spec_t* spec) {
  DevProgram P;
  return build_dev_program(spec, &P);
}

int bgp_spec_num_params(const bgp_kernel_spec_t* spec, int* n_params) {
  DevProgram P;
  BGP_TRY(build_dev_program(spec, &P));
  *n_params = P.n_params_total;
  return BGP_OK;
}

int bgp_dev_alloc(void** p, size_t bytes) {
  BGP_TRY(require_device());
  BGP_CUDA(cudaMalloc(p, bytes));
  return BGP_OK;
}
int bgp_dev_free(void* p) { BGP_CUDA(cudaFree(p)); return BGP_OK; }
int bgp_dev_upload(void* dst, const void* src, size_t bytes) { BGP_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice)); return BGP_OK; }
int bgp_host_alloc_pinned(void** p, size_t bytes) { BGP_CUDA(cudaMallocHost(p, bytes)); return BGP_OK; }
int bgp_host_free_pinned(void* p) { BGP_CUDA(cudaFreeHost(p)); return BGP_OK; }

}  // extern "C"

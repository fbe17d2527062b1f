// hodlr.cu — host orchestration + C ABI of the HODLR solver (replaces src/george/solvers/_hodlr.cpp:36-204 and
// the hodlr::Node recursion of src/george/include/george/hodlr.h).
//
// Pipeline of one compute() (all on the device; the host only builds the O(#nodes) index structure):
//   tree geometry (host, bit-exact with hodlr.h:48-61)
//   -> [stream A] leaf build + LDL^T (K4)      [stream B] ACA of every internal node (K5)
//   -> ranks back to the host (one small D2H), per-level common ranks, panel finalisation
//   -> leaf solves applied to all ancestor columns, then per level bottom-up: gram (K6a) -> LU/solve (K6b) -> update (K6c)
//   -> log-det = sum of leaf and node log-dets.
// solve(): the same three kernels with the right-hand side as target (K7).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "hodlr_kernels.cuh"
#include "hodlr_lu.cuh"
#include "hodlr_aca2.cuh"
#include "hodlr_leaf.cuh"
#include "kernel_eval.cuh"

namespace bgp {
int upload_program(const DevProgram& P, DevBuf<DevProgram>& buf, cudaStream_t s);
int kmat_grad_contract_launch(const DevProgram* dprog, int nd, int np, const unsigned* which_dev, const double* x,
                              int64_t n, const double* M, int64_t ldm, const double* alpha, double ca, double cm,
                              double* g_dev, double* diag_dev, DevBuf<double>& scratch, cudaStream_t s);
int fill_identity_launch(double* A, int64_t n, cudaStream_t s);
bool comm_ready();
int comm_rank();
int comm_world();
int comm_allreduce_sum_f64(double* buf, size_t count, cudaStream_t s);
int comm_allgather_f64(const double* send, double* recv, size_t count, cudaStream_t s);
}
using namespace bgp;

struct HNode {
  int start, size, half, is_leaf, parent, dir, depth;
  int rank = 0, draws = 0, fallback = 0;
  int owned = 1;   // sharding: this process factors the node locally
  int top = 0;     // sharding: node above the shard cut (finished after the exchange)
};

// Factor panels (DESIGN.md §3).  A level owned by one shard only ever touches that shard's rows, so its panels hold
// nloc rows (leading dimension nloc) and are addressed with GLOBAL row indices through a base pointer shifted by the
// shard's first row; the levels above the shard cut span all N rows.  Single-GPU runs have only the "local" set (all rows).
struct PanelSet {
  DevBuf<double> V, U;
  int64_t ld = 0, row_off = 0;
  int vcols = 0, ucols = 0;
  double* vbase() const { return V.p - row_off; }
  double* ubase() const { return U.p - row_off; }
};

struct LevelInfo {
  std::vector<int> nodes;  // pre-order ids of the internal nodes at this depth handled here
  int set = 1;             // 0: level above the shard cut (panel set `top`), 1: owned level (panel set `loc`)
  int cap = 0, max_cap = 0, vcol = 0, r = 0, ucol = 0;  // vcol / ucol: first column of the level in ITS panel set
  int max_half = 0, grow = 0;
  int desc_off = 0;  // offset of this level's NodeDesc block
};

struct AcaGraphKey {  // everything the captured ACA loop depends on
  A2Args a;
  int nn, ncc, nrc, shape, grid;
};

// the cached executable graph of the ACA loop (run_aca2) and the key it was captured for
struct AcaGraph {
  AcaGraphKey key;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  void reset() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    exec = nullptr; graph = nullptr;
  }
  ~AcaGraph() { reset(); }
  AcaGraph() {}
  AcaGraph(const AcaGraph&) = delete;
  AcaGraph& operator=(const AcaGraph&) = delete;
};

struct bgp_hodlr {
  // declared before every DevBuf: streams outlive buffers
  Stream sA, sB, sC;  // sC: capture stream of the ACA graph
  Event ev[8];
  std::vector<Event> prof_events;
  AcaGraph aca;
  ~bgp_hodlr() { sA.sync(); sB.sync(); sC.sync(); }  // no buffer is freed while another stream still uses it
  int64_t n = 0;
  int ndim = 0;
  bgp_hodlr_opts_t opts;
  bool computed = false;
  double log_det = 0.0;
  DevProgram prog;

  std::vector<HNode> nodes;  // pre-order
  std::vector<int> leaves;   // pre-order ids
  std::vector<LevelInfo> levels;
  std::vector<int> piv_off;  // per internal node (by pre-order id) offset into pivot arrays, -1 for leaves
  int max_leaf = 0, cut_depth = 0;
  int64_t row0 = 0, nloc = 0;
  std::vector<int64_t> shard_row0, shard_rows;

  DevBuf<DevProgram> d_prog;
  DevBuf<double> d_x, d_yerr, d_diag, d_L, d_leaf_logdet, d_node_logdet, d_S, d_W, d_scalar, d_rhs;
  PanelSet top, loc;
  const PanelSet& pset(const LevelInfo& L) const { return L.set == 0 ? top : loc; }
  DevBuf<double> d_inv, d_gscratch;          // grad_terms: K^-1 (n x n) and the contraction partials
  DevBuf<double> d_xsend, d_xrecv;           // sharded runs: pack / all-gather staging
  DevBuf<unsigned> d_which;
  LuWorkspace lu_ws;                         // big-rank Woodbury step (hodlr_lu.cuh)
  DevBuf<GemmDesc> d_gram_desc, d_upd_desc;
  std::vector<NodeDesc> h_nodes;             // host copy of d_nodes
  std::vector<int> cap_hint;                 // per-level ACA capacities the previous compute() ended with
  int64_t cap_hint_n = -1;
  int cap_hint_min_size = -1;
  DevBuf<LeafDesc> d_leaves;
  DevBuf<AcaDesc> d_aca;
  DevBuf<AcaOut> d_aca_out;
  DevBuf<NodeDesc> d_nodes;
  DevBuf<int> d_idx, d_piv_rows, d_piv_cols, d_ticket, d_chain_done, d_ncols_by_depth;
  DevBuf<uint32_t> d_chain_state;
  DevBuf<A2Node> d_a2nodes;
  DevBuf<A2State> d_a2states;
  DevBuf<MT19937> d_a2rngs;
  DevBuf<A2EPart> d_epart;
  DevBuf<int> d_cand, d_cand_k, d_cand_words, d_cand_L, d_cand_next, d_cand_live, d_cchunk_node, d_rchunk_node, d_nactive;
  DevBuf<double> d_node_box;
  DevBuf<double2> d_cand_xu;
  DevBuf<unsigned long long> d_cmax, d_stats;
  DevBuf<int4> d_work;
  DevBuf<int> d_work_count, d_iter;
  bool profile = false;
  double prof[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};  // see bgp_hodlr_last_aca_profile
  DevBuf<double> d_vpart, d_upart, d_vmax;
  int aca_iters = 0;
  size_t w_cap = 0;

  double t_ms[5] = {0, 0, 0, 0, 0};
  double work[6] = {0, 0, 0, 0, 0, 0};
};

static int ensure_streams(bgp_hodlr* h) {
  BGP_TRY(h->sA.create());
  BGP_TRY(h->sB.create());
  for (Event& e : h->ev) BGP_TRY(e.create());
  return BGP_OK;
}

// hodlr.h:29-66: pre-order construction; a node splits iff size/2 >= min_size.
static void build_tree(bgp_hodlr* h, int start, int size, int dir, int parent, int depth) {
  HNode nd;
  nd.start = start; nd.size = size; nd.half = size / 2; nd.dir = dir; nd.parent = parent; nd.depth = depth;
  nd.is_leaf = !(nd.half >= h->opts.min_size);
  const int id = (int)h->nodes.size();
  h->nodes.push_back(nd);
  if (!nd.is_leaf) {
    build_tree(h, start, nd.half, 0, id, depth + 1);
    build_tree(h, start + nd.half, size - nd.half, 1, id, depth + 1);
  }
}

static int hodlr_solve_dev(bgp_hodlr* h, double* b, int64_t nrhs, int64_t ldb, cudaStream_t s, bool local_only);
static int hodlr_finish_sharded(bgp_hodlr* h);

static int launch_leaf_solve(bgp_hodlr* h, double* X, int64_t ldx, const int* ncols_by_depth, int ncols_fixed,
                             int max_cols, cudaStream_t s) {
  const int nl = (int)h->leaves.size();
  if (nl == 0 || max_cols == 0) return BGP_OK;
  // only leaves handled locally are in d_leaves; column groups of LS_COLS
  dim3 grid(nl, (max_cols + LS_COLS - 1) / LS_COLS);
  const size_t smem = sizeof(double) * (size_t)h->max_leaf * LS_COLS;
  if (smem > 200 * 1024) { set_error("leaf size %d too large for the leaf solve kernel", h->max_leaf); return BGP_ERR_INVALID; }
  cudaFuncSetAttribute(leaf_solve_kernel<LS_COLS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  leaf_solve_kernel<LS_COLS><<<grid, LS_THREADS, smem, s>>>(h->d_leaves.p, h->d_L.p, X, ldx, ncols_by_depth, ncols_fixed, h->max_leaf);
  BGP_LAUNCH_CHECK();
  return BGP_OK;
}

// one internal level: W = V^T X (both halves), small solve, X -= U T.   factor: up-sweep (X = U panel) vs plain solve
// Two paths: ranks whose 2r x 2r Woodbury matrix fits one CTA's shared memory (the common case) run three batched
// kernels; larger ranks run the Gram / update products on DMMA and the blocked LU of hodlr_lu.cuh.
static int launch_level_big(bgp_hodlr* h, const LevelInfo& L, double* X, int64_t ldx, int ncolsW, int own_off, int factor,
                            int col_lo, int col_hi, cudaStream_t s);

static int launch_level(bgp_hodlr* h, const LevelInfo& L, double* X, int64_t ldx, int ncolsW, int own_off, int factor,
                        int col_lo, int col_hi, cudaStream_t s) {
  const int nn = (int)L.nodes.size();
  if (nn == 0 || L.r == 0) {
    return BGP_OK;
  }
  const int r = L.r;
  const int64_t stride = (int64_t)2 * r * ncolsW;  // one (2r x ncolsW) block per node
  const size_t need = (size_t)nn * stride;
  if (need > h->w_cap) { set_error("internal: W workspace too small (%zu > %zu)", need, h->w_cap); return BGP_ERR_CUDA; }
  BGP_CUDA(cudaMemsetAsync(h->d_W.p, 0, sizeof(double) * need, s));
  // diagnostics: BGP_SMALL_RANK_LIMIT=<2r> lowers the switch-over so the tests can drive every level through the big path
  int small_limit = SS_MAX_N;
  if (const char* e = getenv("BGP_SMALL_RANK_LIMIT")) small_limit = std::min(SS_MAX_N, atoi(e));
  if (2 * r > small_limit) return launch_level_big(h, L, X, ldx, ncolsW, own_off, factor, col_lo, col_hi, s);
  const NodeDesc* nd = h->d_nodes.p + L.desc_off;
  const int max_nh = L.max_half + 1;
  {
    dim3 grid((max_nh + GT_CHUNK - 1) / GT_CHUNK, nn * 2, (ncolsW + GT_TC - 1) / GT_TC);
    gram_tn_kernel<<<grid, GT_THREADS, 0, s>>>(nd, h->pset(L).vbase(), h->pset(L).ld, X, ldx, ncolsW, h->d_W.p, stride);
    BGP_LAUNCH_CHECK();
  }
  {
    const size_t sbytes = sizeof(double) * (size_t)(2 * r) * (2 * r);
    // (the attribute is per device / context: set it on every call, it is cheap)
    cudaFuncSetAttribute(small_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    small_solve_kernel<<<nn, SS_THREADS, sbytes, s>>>(nd, h->d_W.p, stride, ncolsW, own_off, factor, h->d_S.p,
                                                      h->d_node_logdet.p, L.desc_off);
    BGP_LAUNCH_CHECK();
  }
  if (col_hi > col_lo) {
    dim3 grid((max_nh + UP_ROWS - 1) / UP_ROWS, nn * 2, (col_hi - col_lo + UP_TC - 1) / UP_TC);
    update_nn_kernel<<<grid, UP_THREADS, 0, s>>>(nd, h->pset(L).ubase(), h->pset(L).ld, X, ldx, col_lo, col_hi, h->d_W.p, stride, 0);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

static int launch_level_big(bgp_hodlr* h, const LevelInfo& L, double* X, int64_t ldx, int ncolsW, int own_off, int factor,
                            int col_lo, int col_hi, cudaStream_t s) {
  const int nn = (int)L.nodes.size();
  const int r = L.r, n2 = 2 * r;
  const int64_t stride = (int64_t)n2 * ncolsW;
  const int64_t ldv = h->pset(L).ld, ldu = h->pset(L).ld;
  double* W = h->d_W.p;
  constexpr int KCHUNK = 4096;  // rows per split-K slice of the Gram product
  std::vector<LuNode> lun(nn);
  std::vector<GemmDesc> gram, upd;
  int max_nh = 0;
  for (int b = 0; b < nn; ++b) {
    const HNode& nd = h->nodes[L.nodes[b]];
    const int64_t s_off = h->h_nodes[L.desc_off + b].s_off;
    lun[b].S = h->d_S.p + s_off;
    lun[b].piv = reinterpret_cast<int*>(lun[b].S + (int64_t)n2 * n2);
    lun[b].logdet = h->d_node_logdet.p + L.desc_off + b;
    double* Wn = W + (int64_t)b * stride;
    for (int hh = 0; hh < 2; ++hh) {
      const int rs = nd.start + (hh ? nd.half : 0), nh = hh ? (nd.size - nd.half) : nd.half;
      max_nh = std::max(max_nh, nh);
      for (int k0 = 0; k0 < nh; k0 += KCHUNK) {  // W_h (r x ncolsW) += V_h^T X_h
        GemmDesc g;
        g.A = h->pset(L).vbase() + (int64_t)L.vcol * ldv + rs + k0; g.lda = ldv;   // A'(q, i) = V[i + q ldv]
        g.B = X + rs + k0; g.ldb = ldx;                                   // B'(i, c) = X[i + c ldx]
        g.C = Wn + (hh ? 0 : r); g.ldc = n2;
        g.M = r; g.N = ncolsW; g.K = std::min(KCHUNK, nh - k0); g.mode = GD_ATOMIC_ADD;
        gram.push_back(g);
      }
      if (col_hi > col_lo) {  // X_h[:, col_lo:col_hi] -= U_h T_h
        GemmDesc g;
        g.A = h->pset(L).ubase() + (int64_t)L.ucol * ldu + rs; g.lda = ldu;        // A'(i, q) = U[i + q ldu]
        g.B = Wn + (hh ? r : 0) + (int64_t)col_lo * n2; g.ldb = n2;       // B'(q, c) = T[q + c 2r]
        g.C = X + rs + (int64_t)col_lo * ldx; g.ldc = ldx;
        g.M = nh; g.N = col_hi - col_lo; g.K = r; g.mode = GD_SUB;
        upd.push_back(g);
      }
    }
  }
  BGP_TRY(lu_upload(h->d_gram_desc, gram, s));
  BGP_TRY((gemm_dmma_launch<true, true>(h->d_gram_desc.p, (int)gram.size(), r, ncolsW, nullptr, s)));
  if (factor) {
    BGP_TRY(lu_upload(h->lu_ws.d_nodes, lun, s));
    dim3 grid((unsigned)std::min<int64_t>(((int64_t)n2 * n2 + 255) / 256, 4096), nn);
    lu_assemble_kernel<<<grid, 256, 0, s>>>(h->lu_ws.d_nodes.p, W, stride, r, own_off);
    BGP_LAUNCH_CHECK();
    BGP_TRY(lu_factor_batch(h->lu_ws, lun, n2, s));
    // the own columns [own_off, own_off + r) only feed S; the targets are the ancestor columns [col_lo, col_hi)
    if (col_hi > col_lo)
      BGP_TRY(lu_solve_batch(h->lu_ws, lun, n2, W + (int64_t)col_lo * n2, stride, n2, col_hi - col_lo, false, s));
  } else {
    BGP_TRY(lu_solve_batch(h->lu_ws, lun, n2, W, stride, n2, ncolsW, true, s));
  }
  if (!upd.empty()) {
    BGP_TRY(lu_upload(h->d_upd_desc, upd, s));
    BGP_TRY((gemm_dmma_launch<false, true>(h->d_upd_desc.p, (int)upd.size(), max_nh, col_hi - col_lo, nullptr, s)));
  }
  return BGP_OK;
}

// GPU-wide lock-step ACA (hodlr_aca2.cuh).  descs are in launch order; results go to houts[desc.node].
static int run_aca2(bgp_hodlr* h, const std::vector<AcaDesc>& descs, std::vector<AcaOut>& houts, cudaStream_t s) {
  const int nn = (int)descs.size();
  if (nn == 0) return BGP_OK;
  std::vector<A2Node> hn(nn);
  std::vector<int> cchunk_node, rchunk_node;
  int64_t cand_total = 0;
  int capmax = 1;
  for (int i = 0; i < nn; ++i) {
    const AcaDesc& d = descs[i];
    A2Node& a = hn[i];
    a.row0 = d.row0; a.n_rows = d.n_rows; a.col0 = d.col0; a.n_cols = d.n_cols;
    a.vcol = d.vcol; a.cap = d.cap; a.pre_id = d.pre_id; a.node = d.node;
    {
      const PanelSet& ps = h->pset(h->levels[h->nodes[d.pre_id].depth]);
      a.ld = ps.ld;
      a.vbase = ps.vbase() + (int64_t)d.vcol * ps.ld;
    }
    a.idx_off = d.idx_off; a.piv_off = d.piv_off;
    a.cchunk0 = (int)cchunk_node.size(); a.n_cchunks = (d.n_cols + A2_CHUNK - 1) / A2_CHUNK;
    a.rchunk0 = (int)rchunk_node.size(); a.n_rchunks = (d.n_rows + A2_CHUNK - 1) / A2_CHUNK;
    for (int c = 0; c < a.n_cchunks; ++c) cchunk_node.push_back(i);
    for (int c = 0; c < a.n_rchunks; ++c) rchunk_node.push_back(i);
    a.bmax = std::min(A2_BMAX, d.n_rows);
    a.cand_off = cand_total; cand_total += a.bmax;
    capmax = std::max(capmax, d.cap);
  }
  const int ncc = (int)cchunk_node.size(), nrc = (int)rchunk_node.size();
  BGP_TRY(h->d_a2nodes.reserve(nn, s));
  BGP_TRY(h->d_a2states.reserve(nn, s));
  BGP_TRY(h->d_a2rngs.reserve((size_t)2 * nn, s));
  BGP_TRY(h->d_cand.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_cand_k.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_cand_words.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_cand_L.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_cand_next.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_cand_live.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_node_box.reserve((size_t)2 * nn, s));
  BGP_TRY(h->d_cmax.reserve((size_t)cand_total, s));
  BGP_TRY(h->d_epart.reserve((size_t)std::max(ncc, 1) * A2_NSUB, s));
  BGP_TRY(h->d_cchunk_node.reserve(ncc, s));
  BGP_TRY(h->d_rchunk_node.reserve(nrc, s));
  BGP_TRY(h->d_vpart.reserve((size_t)ncc * A2_NSUB * (capmax + 1), s));
  BGP_TRY(h->d_upart.reserve((size_t)nrc * A2_NSUB * (capmax + 1), s));
  const bool cull = shape_has_bound(h->prog.shape) && !getenv("BGP_NO_CULL");  // BGP_NO_CULL: exhaustive scan (tests compare both)
  if (cull) {
    BGP_TRY(h->d_vmax.reserve((size_t)ncc * A2_NGROUP, s));
    BGP_TRY(h->d_cand_xu.reserve((size_t)cand_total, s));
  }
  BGP_TRY(h->d_nactive.reserve(1, s));
  BGP_TRY(h->d_stats.reserve(4, s));
  int64_t work_cap = 0;
  // items per chunk: batches of up to 256 live candidates are cut into blocks of A2_CG, larger ones into A2_CG * A2_ITEM_CB
  for (int i = 0; i < nn; ++i) {
    const int big = (hn[i].bmax + A2_CG * A2_ITEM_CB - 1) / (A2_CG * A2_ITEM_CB);
    const int small = (std::min(hn[i].bmax, 256) + A2_CG - 1) / A2_CG;
    work_cap += (int64_t)hn[i].n_cchunks * std::max(big, small);
  }
  BGP_TRY(h->d_work.reserve((size_t)(2 * work_cap), s));
  BGP_TRY(h->d_work_count.reserve(4, s));  // [0..1] item counters, [2..3] consumption cursors
  BGP_TRY(h->d_iter.reserve(1, s));
  BGP_CUDA(cudaMemsetAsync(h->d_iter.p, 0, sizeof(int), s));
  BGP_CUDA(cudaMemsetAsync(h->d_work_count.p, 0, sizeof(int) * 4, s));
  BGP_CUDA(cudaMemsetAsync(h->d_stats.p, 0, sizeof(unsigned long long) * 4, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_a2nodes.p, hn.data(), sizeof(A2Node) * nn, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_cchunk_node.p, cchunk_node.data(), sizeof(int) * ncc, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_rchunk_node.p, rchunk_node.data(), sizeof(int) * nrc, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(h->d_nactive.p, &nn, sizeof(int), cudaMemcpyHostToDevice, s));
  A2Args a;
  memset(&a, 0, sizeof(a));  // (the struct is also the key of the cached graph: no indeterminate padding)
  a.prog = h->d_prog.p; a.x = h->d_x.p; a.nodes = h->d_a2nodes.p; a.states = h->d_a2states.p; a.rngs = h->d_a2rngs.p; a.n_nodes = nn;
  a.tol = h->opts.tol; a.seed = (uint32_t)h->opts.seed; a.exhaust_mode = h->opts.exhaust_mode;
  a.idx_ws = h->d_idx.p; a.piv_rows = h->d_piv_rows.p; a.piv_cols = h->d_piv_cols.p;
  a.cand = h->d_cand.p; a.cand_k = h->d_cand_k.p; a.cand_words = h->d_cand_words.p; a.cmax = h->d_cmax.p; a.epart = h->d_epart.p;
  a.cchunk_node = h->d_cchunk_node.p; a.rchunk_node = h->d_rchunk_node.p; a.vpart = h->d_vpart.p; a.upart = h->d_upart.p;
  a.vmax = cull ? h->d_vmax.p : nullptr;
  a.cand_xu = cull ? h->d_cand_xu.p : nullptr;
  a.cand_L = h->d_cand_L.p; a.cand_next = h->d_cand_next.p; a.cand_live = h->d_cand_live.p; a.node_box = h->d_node_box.p;
  a.capmax = capmax; a.n_active = h->d_nactive.p; a.stats = h->d_stats.p;
  a.work = h->d_work.p; a.work_count = h->d_work_count.p; a.work_cursor = h->d_work_count.p + 2; a.work_cap = (int)work_cap; a.iter_ptr = h->d_iter.p;
  // (the attribute is per device / context: set it on every call, it is cheap)
  cudaFuncSetAttribute(a2_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(A2NodeSmem));
    cudaFuncSetAttribute(a2_decide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(A2NodeSmem));
    cudaFuncSetAttribute(a2_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(A2NodeSmem));
  a2_init_kernel<<<nn, A2_NODE_THREADS, sizeof(A2NodeSmem), s>>>(a);
  BGP_LAUNCH_CHECK();
  int active = nn, iters = 0;
  const int eval_grid = num_sms() * 6;  // persistent CTAs over the work list (2-3 resident per SM, a few rounds)
  // One lock-step iteration = eval -> decide -> vrow -> pivot -> vnorm|ucol -> finish -> tick.
  auto launch_iteration = [&](cudaStream_t st, cudaGraphConditionalHandle hnd, int use_hnd, int it_prof) -> int {
    auto mark = [&](int slot) -> int {
      if (it_prof < 0) return BGP_OK;
      const size_t need = (size_t)7 * (it_prof + 1);
      while (h->prof_events.size() < need) {
        h->prof_events.emplace_back();
        BGP_TRY(h->prof_events.back().create());
      }
      BGP_CUDA(cudaEventRecord(h->prof_events[(size_t)7 * it_prof + slot], st));
      return BGP_OK;
    };
    BGP_TRY(mark(0));
    a2_eval_launch(h->prog.shape, dim3(eval_grid), st, a);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(1));
    a2_decide_kernel<<<nn, A2_NODE_THREADS, sizeof(A2NodeSmem), st>>>(a);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(2));
    a2_vrow_launch(h->prog.shape, dim3(ncc, A2_NSUB), st, a);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(3));
    a2_pivot_kernel<<<nn, 32, 0, st>>>(a);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(4));
    a2_vnorm_ucol_launch(h->prog.shape, dim3(ncc + nrc, A2_NSUB), st, a, ncc);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(5));
    a2_finish_kernel<<<nn, A2_NODE_THREADS, sizeof(A2NodeSmem), st>>>(a);
    BGP_LAUNCH_CHECK();
    BGP_TRY(mark(6));
    a2_tick_kernel<<<1, 1, 0, st>>>(a.iter_ptr, a.n_active, hnd, use_hnd);
    BGP_LAUNCH_CHECK();
    return BGP_OK;
  };
  const bool use_graph = !h->profile && !getenv("BGP_NO_GRAPH");
  if (use_graph) {
    // The whole loop is ONE graph launch: a WHILE node whose body is one iteration; a2_tick_kernel keeps the condition
    // up to date from the device-side count of active nodes.  The executable graph is cached: a hyper-parameter loop
    // calls compute() with the same shapes and buffers over and over.
    AcaGraphKey key;
    memset(&key, 0, sizeof(key));
    key.a = a; key.nn = nn; key.ncc = ncc; key.nrc = nrc; key.shape = h->prog.shape; key.grid = eval_grid;
    if (!h->aca.exec || memcmp(&key, &h->aca.key, sizeof(key)) != 0) {
      h->aca.reset();
      BGP_CUDA(cudaGraphCreate(&h->aca.graph, 0));
      cudaGraphConditionalHandle hnd;
      BGP_CUDA(cudaGraphConditionalHandleCreate(&hnd, h->aca.graph, 1, cudaGraphCondAssignDefault));
      cudaGraphNodeParams cp = {};
      cp.type = cudaGraphNodeTypeConditional;
      cp.conditional.handle = hnd;
      cp.conditional.type = cudaGraphCondTypeWhile;
      cp.conditional.size = 1;
      cudaGraphNode_t wnode;
      BGP_CUDA(cudaGraphAddNode(&wnode, h->aca.graph, nullptr, 0, &cp));
      cudaGraph_t body = cp.conditional.phGraph_out[0];
      BGP_TRY(h->sC.create());
      BGP_CUDA(cudaStreamBeginCaptureToGraph(h->sC, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
      const int rc = launch_iteration(h->sC, hnd, 1, -1);
      cudaGraph_t captured = nullptr;
      const cudaError_t ce = cudaStreamEndCapture(h->sC, &captured);
      if (rc != BGP_OK) return rc;
      if (ce != cudaSuccess) { set_error("ACA graph capture failed: %s", cudaGetErrorString(ce)); return BGP_ERR_CUDA; }
      BGP_CUDA(cudaGraphInstantiate(&h->aca.exec, h->aca.graph, 0));
      h->aca.key = key;
    }
    BGP_CUDA(cudaGraphLaunch(h->aca.exec, s));
    int it_host = 0;
    BGP_CUDA(cudaMemcpyAsync(&it_host, h->d_iter.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    BGP_CUDA(cudaMemcpyAsync(&active, h->d_nactive.p, sizeof(int), cudaMemcpyDeviceToHost, s));
    BGP_CUDA(cudaStreamSynchronize(s));
    iters = it_host;
    g_launches.fetch_add((uint64_t)7 * (uint64_t)std::max(iters - 1, 0), std::memory_order_relaxed);  // the capture counted one iteration
    if (active > 0) { set_error("ACA did not terminate"); return BGP_ERR_CUDA; }
  } else {
    while (active > 0) {
      for (int rep = 0; rep < 8; ++rep) {
        BGP_TRY(launch_iteration(s, 0, 0, h->profile ? iters : -1));
        iters++;
      }
      BGP_CUDA(cudaMemcpyAsync(&active, h->d_nactive.p, sizeof(int), cudaMemcpyDeviceToHost, s));
      BGP_CUDA(cudaStreamSynchronize(s));
      if (iters > (1 << 22)) { set_error("ACA did not terminate"); return BGP_ERR_CUDA; }
    }
  }
  h->aca_iters = iters;
  {
    unsigned long long st4[4] = {0, 0, 0, 0};
    BGP_CUDA(cudaMemcpyAsync(st4, h->d_stats.p, sizeof(st4), cudaMemcpyDeviceToHost, s));
    BGP_CUDA(cudaStreamSynchronize(s));
    h->prof[1] = iters; h->prof[2] = (double)st4[0]; h->prof[3] = (double)st4[1]; h->prof[4] = (double)st4[2];
    h->prof[5] = (double)st4[3];
    if (h->profile) {
      double tot[6] = {0, 0, 0, 0, 0, 0};
      for (int i = 0; i < iters; ++i)
        for (int k = 0; k < 6; ++k) {
          float ms = 0;
          cudaEventElapsedTime(&ms, h->prof_events[(size_t)7 * i + k], h->prof_events[(size_t)7 * i + k + 1]);
          tot[k] += ms;
        }
      h->prof[0] = tot[0];
      for (int k = 0; k < 6; ++k) h->prof[6 + k] = tot[k];
    }
  }
  if (h->opts.exhaust_mode == BGP_EXHAUST_DENSE) {
    a2_dense_fill_kernel<<<dim3(nn, 64), 256, 0, s>>>(a);
    BGP_LAUNCH_CHECK();
    a2_dense_rank_kernel<<<(nn + 127) / 128, 128, 0, s>>>(a);
    BGP_LAUNCH_CHECK();
  }
  std::vector<A2State> hs(nn);
  BGP_CUDA(cudaMemcpyAsync(hs.data(), h->d_a2states.p, sizeof(A2State) * nn, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  for (int i = 0; i < nn; ++i) {
    AcaOut o;
    o.rank = hs[i].rank; o.draws = hs[i].draws; o.fallback = hs[i].fallback; o.status = hs[i].status;
    houts[descs[i].node] = o;
  }
  return BGP_OK;
}

// log-determinant = sum of the leaf and node log-dets of this process.  A sharded run factors the nodes above the cut on
// every rank but counts them on shard 0 only, so that the sum over the shards counts each node once.
static int sum_log_det(bgp_hodlr* h, cudaStream_t s, double* out) {
  const int nl = (int)h->leaves.size(), nlev = (int)h->levels.size();
  int ndesc = 0;
  for (auto& L : h->levels) ndesc += (int)L.nodes.size();
  std::vector<double> ld_leaf(nl), ld_node(ndesc);
  if (nl) BGP_CUDA(cudaMemcpyAsync(ld_leaf.data(), h->d_leaf_logdet.p, sizeof(double) * nl, cudaMemcpyDeviceToHost, s));
  if (ndesc) BGP_CUDA(cudaMemcpyAsync(ld_node.data(), h->d_node_logdet.p, sizeof(double) * ndesc, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  const int cut = std::min(h->cut_depth, nlev);
  double ld = 0.0;
  for (double v : ld_leaf) ld += v;
  for (int l = 0; l < nlev; ++l) {
    const LevelInfo& L = h->levels[l];
    if (l < cut && h->opts.shard_rank != 0) continue;
    for (size_t i = 0; i < L.nodes.size(); ++i) ld += ld_node[L.desc_off + i];
  }
  *out = ld;
  return BGP_OK;
}

static void record_compute_timing(bgp_hodlr* h) {
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->t_ms[0] = ms;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[2]); h->t_ms[1] = ms;
  cudaEventElapsedTime(&ms, h->ev[6], h->ev[3]); h->t_ms[2] = ms;  // panel finalisation + leaf solves + level sweeps only
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[3]); h->t_ms[3] = ms;
}

static int hodlr_compute_dev_impl(bgp_hodlr* h, const bgp_kernel_spec_t* spec, const double* x_dev, int64_t n,
                                  int32_t ndim, const double* yerr_dev, const bgp_hodlr_opts_t* opts_in) {
  h->computed = false;
  BGP_TRY(require_device());
  BGP_TRY(ensure_streams(h));
  BGP_TRY(build_dev_program(spec, &h->prog));
  if (h->prog.ndim != ndim) { set_error("dimension mismatch: kernel ndim %d, input ndim %d", h->prog.ndim, ndim); return BGP_ERR_DIM; }
  if (ndim > ACA_MAX_NDIM) { set_error("HODLR supports at most %d input dimensions", ACA_MAX_NDIM); return BGP_ERR_INVALID; }
  if (n <= 0 || n > (int64_t)0x7fffffff) { set_error("invalid number of points %lld", (long long)n); return BGP_ERR_INVALID; }
  bgp_hodlr_opts_t o;
  if (opts_in) o = *opts_in; else bgp_hodlr_default_opts(&o);
  if (o.min_size < 1) { set_error("min_size must be >= 1"); return BGP_ERR_INVALID; }
  if (o.shard_count < 1) o.shard_count = 1;
  if (o.shard_count & (o.shard_count - 1)) { set_error("shard_count must be a power of two"); return BGP_ERR_INVALID; }
  if (o.shard_rank < 0 || o.shard_rank >= o.shard_count) { set_error("invalid shard_rank"); return BGP_ERR_INVALID; }
  if (o.shard_count > 1 && o.rng_mode == BGP_RNG_REFERENCE) { set_error("rng_mode=reference serialises the tree and cannot be sharded"); return BGP_ERR_INVALID; }
  if (o.shard_count > 1 && !(comm_ready() && comm_world() == o.shard_count && comm_rank() == o.shard_rank)) {
    set_error("a sharded factorisation is collective: it needs the communicator of bgp_comm_init with world == "
              "opts.shard_count (%d) and rank == opts.shard_rank (%d)", o.shard_count, o.shard_rank);
    return BGP_ERR_INVALID;
  }
  h->opts = o;
  h->n = n;
  h->ndim = ndim;
  cudaStream_t sA = h->sA, sB = h->sB;

  // ---- tree geometry ----
  h->nodes.clear(); h->leaves.clear(); h->levels.clear();
  h->nodes.reserve(2 * (size_t)(n / std::max(1, o.min_size)) + 8);
  build_tree(h, 0, (int)n, 0, -1, 0);
  int cut = 0;
  while ((1 << cut) < o.shard_count) cut++;
  h->cut_depth = cut;
  // sharding: the sub-tree owned by this process is the depth-`cut` node number shard_rank (left-to-right);
  // if the tree is shallower than the cut, everything is "top" work done redundantly.
  int max_depth = 0;
  for (auto& nd : h->nodes) max_depth = std::max(max_depth, nd.depth);
  h->row0 = 0; h->nloc = n;
  if (o.shard_count > 1) {
    int seen = 0; bool found = false;
    h->shard_row0.clear(); h->shard_rows.clear();
    for (size_t i = 0; i < h->nodes.size(); ++i) {
      HNode& nd = h->nodes[i];
      if (nd.depth == cut) {
        if (seen == o.shard_rank) { h->row0 = nd.start; h->nloc = nd.size; found = true; }
        h->shard_row0.push_back(nd.start); h->shard_rows.push_back(nd.size);
        seen++;
      }
    }
    if (!found || seen != o.shard_count) { set_error("tree too shallow to shard %d ways (N=%lld, min_size=%d)", o.shard_count, (long long)n, o.min_size); return BGP_ERR_INVALID; }
    for (auto& nd : h->nodes) {
      nd.top = nd.depth < cut;
      nd.owned = !nd.top && nd.start >= h->row0 && nd.start + nd.size <= h->row0 + h->nloc;
    }
  }
  h->levels.assign(max_depth + 1, LevelInfo());
  for (size_t i = 0; i < h->nodes.size(); ++i) {
    HNode& nd = h->nodes[i];
    if (nd.is_leaf) { if (nd.owned) h->leaves.push_back((int)i); continue; }
    if (!(nd.owned || nd.top)) continue;
    LevelInfo& L = h->levels[nd.depth];
    L.nodes.push_back((int)i);
    L.max_half = std::max(L.max_half, nd.size - nd.half);
  }
  while (!h->levels.empty() && h->levels.back().nodes.empty()) h->levels.pop_back();
  const int nlev = (int)h->levels.size();
  for (int l = 0; l < nlev; ++l) h->levels[l].set = (o.shard_count > 1 && l < cut) ? 0 : 1;
  h->top.ld = n; h->top.row_off = 0;
  h->loc.ld = h->nloc; h->loc.row_off = h->row0;

  // ---- capacities: start from rank_capacity (default 128) per level; levels that overflow are grown and the ACA
  //      stage is repeated (deterministic: the per-node / chained streams restart from the same seeds) ----
  const int rcap0 = o.rank_capacity > 0 ? o.rank_capacity : 128;
  for (auto& L : h->levels) {
    int mh = 0;
    for (int id : L.nodes) mh = std::max(mh, h->nodes[id].half);
    L.max_cap = std::max(1, mh);
    L.cap = std::min(rcap0, L.max_cap);
  }
  // a handle that already factored a tree of this shape starts from the capacities that run ended with (hyper-parameter
  // loops call compute() repeatedly on the same x): no repeated ACA stage in the steady state
  if (o.rank_capacity <= 0 && h->cap_hint_n == n && h->cap_hint_min_size == o.min_size && (int)h->cap_hint.size() == nlev)
    for (int l = 0; l < nlev; ++l) h->levels[l].cap = std::min(h->levels[l].max_cap, std::max(h->levels[l].cap, h->cap_hint[l]));

  // ---- inputs ----
  BGP_TRY(upload_program(h->prog, h->d_prog, sA));
  BGP_TRY(h->d_x.reserve((size_t)n * ndim, sA));
  BGP_TRY(h->d_diag.reserve((size_t)n, sA));
  if (x_dev != h->d_x.p) BGP_CUDA(cudaMemcpyAsync(h->d_x.p, x_dev, sizeof(double) * n * ndim, cudaMemcpyDeviceToDevice, sA));
  square_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1184), 256, 0, sA>>>(yerr_dev, h->d_diag.p, n);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaEventRecord(h->ev[0], sA));  // inputs ready / timing origin

  // ---- leaves (stream A) ----
  const int nl = (int)h->leaves.size();
  std::vector<LeafDesc> hleaves(nl);
  int64_t loff = 0;
  h->max_leaf = 0;
  for (int i = 0; i < nl; ++i) {
    const HNode& nd = h->nodes[h->leaves[i]];
    hleaves[i].start = nd.start; hleaves[i].size = nd.size; hleaves[i].depth = nd.depth; hleaves[i]._pad = 0;
    hleaves[i].off = loff;
    loff += (int64_t)nd.size * nd.size;
    h->max_leaf = std::max(h->max_leaf, nd.size);
  }
  BGP_TRY(h->d_leaves.reserve(std::max(nl, 1), sA));
  BGP_TRY(h->d_L.reserve((size_t)std::max<int64_t>(loff, 1), sA));
  BGP_TRY(h->d_leaf_logdet.reserve(std::max(nl, 1), sA));
  if (nl) {
    BGP_CUDA(cudaMemcpyAsync(h->d_leaves.p, hleaves.data(), sizeof(LeafDesc) * nl, cudaMemcpyHostToDevice, sA));
    if (h->max_leaf <= 768) {
      const int ldp = lf_panel_ld(h->max_leaf);
      const size_t smem = sizeof(double) * (size_t)LF_NB * ldp;
      // (the attribute is per device / context: set it on every call, it is cheap)
      cudaFuncSetAttribute(leaf_factor_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      leaf_factor_dmma_kernel<<<nl, LF_THREADS, smem, sA>>>(h->d_prog.p, h->d_x.p, h->d_diag.p, h->d_leaves.p, h->d_L.p,
                                                            h->d_leaf_logdet.p, ldp);
    } else {
      leaf_build_factor_kernel<<<nl, LEAF_THREADS, 0, sA>>>(h->d_prog.p, h->d_x.p, h->d_diag.p, h->d_leaves.p, h->d_L.p,
                                                            h->d_leaf_logdet.p);
    }
    BGP_LAUNCH_CHECK();
  }
  BGP_CUDA(cudaEventRecord(h->ev[1], sA));  // leaves done

  // ---- ACA (stream B, concurrent with the leaves) ----
  std::vector<AcaDesc> hdesc;
  std::vector<int> desc_node;  // pre-order id per descriptor
  std::vector<AcaOut> houts;
  int64_t idx_total = 0, piv_total = 0;
  int nint = 0;
  BGP_CUDA(cudaStreamWaitEvent(sB, h->ev[0], 0));
  for (int attempt = 0;; ++attempt) {
    int vcols_set[2] = {0, 0};
    for (auto& L : h->levels) { L.vcol = vcols_set[L.set]; vcols_set[L.set] += L.cap; }
    h->top.vcols = vcols_set[0]; h->loc.vcols = vcols_set[1];
    hdesc.clear(); desc_node.clear();
    h->piv_off.assign(h->nodes.size(), -1);
    idx_total = 0; piv_total = 0; nint = 0;
    for (int l = 0; l < nlev; ++l) {
      for (int id : h->levels[l].nodes) {
        const HNode& nd = h->nodes[id];
        AcaDesc d;
        d.row0 = nd.start + nd.half; d.n_rows = nd.size - nd.half; d.col0 = nd.start; d.n_cols = nd.half;
        d.vcol = h->levels[l].vcol; d.cap = h->levels[l].cap; d.pre_id = id; d.node = nint;
        d.idx_off = idx_total; d.piv_off = piv_total;
        h->piv_off[id] = (int)piv_total;
        idx_total += d.n_rows; piv_total += d.cap;
        hdesc.push_back(d); desc_node.push_back(id);
        nint++;
      }
    }
    // launch order: pre-order for the chained reference stream, largest blocks first otherwise
    std::vector<int> order(nint);
    for (int i = 0; i < nint; ++i) order[i] = i;
    if (o.rng_mode == BGP_RNG_REFERENCE) std::sort(order.begin(), order.end(), [&](int a, int b) { return hdesc[a].pre_id < hdesc[b].pre_id; });
    else std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      const int ta = h->nodes[hdesc[a].pre_id].top, tb = h->nodes[hdesc[b].pre_id].top;
      if (ta != tb) return ta > tb;  // nodes above the shard cut first
      return hdesc[a].n_rows > hdesc[b].n_rows;
    });
    std::vector<AcaDesc> hdesc_sorted(nint);
    for (int i = 0; i < nint; ++i) hdesc_sorted[i] = hdesc[order[i]];

    {
      // a capacity that no longer fits: give the old block back to the driver before asking for the larger one (the pool
      // keeps freed blocks cached, and a 2x larger request cannot reuse them: without the trim both would be resident)
      const size_t need_top = (size_t)n * std::max(h->top.vcols, 1), need_loc = (size_t)h->nloc * std::max(h->loc.vcols, 1);
      if ((h->top.V.p && h->top.V.n < need_top) || (h->loc.V.p && h->loc.V.n < need_loc)) {
        if (h->top.V.n < need_top) h->top.V.release();
        if (h->loc.V.n < need_loc) h->loc.V.release();
        h->top.U.release(); h->loc.U.release();
        BGP_CUDA(cudaStreamSynchronize(sA)); BGP_CUDA(cudaStreamSynchronize(sB));
        cudaMemPool_t pool; int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
      }
      BGP_TRY(h->top.V.reserve(need_top, sB));
      BGP_TRY(h->loc.V.reserve(need_loc, sB));
    }
    BGP_TRY(h->d_aca.reserve(std::max(nint, 1), sB));
    BGP_TRY(h->d_aca_out.reserve(std::max(nint, 1), sB));
    BGP_TRY(h->d_idx.reserve((size_t)std::max<int64_t>(idx_total, 1), sB));
    BGP_TRY(h->d_piv_rows.reserve((size_t)std::max<int64_t>(piv_total, 1), sB));
    BGP_TRY(h->d_piv_cols.reserve((size_t)std::max<int64_t>(piv_total, 1), sB));
    BGP_TRY(h->d_ticket.reserve(1, sB));
    BGP_TRY(h->d_chain_state.reserve(640, sB));
    BGP_TRY(h->d_chain_done.reserve(std::max(nint, 1), sB));
    houts.assign(nint, AcaOut());
    if (nint && o.rng_mode != BGP_RNG_REFERENCE) {
      BGP_TRY(run_aca2(h, hdesc_sorted, houts, sB));
    } else if (nint) {
      BGP_CUDA(cudaMemcpyAsync(h->d_aca.p, hdesc_sorted.data(), sizeof(AcaDesc) * nint, cudaMemcpyHostToDevice, sB));
      BGP_CUDA(cudaMemsetAsync(h->d_ticket.p, 0, sizeof(int), sB));
      BGP_CUDA(cudaMemsetAsync(h->d_chain_done.p, 0, sizeof(int) * nint, sB));
      int maxcap = 1;
      for (auto& L : h->levels) maxcap = std::max(maxcap, L.cap);
      const size_t smem = ((sizeof(AcaShared) + 15) & ~size_t(15)) + sizeof(double) * (size_t)maxcap;
      // (the attribute is per device / context: set it on every call, it is cheap)
      cudaFuncSetAttribute(aca_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      if (smem > 200 * 1024) { set_error("rank capacity %d too large", maxcap); return BGP_ERR_RANK_CAPACITY; }
      aca_kernel<<<nint, ACA_THREADS, smem, sB>>>(h->d_prog.p, h->d_x.p, h->d_aca.p, nint, h->loc.vbase(), h->loc.ld, o.tol, (uint32_t)o.seed,
                                                  h->d_idx.p, h->d_piv_rows.p, h->d_piv_cols.p, h->d_aca_out.p,
                                                  h->d_ticket.p, h->d_chain_state.p, h->d_chain_done.p, o.exhaust_mode);
      BGP_LAUNCH_CHECK();
      BGP_CUDA(cudaMemcpyAsync(houts.data(), h->d_aca_out.p, sizeof(AcaOut) * nint, cudaMemcpyDeviceToHost, sB));
    }
    BGP_CUDA(cudaEventRecord(h->ev[2], sB));  // ACA done
    BGP_CUDA(cudaStreamSynchronize(sB));

    // ---- ranks; grow the capacity of overflowing levels and repeat ----
    bool overflow = false;
    for (int i = 0; i < nint; ++i) {
      HNode& nd = h->nodes[desc_node[i]];
      nd.rank = houts[i].rank; nd.draws = houts[i].draws; nd.fallback = houts[i].fallback;
      if (houts[i].status == 2) { set_error("internal: ACA work list overflow"); return BGP_ERR_CUDA; }
      if (houts[i].status != 0) {
        LevelInfo& L = h->levels[nd.depth];
        if (o.rank_capacity > 0 || L.cap >= L.max_cap) {
          set_error("ACA rank capacity exceeded at node [start=%d size=%d] (capacity %d%s); raise rank_capacity", nd.start,
                    nd.size, L.cap, houts[i].fallback ? ", dense fallback" : "");
          return BGP_ERR_RANK_CAPACITY;
        }
        L.grow = houts[i].fallback ? L.max_cap : std::max(L.grow, std::min(L.max_cap, 2 * L.cap));
        overflow = true;
      }
    }
    if (!overflow) {
      h->cap_hint.assign(nlev, 0);
      for (int l = 0; l < nlev; ++l) h->cap_hint[l] = h->levels[l].cap;
      h->cap_hint_n = n; h->cap_hint_min_size = o.min_size;
      break;
    }
    for (auto& L : h->levels) if (L.grow > L.cap) L.cap = L.grow;
    if (attempt > 16) { set_error("ACA capacity growth did not converge"); return BGP_ERR_RANK_CAPACITY; }
  }
  int rtot_set[2] = {0, 0}, ndesc = 0, ndesc_top = 0;
  int64_t s_total = 0;
  size_t w_need = 1;
  std::vector<NodeDesc> hnd;
  for (int l = 0; l < nlev; ++l) {
    LevelInfo& L = h->levels[l];
    L.r = 0;
    for (int id : L.nodes) L.r = std::max(L.r, h->nodes[id].rank);
    L.ucol = rtot_set[L.set];
    rtot_set[L.set] += L.r;
    L.desc_off = ndesc;
    for (int id : L.nodes) {
      const HNode& nd = h->nodes[id];
      NodeDesc d;
      d.start = nd.start; d.size = nd.size; d.half = nd.half; d.depth = nd.depth; d.vcol = L.vcol; d.ucol = L.ucol;
      d.r = L.r; d.rank = nd.rank; d.s_off = s_total;
      s_total += (int64_t)(2 * L.r) * (2 * L.r) + 2 * L.r + 2;
      hnd.push_back(d);
      ndesc++;
      if (L.set == 0) ndesc_top++;
    }
    w_need = std::max(w_need, (size_t)L.nodes.size() * 2 * (size_t)L.r * (size_t)(L.ucol + L.r));
  }
  h->top.ucols = rtot_set[0]; h->loc.ucols = rtot_set[1];
  const int rtot = rtot_set[0] + rtot_set[1];
  // per-depth number of LOCAL ancestor columns a leaf (or node) at that depth sees (levels above the cut live in the top
  // panel set and receive this shard's sub-tree inverse in a separate pass, below)
  std::vector<int> ncols_by_depth(max_depth + 2, h->loc.ucols);
  for (int dpt = 0; dpt <= max_depth + 1; ++dpt)
    ncols_by_depth[dpt] = dpt < nlev ? (h->levels[dpt].set == 1 ? h->levels[dpt].ucol : 0) : h->loc.ucols;

  BGP_CUDA(cudaEventRecord(h->ev[6], sA));  // ranks known, both streams drained up to here: the up-sweep starts
  BGP_TRY(h->d_nodes.reserve(std::max(ndesc, 1), sA));
  BGP_TRY(h->d_node_logdet.reserve(std::max(ndesc, 1), sA));
  BGP_TRY(h->top.U.reserve((size_t)n * std::max(h->top.ucols, 1), sA));
  BGP_TRY(h->loc.U.reserve((size_t)h->nloc * std::max(h->loc.ucols, 1), sA));
  BGP_TRY(h->d_S.reserve((size_t)std::max<int64_t>(s_total, 1), sA));
  // solve() needs 2*r*nrhs per node; keep room for 64 right-hand sides per batch
  for (auto& L : h->levels) w_need = std::max(w_need, (size_t)L.nodes.size() * 2 * (size_t)L.r * 64);
  BGP_TRY(h->d_W.reserve(w_need, sA));
  h->w_cap = h->d_W.n;
  BGP_TRY(h->d_ncols_by_depth.reserve(ncols_by_depth.size(), sA));
  BGP_TRY(h->d_scalar.reserve(4, sA));
  BGP_CUDA(cudaMemcpyAsync(h->d_ncols_by_depth.p, ncols_by_depth.data(), sizeof(int) * ncols_by_depth.size(), cudaMemcpyHostToDevice, sA));
  if (ndesc) {
    BGP_CUDA(cudaMemcpyAsync(h->d_nodes.p, hnd.data(), sizeof(NodeDesc) * ndesc, cudaMemcpyHostToDevice, sA));
    h->h_nodes = hnd;
    BGP_CUDA(cudaMemsetAsync(h->d_node_logdet.p, 0, sizeof(double) * ndesc, sA));
    // the levels above the cut come first in the descriptor list: one launch per panel set
    int rmax_set[2] = {0, 0};
    for (auto& L : h->levels) rmax_set[L.set] = std::max(rmax_set[L.set], L.r);
    if (ndesc_top > 0 && rmax_set[0] > 0) {
      finalize_panels_kernel<<<dim3(ndesc_top, rmax_set[0]), 256, 0, sA>>>(h->d_nodes.p, h->top.vbase(), h->top.ld, h->top.ubase(), h->top.ld);
      BGP_LAUNCH_CHECK();
    }
    if (ndesc > ndesc_top && rmax_set[1] > 0) {
      finalize_panels_kernel<<<dim3(ndesc - ndesc_top, rmax_set[1]), 256, 0, sA>>>(h->d_nodes.p + ndesc_top, h->loc.vbase(), h->loc.ld,
                                                                                  h->loc.ubase(), h->loc.ld);
      BGP_LAUNCH_CHECK();
    }
  }

  // ---- up-sweep (stream A; leaves are already ordered before this on the same stream) ----
  // (1) the owned sub-tree against its own (local) ancestor columns
  if (h->loc.ucols > 0) BGP_TRY(launch_leaf_solve(h, h->loc.ubase(), h->loc.ld, h->d_ncols_by_depth.p, 0, h->loc.ucols, sA));
  const int stop_level = (o.shard_count > 1) ? h->cut_depth : 0;
  for (int l = nlev - 1; l >= stop_level; --l) {
    const LevelInfo& L = h->levels[l];
    BGP_TRY(launch_level(h, L, h->loc.ubase(), h->loc.ld, L.ucol + L.r, L.ucol, 1, 0, L.ucol, sA));
  }
  // (2) sharded: the factored sub-tree applied to this shard's rows of the top-level factor columns (hodlr.h:95-102 for
  //     the ancestors above the cut) — the same kernels as a solve with the top panel as right-hand sides
  if (o.shard_count > 1 && h->top.ucols > 0) BGP_TRY(hodlr_solve_dev(h, h->top.U.p, h->top.ucols, n, sA, true));
  BGP_CUDA(cudaEventRecord(h->ev[3], sA));
  if (o.shard_count > 1) return hodlr_finish_sharded(h);

  BGP_TRY(sum_log_det(h, sA, &h->log_det));
  h->computed = true;
  record_compute_timing(h);

  // algorithmic work (SURVEY.md §8d)
  {
    double evals = 0, bytes = 0, flops = 0, R = rtot;
    for (int id : h->leaves) { const double m = h->nodes[id].size; evals += m * (m + 1) / 2; bytes += 8 * m * m; flops += m * m * m / 3 + 2 * m * m * ncols_by_depth[h->nodes[id].depth]; }
    for (int l = 0; l < nlev; ++l) {
      const LevelInfo& L = h->levels[l];
      for (int id : L.nodes) {
        const HNode& nd = h->nodes[id];
        evals += (double)nd.size * nd.draws;  // one row + one column of the block per accepted/rejected draw (upper bound)
        bytes += 16.0 * nd.size * nd.rank;
        flops += 4.0 * nd.size * L.r * L.ucol + 2.0 * nd.size * L.r * L.r + 2.0 * nd.size * nd.rank * nd.rank;
      }
    }
    h->work[0] = evals; h->work[1] = bytes; h->work[2] = flops; h->work[3] = R; h->work[4] = h->max_leaf; h->work[5] = nlev;
  }
  return BGP_OK;
}

// all-gather of the shards' row slices of `cols` columns of a column-major matrix P (leading dimension ld): every rank
// ends up with all rows.  pack -> ncclAllGather -> unpack on one stream, no host synchronisation.
static int exchange_rows(bgp_hodlr* h, double* P, int64_t ld, int64_t cols, cudaStream_t s) {
  if (cols <= 0) return BGP_OK;
  const int world = h->opts.shard_count;
  int64_t rows_pad = 0;
  for (int64_t r : h->shard_rows) rows_pad = std::max(rows_pad, r);
  const size_t per = (size_t)cols * rows_pad;
  BGP_TRY(h->d_xsend.reserve(per, s));
  BGP_TRY(h->d_xrecv.reserve(per * world, s));
  if (h->nloc < rows_pad) BGP_CUDA(cudaMemsetAsync(h->d_xsend.p, 0, sizeof(double) * per, s));
  pack_rows_kernel<<<1184, 256, 0, s>>>(P, ld, h->row0, h->nloc, cols, h->d_xsend.p, rows_pad);
  BGP_LAUNCH_CHECK();
  BGP_TRY(comm_allgather_f64(h->d_xsend.p, h->d_xrecv.p, per, s));
  for (int sh = 0; sh < world; ++sh) {
    if (sh == h->opts.shard_rank) continue;  // own rows are already in place
    unpack_rows_kernel<<<1184, 256, 0, s>>>(P, ld, h->shard_row0[sh], h->shard_rows[sh], cols, h->d_xrecv.p + (size_t)sh * per, rows_pad);
    BGP_LAUNCH_CHECK();
  }
  return BGP_OK;
}

// local_only: the leaves and the levels at or below the shard cut, without the exchange (compute() applies the owned
// sub-tree to the top panel this way).  Otherwise the whole solve; a sharded one all-gathers the locally solved rows
// before the levels above the cut (replicated right-hand side: every rank needs all rows).
static int hodlr_solve_dev(bgp_hodlr* h, double* b, int64_t nrhs, int64_t ldb, cudaStream_t s, bool local_only) {
  const int nlev = (int)h->levels.size();
  const bool sharded = h->opts.shard_count > 1;
  const int cut = sharded ? h->cut_depth : 0;
  for (int64_t c0 = 0; c0 < nrhs; c0 += 64) {
    const int nc = (int)std::min<int64_t>(64, nrhs - c0);
    double* X = b + c0 * ldb;
    BGP_TRY(launch_leaf_solve(h, X, ldb, nullptr, nc, nc, s));
    for (int l = nlev - 1; l >= cut; --l) BGP_TRY(launch_level(h, h->levels[l], X, ldb, nc, 0, 0, 0, nc, s));
    if (local_only) continue;
    if (sharded) BGP_TRY(exchange_rows(h, X, ldb, nc, s));
    for (int l = std::min(cut, nlev) - 1; l >= 0; --l) BGP_TRY(launch_level(h, h->levels[l], X, ldb, nc, 0, 0, 0, nc, s));
  }
  return BGP_OK;
}

// The collective tail of a sharded compute(): all-gather of the locally solved rows of the top-level factor panel (the
// ONE data-path collective of compute(), SURVEY.md §8e), Gram / LU / log-det / update of the nodes above the shard cut
// (every rank does all of them: they are tiny), then the log-determinant: owned leaves + owned nodes, the top nodes
// counted once (by shard 0), the partial sums added over the ranks on the device (one double).
static int hodlr_finish_sharded(bgp_hodlr* h) {
  cudaStream_t s = h->sA;
  BGP_TRY(exchange_rows(h, h->top.U.p, h->n, h->top.ucols, s));
  const int cut = std::min(h->cut_depth, (int)h->levels.size());
  for (int l = cut - 1; l >= 0; --l) {
    const LevelInfo& L = h->levels[l];
    BGP_TRY(launch_level(h, L, h->top.U.p, h->n, L.ucol + L.r, L.ucol, 1, 0, L.ucol, s));
  }
  double ld = 0.0;
  BGP_TRY(sum_log_det(h, s, &ld));
  BGP_CUDA(cudaMemcpyAsync(h->d_scalar.p, &ld, sizeof(double), cudaMemcpyHostToDevice, s));
  BGP_TRY(comm_allreduce_sum_f64(h->d_scalar.p, 1, s));
  BGP_CUDA(cudaMemcpyAsync(&ld, h->d_scalar.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  h->log_det = ld;
  h->computed = true;
  record_compute_timing(h);
  return BGP_OK;
}

extern "C" {

void bgp_hodlr_default_opts(bgp_hodlr_opts_t* o) {
  o->min_size = 100; o->seed = 42; o->tol = 0.1;  // _hodlr.cpp:202
  o->rng_mode = BGP_RNG_REFERENCE;  // at the default tol the answer depends on the pivots: reproduce the reference's order
  o->rank_capacity = 0; o->shard_rank = 0; o->shard_count = 1; o->exhaust_mode = BGP_EXHAUST_DENSE;
}

int bgp_hodlr_create(bgp_hodlr_t** out) {
  *out = new (std::nothrow) bgp_hodlr();
  if (!*out) { set_error("out of host memory"); return BGP_ERR_NOMEM; }
  bgp_hodlr_default_opts(&(*out)->opts);
  return BGP_OK;
}

void bgp_hodlr_destroy(bgp_hodlr_t* h) {
  if (!h) return;
  delete h;
}

int bgp_hodlr_compute_dev(bgp_hodlr_t* h, const bgp_kernel_spec_t* spec, const double* x_dev, int64_t n, int32_t ndim,
                          const double* yerr_dev, const bgp_hodlr_opts_t* opts) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  return hodlr_compute_dev_impl(h, spec, x_dev, n, ndim, yerr_dev, opts);
}

int bgp_hodlr_compute(bgp_hodlr_t* h, const bgp_kernel_spec_t* spec, const double* x, int64_t n, int32_t ndim,
                      const double* yerr, const bgp_hodlr_opts_t* opts) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  h->computed = false;
  BGP_TRY(require_device());
  BGP_TRY(ensure_streams(h));
  if (n <= 0 || ndim <= 0) { set_error("invalid input shape (%lld, %d)", (long long)n, ndim); return BGP_ERR_INVALID; }
  BGP_TRY(h->d_x.reserve((size_t)n * ndim, h->sA));
  BGP_TRY(h->d_yerr.reserve((size_t)n, h->sA));
  BGP_CUDA(cudaMemcpyAsync(h->d_x.p, x, sizeof(double) * n * ndim, cudaMemcpyHostToDevice, h->sA));
  BGP_CUDA(cudaMemcpyAsync(h->d_yerr.p, yerr, sizeof(double) * n, cudaMemcpyHostToDevice, h->sA));
  return hodlr_compute_dev_impl(h, spec, h->d_x.p, n, ndim, h->d_yerr.p, opts);
}

int bgp_hodlr_computed(const bgp_hodlr_t* h) { return h && h->computed ? 1 : 0; }

int bgp_hodlr_log_determinant(const bgp_hodlr_t* h, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  *out = h->log_det;
  return BGP_OK;
}

int bgp_hodlr_apply_inverse(bgp_hodlr_t* h, double* b, int64_t nrhs, int64_t ldb) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  if (nrhs <= 0) return BGP_OK;
  if (ldb < h->n) { set_error("dimension mismatch: ldb < n"); return BGP_ERR_DIM; }
  cudaStream_t s = h->sA;
  const int64_t n = h->n;
  // process in slabs of columns to bound device memory
  const int64_t slab = std::max<int64_t>(1, std::min<int64_t>(nrhs, (int64_t)(1ull << 28) / n));
  BGP_TRY(h->d_rhs.reserve((size_t)n * slab, s));
  for (int64_t c0 = 0; c0 < nrhs; c0 += slab) {
    const int64_t nc = std::min(slab, nrhs - c0);
    BGP_CUDA(cudaMemcpy2DAsync(h->d_rhs.p, sizeof(double) * n, b + c0 * ldb, sizeof(double) * ldb, sizeof(double) * n, nc, cudaMemcpyHostToDevice, s));
    BGP_CUDA(cudaEventRecord(h->ev[4], s));
    BGP_TRY(hodlr_solve_dev(h, h->d_rhs.p, nc, n, s, false));
    BGP_CUDA(cudaEventRecord(h->ev[5], s));
    BGP_CUDA(cudaMemcpy2DAsync(b + c0 * ldb, sizeof(double) * ldb, h->d_rhs.p, sizeof(double) * n, sizeof(double) * n, nc, cudaMemcpyDeviceToHost, s));
    BGP_CUDA(cudaStreamSynchronize(s));
  }
  float ms = 0; cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]); h->t_ms[4] = ms;
  return BGP_OK;
}

int bgp_hodlr_dot_solve_dev(bgp_hodlr_t* h, const double* y_dev, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  cudaStream_t s = h->sA;
  const int64_t n = h->n;
  BGP_TRY(h->d_rhs.reserve((size_t)n, s));
  BGP_CUDA(cudaEventRecord(h->ev[4], s));
  BGP_CUDA(cudaMemcpyAsync(h->d_rhs.p, y_dev, sizeof(double) * n, cudaMemcpyDeviceToDevice, s));
  BGP_TRY(hodlr_solve_dev(h, h->d_rhs.p, 1, n, s, false));
  BGP_CUDA(cudaMemsetAsync(h->d_scalar.p, 0, sizeof(double), s));
  dot_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 592), 256, 0, s>>>(y_dev, h->d_rhs.p, n, h->d_scalar.p);
  BGP_LAUNCH_CHECK();
  BGP_CUDA(cudaEventRecord(h->ev[5], s));
  BGP_CUDA(cudaMemcpyAsync(out, h->d_scalar.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  float ms = 0; cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]); h->t_ms[4] = ms;
  return BGP_OK;
}

int bgp_hodlr_dot_solve(bgp_hodlr_t* h, const double* y, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  cudaStream_t s = h->sA;
  BGP_TRY(h->d_yerr.reserve((size_t)h->n, s));  // reuse as staging for y
  BGP_CUDA(cudaMemcpyAsync(h->d_yerr.p, y, sizeof(double) * h->n, cudaMemcpyHostToDevice, s));
  return bgp_hodlr_dot_solve_dev(h, h->d_yerr.p, out);
}

int bgp_hodlr_get_inverse(bgp_hodlr_t* h, double* out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  const int64_t n = h->n;
  for (int64_t j = 0; j < n; ++j) {
    double* c = out + j * n;
    memset(c, 0, sizeof(double) * n);
    c[j] = 1.0;
  }
  return bgp_hodlr_apply_inverse(h, out, n, n);  // COLUMN-major K^-1 (symmetric only to tol: the host transposes)
}

// alpha = K^-1 r, g_p = sum_ij (alpha alpha^T - K^-1)_ij dK_ij/dtheta_p, diag(alpha alpha^T - K^-1): everything
// GP.grad_log_likelihood (gp.py:406-468) needs from the solver, with K^-1 (solve against the identity, _hodlr.cpp:193-199)
// and the gradient contraction staying on the device.
int bgp_hodlr_grad_terms(bgp_hodlr_t* h, const uint32_t* which, const double* r, double* alpha_out, double* g_out,
                         double* diag_out) {
  if (!h || !h->computed) { set_error("the solver has not been computed"); return BGP_ERR_NOT_COMPUTED; }
  if (h->opts.shard_count > 1) { set_error("grad_terms is not available on a sharded factorisation"); return BGP_ERR_INVALID; }
  const int64_t n = h->n;
  const int np = h->prog.n_params_total;
  if (np > 64) { set_error("gradient supports at most 64 hyper-parameters"); return BGP_ERR_INVALID; }
  cudaStream_t s = h->sA;
  BGP_TRY(h->d_rhs.reserve((size_t)n * 2 + 64, s));
  double* alpha = h->d_rhs.p;
  double* dg = h->d_rhs.p + n;
  double* ddiag = h->d_rhs.p + n + 64;
  BGP_CUDA(cudaMemcpyAsync(alpha, r, sizeof(double) * n, cudaMemcpyHostToDevice, s));
  BGP_TRY(hodlr_solve_dev(h, alpha, 1, n, s, false));
  if (alpha_out) BGP_CUDA(cudaMemcpyAsync(alpha_out, alpha, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  BGP_TRY(h->d_inv.reserve((size_t)n * n, s));
  BGP_TRY(fill_identity_launch(h->d_inv.p, n, s));
  BGP_TRY(hodlr_solve_dev(h, h->d_inv.p, n, n, s, false));
  BGP_TRY(h->d_which.reserve(std::max(np, 1), s));
  if (np) BGP_CUDA(cudaMemcpyAsync(h->d_which.p, which, sizeof(unsigned) * np, cudaMemcpyHostToDevice, s));
  BGP_TRY(kmat_grad_contract_launch(h->d_prog.p, h->ndim, np, h->d_which.p, h->d_x.p, n, h->d_inv.p, n, alpha, 1.0, -1.0, dg,
                                    diag_out ? ddiag : nullptr, h->d_gscratch, s));
  if (np && g_out) BGP_CUDA(cudaMemcpyAsync(g_out, dg, sizeof(double) * np, cudaMemcpyDeviceToHost, s));
  if (diag_out) BGP_CUDA(cudaMemcpyAsync(diag_out, ddiag, sizeof(double) * n, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_hodlr_num_nodes(const bgp_hodlr_t* h, int64_t* out) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  *out = (int64_t)h->nodes.size();
  return BGP_OK;
}

int bgp_hodlr_node_info(const bgp_hodlr_t* h, bgp_hodlr_node_info_t* out) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  for (size_t i = 0; i < h->nodes.size(); ++i) {
    const HNode& nd = h->nodes[i];
    out[i].start = nd.start; out[i].size = nd.size; out[i].half = nd.half; out[i].is_leaf = nd.is_leaf;
    out[i].parent = nd.parent; out[i].direction = nd.dir; out[i].depth = nd.depth; out[i].rank = nd.rank;
    out[i].rng_draws = nd.draws; out[i].dense_fallback = nd.fallback;
  }
  return BGP_OK;
}

int bgp_hodlr_node_pivots(const bgp_hodlr_t* hc, int64_t node, int32_t* rows, int32_t* cols) {
  bgp_hodlr_t* h = const_cast<bgp_hodlr_t*>(hc);
  if (!h || node < 0 || node >= (int64_t)h->nodes.size()) { set_error("node index out of range"); return BGP_ERR_INDEX; }
  const HNode& nd = h->nodes[node];
  // dense fallback nodes (exhaust_mode = dense) have no pivot list: their factors are the identity / the block itself
  if (nd.is_leaf || h->piv_off[node] < 0 || nd.rank == 0 ||
      (nd.fallback && h->opts.exhaust_mode == BGP_EXHAUST_DENSE))
    return BGP_OK;
  BGP_CUDA(cudaMemcpy(rows, h->d_piv_rows.p + h->piv_off[node], sizeof(int) * nd.rank, cudaMemcpyDeviceToHost));
  BGP_CUDA(cudaMemcpy(cols, h->d_piv_cols.p + h->piv_off[node], sizeof(int) * nd.rank, cudaMemcpyDeviceToHost));
  return BGP_OK;
}

int bgp_hodlr_last_timing(const bgp_hodlr_t* h, double* ms5) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  for (int i = 0; i < 5; ++i) ms5[i] = h->t_ms[i];
  return BGP_OK;
}
int bgp_hodlr_set_profiling(bgp_hodlr_t* h, int on) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  h->profile = on != 0;
  return BGP_OK;
}
int bgp_hodlr_last_aca_profile(const bgp_hodlr_t* h, double* p12) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  for (int i = 0; i < 12; ++i) p12[i] = h->prof[i];
  return BGP_OK;
}
int bgp_hodlr_last_work(const bgp_hodlr_t* h, double* w6) {
  if (!h) { set_error("null handle"); return BGP_ERR_INVALID; }
  for (int i = 0; i < 6; ++i) w6[i] = h->work[i];
  return BGP_OK;
}

// ---- diagnostics: the dense building blocks of the big-rank path, callable on their own (tests/test_gpu_linalg.py) ----
int bgp_selftest_lu(int32_t n, int32_t nrhs, const double* S_host, double* R_host, double* logdet) {
  BGP_TRY(require_device());
  if (n <= 0 || nrhs < 0) { set_error("bgp_selftest_lu: bad sizes"); return BGP_ERR_INVALID; }
  cudaStream_t s = 0;
  DevBuf<double> dS, dR, dld;
  LuWorkspace ws;
  BGP_TRY(dS.alloc((size_t)n * n + n, s));
  BGP_TRY(dR.alloc(std::max<size_t>((size_t)n * nrhs, 1), s));
  BGP_TRY(dld.alloc(1, s));
  BGP_CUDA(cudaMemcpyAsync(dS.p, S_host, sizeof(double) * n * n, cudaMemcpyHostToDevice, s));
  if (nrhs) BGP_CUDA(cudaMemcpyAsync(dR.p, R_host, sizeof(double) * n * nrhs, cudaMemcpyHostToDevice, s));
  std::vector<LuNode> nodes(1);
  nodes[0].S = dS.p; nodes[0].piv = reinterpret_cast<int*>(dS.p + (size_t)n * n); nodes[0].logdet = dld.p;
  BGP_TRY(lu_factor_batch(ws, nodes, n, s));
  BGP_TRY(lu_solve_batch(ws, nodes, n, dR.p, 0, n, nrhs, false, s));
  if (nrhs) BGP_CUDA(cudaMemcpyAsync(R_host, dR.p, sizeof(double) * n * nrhs, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaMemcpyAsync(logdet, dld.p, sizeof(double), cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

int bgp_selftest_gemm(int32_t a_kcontig, int32_t b_kcontig, int32_t m, int32_t n, int32_t k, const double* A_host,
                      int64_t lda, const double* B_host, int64_t ldb, double* C_host, int64_t ldc, int32_t atomic_add) {
  BGP_TRY(require_device());
  if (m <= 0 || n <= 0 || k <= 0) { set_error("bgp_selftest_gemm: bad sizes"); return BGP_ERR_INVALID; }
  cudaStream_t s = 0;
  const size_t na = (size_t)(a_kcontig ? m : k) * lda, nb = (size_t)(b_kcontig ? n : k) * ldb, nc = (size_t)n * ldc;
  DevBuf<double> dA, dB, dC;
  DevBuf<GemmDesc> dd;
  BGP_TRY(dA.alloc(na, s)); BGP_TRY(dB.alloc(nb, s)); BGP_TRY(dC.alloc(nc, s)); BGP_TRY(dd.alloc(1, s));
  BGP_CUDA(cudaMemcpyAsync(dA.p, A_host, sizeof(double) * na, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(dB.p, B_host, sizeof(double) * nb, cudaMemcpyHostToDevice, s));
  BGP_CUDA(cudaMemcpyAsync(dC.p, C_host, sizeof(double) * nc, cudaMemcpyHostToDevice, s));
  GemmDesc g;
  g.A = dA.p; g.B = dB.p; g.C = dC.p; g.M = m; g.N = n; g.K = k; g.mode = atomic_add ? GD_ATOMIC_ADD : GD_SUB;
  g.lda = lda; g.ldb = ldb; g.ldc = ldc;
  BGP_CUDA(cudaMemcpyAsync(dd.p, &g, sizeof(g), cudaMemcpyHostToDevice, s));
  if (a_kcontig && b_kcontig) BGP_TRY((gemm_dmma_launch<true, true>(dd.p, 1, m, n, nullptr, s)));
  else if (!a_kcontig && b_kcontig) BGP_TRY((gemm_dmma_launch<false, true>(dd.p, 1, m, n, nullptr, s)));
  else { set_error("bgp_selftest_gemm: only the (A K-contiguous | M-contiguous) x (B K-contiguous) variants are built here"); return BGP_ERR_INVALID; }
  BGP_CUDA(cudaMemcpyAsync(C_host, dC.p, sizeof(double) * nc, cudaMemcpyDeviceToHost, s));
  BGP_CUDA(cudaStreamSynchronize(s));
  return BGP_OK;
}

}  // extern "C"

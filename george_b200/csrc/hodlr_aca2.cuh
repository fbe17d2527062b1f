// hodlr_aca2.cuh — K5, GPU-wide version: every internal node's ACA advances in lock-step and each step's work is spread
// over the whole chip as (node, chunk-of-1024-columns/rows) items.
//
// Same algorithm as hodlr.h:136-221 (and as aca_kernel in hodlr_kernels.cuh, which is kept for the chained
// rng_mode = reference): random row -> residual -> arg-max pivot -> retry while |pivot| < 1e-14 -> column residual ->
// stopping rule.  What changes is the schedule:
//   * while a node looks for a usable pivot row, the factors do not change, so the next B candidate rows of its RNG
//     sequence are evaluated SPECULATIVELY in one launch; the first candidate (in sequence order) with
//     max|residual| >= 1e-14 wins and the RNG / row-index list are committed up to exactly that draw — bit-identical
//     to the one-at-a-time loop.  B doubles after a fully rejected batch.  Kernels that are exactly low rank
//     (Matern-3/2 in 1-D) reject EVERY row of most nodes; this turns that O(n_rows * n_cols) scan into a dense,
//     perfectly parallel evaluation instead of n_rows dependent steps.
//   * one iteration = 6 small launches shared by all nodes:
//       eval (persistent CTAs over a work list of (column chunk, candidate block) items; only per-candidate maxima
//       leave the kernel, through atomicMax) -> decide (first usable candidate; RNG / row list committed to that draw)
//       -> vrow (winning row's residual + chunk arg-max) -> pivot -> vnorm || ucol (one launch) -> finish (stopping
//       rule, next candidates).  The host reads one "active nodes" counter every 8 iterations.
//   * sharded runs: every rank scans the nodes above the cut itself.  With bound culling and one-candidate batches the
//     scans are cheap, and a collective inside the lock-step loop would put a latency on every step.
#pragma once

#include "hodlr_kernels.cuh"

namespace bgp {

constexpr int A2_CHUNK = 1024;    // rows / columns per work item
constexpr int A2_THREADS = 256;
constexpr int A2_NODE_THREADS = 1024;  // per-node kernels (init / decide / finish): one CTA per node whose work is a chain
                                       // of short, latency-bound phases over up to A2_BMAX candidates — more threads per phase
constexpr int A2_EPT = A2_CHUNK / A2_THREADS;  // elements per thread
constexpr int A2_CG = 4;          // candidates evaluated together (register blocking)
constexpr int A2_ITEM_CB = 8;      // candidate blocks (of A2_CG rows) per eval work item
constexpr int A2_BMAX = 8192;     // max speculative candidates per iteration (bounded by the per-node CTA's shared memory)
constexpr int A2_BGROW = 8;       // batch growth after a fully rejected batch: 4, 32, 256, 2048, 8192
constexpr int A2_NSUB = 4;        // the residual kernels (vrow / ucol / vnorm) split a chunk into sub-chunks of A2_THREADS
constexpr int A2_GROUP = A2_CHUNK / (A2_THREADS / 32);  // 128 columns: what one warp of a2_eval sweeps (bound granularity)
constexpr int A2_NGROUP = A2_CHUNK / A2_GROUP;           // 8 groups per chunk
static_assert(A2_NSUB * A2_THREADS == A2_CHUNK, "sub-chunks tile a chunk");
constexpr int A2_HASH = 16384;    // open-addressing slots of the swap-pop multimap (>= 2 * A2_BMAX)
static_assert(A2_BMAX <= 65536, "multimap values are 16-bit draw numbers");
constexpr int A2_XWORDS = 64;     // room for the extra words consumed by Lemire rejections inside one batch

struct A2Node {  // static description
  int row0, n_rows, col0, n_cols;
  int vcol, cap, pre_id, node;
  int cchunk0, n_cchunks, rchunk0, n_rchunks;
  int bmax;
  int64_t idx_off, piv_off, cand_off;
  double* vbase;   // column 0 of this node's level in ITS factor panel, addressed by GLOBAL row index: the panel of a level
                   // owned by one shard holds only that shard's rows (leading dimension ld = rows of the shard) and vbase
                   // points row0_shard entries before its allocation; levels above the shard cut span all N rows
  int64_t ld;
};

struct A2State {  // dynamic
  int rank, draws, n_index, fallback, status, active;
  int phase;  // 0 = candidates pending evaluation, 1 = pivot accepted (vnorm/ucol run), 2 = done
  int B, ncand, piv_i, piv_j;
  int end_words;  // mt19937 words drawn for the pending batch (a.rngs[2*node+1] is the stream after exactly that many)
  int deferred;   // the pending batch is ONE live candidate whose acceptance test is left to a2_vrow / a2_pivot
  double pivot, norm;
};

struct A2EPart {
  double val;  // signed residual entry of largest magnitude in (candidate, chunk)
  int idx;     // its column (block-relative), lowest on ties
  int _pad;
};

enum { A2_SELECT = 0, A2_ACCEPT = 1, A2_DONE = 2, A2_LATE_REJECT = 3 };
// A2_LATE_REJECT: a one-candidate batch is not evaluated by a2_eval at all — a2_vrow computes that row anyway when it is
// accepted, and its arg-max IS the acceptance test (hodlr.h:191); a2_pivot turns the provisional accept into a reject when
// |pivot| < 1e-14 and a2_finish draws the next batch.  One pass over the factor panel less per step for kernels whose rows
// are all usable (the high-rank regime, where a step is bound by exactly those passes).

// cooperative 625-word copy of an mt19937 state (all threads of the CTA; caller synchronises)
__device__ __forceinline__ void mt_copy(MT19937* dst, const MT19937* src) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  for (int i = threadIdx.x; i < (int)(sizeof(MT19937) / 4); i += blockDim.x) d[i] = s[i];
}

// cooperative twist of the whole state: 3 dependent phases of <= 227 independent elements + the last word.  Element i
// needs the OLD mt[i + 1], which the neighbouring thread overwrites in the same phase: every phase computes into
// registers, synchronises, then stores.
__device__ __forceinline__ void mt_twist_coop(MT19937& g) {
  auto value = [&](uint32_t a, uint32_t b, uint32_t m) {
    const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return m ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
  };
  auto phase = [&](int lo, int hi, int moff) {  // elements [lo, hi), partner mt[i + moff]
    for (int base = lo; base < hi; base += blockDim.x) {  // (one trip for blockDim >= 227)
      const int i = base + threadIdx.x;
      uint32_t v = 0;
      if (i < hi) v = value(g.mt[i], g.mt[i + 1], g.mt[i + moff]);
      __syncthreads();
      if (i < hi) g.mt[i] = v;
      __syncthreads();
    }
  };
  phase(0, 227, 397);
  phase(227, 454, -227);
  phase(454, 623, -227);
  if (threadIdx.x == 0) { g.mt[623] = value(g.mt[623], g.mt[0], g.mt[396]); g.idx = 0; }
  __syncthreads();
}
__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= (y >> 11);
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= (y >> 18);
  return y;
}
// the next `n` tempered words of the stream into out[] (state advanced); all threads of the CTA
__device__ inline void mt_fill_coop(MT19937& g, uint32_t* out, int n) {
  int done = 0;
  __syncthreads();
  while (done < n) {
    if (g.idx >= 624) mt_twist_coop(g);
    const int idx = g.idx;
    const int take = min(n - done, 624 - idx);
    for (int t = threadIdx.x; t < take; t += blockDim.x) out[done + t] = mt_temper(g.mt[idx + t]);
    __syncthreads();
    if (threadIdx.x == 0) g.idx = idx + take;
    __syncthreads();
    done += take;
  }
}
// skip `n` words of the stream (state advanced); all threads of the CTA
__device__ inline void mt_skip_coop(MT19937& g, int n) {
  __syncthreads();
  while (n > 0) {
    if (g.idx >= 624) mt_twist_coop(g);
    const int idx = g.idx;
    const int take = min(n, 624 - idx);
    __syncthreads();
    if (threadIdx.x == 0) g.idx = idx + take;
    __syncthreads();
    n -= take;
  }
}

struct A2Args {
  const DevProgram* prog;
  const double* x;
  const A2Node* nodes;
  A2State* states;
  MT19937* rngs;   // [2 * node]: committed stream, [2 * node + 1]: stream after the whole pending batch
  int n_nodes;
  double tol;
  uint32_t seed;
  int exhaust_mode;
  int* idx_ws;
  int* piv_rows;
  int* piv_cols;
  int* cand;       // candidate rows          [cand_off + c]
  int* cand_k;     // drawn positions
  int* cand_words; // cumulative words
  int* cand_L;     // value the swap-pop of draw c writes to position cand_k[c] (the list entry that was last at that time)
  int* cand_next;  // next draw of the batch that writes the same position (0x7fffffff: none): commit rule of a2_decide
  int* cand_live;  // indices (into the batch) of the candidates that need evaluation, compacted; see a2_generate
  double* node_box;  // [2 * node]: min / max coordinate of the node's columns (1-D bound culling)
  unsigned long long* cmax;  // per candidate: bit pattern of max |residual| over all chunks (atomicMax)
  A2EPart* epart;  // one slot per column sub-chunk: arg-max of the winning row's residual there
  const int* cchunk_node;  // chunk -> node
  const int* rchunk_node;
  double* vpart;   // per column sub-chunk: [(chunk * A2_NSUB + sub) * (capmax + 1)] : vn2 then dots[k]
  double* upart;   // per row sub-chunk
  double* vmax;    // per (column chunk, 128-column group): max over the factors q and the group's columns j of |V(j, q)|
                   // [chunk * 8 + g]  (bound culling of a2_eval; nullptr when the program has no distance bound)
  double2* cand_xu;  // per candidate: (coordinate of its row, sum_q |U(row, q)|), written by a2_generate for a2_eval
  int capmax;
  int* n_active;
  int4* work;          // eval work items (chunk, first candidate, #candidates, node), two buffers of work_cap
  int* work_count;     // [2] item counters (buffer i%2 is consumed by iteration i and refilled for i+2)
  int* work_cursor;    // [2] next (item, group) unit of the buffer being consumed (a2_eval pulls work dynamically)
  int work_cap;
  int* iter_ptr;       // device counter: lock-step iteration number (selects the buffers); advanced by a2_tick_kernel
  unsigned long long* stats;  // [0] candidate-row entries verified (pairs), [1] residual-update FMAs executed, [2] candidates,
                              // [3] entries actually evaluated by a2_eval (the rest were bounded < 1e-14 without evaluation)
};

// shared-memory workspace of the per-node kernels (dynamic shared memory)
struct A2NodeSmem {
  MT19937 rng;
  int k[A2_BMAX];       // drawn positions
  int ol[A2_BMAX];      // index[n_index-1-c] before this batch
  int hkey[A2_HASH];    // multimap position -> draws that write it (one slot per draw)
  unsigned short hval[A2_HASH];
  uint32_t raw[A2_BMAX + A2_XWORDS]; // raw mt19937 words of the batch (+ the extra words of Lemire rejections); then
                                     // wl[c] = most recent earlier draw writing position last_c
  double red[32];
  int redi[32];
  int flag;
  int n_live;
  int extra;
};

__device__ __forceinline__ unsigned a2_hash(int pos) { return ((unsigned)pos * 2654435761u) & (A2_HASH - 1); }
// most recent draw before `c` that wrote position `pos` (-1: none)
__device__ __forceinline__ int a2_prev_writer(const A2NodeSmem& S, int pos, int c) {
  int best = -1;
  unsigned h = a2_hash(pos);
  while (true) {
    const int key = S.hkey[h];
    if (key == -1) break;
    if (key == pos) { const int v = S.hval[h]; if (v < c && v > best) best = v; }
    h = (h + 1) & (A2_HASH - 1);
  }
  return best;
}
// first draw after `c` that writes position `pos` (0x7fffffff: none)
__device__ __forceinline__ int a2_next_writer(const A2NodeSmem& S, int pos, int c) {
  int best = 0x7fffffff;
  unsigned h = a2_hash(pos);
  while (true) {
    const int key = S.hkey[h];
    if (key == -1) break;
    if (key == pos) { const int v = S.hval[h]; if (v > c && v < best) best = v; }
    h = (h + 1) & (A2_HASH - 1);
  }
  return best;
}

// upper bound of |k| at distance >= gap for the program's shape (+inf when the program has no decreasing bound)
__device__ __forceinline__ double program_bound(const DevProgram* g, double gap) {
  switch (g->shape) {
    case BGP_SHAPE_EXPSQ: return ScaledProfile1D<BGP_SHAPE_EXPSQ>(*g).bound(gap);
    case BGP_SHAPE_M32: return ScaledProfile1D<BGP_SHAPE_M32>(*g).bound(gap);
    case BGP_SHAPE_M52: return ScaledProfile1D<BGP_SHAPE_M52>(*g).bound(gap);
    case BGP_SHAPE_EXP: return ScaledProfile1D<BGP_SHAPE_EXP>(*g).bound(gap);
    case BGP_SHAPE_PROD_EXPSQ_ES2: return ScaledProfile1D<BGP_SHAPE_PROD_EXPSQ_ES2>(*g).bound(gap);
    case BGP_SHAPE_PROD_M32_ES2: return ScaledProfile1D<BGP_SHAPE_PROD_M32_ES2>(*g).bound(gap);
    default: return __longlong_as_double(0x7ff0000000000000ll);
  }
}

// Draw the next min(B, bmax, n_index) candidate rows speculatively: k_c = uniform(0, n_index-1-c) from `S.rng`
// (advanced), swap-pop on the index list (hodlr.h:179-183):  cand[c] = A[k_c];  A[k_c] = A[n_index-1-c].
// The positions depend on the RNG only, so the whole batch is resolved in parallel: a position's content at time c is
// the original list entry unless an earlier draw of the batch wrote it, and what a draw writes is the content of ITS
// "last" slot at ITS time — a chain towards earlier draws that is almost always empty (two draws of a batch touch the same
// slot with probability ~ B / n_index).  A shared-memory multimap position -> draws gives every thread the most recent
// earlier writer of the two slots it reads; chains are followed to their root.  The index list itself is NOT modified
// here: a2_decide commits exactly the draws that were consumed (L[c], next[c] below), so nothing has to be undone.
// cand[c] = row, cand_k[c] = position, words[c] = mt19937 words consumed up to and including draw c.
//
// Candidate-level bound culling (programs with a decreasing bound, 1-D): |residual(i, j)| <= bound(gap(x_i, node's
// columns)) + sum_q |U(i, q)| for EVERY column (|V| <= 1: rows are normalised by their largest entry, hodlr.h:194), so a
// candidate whose right-hand side is < 1e-14 is rejected without any evaluation; only the others ("live") get eval work.
__device__ inline void a2_generate(const A2Args& a, A2State& st, A2NodeSmem& S, const A2Node& nd, int nid, int nb) {
  int* __restrict__ index = a.idx_ws + nd.idx_off;
  int* __restrict__ cand = a.cand + nd.cand_off;
  int* __restrict__ cand_k = a.cand_k + nd.cand_off;
  int* __restrict__ words = a.cand_words + nd.cand_off;
  int* __restrict__ cand_L = a.cand_L + nd.cand_off;
  int* __restrict__ cand_next = a.cand_next + nd.cand_off;
  int* __restrict__ live = a.cand_live + nd.cand_off;
  unsigned long long* __restrict__ cmax = a.cmax + nd.cand_off;
  const int n_index = st.n_index;
  int B = min(min(st.B, nd.bmax), n_index);
  MT19937* rng_commit = a.rngs + 2 * (int64_t)nid;
  MT19937* rng_end = rng_commit + 1;
  // Lemire's multiply-shift (libstdc++ uniform_int_distribution) rejects a word with probability srange / 2^32 and then
  // takes the NEXT word of the stream for the same draw, which shifts every later draw by one word.  The batch is drawn
  // in parallel assuming no rejection; the first draw that rejects (if any) is redone one word at a time and the tail of
  // the batch is recomputed with the new offset.  Expected number of passes: 1 + B * n_index / 2^32.
  if (threadIdx.x == 0) { S.flag = 0x7fffffff; S.n_live = 0; S.extra = 0; }
  mt_fill_coop(S.rng, S.raw, B);
  int start = 0;
  bool truncated = false;
  while (true) {
    const int extra = S.extra;
    for (int c = start + threadIdx.x; c < B; c += blockDim.x) {
      const uint32_t srange = (uint32_t)(n_index - c);
      const uint64_t prod = (uint64_t)S.raw[c + extra] * (uint64_t)srange;
      const uint32_t low = (uint32_t)prod;
      if (low < srange && low < (0u - srange) % srange) atomicMin(&S.flag, c);
      S.k[c] = (int)(prod >> 32);
      words[c] = c + 1 + extra;
      cmax[c] = 0ull;
    }
    __syncthreads();
    const int c0 = S.flag;
    if (c0 == 0x7fffffff) break;
    __syncthreads();  // every thread has read S.flag before thread 0 rewrites it below
    // redo draw c0: words raw[c0 + extra + 1], ... until one is accepted (they were already generated for later draws)
    if (threadIdx.x == 0) {
      const uint32_t srange = (uint32_t)(n_index - c0);
      const uint32_t thr = (0u - srange) % srange;
      int e = extra;
      int kk = -1;
      while (e + 1 < A2_XWORDS && c0 + e + 1 < B + extra) {  // only words that exist; the rest follows below
        ++e;
        const uint64_t prod = (uint64_t)S.raw[c0 + e] * (uint64_t)srange;
        if ((uint32_t)prod >= thr) { kk = (int)(prod >> 32); break; }
      }
      if (kk >= 0) { S.k[c0] = kk; words[c0] = c0 + 1 + e; S.extra = e; S.flag = 0x7fffffff; }
      else S.flag = -1 - c0;  // ran out of generated words / budget: truncate the batch before this draw
    }
    __syncthreads();
    if (S.flag < 0) {  // (practically unreachable) keep the draws before c0; with none left, draw c0 alone, sequentially
      const int c0t = -1 - S.flag;
      __syncthreads();
      if (c0t > 0) { B = c0t; truncated = true; break; }
      mt_copy(&S.rng, rng_commit);
      __syncthreads();
      if (threadIdx.x == 0) { int w = 0; S.k[0] = mt_uniform(S.rng, (uint32_t)n_index, &w); words[0] = w; cmax[0] = 0ull; S.extra = -1; }
      __syncthreads();
      B = 1;
      break;
    }
    // the stream needs as many more words as the offset grew
    {
      const int grown = S.extra - extra;
      mt_fill_coop(S.rng, S.raw + B + extra, grown);
    }
    start = c0 + 1;
  }
  // S.rng is now the stream after the words of the whole batch (unless the batch was truncated): decide copies it
  // instead of replaying the twists when the whole batch is consumed
  __syncthreads();
  mt_copy(rng_end, &S.rng);
  if (threadIdx.x == 0) {
    st.ncand = B;
    st.end_words = (!truncated && S.extra >= 0 && B > 0 && words[B - 1] == B + S.extra) ? B + S.extra : -1;
  }
  for (int t = threadIdx.x; t < A2_HASH; t += blockDim.x) S.hkey[t] = -1;
  __syncthreads();
  for (int c = threadIdx.x; c < B; c += blockDim.x) {
    const int pos = S.k[c];
    S.ol[c] = index[n_index - 1 - c];
    unsigned h = a2_hash(pos);
    while (atomicCAS(&S.hkey[h], -1, pos) != -1) h = (h + 1) & (A2_HASH - 1);
    S.hval[h] = (unsigned short)c;
  }
  __syncthreads();
  int* wl = reinterpret_cast<int*>(S.raw);
  for (int c = threadIdx.x; c < B; c += blockDim.x) wl[c] = a2_prev_writer(S, n_index - 1 - c, c);
  __syncthreads();
  auto last_value = [&](int c) {  // content of slot n_index-1-c at time c
    int w = wl[c];
    while (w >= 0) { c = w; w = wl[c]; }
    return S.ol[c];
  };
  for (int c = threadIdx.x; c < B; c += blockDim.x) {
    const int pos = S.k[c];
    const int wk = a2_prev_writer(S, pos, c);
    const int row = (wk < 0) ? index[pos] : last_value(wk);  // (the list itself is untouched until a2_decide commits)
    cand[c] = row;
    cand_k[c] = pos;
    cand_L[c] = last_value(c);
    cand_next[c] = a2_next_writer(S, pos, c);
  }
  const bool cull = a.vmax != nullptr;
  const int rank = st.rank;
  if (!cull) {
    for (int c = threadIdx.x; c < B; c += blockDim.x) live[c] = c;
    if (threadIdx.x == 0) S.n_live = B;
  } else {
    const double clo = a.node_box[2 * nid], chi = a.node_box[2 * nid + 1];
    const double* Ucol = nd.vbase + nd.row0;
    const double* xr = a.x + nd.row0;
    constexpr int G = 4;  // candidates per trip: their (dependent, uncoalesced) loads are issued together
    for (int c0 = threadIdx.x; c0 < B; c0 += G * blockDim.x) {
      int row[G];
      double xi[G], b[G];
#pragma unroll
      for (int j = 0; j < G; ++j) { const int c = c0 + j * blockDim.x; row[j] = cand[(c < B) ? c : c0]; }  // written above by this thread
#pragma unroll
      for (int j = 0; j < G; ++j) xi[j] = xr[row[j]];
#pragma unroll
      for (int j = 0; j < G; ++j) b[j] = 0.0;
      for (int q = 0; q < rank; ++q) {
        double u[G];
#pragma unroll
        for (int j = 0; j < G; ++j) u[j] = __ldcg(Ucol + (int64_t)q * nd.ld + row[j]);
#pragma unroll
        for (int j = 0; j < G; ++j) b[j] += fabs(u[j]);
      }
#pragma unroll
      for (int j = 0; j < G; ++j) {
        const int c = c0 + j * blockDim.x;
        if (c < B) {
          const double bb = b[j] + program_bound(a.prog, fmax(0.0, fmax(clo - xi[j], xi[j] - chi)));
          if (!(bb * 1.000001 < 1e-14)) {  // NaN keeps the candidate
            live[atomicAdd(&S.n_live, 1)] = c;
            a.cand_xu[nd.cand_off + c] = make_double2(xi[j], b[j]);
          }
        }
      }
    }
  }
  __syncthreads();
  // publish the evaluation work of the NEXT eval launch: one item = (column chunk, up to A2_CG * A2_ITEM_CB live candidates)
  {
    int n_live = S.n_live;
    const bool defer = (B == 1 && n_live == 1);
    if (threadIdx.x == 0) st.deferred = defer ? 1 : 0;
    if (defer) n_live = 0;  // no eval work: see A2_LATE_REJECT
    // few live candidates: one block of A2_CG per item, so that the sweep has no sequential depth inside an item
    const int ipc = (n_live <= 256) ? A2_CG : A2_CG * A2_ITEM_CB;
    const int per_chunk = (n_live + ipc - 1) / ipc;
    const int n_items = nd.n_cchunks * per_chunk;
    int4* work_next = a.work + (int64_t)nb * a.work_cap;
    __syncthreads();
    if (threadIdx.x == 0) {
      S.flag = n_items ? atomicAdd(a.work_count + nb, n_items) : 0;
      if (S.flag + n_items > a.work_cap) st.status = 2;  // cannot happen (the host sizes the list for the worst case): fail loudly
    }
    __syncthreads();
    const int base = S.flag;
    for (int t = threadIdx.x; t < n_items; t += blockDim.x) {
      const int ci = t / per_chunk, pi = t % per_chunk;
      const int c0 = pi * ipc;
      if (base + t < a.work_cap) work_next[base + t] = make_int4(nd.cchunk0 + ci, c0, min(ipc, n_live - c0), nid);
    }
  }
  __syncthreads();
}

// ---- init: index list, RNG seed, first candidates -------------------------------------------------------------
__global__ void __launch_bounds__(A2_NODE_THREADS) a2_init_kernel(A2Args a) {
  extern __shared__ __align__(16) unsigned char a2_smem_raw[];
  A2NodeSmem& S = *reinterpret_cast<A2NodeSmem*>(a2_smem_raw);
  const int nid = blockIdx.x;
  const A2Node nd = a.nodes[nid];
  A2State& st = a.states[nid];
  int* index = a.idx_ws + nd.idx_off;
  for (int n = threadIdx.x; n < nd.n_rows; n += blockDim.x) index[n] = n;
  if (threadIdx.x == 0) {
    mt_seed(S.rng, node_seed(a.seed, nd.pre_id));
    st.rank = 0; st.draws = 0; st.n_index = nd.n_rows; st.fallback = 0; st.status = 0; st.active = 1;
    st.phase = A2_SELECT; st.B = 4; st.norm = 0.0; st.pivot = 0.0; st.piv_i = 0; st.piv_j = 0; st.ncand = 0;
  }
  __syncthreads();
  mt_copy(a.rngs + 2 * (int64_t)nid, &S.rng);  // committed = state before the speculative draws
  __syncthreads();
  if (nd.cap <= 0) {
    if (threadIdx.x == 0) { st.status = 1; st.phase = A2_DONE; st.active = 0; atomicSub(a.n_active, 1); }
    return;
  }
  // bounding interval of the node's columns (candidate-level bound culling; 1-D programs with a distance bound only)
  if (a.vmax) {
    double lo = __longlong_as_double(0x7ff0000000000000ll), hi = -lo;
    for (int n = threadIdx.x; n < nd.n_cols; n += blockDim.x) { const double xv = a.x[nd.col0 + n]; lo = fmin(lo, xv); hi = fmax(hi, xv); }
    lo = -block_max_signed(-lo, S.red);
    hi = block_max_signed(hi, S.red);
    if (threadIdx.x == 0) { a.node_box[2 * nid] = lo; a.node_box[2 * nid + 1] = hi; }
    __syncthreads();
  }
  a2_generate(a, st, S, nd, nid, 0);
}

// ---- eval: residual maxima of the pending candidate rows ------------------------------------------------------
// Warp-autonomous: each warp owns 128 columns of the chunk (4 per lane, coalesced) and walks the candidate rows in
// blocks of A2_CG with no block-level synchronisation and no shared memory: the candidate's coordinates and its U row
// are warp-uniform (broadcast) loads, the arg-max is a shuffle reduction and one atomicMax per (candidate, warp).
//
// Bound culling (CULL; 1-D inputs, programs whose |k| has a decreasing bound in the distance).  The only consumer of the
// maxima is the test  max_j |residual(i, j)| >= 1e-14  (hodlr.h:191).  For a candidate row i and this warp's 128 columns
//     |residual(i, j)| <= |k(x_i, x_j)| + sum_q |U(i, q)| |V(j, q)| <= bound(gap(x_i, group)) + (sum_q |U(i, q)|) vmax(group)
// and when the right-hand side (with a 1e-6 relative margin for the rounding of both sides) is below 1e-14 the group
// cannot change the outcome of that test, so it is not evaluated.  Lane c works out the bound of candidate c; the warp
// then sweeps only the surviving candidates.  The decisions — hence pivots, ranks and RNG draws — are exactly those of
// the exhaustive scan; what disappears is the O(rows x cols) evaluation of entries that are provably negligible
// (Matern / squared-exponential tails: everything farther than a few dozen length scales from the block's corner).
template <class KFn, bool CULL>
__device__ __forceinline__ void a2_eval_body(const A2Args& a, const A2Node& nd, int rank, int chunk, int c_first,
                                             int c_count, int ndim, KFn fn, int warp, unsigned long long& n_eval,
                                             unsigned long long& n_fma) {
  const int lc = chunk - nd.cchunk0;
  const int lane = threadIdx.x & 31;
  const int w_lo = lc * A2_CHUNK + warp * A2_GROUP;  // first column of this warp
  const int w_n = min(A2_GROUP, nd.n_cols - w_lo);
  if (w_n <= 0) return;
  const double* Vcols = nd.vbase;
  const double* xr = a.x + (int64_t)nd.row0 * ndim;
  const double* xc = a.x + (int64_t)(nd.col0 + w_lo) * ndim;
  const int* cand = a.cand + nd.cand_off;
  const int* live_list = a.cand_live + nd.cand_off;
  unsigned long long* cmax = a.cmax + nd.cand_off;
  int ncol[A2_EPT];
#pragma unroll
  for (int e = 0; e < A2_EPT; ++e) ncol[e] = min(lane + 32 * e, w_n - 1);  // clamped (masked in the arg-max)

  double glo = 0.0, ghi = 0.0;
  const double* vmaxg = nullptr;
  const bool cull = CULL && a.vmax != nullptr;  // runtime switch: BGP_NO_CULL runs the exhaustive scan
  double vg = 0.0;
  if constexpr (CULL) if (cull) {
    glo = __longlong_as_double(0x7ff0000000000000ll); ghi = -glo;
#pragma unroll
    for (int e = 0; e < A2_EPT; ++e) { const double xv = xc[ncol[e]]; glo = fmin(glo, xv); ghi = fmax(ghi, xv); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      glo = fmin(glo, __shfl_xor_sync(0xffffffffu, glo, o));
      ghi = fmax(ghi, __shfl_xor_sync(0xffffffffu, ghi, o));
    }
    vmaxg = a.vmax + ((int64_t)chunk * A2_NGROUP + warp);
    vg = __ldcg(vmaxg);
  }

  const int ncand = c_first + c_count;
  for (int cb0 = c_first; cb0 < ncand; cb0 += 32) {
    const bool valid = cb0 + lane < ncand;
    const int myc = valid ? live_list[cb0 + lane] : 0;  // index of the candidate in the node's batch
    const int myrow = valid ? cand[myc] : 0;
    unsigned live = __ballot_sync(0xffffffffu, valid);
    if constexpr (CULL) if (cull) {
      bool keep = valid;
      if (valid) {
        const double2 xu = __ldcg(a.cand_xu + nd.cand_off + myc);  // (x_i, sum_q |U(i, q)|) from a2_generate
        const double gap = fmax(0.0, fmax(glo - xu.x, xu.x - ghi));
        const double b = fn.bound(gap) + xu.y * vg;
        keep = !(b * 1.000001 < 1e-14);  // NaN keeps the candidate
      }
      live = __ballot_sync(0xffffffffu, keep);
    }
    n_eval += (unsigned long long)__popc(live) * (unsigned long long)w_n;
    n_fma += (unsigned long long)__popc(live) * (unsigned long long)w_n * (unsigned long long)rank;
    while (live) {
      int sel[A2_CG], row[A2_CG], cidx[A2_CG];
      int ncb = 0;
#pragma unroll
      for (int c = 0; c < A2_CG; ++c) {
        if (live) { sel[c] = __ffs(live) - 1; live &= live - 1; ncb = c + 1; }
        else sel[c] = sel[0];
        row[c] = __shfl_sync(0xffffffffu, myrow, sel[c]);
        cidx[c] = __shfl_sync(0xffffffffu, myc, sel[c]);
      }
      double vals[A2_CG][A2_EPT];
#pragma unroll
      for (int e = 0; e < A2_EPT; ++e) {
        const double* x2 = xc + (int64_t)ncol[e] * ndim;
#pragma unroll
        for (int c = 0; c < A2_CG; ++c) vals[c][e] = fn(xr + (int64_t)row[c] * ndim, x2);
      }
      int k = 0;
      for (; k + 2 <= rank; k += 2) {  // two factor columns per trip: the loads of the second overlap the FMAs of the first
        const double* vc0 = Vcols + (int64_t)k * nd.ld;
        const double* vc1 = vc0 + nd.ld;
        double vk0[A2_EPT], vk1[A2_EPT], u0[A2_CG], u1[A2_CG];
#pragma unroll
        for (int c = 0; c < A2_CG; ++c) { u0[c] = __ldcg(vc0 + nd.row0 + row[c]); u1[c] = __ldcg(vc1 + nd.row0 + row[c]); }
#pragma unroll
        for (int e = 0; e < A2_EPT; ++e) { vk0[e] = vc0[nd.col0 + w_lo + ncol[e]]; vk1[e] = vc1[nd.col0 + w_lo + ncol[e]]; }
#pragma unroll
        for (int c = 0; c < A2_CG; ++c)
#pragma unroll
          for (int e = 0; e < A2_EPT; ++e) { vals[c][e] -= u0[c] * vk0[e]; vals[c][e] -= u1[c] * vk1[e]; }
      }
      for (; k < rank; ++k) {
        const double* vcol = Vcols + (int64_t)k * nd.ld;
        double vk[A2_EPT], u[A2_CG];
#pragma unroll
        for (int c = 0; c < A2_CG; ++c) u[c] = __ldcg(vcol + nd.row0 + row[c]);
#pragma unroll
        for (int e = 0; e < A2_EPT; ++e) vk[e] = vcol[nd.col0 + w_lo + ncol[e]];
#pragma unroll
        for (int c = 0; c < A2_CG; ++c)
#pragma unroll
          for (int e = 0; e < A2_EPT; ++e) vals[c][e] -= u[c] * vk[e];
      }
#pragma unroll
      for (int c = 0; c < A2_CG; ++c) {
        double best = 0.0;
        bool isnan_any = false;
#pragma unroll
        for (int e = 0; e < A2_EPT; ++e) {
          const double av = fabs(vals[c][e]);
          if (lane + 32 * e < w_n) { best = fmax(best, av); isnan_any |= (av != av); }
        }
        if (isnan_any) best = __longlong_as_double(0x7ff8000000000000ll);
        unsigned long long bits = (unsigned long long)__double_as_longlong(best);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const unsigned long long ob = __shfl_xor_sync(0xffffffffu, bits, o);
          bits = ob > bits ? ob : bits;
        }
        if (lane == 0 && c < ncb && bits != 0ull) atomicMax(cmax + cidx[c], bits);
      }
    }
  }
}

// one instantiation per program shape: the specialised ones carry no interpreter and need far fewer registers.
// Register allocation for 3 CTAs per SM on the specialised shapes (80 registers and a few spilled temporaries of the
// software exp / sqrt chains, but 24 instead of 16 warps per SM to hide their latency), 2 on the interpreter (128, no spills)
template <int SHAPE>
__global__ void __launch_bounds__(A2_THREADS, SHAPE == BGP_SHAPE_GENERIC ? 2 : 3) a2_eval_kernel(A2Args a) {
  __shared__ DevProgram P;
  // persistent CTAs sweep the work list published by the node kernels of the previous step: perfectly balanced over
  // the chip whatever mix of nodes is still active, and no empty CTAs
  const int buf = *a.iter_ptr & 1;
  const int n_items = min(a.work_count[buf], a.work_cap);
  const int4* items = a.work + (int64_t)buf * a.work_cap;
  if (blockIdx.x == 0 && threadIdx.x == 0) a.work_count[buf ^ 1] = 0;  // refilled by decide / finish of this iteration
  if constexpr (SHAPE == BGP_SHAPE_GENERIC) {
    stage_program(&P, a.prog);
    __syncthreads();
  }
  const auto fn = ShapeEval<SHAPE>::make(&P, a.prog);
  constexpr bool CULL = shape_has_bound(SHAPE);
  unsigned long long n_eval = 0ull, n_fma = 0ull;
  // work unit = (item, 128-column group); every WARP pulls its next unit from a global cursor: items differ wildly in cost
  // (fully culled ... 32 candidate rows to evaluate), a static deal leaves most of the chip idle behind the few heavy ones
  int* cursor = a.work_cursor + buf;
  if (blockIdx.x == 0 && threadIdx.x == 0) a.work_cursor[buf ^ 1] = 0;
  const int n_units = n_items * A2_NGROUP;
  while (true) {
    int u = 0;
    if ((threadIdx.x & 31) == 0) u = atomicAdd(cursor, 1);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= n_units) break;
    const int4 w = items[u / A2_NGROUP];
    const int grp = u % A2_NGROUP;
    const A2Node& nd = a.nodes[w.w];
    const int rank = a.states[w.w].rank;
    if constexpr (SHAPE == BGP_SHAPE_GENERIC) a2_eval_body<decltype(fn), false>(a, nd, rank, w.x, w.y, w.z, P.ndim, fn, grp, n_eval, n_fma);
    else a2_eval_body<decltype(fn), CULL>(a, nd, rank, w.x, w.y, w.z, 1, fn, grp, n_eval, n_fma);
  }
  if ((threadIdx.x & 31) == 0 && n_eval) { atomicAdd(a.stats + 3, n_eval); atomicAdd(a.stats + 1, n_fma); }
}
inline void a2_eval_launch(int shape, dim3 grid, cudaStream_t s, const A2Args& a) {
  BGP_SHAPE_SWITCH(shape, (a2_eval_kernel<SHAPE><<<grid, A2_THREADS, 0, s>>>(a)));
}

// ---- decide: first usable candidate wins; commit the RNG / index list up to it ----------------------------------
__global__ void __launch_bounds__(A2_NODE_THREADS) a2_decide_kernel(A2Args a) {
  extern __shared__ __align__(16) unsigned char a2_smem_raw[];
  A2NodeSmem& S = *reinterpret_cast<A2NodeSmem*>(a2_smem_raw);
  __shared__ int s_winner;
  const int nid = blockIdx.x;
  A2State& st = a.states[nid];
  if (st.phase != A2_SELECT || !st.active) return;
  const A2Node nd = a.nodes[nid];
  const int ncand = st.ncand;
  int* cand = a.cand + nd.cand_off;
  int* cand_k = a.cand_k + nd.cand_off;
  int* words = a.cand_words + nd.cand_off;
  int* index = a.idx_ws + nd.idx_off;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    s_winner = 0x7fffffff;
  }
  __syncthreads();
  // first candidate (sequence order) whose max |residual| over all chunks is >= 1e-14 (hodlr.h:191; a NaN also
  // leaves the reference's loop): the per-candidate maxima were reduced across chunks by atomicMax in a2_eval.
  // A deferred one-candidate batch is accepted provisionally (a2_pivot applies the test to the row a2_vrow computes).
  const bool deferred = st.deferred != 0;
  if (deferred) {
    if (threadIdx.x == 0) { s_winner = 0; atomicAdd(a.stats + 3, (unsigned long long)nd.n_cols); }
  } else {
    const unsigned long long* cmax = a.cmax + nd.cand_off;
    int mine = 0x7fffffff;
    for (int c = threadIdx.x; c < ncand; c += blockDim.x) {
      const double m = __longlong_as_double((long long)cmax[c]);
      if (!(m < 1e-14)) { mine = c; break; }
    }
    if (mine != 0x7fffffff) atomicMin(&s_winner, mine);
  }
  __syncthreads();
  const int p = s_winner;
  // commit the stream: the words consumed up to the winner (or the whole batch).  When that is the whole batch the
  // stream after it was saved by a2_generate; otherwise replay the words from the committed state.
  {
    MT19937* rng_commit = a.rngs + 2 * (int64_t)nid;
    const int w = (p != 0x7fffffff) ? words[p] : (ncand > 0 ? words[ncand - 1] : 0);
    if (w == st.end_words) {
      mt_copy(&S.rng, rng_commit + 1);
    } else {
      mt_copy(&S.rng, rng_commit);
      __syncthreads();
      mt_skip_coop(S.rng, w);
    }
    if (threadIdx.x == 0) st.draws += w;
    __syncthreads();
    mt_copy(rng_commit, &S.rng);
  }
  // commit the swap-pops of the consumed draws 0..last: position cand_k[c] ends up with the value of the LAST consumed draw
  // that wrote it (a2_generate left the list untouched and recorded, per draw, its value and the next writer of its slot)
  {
    const int last = (p != 0x7fffffff) ? p : ncand - 1;
    if (threadIdx.x == 0) {  // consumed candidate rows: each one is a row of the block verified against the 1e-14 threshold
      atomicAdd(a.stats + 0, (unsigned long long)(last + 1) * (unsigned long long)nd.n_cols);
      atomicAdd(a.stats + 2, (unsigned long long)(last + 1));
    }
    const int* cand_L = a.cand_L + nd.cand_off;
    const int* cand_next = a.cand_next + nd.cand_off;
    for (int c = threadIdx.x; c <= last; c += blockDim.x)
      if (cand_next[c] > last) index[cand_k[c]] = cand_L[c];
  }
  __syncthreads();
  if (p != 0x7fffffff) {
    if (threadIdx.x == 0) {
      st.n_index -= (p + 1);
      st.piv_i = cand[p];
      st.phase = A2_ACCEPT;  // pivot column / value follow from a2_vrow + a2_pivot
      // next batch: a kernel whose rows are all usable settles at ONE candidate per step (every speculative row costs a
      // pass over the factor panel); otherwise twice what this pivot search needed
      st.B = (p == 0) ? 1 : max(1, min(st.B, 2 * (p + 1)));
    }
    return;
  }
  if (threadIdx.x == 0) {
    st.n_index -= ncand;
    st.B = min(A2_BGROW * st.B, A2_BMAX);
    if (st.n_index == 0) {
      st.fallback = 1;  // rows exhausted (hodlr.h:161); dense fill (if requested) happens after the loop
      st.phase = A2_DONE; st.active = 0;
      atomicSub(a.n_active, 1);
    }
  }
  __syncthreads();
  if (st.n_index == 0) return;
  a2_generate(a, st, S, nd, nid, (*a.iter_ptr + 1) & 1);
}

// ---- residual of one row (vrow) or one column (ucol) of the block over a sub-chunk of A2_THREADS entries ------------
// One entry per thread; the factor columns are streamed with A2_KU loads in flight per thread and subtracted in the
// order q = 0, 1, ... (the order of hodlr.h:188 / :199 and of the oracle), so the value does not depend on the schedule.
constexpr int A2_KU = 8;
template <class KFn>
__device__ __forceinline__ double a2_resid_entry(const KFn& fn, const double* xa, const double* xb, int rank,
                                                 const double* __restrict__ pcol,  // &panel[0][this entry]
                                                 int64_t ld, const double* __restrict__ coef_g,  // coef[q] = coef_g[q * ld]
                                                 double* s_coef, bool active) {
  double val = active ? fn(xa, xb) : 0.0;
  for (int k0 = 0; k0 < rank; k0 += 128) {
    const int nk = min(128, rank - k0);
    __syncthreads();
    for (int k = threadIdx.x; k < nk; k += A2_THREADS) s_coef[k] = __ldcg(coef_g + (int64_t)(k0 + k) * ld);
    __syncthreads();
    if (active) {
      const double* pc = pcol + (int64_t)k0 * ld;
      int k = 0;
      for (; k + A2_KU <= nk; k += A2_KU) {
        double pv[A2_KU];
#pragma unroll
        for (int q = 0; q < A2_KU; ++q) pv[q] = pc[(int64_t)(k + q) * ld];
#pragma unroll
        for (int q = 0; q < A2_KU; ++q) val -= s_coef[k + q] * pv[q];
      }
      for (; k < nk; ++k) val -= s_coef[k] * pc[(int64_t)k * ld];
    }
  }
  return val;
}

// ---- vrow: residual of the winning row over one column sub-chunk, stored UN-normalised in panel column `rank`, plus
//      the sub-chunk's arg-max (hodlr.h:186-189).  Same evaluator as a2_eval (one shape, one arithmetic).
template <int SHAPE>
__global__ void __launch_bounds__(A2_THREADS) a2_vrow_kernel(A2Args a) {
  __shared__ DevProgram P;
  __shared__ double s_x[ACA_MAX_NDIM];
  __shared__ double s_u[128];
  __shared__ double s_red[A2_THREADS / 32];
  __shared__ int s_redi[A2_THREADS / 32];
  const int chunk = blockIdx.x, sub = blockIdx.y;
  const int nid = a.cchunk_node[chunk];
  const A2State& st = a.states[nid];
  if (st.phase != A2_ACCEPT || !st.active) return;
  const A2Node nd = a.nodes[nid];
  const int lc = chunk - nd.cchunk0;
  const int c_lo = lc * A2_CHUNK + sub * A2_THREADS;
  if (c_lo >= nd.n_cols) return;
  if constexpr (SHAPE == BGP_SHAPE_GENERIC) stage_program(&P, a.prog);
  const int ndim = a.prog->ndim;
  const int rank = st.rank;
  const int c_n = min(A2_THREADS, nd.n_cols - c_lo);
  double* Vcols = nd.vbase;
  const int i = st.piv_i;
  for (int q = threadIdx.x; q < ndim; q += A2_THREADS) s_x[q] = a.x[(int64_t)(nd.row0 + i) * ndim + q];
  __syncthreads();
  const auto fn = ShapeEval<SHAPE>::make(&P, a.prog);
  const int n = threadIdx.x;
  const bool act = n < c_n;
  const int nn = act ? n : 0;
  const double val = a2_resid_entry(fn, s_x, a.x + (int64_t)(nd.col0 + c_lo + nn) * ndim, rank, Vcols + nd.col0 + c_lo + nn,
                                    nd.ld, Vcols + nd.row0 + i, s_u, act);
  double best = -1.0, bval = 0.0;
  int bidx = 0x7fffffff;
  if (act) {
    Vcols[(int64_t)rank * nd.ld + nd.col0 + c_lo + n] = val;
    best = fabs(val); bidx = c_lo + n; bval = val;
    if (val != val) best = __longlong_as_double(0x7ff0000000000000ll);  // a NaN wins the arg-max (it ends the reference's loop)
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const double ov = __shfl_xor_sync(0xffffffffu, bval, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
    if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; bval = ov; }
  }
  if (lane == 0) { s_red[warp] = bval; s_redi[warp] = bidx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < A2_THREADS / 32; ++w) {
      const double ov = s_red[w];
      const int oi = s_redi[w];
      if (oi == 0x7fffffff) continue;
      if (bidx == 0x7fffffff || fabs(ov) > fabs(bval) || (fabs(ov) == fabs(bval) && oi < bidx) || (ov != ov && !(bval != bval))) { bval = ov; bidx = oi; }
    }
    A2EPart p;
    p.val = bval; p.idx = bidx; p._pad = 0;
    a.epart[(int64_t)(nd.cchunk0 + lc) * A2_NSUB + sub] = p;
  }
}

// ---- pivot: arg-max over the sub-chunks of the winning row (first maximum, as Eigen's maxCoeff) ---------------------
__global__ void __launch_bounds__(32) a2_pivot_kernel(A2Args a) {
  const int nid = blockIdx.x;
  A2State& st = a.states[nid];
  if (st.phase != A2_ACCEPT || !st.active) return;
  const A2Node nd = a.nodes[nid];
  const int lane = threadIdx.x;
  double bval = 0.0;
  int bidx = 0x7fffffff;
  const int nsub = (nd.n_cols + A2_THREADS - 1) / A2_THREADS;  // sub-chunks that exist (slot = chunk * A2_NSUB + sub, contiguous)
  for (int ch = lane; ch < nsub; ch += 32) {
    const A2EPart q = a.epart[(int64_t)nd.cchunk0 * A2_NSUB + ch];
    if (q.idx == 0x7fffffff) continue;
    if (bidx == 0x7fffffff || fabs(q.val) > fabs(bval) || (fabs(q.val) == fabs(bval) && q.idx < bidx) || (q.val != q.val && !(bval != bval))) { bval = q.val; bidx = q.idx; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, bval, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bidx, o);
    if (oi == 0x7fffffff) continue;
    if (bidx == 0x7fffffff || fabs(ov) > fabs(bval) || (fabs(ov) == fabs(bval) && oi < bidx) || (ov != ov && !(bval != bval))) { bval = ov; bidx = oi; }
  }
  if (lane == 0) {
    st.piv_j = bidx; st.pivot = bval;
    if (st.deferred && fabs(bval) < 1e-14) st.phase = A2_LATE_REJECT;  // hodlr.h:191 (a NaN pivot leaves the loop: accepted)
  }
}

// partial dot products  part[1 + q] = sum_n P[q][n] * s_vec[n]  over this CTA's `cnt` entries, for q < rank: warp w takes
// q = w, w + W, ... four at a time (their loads are independent: 32 in flight per lane)
__device__ __forceinline__ void a2_partial_dots(const double* __restrict__ pbase, int64_t ld, int rank, const double* s_vec,
                                                int cnt, double* __restrict__ part) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int W = A2_THREADS / 32, QU = 4;
  for (int q0 = warp * QU; q0 < rank; q0 += W * QU) {
    double acc[QU];
#pragma unroll
    for (int u = 0; u < QU; ++u) acc[u] = 0.0;
    for (int n = lane; n < cnt; n += 32) {
      const double sv = s_vec[n];
      double pv[QU];
#pragma unroll
      for (int u = 0; u < QU; ++u) pv[u] = (q0 + u < rank) ? pbase[(int64_t)(q0 + u) * ld + n] : 0.0;
#pragma unroll
      for (int u = 0; u < QU; ++u) acc[u] += pv[u] * sv;
    }
#pragma unroll
    for (int u = 0; u < QU; ++u) {
      const double r = warp_sum(acc[u]);
      if (lane == 0 && q0 + u < rank) part[1 + q0 + u] = r;
    }
  }
}

// ---- vnorm: normalise the stored row residual (hodlr.h:194), partial ||v||^2 and V_prev^T v, group maxima ------------
__device__ __forceinline__ void a2_vnorm_body(const A2Args& a, int chunk, int sub, double* s_v, double* red) {
  const int nid = a.cchunk_node[chunk];
  const A2State& st = a.states[nid];
  if (st.phase != A2_ACCEPT || !st.active) return;
  const A2Node nd = a.nodes[nid];
  const int rank = st.rank;
  const int lc = chunk - nd.cchunk0;
  const int c_lo = lc * A2_CHUNK + sub * A2_THREADS;
  if (c_lo >= nd.n_cols) return;
  const int c_n = min(A2_THREADS, nd.n_cols - c_lo);
  double* Vcols = nd.vbase;
  const double pivot = st.pivot;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double vn2 = 0.0, av = 0.0;
  {
    const int n = threadIdx.x;
    double v = 0.0;
    if (n < c_n) {
      double* pv = Vcols + (int64_t)rank * nd.ld + nd.col0 + c_lo + n;
      v = *pv / pivot;
      *pv = v;
      vn2 = v * v;
      av = fabs(v);
      if (v != v) av = __longlong_as_double(0x7ff0000000000000ll);
    }
    s_v[n] = v;
  }
  if (a.vmax) {  // max |v| of the two 128-column groups of this sub-chunk (warps 0-3 | 4-7)
    av = warp_max(av);
    if (lane == 0) red[16 + warp] = av;
  }
  vn2 = block_sum(vn2, red);  // (two barriers: s_v and red[16..] visible)
  if (a.vmax && threadIdx.x < 2) {
    const int g = threadIdx.x;
    const double m = fmax(fmax(red[16 + 4 * g], red[17 + 4 * g]), fmax(red[18 + 4 * g], red[19 + 4 * g]));
    double* slot = a.vmax + ((int64_t)chunk * A2_NGROUP + sub * 2 + g);
    if (rank == 0 || m > *slot || m != m) *slot = m;  // running maximum over the factors (first factor: overwrite)
  }
  double* part = a.vpart + ((int64_t)chunk * A2_NSUB + sub) * (a.capmax + 1);
  if (threadIdx.x == 0) part[0] = vn2;
  a2_partial_dots(Vcols + nd.col0 + c_lo, nd.ld, rank, s_v, c_n, part);
}

// ---- ucol: column residual -> panel column `rank` (row part), partial ||u||^2 and U_prev^T u --------------------
// vnorm (column sub-chunks) and ucol (row sub-chunks) are independent: one launch, blocks [0, n_cchunks) normalise, the
// rest compute the column residual.
template <int SHAPE>
__global__ void __launch_bounds__(A2_THREADS) a2_vnorm_ucol_kernel(A2Args a, int n_cchunks_total) {
  __shared__ DevProgram P;
  __shared__ double s_x[ACA_MAX_NDIM];
  __shared__ double s_vr[128];
  __shared__ double s_u[A2_THREADS];
  __shared__ double red[32];
  const int sub = blockIdx.y;
  if ((int)blockIdx.x < n_cchunks_total) { a2_vnorm_body(a, blockIdx.x, sub, s_u, red); return; }
  const int chunk = blockIdx.x - n_cchunks_total;
  const int nid = a.rchunk_node[chunk];
  const A2State& st = a.states[nid];
  if (st.phase != A2_ACCEPT || !st.active) return;
  const A2Node nd = a.nodes[nid];
  const int lr = chunk - nd.rchunk0;
  const int r_lo = lr * A2_CHUNK + sub * A2_THREADS;
  if (r_lo >= nd.n_rows) return;
  if constexpr (SHAPE == BGP_SHAPE_GENERIC) stage_program(&P, a.prog);
  const int ndim = a.prog->ndim;
  const int rank = st.rank;
  const int r_n = min(A2_THREADS, nd.n_rows - r_lo);
  double* Vcols = nd.vbase;
  const int j = st.piv_j;
  for (int q = threadIdx.x; q < ndim; q += A2_THREADS) s_x[q] = a.x[(int64_t)(nd.col0 + j) * ndim + q];
  __syncthreads();
  const auto fn = ShapeEval<SHAPE>::make(&P, a.prog);
  const int n = threadIdx.x;
  const bool act = n < r_n;
  const int nn = act ? n : 0;
  // V(j, q) for q < rank: columns already normalised in earlier iterations
  const double val = a2_resid_entry(fn, a.x + (int64_t)(nd.row0 + r_lo + nn) * ndim, s_x, rank, Vcols + nd.row0 + r_lo + nn, nd.ld,
                                    Vcols + nd.col0 + j, s_vr, act);
  double un2 = 0.0;
  if (act) {
    Vcols[(int64_t)rank * nd.ld + nd.row0 + r_lo + n] = val;
    un2 = val * val;
  }
  s_u[n] = act ? val : 0.0;
  un2 = block_sum(un2, red);
  double* part = a.upart + ((int64_t)chunk * A2_NSUB + sub) * (a.capmax + 1);
  if (threadIdx.x == 0) part[0] = un2;
  a2_partial_dots(Vcols + nd.row0 + r_lo, nd.ld, rank, s_u, r_n, part);
}
inline void a2_vrow_launch(int shape, dim3 grid, cudaStream_t s, const A2Args& a) {
  BGP_SHAPE_SWITCH(shape, (a2_vrow_kernel<SHAPE><<<grid, A2_THREADS, 0, s>>>(a)));
}
inline void a2_vnorm_ucol_launch(int shape, dim3 grid, cudaStream_t s, const A2Args& a, int ncc) {
  BGP_SHAPE_SWITCH(shape, (a2_vnorm_ucol_kernel<SHAPE><<<grid, A2_THREADS, 0, s>>>(a, ncc)));
}

// ---- finish: stopping rule (hodlr.h:202-214), next candidates -----------------------------------------------------
__global__ void __launch_bounds__(A2_NODE_THREADS) a2_finish_kernel(A2Args a) {
  extern __shared__ __align__(16) unsigned char a2_smem_raw[];
  A2NodeSmem& S = *reinterpret_cast<A2NodeSmem*>(a2_smem_raw);
  __shared__ int s_done;
  const int nid = blockIdx.x;
  A2State& st = a.states[nid];
  if (!st.active) return;
  if (st.phase == A2_LATE_REJECT) {  // the deferred candidate failed the pivot test: same bookkeeping as a rejected batch
    const A2Node nd = a.nodes[nid];
    __syncthreads();
    if (threadIdx.x == 0) {
      st.B = min(A2_BGROW * st.B, A2_BMAX);
      if (st.n_index == 0) {
        st.fallback = 1;
        st.phase = A2_DONE; st.active = 0;
        atomicSub(a.n_active, 1);
      } else {
        st.phase = A2_SELECT;
      }
    }
    __syncthreads();
    if (st.phase == A2_DONE) return;
    mt_copy(&S.rng, a.rngs + 2 * (int64_t)nid);
    __syncthreads();
    a2_generate(a, st, S, nd, nid, (*a.iter_ptr + 1) & 1);
    return;
  }
  if (st.phase != A2_ACCEPT) return;
  const A2Node nd = a.nodes[nid];
  const int rank = st.rank;
  double vn2 = 0.0, un2 = 0.0;
  // sub-chunk slots of a node are contiguous: slot = chunk * A2_NSUB + sub; the ones past the node's end were never written
  const int nvs = (nd.n_cols + A2_THREADS - 1) / A2_THREADS, nus = (nd.n_rows + A2_THREADS - 1) / A2_THREADS;
  const double* vp0 = a.vpart + (int64_t)nd.cchunk0 * A2_NSUB * (a.capmax + 1);
  const double* up0 = a.upart + (int64_t)nd.rchunk0 * A2_NSUB * (a.capmax + 1);
  for (int c = threadIdx.x; c < nvs; c += blockDim.x) vn2 += vp0[(int64_t)c * (a.capmax + 1)];
  for (int c = threadIdx.x; c < nus; c += blockDim.x) un2 += up0[(int64_t)c * (a.capmax + 1)];
  vn2 = block_sum(vn2, S.red);
  un2 = block_sum(un2, S.red);
  double vdot = 0.0, udot = 0.0;
  for (int k = threadIdx.x; k < rank; k += blockDim.x) {
    double sv = 0.0, su = 0.0;
    for (int c = 0; c < nvs; ++c) sv += vp0[(int64_t)c * (a.capmax + 1) + 1 + k];
    for (int c = 0; c < nus; ++c) su += up0[(int64_t)c * (a.capmax + 1) + 1 + k];
    vdot = fmax(vdot, fabs(sv));
    udot = fmax(udot, fabs(su));
  }
  vdot = block_max(vdot, S.red);
  udot = block_max(udot, S.red);
  mt_copy(&S.rng, a.rngs + 2 * (int64_t)nid);
  if (threadIdx.x == 0) {
    a.piv_rows[nd.piv_off + rank] = st.piv_i;
    a.piv_cols[nd.piv_off + rank] = st.piv_j;
    const int new_rank = rank + 1;
    st.rank = new_rank;
    const int max_rank = min(nd.n_rows, nd.n_cols);
    bool done = false;
    if (new_rank >= max_rank) done = true;  // hodlr.h:203
    else {
      const double rowcol = un2 * vn2;
      if (rowcol < a.tol * a.tol * st.norm) done = true;  // hodlr.h:207
      else {
        st.norm += rowcol;
        if (new_rank > 1) st.norm += 2.0 * udot + 2.0 * vdot;
        if (new_rank >= nd.cap) { st.status = 1; done = true; }       // no room for another column
        else if (st.n_index == 0) { st.fallback = 1; done = true; }  // next pass of the do-loop would find no rows
      }
    }
    if (done) {
      st.phase = A2_DONE; st.active = 0;
      atomicSub(a.n_active, 1);
    } else {
      st.phase = A2_SELECT;
    }
    s_done = done ? 1 : 0;
  }
  __syncthreads();
  if (s_done) return;
  a2_generate(a, st, S, nd, nid, (*a.iter_ptr + 1) & 1);
}

// ---- tick: end of a lock-step iteration.  Advances the iteration counter and, inside the captured loop (CUDA graph WHILE
//      node), tells the graph whether another iteration is needed: no host round trip between iterations. ----
__global__ void a2_tick_kernel(int* iter_ptr, const int* n_active, cudaGraphConditionalHandle handle, int use_handle) {
  const int it = *iter_ptr + 1;
  *iter_ptr = it;
  if (use_handle) cudaGraphSetConditional(handle, (*n_active > 0 && it < (1 << 22)) ? 1u : 0u);
}

// ---- dense fallback fill (hodlr.h:161-176): V = I, U = K(rows, cols) ---------------------------------------------
// grid = (node, column m); nodes without the fallback flag (or in low-rank exhaust mode) return at once.
__global__ void __launch_bounds__(256) a2_dense_fill_kernel(A2Args a) {
  __shared__ DevProgram P;
  const int nid = blockIdx.x;
  A2State& st = a.states[nid];
  if (!st.fallback || a.exhaust_mode != BGP_EXHAUST_DENSE || st.status) return;
  const A2Node nd = a.nodes[nid];
  const int max_rank = min(nd.n_rows, nd.n_cols);
  if (max_rank > nd.cap) {
    if (blockIdx.y == 0 && threadIdx.x == 0) st.status = 1;
    return;
  }
  stage_program(&P, a.prog);
  __syncthreads();
  const int ndim = P.ndim;
  const double* xr = a.x + (int64_t)nd.row0 * ndim;
  const double* xc = a.x + (int64_t)nd.col0 * ndim;
  for (int m = blockIdx.y; m < nd.n_cols; m += gridDim.y) {
    double* vc = nd.vbase + (int64_t)m * nd.ld;
    for (int n = threadIdx.x; n < nd.n_cols; n += blockDim.x) vc[nd.col0 + n] = (n == m) ? 1.0 : 0.0;
    for (int n = threadIdx.x; n < nd.n_rows; n += blockDim.x)
      vc[nd.row0 + n] = kernel_value(P, xr + (int64_t)n * ndim, xc + (int64_t)m * ndim);
  }
}
__global__ void a2_dense_rank_kernel(A2Args a) {
  const int nid = blockIdx.x * blockDim.x + threadIdx.x;
  if (nid >= a.n_nodes) return;
  A2State& st = a.states[nid];
  if (st.fallback && a.exhaust_mode == BGP_EXHAUST_DENSE && !st.status) {
    const A2Node nd = a.nodes[nid];
    st.rank = min(nd.n_rows, nd.n_cols);
  }
}

}  // namespace bgp

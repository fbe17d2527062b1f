// comm.cu — NCCL plumbing of the sharded HODLR solver (SURVEY.md §8e): ONE communicator owned by the library carries
// the data-path collectives — the all-gather of the top-level factor rows after the local sub-trees are factored, the
// all-gather of the right-hand-side slices in a solve, and the one-double log-det all-reduce — on the solver's own
// stream, without a host round trip between the pack kernel, the collective and the unpack kernel.  The Python host
// (george_b200/parallel.py) only bootstraps it (broadcast of the 128-byte unique id over its process group).
//
// The process already has NCCL loaded (torch links libnccl.so.2), so the library is reached through dlopen/dlsym
// instead of being linked a second time; the communicator is created from a unique id that rank 0 makes and the host
// broadcasts over its own process group.
#include <dlfcn.h>

#include "common.cuh"

namespace bgp {

typedef struct { char internal[128]; } nccl_unique_id_t;
typedef void* nccl_comm_t;
typedef int (*fn_get_unique_id)(nccl_unique_id_t*);
typedef int (*fn_comm_init_rank)(nccl_comm_t*, int, nccl_unique_id_t, int);
typedef int (*fn_all_reduce)(const void*, void*, size_t, int, int, nccl_comm_t, cudaStream_t);
typedef int (*fn_all_gather)(const void*, void*, size_t, int, nccl_comm_t, cudaStream_t);
typedef int (*fn_comm_destroy)(nccl_comm_t);
typedef const char* (*fn_get_error_string)(int);

static void* g_nccl = nullptr;
static fn_get_unique_id p_get_unique_id = nullptr;
static fn_comm_init_rank p_comm_init_rank = nullptr;
static fn_all_reduce p_all_reduce = nullptr;
static fn_all_gather p_all_gather = nullptr;
static fn_comm_destroy p_comm_destroy = nullptr;
static fn_get_error_string p_error_string = nullptr;
static nccl_comm_t g_comm = nullptr;
static int g_rank = 0, g_world = 1;

static int load_nccl(const char* path) {
  if (g_nccl) return BGP_OK;
  const char* names[] = {path, "libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    if (!nm || !nm[0]) continue;
    g_nccl = dlopen(nm, RTLD_NOW | RTLD_NOLOAD);  // the copy torch already loaded, if any
    if (!g_nccl) g_nccl = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl) break;
  }
  if (!g_nccl) { set_error("cannot load NCCL: %s", dlerror()); return BGP_ERR_CUDA; }
  p_get_unique_id = (fn_get_unique_id)dlsym(g_nccl, "ncclGetUniqueId");
  p_comm_init_rank = (fn_comm_init_rank)dlsym(g_nccl, "ncclCommInitRank");
  p_all_reduce = (fn_all_reduce)dlsym(g_nccl, "ncclAllReduce");
  p_all_gather = (fn_all_gather)dlsym(g_nccl, "ncclAllGather");
  p_comm_destroy = (fn_comm_destroy)dlsym(g_nccl, "ncclCommDestroy");
  p_error_string = (fn_get_error_string)dlsym(g_nccl, "ncclGetErrorString");
  if (!p_get_unique_id || !p_comm_init_rank || !p_all_reduce || !p_all_gather || !p_comm_destroy) {
    set_error("NCCL symbols missing");
    return BGP_ERR_CUDA;
  }
  return BGP_OK;
}

bool comm_ready() { return g_comm != nullptr && g_world > 1; }
int comm_rank() { return g_rank; }
int comm_world() { return g_world; }

// in-place SUM all-reduce of `count` doubles (ncclFloat64 = 8, ncclSum = 0)
int comm_allreduce_sum_f64(double* buf, size_t count, cudaStream_t s) {
  if (!comm_ready()) { set_error("no communicator"); return BGP_ERR_INVALID; }
  const int rc = p_all_reduce(buf, buf, count, 8, 0, g_comm, s);
  if (rc != 0) { set_error("ncclAllReduce failed: %s", p_error_string ? p_error_string(rc) : "?"); return BGP_ERR_CUDA; }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return BGP_OK;
}

// all-gather of `count` doubles per rank: recv holds world * count doubles, rank r's block at r * count
int comm_allgather_f64(const double* send, double* recv, size_t count, cudaStream_t s) {
  if (!comm_ready()) { set_error("no communicator"); return BGP_ERR_INVALID; }
  const int rc = p_all_gather(send, recv, count, 8, g_comm, s);
  if (rc != 0) { set_error("ncclAllGather failed: %s", p_error_string ? p_error_string(rc) : "?"); return BGP_ERR_CUDA; }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return BGP_OK;
}

}  // namespace bgp

using namespace bgp;

extern "C" {

int bgp_comm_unique_id(void* out128, const char* nccl_path) {
  BGP_TRY(load_nccl(nccl_path));
  nccl_unique_id_t id;
  const int rc = p_get_unique_id(&id);
  if (rc != 0) { set_error("ncclGetUniqueId failed: %s", p_error_string ? p_error_string(rc) : "?"); return BGP_ERR_CUDA; }
  memcpy(out128, &id, sizeof(id));
  return BGP_OK;
}

int bgp_comm_init(const void* id128, int rank, int world, const char* nccl_path) {
  BGP_TRY(require_device());
  BGP_TRY(load_nccl(nccl_path));
  if (g_comm) { p_comm_destroy(g_comm); g_comm = nullptr; }
  nccl_unique_id_t id;
  memcpy(&id, id128, sizeof(id));
  const int rc = p_comm_init_rank(&g_comm, world, id, rank);
  if (rc != 0) { set_error("ncclCommInitRank failed: %s", p_error_string ? p_error_string(rc) : "?"); g_comm = nullptr; return BGP_ERR_CUDA; }
  g_rank = rank; g_world = world;
  return BGP_OK;
}

int bgp_comm_destroy(void) {
  if (g_comm && p_comm_destroy) p_comm_destroy(g_comm);
  g_comm = nullptr; g_world = 1; g_rank = 0;
  return BGP_OK;
}

}  // extern "C"

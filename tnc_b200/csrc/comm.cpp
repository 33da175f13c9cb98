// Partitioned fan-in over NCCL point-to-point: replaces tnc/src/mpi/communication.rs
// (send_tensor/receive_tensor :72-85, the fan-in loop :199-249) and the postcard + 192-byte
// blob wire format of mpi/serialization.rs:43-79.  A boundary tensor travels GPU->GPU as its
// raw complex128 buffer (2*elems doubles) on the context stream; legs and dims are derived
// from the broadcast plan on every rank, so nothing is serialised.
//
// libnccl is resolved with dlopen at first use: the library stays loadable on hosts without
// NCCL, and inside a PyTorch process it binds to the libnccl.so.2 torch already loaded.
#include "internal.h"
#include <dlfcn.h>
#include <algorithm>
#include <cstring>
#include <mutex>
#include <vector>

namespace tncb {

struct Uid { char internal[128]; }; // ncclUniqueId
struct NcclFns {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /*ncclUniqueId by value*/ Uid, int) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
};

static NcclFns g_nccl;
static std::once_flag g_nccl_once;
static std::string g_nccl_err;

static void load_nccl() {
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    h = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL); // already in the process (torch)?
    if (h) break;
  }
  if (!h) for (const char* n : names) { h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
  if (!h) { g_nccl_err = std::string("cannot load libnccl: ") + dlerror(); return; }
  g_nccl.handle = h;
#define LOAD(field, sym)                                                   \
  *(void**)(&g_nccl.field) = dlsym(h, sym);                                \
  if (!g_nccl.field) { g_nccl_err = std::string("missing symbol ") + sym; return; }
  LOAD(GetUniqueId, "ncclGetUniqueId");
  LOAD(CommInitRank, "ncclCommInitRank");
  LOAD(Send, "ncclSend");
  LOAD(Recv, "ncclRecv");
  LOAD(CommDestroy, "ncclCommDestroy");
  LOAD(GetErrorString, "ncclGetErrorString");
  LOAD(GroupStart, "ncclGroupStart");
  LOAD(GroupEnd, "ncclGroupEnd");
  LOAD(AllReduce, "ncclAllReduce");
#undef LOAD
}

static int nccl_ready() {
  std::call_once(g_nccl_once, load_nccl);
  if (!g_nccl.handle || !g_nccl_err.empty()) return fail(TNCB_ERR_NCCL, g_nccl_err.empty() ? "libnccl not available" : g_nccl_err);
  return TNCB_OK;
}

#define TNCB_NCCL(call)                                                                         \
  do {                                                                                          \
    int _r = (call);                                                                            \
    if (_r != 0) return fail(TNCB_ERR_NCCL, std::string(#call) + ": " + g_nccl.GetErrorString(_r)); \
  } while (0)

constexpr int kNcclFloat64 = 8; // ncclFloat64 / ncclDouble

} // namespace tncb

using namespace tncb;

extern "C" {

int tncb_comm_unique_id(uint8_t id_out[128]) {
  if (!id_out) return fail(TNCB_ERR_INVALID, "null argument");
  int rc = nccl_ready();
  if (rc) return rc;
  Uid id;
  TNCB_NCCL(g_nccl.GetUniqueId(&id));
  std::memcpy(id_out, id.internal, 128);
  return TNCB_OK;
}

int tncb_comm_init(tncb_ctx* ctx, int world_size, int rank, const uint8_t id_in[128]) {
  if (!ctx || !id_in || world_size < 1 || rank < 0 || rank >= world_size) return fail(TNCB_ERR_INVALID, "bad argument");
  int rc = nccl_ready();
  if (rc) return rc;
  TNCB_CUDA(cudaSetDevice(ctx->device));
  Uid id;
  std::memcpy(id.internal, id_in, 128);
  void* comm = nullptr;
  TNCB_NCCL(g_nccl.CommInitRank(&comm, world_size, id, rank));
  ctx->nccl_comm = comm; ctx->world = world_size; ctx->rank = rank;
  return TNCB_OK;
}

int tncb_comm_send(tncb_ctx* ctx, const tncb_tensor* t, int peer) {
  if (!ctx || !t) return fail(TNCB_ERR_INVALID, "null argument");
  if (t->dtype != TNCB_C128) return fail(TNCB_ERR_UNSUPPORTED, "NCCL transfers of complex64 tensors are not supported");
  if (!ctx->nccl_comm) return fail(TNCB_ERR_NCCL, "communicator not initialised");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_NCCL(g_nccl.Send(t->ptr, (size_t)t->elems * 2, kNcclFloat64, peer, ctx->nccl_comm, ctx->stream));
  return TNCB_OK;
}

int tncb_comm_recv(tncb_ctx* ctx, int rank_dims, const uint64_t* dims, int peer, tncb_tensor** out) {
  if (!ctx || !out) return fail(TNCB_ERR_INVALID, "null argument");
  if (!ctx->nccl_comm) return fail(TNCB_ERR_NCCL, "communicator not initialised");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  tncb_tensor* t = nullptr;
  int rc = tensor_new(ctx, rank_dims, dims, &t);
  if (rc) return rc;
  int r = g_nccl.Recv(t->ptr, (size_t)t->elems * 2, kNcclFloat64, peer, ctx->nccl_comm, ctx->stream);
  if (r != 0) { tncb_tensor_free(ctx, t); return fail(TNCB_ERR_NCCL, std::string("ncclRecv: ") + g_nccl.GetErrorString(r)); }
  *out = t;
  return TNCB_OK;
}

int tncb_comm_allreduce_sum(tncb_ctx* ctx, tncb_tensor* t) {
  if (!ctx || !t) return fail(TNCB_ERR_INVALID, "null argument");
  if (t->dtype != TNCB_C128) return fail(TNCB_ERR_UNSUPPORTED, "NCCL transfers of complex64 tensors are not supported");
  if (!ctx->nccl_comm) return fail(TNCB_ERR_NCCL, "communicator not initialised");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_NCCL(g_nccl.AllReduce(t->ptr, t->ptr, (size_t)t->elems * 2, kNcclFloat64, /*ncclSum*/ 0, ctx->nccl_comm, ctx->stream));
  return TNCB_OK;
}

int tncb_comm_destroy(tncb_ctx* ctx) {
  if (!ctx || !ctx->nccl_comm) return TNCB_OK;
  cudaStreamSynchronize(ctx->stream);
  g_nccl.CommDestroy(ctx->nccl_comm);
  ctx->nccl_comm = nullptr;
  return TNCB_OK;
}

// Iteration order of `FxHashMap<usize, _>::from_iter(keys)` as the reference builds `path.nested`
// (contractionpath.rs:40-47): rustc-hash 2.1.1 (hash = rotl((0 + key) * 0xf1357aea2e62a9c5, 26), tnc/Cargo.toml:32)
// on hashbrown's SwissTable (Cargo.lock): buckets = capacity_to_buckets(n), a key goes to the first EMPTY
// control byte of the 16-wide group probe starting at hash & mask (triangular stride; tables smaller than a
// group rescan from 0 when the hit lands in the mirror bytes), and iteration walks the buckets in ascending
// index.  Restated from the published crates (both absent from /root/reference); pinned by the reference's
// own KAT communication.rs:257-279 (keys 0,1,2 iterate as 0,2,1).
static std::vector<size_t> fxhashmap_iteration_order(const uint64_t* keys, size_t n) {
  size_t buckets = n < 4 ? 4 : (n < 8 ? 8 : 1);
  if (n >= 8) { size_t adj = n * 8 / 7; while (buckets < adj) buckets <<= 1; }
  const size_t mask = buckets - 1, W = 16;
  std::vector<char> full(buckets, 0);
  std::vector<size_t> owner(buckets, 0);
  for (size_t q = 0; q < n; q++) {
    const uint64_t m = keys[q] * 0xf1357aea2e62a9c5ull;
    const uint64_t h = (m << 26) | (m >> 38);
    size_t pos = (size_t)h & mask, stride = 0, slot = buckets;
    while (slot == buckets) {
      for (size_t b = 0; b < W && slot == buckets; b++) {
        const size_t i = pos + b;           // control bytes [buckets, buckets+W) mirror the start (or are EMPTY)
        if (i < buckets) { if (!full[i]) slot = i; }
        else if (buckets < W) {             // small table: bytes buckets..W-1 are always EMPTY -> masked index, then the fix-up
          size_t idx = i & mask;
          if (full[idx]) { idx = 0; while (full[idx]) idx++; }
          slot = idx;
        } else if (!full[i & mask]) slot = i & mask;
      }
      stride += W; pos = (pos + stride) & mask;
    }
    full[slot] = 1; owner[slot] = q;
  }
  std::vector<size_t> order;
  for (size_t i = 0; i < buckets; i++) if (full[i]) order.push_back(owner[i]);
  return order;
}

// get_tensor_mapping (mpi/communication.rs:89-115): walk `path.nested.keys()` (FxHashMap order, see above;
// `partition_index` is the insertion order, ascending in every caller here and in the reference's finders),
// the partition on the left of the last top-level pair gets rank 0, the others 1, 2, ... in walk order.
int tncb_fanin_mapping(size_t n_partitions, const uint64_t* partition_index, size_t n_pairs,
                       const uint64_t* toplevel_pairs, int world_size, int* rank_of_partition) {
  if ((n_partitions && (!partition_index || !rank_of_partition)) || (n_pairs && !toplevel_pairs))
    return fail(TNCB_ERR_INVALID, "null argument");
  if (n_pairs == 0) { // empty top-level path: at most one partition, goes to rank 0
    for (size_t p = 0; p < n_partitions; p++) rank_of_partition[p] = 0;
    return TNCB_OK;
  }
  const uint64_t final_tensor = toplevel_pairs[2 * (n_pairs - 1)];
  int used = 1;
  for (size_t q : fxhashmap_iteration_order(partition_index, n_partitions)) {
    if (partition_index[q] == final_tensor) rank_of_partition[q] = 0;
    else rank_of_partition[q] = used++;
  }
  if (used > world_size)
    return fail(TNCB_ERR_INVALID, "Not enough ranks available, got " + std::to_string(world_size) + " but need " + std::to_string(used) + "!");
  return TNCB_OK;
}

} // extern "C"

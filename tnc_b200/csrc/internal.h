// Internal definitions shared by the host runtime and the CUDA kernels of libtncb200.
#pragma once
#include <cstdint>
#include <cstddef>
#include <string>
#include <vector>
#include <map>
#include <cuda_runtime.h>
#include "../../include/tncb.h"

namespace tncb {

constexpr int kMaxLegs = 64;   // max rank of a tensor accepted at the ABI
constexpr int kMaxGroups = 40; // max fused leg groups per list passed to a kernel

// A list of (fused) legs of one index class, outermost first, innermost last.
struct LegList {
  int n;
  int _pad;
  long long dim[kMaxGroups];
  long long sa[kMaxGroups]; // element stride in operand A (or in the only operand)
  long long sb[kMaxGroups]; // element stride in operand B (K-list only)
};

// The GEMM view of one pairwise contraction  C[N,M] = sum_K Bt[N,K] * At[K,M]
// (SURVEY 3.4): M = legs(a)\legs(b) in a's order, N = legs(b)\legs(a) in b's
// order, K = shared legs.  C is plain row-major [N][M], which *is* the
// reference's output layout (b\a)++(a\b) (tensor.rs:463-479).
struct PairPlan {
  std::vector<uint64_t> out_legs, out_dims;
  long long M = 1, N = 1, K = 1;
  LegList m{}, n{}, k{};  // m: strides in A; n: strides in B (stored in .sa); k: sa=A, sb=B
  int kernel_class = 0;   // 0 = K0, 1 = K1 (K1' above a size threshold), 2 = K2 streaming (big x tiny)
  bool k2_big_is_a = true; // K2: which operand is the big one
  // K1 loader modes: true = consecutive threads walk the K index, false = the free index
  bool a_kfast = false, b_kfast = true;
  double flops() const { return 8.0 * (double)M * (double)N * (double)K; }
  double bytes() const { return 16.0 * ((double)M * K + (double)K * N + (double)M * N); }
};

// Returns TNCB_OK or an error; fills plan. Pure host code (no CUDA calls).
int plan_pair(int n_a, const uint64_t* a_legs, const uint64_t* a_dims,
              int n_b, const uint64_t* b_legs, const uint64_t* b_dims, PairPlan& plan);

void set_error(const std::string& msg);
int fail(int status, const std::string& msg);

// ---- device arena -------------------------------------------------------------------
struct Slab { char* base; size_t size; std::map<size_t, size_t> free_by_off; };

struct Arena {
  std::vector<Slab> slabs;
  size_t capacity_limit = 0; // 0 = device free memory
  size_t reserved = 0, live = 0, peak = 0;
  size_t next_slab = (size_t)256 << 20;
  int alloc(size_t bytes, void** out);
  void free(void* p, size_t bytes);
  void release_all();
  size_t trim();             // cudaFree every slab that holds no live block; returns the bytes given back
};

} // namespace tncb

struct tncb_tensor {
  double2* ptr = nullptr;   // float2 data for TNCB_C64 (see dtype)
  int rank = 0;
  int dtype = TNCB_C128;
  uint64_t dims[tncb::kMaxLegs];
  uint64_t elems = 1;
  size_t bytes = 0;      // arena bytes (0 = not owned by the arena)
  bool owned = true;
};

struct NcclApi;

struct tncb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  tncb::Arena arena;
  uint64_t launches = 0;
  int oz_slices = 8;  // 0 = DMMA only; otherwise the tcgen05 int8 engine (K1') takes large pairs (digit-slicing engine: #slices)
  int oz_engine = 0;  // 0 = CRT / modular engine (crt.cu, default), 1 = 7-bit digit slicing (ozaki.cu, kept for A/B)
  long long oz_min_tiles = 96, oz_min_k = 1536;   // thresholds of the digit-slicing engine
  // CRT engine: operand bits (53 = full mantissa) or a requested tolerance, forced modulus count, thresholds, workspace
  int crt_bits = 53; double crt_tol = 0.0; int crt_nmod_force = 0;
  long long crt_min_k = 256; double crt_min_mnk = 268435456.0;   // K >= 256 and M*N*K >= 2^28
  size_t crt_ws_bytes = (size_t)12 << 30; int crt_group = 8;
  double last_int8_ops = 0.0; int last_nmod = 0; int last_products = 0;
  int crt_products = 0;            // real int8 products per complex product: 0 = auto (3 when K >= crt_kara_min_k), 3, 4
  long long crt_kara_min_k = 4096;
  uint64_t engine_count[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // K0, K0 split-K, K1 DMMA, K1 DMMA split-K, K1' tcgen05, K2, permute, -
  // dominant-kernel timing: 0 off, 1 keep the last launch (gemm_ev0/1), 2 accumulate every launch (event pool)
  int time_gemm = 0; cudaEvent_t gemm_ev0 = nullptr, gemm_ev1 = nullptr; bool gemm_ev_valid = false;
  std::vector<cudaEvent_t> gemm_pool; size_t gemm_used = 0; std::vector<double> gemm_ops;
  int sm_count = 148;
  // pinned staging for leaf uploads
  void* stage_host = nullptr; size_t stage_bytes = 0;
  // K1 offset-table workspace (grown on demand, stream-ordered reuse)
  long long* tab = nullptr; size_t tab_elems = 0;
  // signature of the tables currently in `tab` (they depend on the plan only, like a TMA
  // descriptor): an identical consecutive pair re-uses them without a rebuild
  bool tab_valid = false; tncb::LegList tab_m{}, tab_n{}, tab_k{};
  // split-K partial workspace
  double2* partial = nullptr; size_t partial_elems = 0;
  double2* partial_override = nullptr; size_t partial_override_elems = 0;  // set while a plan graph is captured
  // NCCL
  void* nccl_comm = nullptr; int world = 1, rank = 0;
  // host pipeline (tncb_contract_pair_host): 3 in-flight jobs, each with its own device operands/result and events;
  // copies run on their own streams so that H2D of pair j+1, the kernels of pair j and D2H of pair j-1 overlap
  struct HostSlot { void* buf[3] = {nullptr, nullptr, nullptr}; size_t bytes[3] = {0, 0, 0};
                    cudaEvent_t in_done = nullptr, comp_done = nullptr, out_done = nullptr; bool busy = false; };
  HostSlot host_slot[3]; uint64_t host_jobs = 0;
  cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
  // plans that hold device state (graph, workspace) on this context; detached by tncb_ctx_destroy
  std::vector<struct tncb_plan*> plans;
  // structure-keyed cache of plans behind tncb_contract_tensor_network (most recently used last)
  struct CachedPlan { std::vector<uint64_t> key; struct tncb_plan* plan; };
  std::vector<CachedPlan> plan_cache;
};

extern "C" void tncb_plan_release_device_state(struct tncb_plan* plan);

namespace tncb {
// bytes per element of a tncb_dtype (0: not a dtype)
inline size_t dtype_size(int dtype) { return dtype == TNCB_C128 ? 16 : dtype == TNCB_C64 ? 8 : 0; }

// ---- kernel launchers (kernels.cu) ---------------------------------------------------
// Operands and results are complex128 (double2) or, for dtype TNCB_C64, complex64 (float2); split-K partials are
// double2 for both.  Kernel and configuration choices never depend on the dtype.
int launch_pair(tncb_ctx* ctx, const PairPlan& p, const void* A, const void* B, void* C, int dtype = TNCB_C128);
int launch_permute(tncb_ctx* ctx, const void* in, void* out, int rank,
                   const uint64_t* in_dims, const int* perm, int dtype = TNCB_C128);
int launch_conj(tncb_ctx* ctx, void* data, uint64_t elems, int dtype = TNCB_C128);
int launch_add(tncb_ctx* ctx, void* dst, const void* src, uint64_t elems, int dtype = TNCB_C128);
int ensure_tab(tncb_ctx* ctx, size_t elems);
// K1': tcgen05 int8-sliced ZGEMM (ozaki.cu); tables as built by launch_k1
int launch_k1_ozaki(tncb_ctx* ctx, const PairPlan& p, const double2* A, const double2* B, double2* C, int S,
                    const long long* offAm, const long long* offBn, const long long* offAk, const long long* offBk);

// K1' default engine: tcgen05 int8 GEMMs over coprime moduli + CRT reconstruction (crt.cu)
int launch_k1_crt(tncb_ctx* ctx, const PairPlan& p, const void* A, const void* B, void* C,
                  const long long* offAm, const long long* offBn, const long long* offAk, const long long* offBk,
                  int dtype = TNCB_C128);
constexpr int kCrtBitsC64 = 28;   // default operand bits of complex64 pairs: bound 2^-24 K max|b[n,:]| max|a[m,:]|
void crt_choose(long long K, int want_bits, int nmod_force, int* nmod, int* bits_a, int* bits_b);
int crt_bits_for_tolerance(long long K, double tol);
int crt_export_tables(int nmod, int* moduli, double* rho1, double* rho2, double* log2_product);

void gemm_timer_begin(tncb_ctx* ctx);              // brackets one launch of the dominant GEMM kernel (K1 / K1')
void gemm_timer_end(tncb_ctx* ctx, double ops);    // ops: executed int8 ops (K1') or flops (K1) of that launch

int ensure_partial(tncb_ctx* ctx, size_t elems);
size_t k0_partial_elems(int sm_count, const PairPlan& p);

// ---- batched tiny pairs: every independent K0 pair of one tree level in ONE launch (plans with a static layout) ----
constexpr int kBatchGroups = 8;
struct CompactLegs { int n; int _pad; long long dim[kBatchGroups]; long long sa[kBatchGroups]; long long sb[kBatchGroups]; };
struct K0BatchItem {
  long long offA, offB, offC;   // byte offsets into the plan workspace
  long long M, N, K;
  int G, _pad;                  // lanes per output element: the value k0_config picks for the single-pair kernel (bit-identical sums)
  CompactLegs m, n, k;
};
bool k0_batch_eligible(int sm_count, const PairPlan& p);
int k0_batch_fill(int sm_count, const PairPlan& p, K0BatchItem* item);   // returns the number of 256-thread blocks of the item
int launch_k0_batch(tncb_ctx* ctx, const K0BatchItem* d_items, const int* d_block_start, int n_items, int total_blocks, char* ws,
                    int dtype = TNCB_C128);

int tensor_new(tncb_ctx* ctx, int rank, const uint64_t* dims, tncb_tensor** out, int dtype = TNCB_C128);

// TensorData::File leaf (hdf5io.cpp): first member of /tensors, optionally adjointed, checked against the leaf's dims
namespace h5 { int load_file_leaf(const char* path, bool adjoint, int rank, const uint64_t* dims, double* out_re_im); }
} // namespace tncb

#define TNCB_CUDA(call)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (call);                                                              \
    if (_e != cudaSuccess)                                                                \
      return tncb::fail(TNCB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
  } while (0)

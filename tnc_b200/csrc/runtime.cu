// Context, device arena, tensor handles and the single-pair entry points of libtncb200.
#include "internal.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>

namespace tncb {

// ---- arena: first-fit free lists over cudaMalloc'd slabs, 256-byte granularity --------------
static inline size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int Arena::alloc(size_t bytes, void** out) {
  bytes = round_up(std::max<size_t>(bytes, 256), 256);
  for (Slab& s : slabs) {
    for (auto it = s.free_by_off.begin(); it != s.free_by_off.end(); ++it) {
      if (it->second >= bytes) {
        size_t off = it->first, sz = it->second;
        s.free_by_off.erase(it);
        if (sz > bytes) s.free_by_off[off + bytes] = sz - bytes;
        *out = s.base + off;
        live += bytes; peak = std::max(peak, live);
        return TNCB_OK;
      }
    }
  }
  // new slab
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) return fail(TNCB_ERR_CUDA, "cudaMemGetInfo failed");
  size_t limit = capacity_limit ? capacity_limit : reserved + (free_b > ((size_t)1 << 30) ? free_b - ((size_t)1 << 30) : 0);
  if (reserved + bytes > limit)
    return fail(TNCB_ERR_OOM, "device arena exhausted: need " + std::to_string(bytes) + " B, reserved " +
                                  std::to_string(reserved) + " B, limit " + std::to_string(limit) + " B");
  size_t want = std::max(bytes, std::min(next_slab, limit - reserved));
  want = round_up(want, (size_t)2 << 20);
  if (reserved + want > limit) want = bytes;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess && want > bytes) { cudaGetLastError(); want = bytes; e = cudaMalloc(&p, want); }
  if (e != cudaSuccess) { cudaGetLastError(); return fail(TNCB_ERR_OOM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
  reserved += want;
  if (std::getenv("TNCB_TRACE")) fprintf(stderr, "TNCB_TRACE arena: new slab %.1f MiB for a %.1f MiB request (reserved %.1f MiB, live %.1f MiB)\n",
                                         want / 1048576.0, bytes / 1048576.0, reserved / 1048576.0, live / 1048576.0);
  next_slab = std::min(next_slab * 2, (size_t)16 << 30);
  Slab s; s.base = (char*)p; s.size = want;
  if (want > bytes) s.free_by_off[bytes] = want - bytes;
  slabs.push_back(std::move(s));
  *out = p;
  live += bytes; peak = std::max(peak, live);
  return TNCB_OK;
}

void Arena::free(void* p, size_t bytes) {
  if (!p) return;
  bytes = round_up(std::max<size_t>(bytes, 256), 256);
  for (Slab& s : slabs) {
    if ((char*)p >= s.base && (char*)p < s.base + s.size) {
      size_t off = (char*)p - s.base;
      auto it = s.free_by_off.emplace(off, bytes).first;
      // coalesce with next
      auto nx = std::next(it);
      if (nx != s.free_by_off.end() && it->first + it->second == nx->first) { it->second += nx->second; s.free_by_off.erase(nx); }
      if (it != s.free_by_off.begin()) {
        auto pv = std::prev(it);
        if (pv->first + pv->second == it->first) { pv->second += it->second; s.free_by_off.erase(it); }
      }
      live -= bytes;
      return;
    }
  }
}

void Arena::release_all() {
  for (Slab& s : slabs) cudaFree(s.base);
  slabs.clear(); reserved = live = 0;
}

size_t Arena::trim() {
  size_t freed = 0;
  for (size_t i = 0; i < slabs.size();) {
    Slab& s = slabs[i];
    if (s.free_by_off.size() == 1 && s.free_by_off.begin()->first == 0 && s.free_by_off.begin()->second == s.size) {
      cudaFree(s.base);
      freed += s.size; reserved -= s.size;
      slabs.erase(slabs.begin() + i);
    } else i++;
  }
  if (slabs.empty()) next_slab = (size_t)256 << 20;
  return freed;
}

void gemm_timer_begin(tncb_ctx* ctx) {
  if (ctx->time_gemm == 1) cudaEventRecord(ctx->gemm_ev0, ctx->stream);
  else if (ctx->time_gemm == 2) {
    if (ctx->gemm_used + 2 > ctx->gemm_pool.size()) {
      cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
      ctx->gemm_pool.push_back(a); ctx->gemm_pool.push_back(b);
    }
    cudaEventRecord(ctx->gemm_pool[ctx->gemm_used], ctx->stream);
  }
}

void gemm_timer_end(tncb_ctx* ctx, double ops) {
  if (ctx->time_gemm == 1) { cudaEventRecord(ctx->gemm_ev1, ctx->stream); ctx->gemm_ev_valid = true; }
  else if (ctx->time_gemm == 2) {
    cudaEventRecord(ctx->gemm_pool[ctx->gemm_used + 1], ctx->stream);
    ctx->gemm_used += 2; ctx->gemm_ops.push_back(ops);
  }
}

int tensor_new(tncb_ctx* ctx, int rank, const uint64_t* dims, tncb_tensor** out, int dtype) {
  if (rank < 0 || rank > kMaxLegs) return fail(TNCB_ERR_INVALID, "tensor rank out of range");
  if (!dtype_size(dtype)) return fail(TNCB_ERR_INVALID, "dtype must be TNCB_C128 or TNCB_C64");
  tncb_tensor* t = new tncb_tensor();
  t->rank = rank; t->elems = 1; t->dtype = dtype;
  for (int i = 0; i < rank; i++) { t->dims[i] = dims[i]; t->elems *= dims[i]; }
  t->bytes = std::max<size_t>(t->elems * dtype_size(dtype), 16);
  void* p = nullptr;
  int rc = ctx->arena.alloc(t->bytes, &p);
  if (rc) { delete t; return rc; }
  t->ptr = (double2*)p;
  *out = t;
  return TNCB_OK;
}

} // namespace tncb

using namespace tncb;

extern "C" {

int tncb_ctx_create(int device, size_t arena_bytes, tncb_ctx** out) {
  if (!out) return fail(TNCB_ERR_INVALID, "out is null");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    return fail(TNCB_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) +
                                   "); libtncb200 has no CPU fallback");
  }
  if (device < 0 || device >= count) return fail(TNCB_ERR_INVALID, "device index out of range");
  TNCB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  TNCB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(TNCB_ERR_CUDA, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
                                   ", libtncb200 is built for sm_100a only");
  tncb_ctx* ctx = new tncb_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->arena.capacity_limit = arena_bytes;
  if (const char* e = std::getenv("TNCB_OZAKI_SLICES")) ctx->oz_slices = std::max(0, std::min(8, atoi(e)));
  if (const char* e = std::getenv("TNCB_TCGEN05_ENGINE")) ctx->oz_engine = atoi(e) == 1 ? 1 : 0;
  if (const char* e = std::getenv("TNCB_CRT_MODULI")) ctx->crt_nmod_force = std::max(0, std::min(20, atoi(e)));
  if (const char* e = std::getenv("TNCB_CRT_PRODUCTS")) { const int v = atoi(e); ctx->crt_products = (v == 3 || v == 4) ? v : 0; }
  if (const char* e = std::getenv("TNCB_CRT_MIN_K3")) ctx->crt_kara_min_k = std::max(1, atoi(e));
  if (const char* e = std::getenv("TNCB_CRT_GROUP")) ctx->crt_group = std::max(1, atoi(e));
  if (const char* e = std::getenv("TNCB_CRT_WS_GB")) ctx->crt_ws_bytes = (size_t)std::max(1, atoi(e)) << 30;
  cudaError_t se = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (se != cudaSuccess) { delete ctx; return fail(TNCB_ERR_CUDA, cudaGetErrorString(se)); }
  // keep freed workspace memory in the stream-ordered pool
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  *out = ctx;
  return TNCB_OK;
}

void tncb_ctx_destroy(tncb_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& c : ctx->plan_cache) tncb_plan_destroy(c.plan);                         // the contract_tensor_network plan cache
  ctx->plan_cache.clear();
  while (!ctx->plans.empty()) tncb_plan_release_device_state(ctx->plans.back());   // plans may outlive the ctx
  tncb_comm_destroy(ctx);
  if (ctx->tab) cudaFree(ctx->tab);
  if (ctx->partial) cudaFree(ctx->partial);
  if (ctx->stage_host) cudaFreeHost(ctx->stage_host);
  if (ctx->gemm_ev0) { cudaEventDestroy(ctx->gemm_ev0); cudaEventDestroy(ctx->gemm_ev1); }
  for (cudaEvent_t e : ctx->gemm_pool) cudaEventDestroy(e);
  if (ctx->h2d_stream) {
    cudaStreamSynchronize(ctx->h2d_stream); cudaStreamSynchronize(ctx->d2h_stream);
    for (auto& sl : ctx->host_slot) {
      for (int i = 0; i < 3; i++) if (sl.buf[i]) cudaFree(sl.buf[i]);
      cudaEventDestroy(sl.in_done); cudaEventDestroy(sl.comp_done); cudaEventDestroy(sl.out_done);
    }
    cudaStreamDestroy(ctx->h2d_stream); cudaStreamDestroy(ctx->d2h_stream);
  }
  ctx->arena.release_all();
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int tncb_ctx_synchronize(tncb_ctx* ctx) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ctx->d2h_stream) {   // results of tncb_contract_pair_host still travelling to the host
    TNCB_CUDA(cudaStreamSynchronize(ctx->h2d_stream));
    TNCB_CUDA(cudaStreamSynchronize(ctx->d2h_stream));
    for (auto& sl : ctx->host_slot) sl.busy = false;
  }
  return TNCB_OK;
}

// tetra::contract for HOST operands, pipelined: the call only enqueues (H2D of a and b on a copy stream, the pair
// kernels on the ctx stream, D2H of the result on a second copy stream) and returns; with back-to-back calls the upload
// of pair j+1, the contraction of pair j and the download of pair j-1 overlap (PCIe is full duplex), so the steady-state
// cost per pair is max(H2D, kernels, D2H) instead of their sum.  Host buffers must be pinned (cudaHostAlloc /
// torch pin_memory) for the copies to be asynchronous; they may be touched again after tncb_ctx_synchronize.
int tncb_contract_pair_host(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const uint64_t* a_dims, const double* host_a,
                            int n_b, const uint64_t* b_legs, const uint64_t* b_dims, const double* host_b, double* host_c) {
  if (!ctx || !host_a || !host_b || !host_c) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  PairPlan P;
  int rc = plan_pair(n_a, a_legs, a_dims, n_b, b_legs, b_dims, P);
  if (rc) return rc;
  size_t ea = 1, eb = 1;
  for (int i = 0; i < n_a; i++) ea *= a_dims[i];
  for (int i = 0; i < n_b; i++) eb *= b_dims[i];
  const size_t need[3] = {std::max<size_t>(ea * 16, 16), std::max<size_t>(eb * 16, 16), std::max<size_t>((size_t)(P.M * P.N) * 16, 16)};
  if (!ctx->h2d_stream) {
    TNCB_CUDA(cudaStreamCreateWithFlags(&ctx->h2d_stream, cudaStreamNonBlocking));
    TNCB_CUDA(cudaStreamCreateWithFlags(&ctx->d2h_stream, cudaStreamNonBlocking));
    for (auto& sl : ctx->host_slot) {
      TNCB_CUDA(cudaEventCreateWithFlags(&sl.in_done, cudaEventDisableTiming));
      TNCB_CUDA(cudaEventCreateWithFlags(&sl.comp_done, cudaEventDisableTiming));
      TNCB_CUDA(cudaEventCreateWithFlags(&sl.out_done, cudaEventDisableTiming));
    }
  }
  tncb_ctx::HostSlot& sl = ctx->host_slot[ctx->host_jobs % 3];
  if (sl.busy) TNCB_CUDA(cudaEventSynchronize(sl.out_done));        // the job that used this slot three calls ago
  for (int i = 0; i < 3; i++)
    if (sl.bytes[i] < need[i]) {                                     // private buffers (not the arena: they are touched by three streams)
      if (sl.buf[i]) TNCB_CUDA(cudaFree(sl.buf[i]));
      sl.buf[i] = nullptr; sl.bytes[i] = 0;
      cudaError_t e = cudaMalloc(&sl.buf[i], need[i]);
      if (e != cudaSuccess) { cudaGetLastError(); return fail(TNCB_ERR_OOM, std::string("cudaMalloc (host pipeline): ") + cudaGetErrorString(e)); }
      sl.bytes[i] = need[i];
    }
  TNCB_CUDA(cudaMemcpyAsync(sl.buf[0], host_a, ea * 16, cudaMemcpyHostToDevice, ctx->h2d_stream));
  TNCB_CUDA(cudaMemcpyAsync(sl.buf[1], host_b, eb * 16, cudaMemcpyHostToDevice, ctx->h2d_stream));
  TNCB_CUDA(cudaEventRecord(sl.in_done, ctx->h2d_stream));
  TNCB_CUDA(cudaStreamWaitEvent(ctx->stream, sl.in_done, 0));
  if ((rc = launch_pair(ctx, P, (const double2*)sl.buf[0], (const double2*)sl.buf[1], (double2*)sl.buf[2]))) return rc;
  TNCB_CUDA(cudaEventRecord(sl.comp_done, ctx->stream));
  TNCB_CUDA(cudaStreamWaitEvent(ctx->d2h_stream, sl.comp_done, 0));
  TNCB_CUDA(cudaMemcpyAsync(host_c, sl.buf[2], (size_t)(P.M * P.N) * 16, cudaMemcpyDeviceToHost, ctx->d2h_stream));
  TNCB_CUDA(cudaEventRecord(sl.out_done, ctx->d2h_stream));
  // the next upload into THIS slot's operands must not overtake these kernels: ordered by out_done (waited above)
  sl.busy = true;
  ctx->host_jobs++;
  return TNCB_OK;
}

void* tncb_ctx_stream(tncb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int tncb_ctx_trim(tncb_ctx* ctx, uint64_t* freed_bytes, uint64_t* reserved_bytes) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));      // stream-ordered reuse: nothing may still be running in a freed block
  for (auto& c : ctx->plan_cache) tncb_plan_destroy(c.plan);   // the internal plans behind tncb_contract_tensor_network
  ctx->plan_cache.clear();
  const size_t f = ctx->arena.trim();
  if (freed_bytes) *freed_bytes = f;
  if (reserved_bytes) *reserved_bytes = ctx->arena.reserved;
  return TNCB_OK;
}

int tncb_ctx_stats(tncb_ctx* ctx, uint64_t* kernel_launches, uint64_t* arena_peak_bytes, uint64_t* arena_live_bytes) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  if (kernel_launches) *kernel_launches = ctx->launches;
  if (arena_peak_bytes) *arena_peak_bytes = ctx->arena.peak;
  if (arena_live_bytes) *arena_live_bytes = ctx->arena.live;
  return TNCB_OK;
}

int tncb_ctx_reset_stats(tncb_ctx* ctx) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  ctx->launches = 0; ctx->arena.peak = ctx->arena.live;
  for (int i = 0; i < 8; i++) ctx->engine_count[i] = 0;
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_slices(tncb_ctx* ctx, int slices) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  if (slices != 0 && (slices < 2 || slices > 8)) return fail(TNCB_ERR_INVALID, "slices must be 0 or in [2, 8]");
  ctx->oz_slices = slices;
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_engine(tncb_ctx* ctx, int engine) {
  if (!ctx || (engine != 0 && engine != 1)) return fail(TNCB_ERR_INVALID, "engine must be 0 (modular / CRT) or 1 (digit slicing)");
  ctx->oz_engine = engine;
  return TNCB_OK;
}

int tncb_ctx_set_tolerance(tncb_ctx* ctx, double rel) {
  if (!ctx || !(rel >= 0.0) || rel >= 1.0) return fail(TNCB_ERR_INVALID, "tolerance must be in [0, 1)");
  ctx->crt_tol = rel;
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_moduli(tncb_ctx* ctx, int n_moduli) {
  if (!ctx || (n_moduli != 0 && (n_moduli < 2 || n_moduli > 20))) return fail(TNCB_ERR_INVALID, "n_moduli must be 0 (auto) or in [2, 20]");
  ctx->crt_nmod_force = n_moduli;
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_products(tncb_ctx* ctx, int products, long long min_k3) {
  if (!ctx || (products != 0 && products != 3 && products != 4)) return fail(TNCB_ERR_INVALID, "products must be 0 (auto), 3 or 4");
  ctx->crt_products = products;
  if (min_k3 > 0) ctx->crt_kara_min_k = min_k3;
  return TNCB_OK;
}

int tncb_ctx_last_tcgen05_products(tncb_ctx* ctx, int* products) {
  if (!ctx || !products) return fail(TNCB_ERR_INVALID, "null argument");
  *products = ctx->last_products;
  return TNCB_OK;
}

int tncb_tcgen05_bound(uint64_t k, double rel, int n_moduli_force, int* n_moduli, int* bits_a, int* bits_b, double* bound) {
  if (k == 0 || (n_moduli_force != 0 && (n_moduli_force < 2 || n_moduli_force > 20))) return fail(TNCB_ERR_INVALID, "bad argument");
  int n, a, b;
  crt_choose((long long)k, crt_bits_for_tolerance((long long)k, rel), n_moduli_force, &n, &a, &b);
  if (n_moduli) *n_moduli = n;
  if (bits_a) *bits_a = a;
  if (bits_b) *bits_b = b;
  // truncation of a: < 2^(eA-a) per part, of b: < 2^(eB-b); 2K real products each way per real output; 2^e <= 2 max
  if (bound) *bound = 4.0 * (double)k * (std::ldexp(1.0, 1 - a) + std::ldexp(1.0, 1 - b));
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_workspace(tncb_ctx* ctx, size_t bytes) {
  if (!ctx || bytes < ((size_t)1 << 20)) return fail(TNCB_ERR_INVALID, "workspace must be >= 1 MiB");
  ctx->crt_ws_bytes = bytes;
  return TNCB_OK;
}

int tncb_tcgen05_tables(int n_moduli, int* moduli, double* rho1, double* rho2, double* log2_product) {
  if (n_moduli < 2 || n_moduli > 20) return fail(TNCB_ERR_INVALID, "n_moduli must be in [2, 20]");
  return crt_export_tables(n_moduli, moduli, rho1, rho2, log2_product);
}

int tncb_ctx_engine_counts(tncb_ctx* ctx, uint64_t counts[8]) {
  if (!ctx || !counts) return fail(TNCB_ERR_INVALID, "null argument");
  for (int i = 0; i < 8; i++) counts[i] = ctx->engine_count[i];
  return TNCB_OK;
}

int tncb_ctx_last_tcgen05_info(tncb_ctx* ctx, double* int8_ops, int* n_moduli) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  if (int8_ops) *int8_ops = ctx->last_int8_ops;
  if (n_moduli) *n_moduli = ctx->last_nmod;
  return TNCB_OK;
}

int tncb_ctx_set_tcgen05_threshold(tncb_ctx* ctx, long long min_tiles, long long min_k) {
  if (!ctx || min_tiles < 1 || min_k < 1) return fail(TNCB_ERR_INVALID, "bad argument");
  ctx->oz_min_tiles = min_tiles; ctx->oz_min_k = min_k;
  // the modular engine: the same call routes every pair with M, N >= 128 and K >= min_k to it when min_tiles == 1
  ctx->crt_min_k = min_k;
  ctx->crt_min_mnk = min_tiles <= 1 ? 0.0 : 268435456.0;
  return TNCB_OK;
}

int tncb_ctx_time_gemm(tncb_ctx* ctx, int enable) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  if (enable < 0 || enable > 2) return fail(TNCB_ERR_INVALID, "enable must be 0, 1 (last launch) or 2 (accumulate)");
  if (enable && !ctx->gemm_ev0) { TNCB_CUDA(cudaEventCreate(&ctx->gemm_ev0)); TNCB_CUDA(cudaEventCreate(&ctx->gemm_ev1)); }
  ctx->time_gemm = enable; ctx->gemm_ev_valid = false; ctx->gemm_used = 0; ctx->gemm_ops.clear();
  return TNCB_OK;
}

int tncb_ctx_gemm_totals(tncb_ctx* ctx, double* ms, double* ops, uint64_t* launches) {
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  double tms = 0.0, tops = 0.0;
  for (size_t i = 0; i + 1 < ctx->gemm_used; i += 2) {
    float t = 0.f;
    TNCB_CUDA(cudaEventElapsedTime(&t, ctx->gemm_pool[i], ctx->gemm_pool[i + 1]));
    tms += t; tops += ctx->gemm_ops[i / 2];
  }
  if (ms) *ms = tms;
  if (ops) *ops = tops;
  if (launches) *launches = ctx->gemm_used / 2;
  ctx->gemm_used = 0; ctx->gemm_ops.clear();
  return TNCB_OK;
}

int tncb_ctx_last_gemm_ms(tncb_ctx* ctx, float* ms) {
  if (!ctx || !ms) return fail(TNCB_ERR_INVALID, "null argument");
  if (!ctx->gemm_ev_valid) return fail(TNCB_ERR_INVALID, "no timed GEMM kernel yet");
  TNCB_CUDA(cudaEventSynchronize(ctx->gemm_ev1));
  TNCB_CUDA(cudaEventElapsedTime(ms, ctx->gemm_ev0, ctx->gemm_ev1));
  return TNCB_OK;
}

int tncb_tensor_alloc_dt(tncb_ctx* ctx, int rank, const uint64_t* dims, int dtype, tncb_tensor** out) {
  if (!ctx || !out || (rank > 0 && !dims)) return fail(TNCB_ERR_INVALID, "null argument");
  if (!dtype_size(dtype)) return fail(TNCB_ERR_INVALID, "dtype must be TNCB_C128 or TNCB_C64");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  return tensor_new(ctx, rank, dims, out, dtype);
}

int tncb_tensor_alloc(tncb_ctx* ctx, int rank, const uint64_t* dims, tncb_tensor** out) {
  return tncb_tensor_alloc_dt(ctx, rank, dims, TNCB_C128, out);
}

int tncb_tensor_upload_dt(tncb_ctx* ctx, int rank, const uint64_t* dims, int dtype, const void* host, tncb_tensor** out) {
  if (!host) return fail(TNCB_ERR_INVALID, "host buffer is null");
  int rc = tncb_tensor_alloc_dt(ctx, rank, dims, dtype, out);
  if (rc) return rc;
  tncb_tensor* t = *out;
  // pageable or pinned host memory both work; the copy is ordered on the ctx stream
  TNCB_CUDA(cudaMemcpyAsync(t->ptr, host, t->elems * dtype_size(dtype), cudaMemcpyHostToDevice, ctx->stream));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  return TNCB_OK;
}

int tncb_tensor_upload(tncb_ctx* ctx, int rank, const uint64_t* dims, const double* host, tncb_tensor** out) {
  return tncb_tensor_upload_dt(ctx, rank, dims, TNCB_C128, host, out);
}

int tncb_tensor_dtype(const tncb_tensor* t) { return t ? t->dtype : TNCB_ERR_INVALID; }

// raw copies in the tensor's own dtype
int tncb_tensor_download(tncb_ctx* ctx, const tncb_tensor* t, double* host) {
  if (!ctx || !t || !host) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaMemcpyAsync(host, t->ptr, t->elems * dtype_size(t->dtype), cudaMemcpyDeviceToHost, ctx->stream));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  return TNCB_OK;
}

int tncb_tensor_write(tncb_ctx* ctx, tncb_tensor* t, const double* host) {
  if (!ctx || !t || !host) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaMemcpyAsync(t->ptr, host, t->elems * dtype_size(t->dtype), cudaMemcpyHostToDevice, ctx->stream));
  return TNCB_OK;
}

int tncb_tensor_read(tncb_ctx* ctx, const tncb_tensor* t, double* host) {
  if (!ctx || !t || !host) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  TNCB_CUDA(cudaMemcpyAsync(host, t->ptr, t->elems * dtype_size(t->dtype), cudaMemcpyDeviceToHost, ctx->stream));
  return TNCB_OK;
}

int tncb_tensor_free(tncb_ctx* ctx, tncb_tensor* t) {
  if (!t) return TNCB_OK;
  if (!ctx) return fail(TNCB_ERR_INVALID, "ctx is null");
  // Stream-ordered reuse: every kernel of this ctx runs on ctx->stream, so a later
  // allocation of the same bytes is only ever touched by later kernels.
  if (t->owned && t->ptr) ctx->arena.free(t->ptr, t->bytes);
  delete t;
  return TNCB_OK;
}

int tncb_tensor_rank(const tncb_tensor* t) { return t ? t->rank : TNCB_ERR_INVALID; }
int tncb_tensor_dims(const tncb_tensor* t, uint64_t* dims_out) {
  if (!t || !dims_out) return fail(TNCB_ERR_INVALID, "null argument");
  for (int i = 0; i < t->rank; i++) dims_out[i] = t->dims[i];
  return TNCB_OK;
}
uint64_t tncb_tensor_elements(const tncb_tensor* t) { return t ? t->elems : 0; }
void* tncb_tensor_device_ptr(const tncb_tensor* t) { return t ? (void*)t->ptr : nullptr; }

static int check_tensor_legs(const tncb_tensor* t, int n, const char* who) {
  if (!t) return fail(TNCB_ERR_UNCONTRACTED, std::string("tensor ") + who + " is null");
  if (n != t->rank) return fail(TNCB_ERR_INVALID, std::string("leg count of ") + who + " != tensor rank");
  return TNCB_OK;
}

// no implicit promotion: every tensor of one call has the same dtype
static int check_same_dtype(const tncb_tensor* a, const tncb_tensor* b) {
  if (a->dtype != b->dtype) return fail(TNCB_ERR_INVALID, "operands have different dtypes (complex64 vs complex128)");
  return TNCB_OK;
}

int tncb_contract_pair_into(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const tncb_tensor* a,
                            int n_b, const uint64_t* b_legs, const tncb_tensor* b, tncb_tensor* out) {
  if (!ctx || !out) return fail(TNCB_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_tensor_legs(a, n_a, "a")) || (rc = check_tensor_legs(b, n_b, "b"))) return rc;
  if ((rc = check_same_dtype(a, b)) || (rc = check_same_dtype(a, out))) return rc;
  TNCB_CUDA(cudaSetDevice(ctx->device));
  PairPlan P;
  if ((rc = plan_pair(n_a, a_legs, a->dims, n_b, b_legs, b->dims, P))) return rc;
  if ((uint64_t)(P.M * P.N) != out->elems) return fail(TNCB_ERR_SHAPE, "output tensor has the wrong number of elements");
  return launch_pair(ctx, P, a->ptr, b->ptr, out->ptr, a->dtype);
}

int tncb_contract_pair_keep(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const tncb_tensor* a,
                            int n_b, const uint64_t* b_legs, const tncb_tensor* b, tncb_tensor** out) {
  if (!ctx || !out) return fail(TNCB_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_tensor_legs(a, n_a, "a")) || (rc = check_tensor_legs(b, n_b, "b"))) return rc;
  if ((rc = check_same_dtype(a, b))) return rc;
  TNCB_CUDA(cudaSetDevice(ctx->device));
  PairPlan P;
  if ((rc = plan_pair(n_a, a_legs, a->dims, n_b, b_legs, b->dims, P))) return rc;
  tncb_tensor* c = nullptr;
  if ((rc = tensor_new(ctx, (int)P.out_dims.size(), P.out_dims.data(), &c, a->dtype))) return rc;
  if ((rc = launch_pair(ctx, P, a->ptr, b->ptr, c->ptr, a->dtype))) { tncb_tensor_free(ctx, c); return rc; }
  *out = c;
  return TNCB_OK;
}

int tncb_contract_pair(tncb_ctx* ctx, int n_out, const uint64_t* out_legs,
                       int n_a, const uint64_t* a_legs, tncb_tensor* a,
                       int n_b, const uint64_t* b_legs, tncb_tensor* b, tncb_tensor** out) {
  if (!ctx || !out) return fail(TNCB_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_tensor_legs(a, n_a, "a")) || (rc = check_tensor_legs(b, n_b, "b"))) return rc;
  if (a == b) return fail(TNCB_ERR_INVALID, "a and b are the same tensor");
  if ((rc = check_same_dtype(a, b))) return rc;
  if (out_legs) {
    PairPlan P;
    if ((rc = plan_pair(n_a, a_legs, a->dims, n_b, b_legs, b->dims, P))) return rc;
    bool same = (int)P.out_legs.size() == n_out;
    for (int i = 0; same && i < n_out; i++) same = P.out_legs[i] == out_legs[i];
    if (!same) return fail(TNCB_ERR_INVALID, "out_legs must equal (b \\ a) ++ (a \\ b)");
  }
  rc = tncb_contract_pair_keep(ctx, n_a, a_legs, a, n_b, b_legs, b, out);
  if (rc) return rc;
  // ownership moved to the callee, exactly like the Rust by-value call (contraction.rs:78-84)
  tncb_tensor_free(ctx, a);
  tncb_tensor_free(ctx, b);
  return TNCB_OK;
}

int tncb_permute(tncb_ctx* ctx, tncb_tensor* t, const int* perm, tncb_tensor** out) {
  if (!ctx || !t || !out || (t->rank > 0 && !perm)) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  bool seen[kMaxLegs] = {false};
  uint64_t odims[kMaxLegs];
  for (int i = 0; i < t->rank; i++) {
    if (perm[i] < 0 || perm[i] >= t->rank || seen[perm[i]]) return fail(TNCB_ERR_INVALID, "perm is not a permutation");
    seen[perm[i]] = true; odims[i] = t->dims[perm[i]];
  }
  tncb_tensor* o = nullptr;
  int rc = tensor_new(ctx, t->rank, odims, &o, t->dtype);
  if (rc) return rc;
  if ((rc = launch_permute(ctx, t->ptr, o->ptr, t->rank, t->dims, perm, t->dtype))) { tncb_tensor_free(ctx, o); return rc; }
  tncb_tensor_free(ctx, t);
  *out = o;
  return TNCB_OK;
}

int tncb_tensor_add(tncb_ctx* ctx, tncb_tensor* dst, const tncb_tensor* src) {
  if (!ctx || !dst || !src) return fail(TNCB_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_same_dtype(dst, src))) return rc;
  if (dst->elems != src->elems) return fail(TNCB_ERR_SHAPE, "tensor_add: element counts differ");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  return launch_add(ctx, dst->ptr, src->ptr, dst->elems, dst->dtype);
}

int tncb_conjugate(tncb_ctx* ctx, tncb_tensor* t) {
  if (!ctx || !t) return fail(TNCB_ERR_INVALID, "null argument");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  return launch_conj(ctx, t->ptr, t->elems, t->dtype);
}

} // extern "C"

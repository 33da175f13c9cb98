// sm_100a kernels of the pairwise-contraction hot path (replaces tetra::contract, called at
// tnc/src/tensornetwork/contraction.rs:78-84, i.e. HPTT transposes + faer/MKL ZGEMM).
//
//   C[n, m] = sum_k Bt[n, k] * At[k, m]      (complex128, C row-major [N][M])
//   Bt[n, k] = B[offBn(n) + offBk(k)],  At[k, m] = A[offAm(m) + offAk(k)]
//
// The permutes of the reference's TTGT are never materialised: both operands are gathered
// through separable mixed-radix offset functions while the tile is staged into shared memory.
//
//   K0  strided kernel: G lanes per output element cooperate over K (shuffle reduction),
//       optional deterministic split-K; for tiny and for low-intensity pairs.
//   K1  fused gather + ZGEMM: cp.async 16-byte gathers into a fragment-ordered shared-memory
//       ring, FP64 tensor-core DMMA (mma.sync.m8n8k4.f64, 4 real MMAs per complex tile).
//       tcgen05.mma has no f64 kind, so the FP64 tensor path on sm_100a is DMMA; measured
//       peak 37.2 TFLOP/s (profiles/r01_fp64_peak_microbench.txt).
//
// complex64 (TNCB_C64): every kernel has a float2 instantiation that reads the 8-byte operands, widens them exactly to
// f64, runs the f64 arithmetic of the complex128 kernel in the same order and rounds once at the final store (split-K
// partials stay f64).  Launch configurations are chosen from the pair alone, so the complex64 result is bit for bit
// complex64(complex128 kernel(widen(a), widen(b))).
#include "internal.h"
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <nvtx3/nvToolsExt.h>   // header-only NVTX v3: no link dependency, no cost unless a tool is attached

namespace tncb {

// TNCB_NVTX=1: one NVTX range per pairwise contraction ("K1' M=.. N=.. K=..") around its launches, so that a timeline
// (nsys / ncu --nvtx) shows the path step by step -- the counterpart of the reference's per-contraction flame-graph spans.
struct NvtxPairRange {
  bool on;
  NvtxPairRange(const PairPlan& P) {
    static const bool enabled = std::getenv("TNCB_NVTX") != nullptr;
    on = enabled;
    if (on) {
      char buf[96];
      snprintf(buf, sizeof buf, "pair K%d M=%lld N=%lld K=%lld", P.kernel_class, P.M, P.N, P.K);
      nvtxRangePushA(buf);
    }
  }
  ~NvtxPairRange() { if (on) nvtxRangePop(); }
};

// ------------------------------------------------------------------------------------------
// element access: load + exact widening to f64, one rounding at the store
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 widen(const double2 v) { return v; }
__device__ __forceinline__ double2 widen(const float2 v) { return make_double2((double)v.x, (double)v.y); }
template <typename T>
__device__ __forceinline__ double2 ldg_wide(const T* p) { return widen(__ldg(p)); }
__device__ __forceinline__ void st_round(double2* p, double x, double y) { *p = make_double2(x, y); }
__device__ __forceinline__ void st_round(float2* p, double x, double y) { *p = make_float2((float)x, (float)y); }

// ------------------------------------------------------------------------------------------
// index helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ long long decomp_a(long long idx, const LegList& L) {
  long long off = 0;
  for (int g = L.n - 1; g > 0; --g) {
    long long d = L.dim[g];
    long long q = idx / d;
    off += (idx - q * d) * L.sa[g];
    idx = q;
  }
  if (L.n > 0) off += idx * L.sa[0];
  return off;
}

__device__ __forceinline__ void decomp_ab(long long idx, const LegList& L, long long& oa, long long& ob) {
  long long a = 0, b = 0;
  for (int g = L.n - 1; g > 0; --g) {
    long long d = L.dim[g];
    long long q = idx / d;
    long long r = idx - q * d;
    a += r * L.sa[g];
    b += r * L.sb[g];
    idx = q;
  }
  if (L.n > 0) { a += idx * L.sa[0]; b += idx * L.sb[0]; }
  oa = a; ob = b;
}

// ------------------------------------------------------------------------------------------
// K0: strided kernel with G cooperating lanes per output and optional split-K
// ------------------------------------------------------------------------------------------
struct K0Args {
  LegList m, n, k;
  long long M, N, K;
  long long kchunk; // K range handled by one blockIdx.y
};

constexpr int K0_THREADS = 256;
constexpr int K0_KT = 1024;

// T: operand type, TO: output type (double2 for split-K partials)
template <int G, typename T, typename TO>
__global__ void __launch_bounds__(K0_THREADS)
k0_kernel(const T* __restrict__ A, const T* __restrict__ B, TO* __restrict__ dst,
          const __grid_constant__ K0Args p) {
  __shared__ long long s_ka[K0_KT];
  __shared__ long long s_kb[K0_KT];
  const int tid = threadIdx.x;
  const int lane_g = tid % G;
  const long long MN = p.M * p.N;
  const long long o = (long long)blockIdx.x * (K0_THREADS / G) + tid / G;
  const bool valid = o < MN;
  long long n = 0, m = 0;
  if (valid) { n = o / p.M; m = o - n * p.M; }
  const long long offA0 = decomp_a(m, p.m);
  const long long offB0 = decomp_a(n, p.n);
  const long long kbeg = (long long)blockIdx.y * p.kchunk;
  const long long kend = min(p.K, kbeg + p.kchunk);
  double cr = 0.0, ci = 0.0;
  for (long long kb = kbeg; kb < kend; kb += K0_KT) {
    const int cnt = (int)min((long long)K0_KT, kend - kb);
    __syncthreads();
    for (int i = tid; i < cnt; i += K0_THREADS) {
      long long oa, ob;
      decomp_ab(kb + i, p.k, oa, ob);
      s_ka[i] = oa; s_kb[i] = ob;
    }
    __syncthreads();
    if (valid) {
#pragma unroll 4
      for (int i = lane_g; i < cnt; i += G) {
        const double2 a = ldg_wide(A + offA0 + s_ka[i]);
        const double2 b = ldg_wide(B + offB0 + s_kb[i]);
        cr = fma(b.x, a.x, cr); cr = fma(-b.y, a.y, cr);
        ci = fma(b.x, a.y, ci); ci = fma(b.y, a.x, ci);
      }
    }
  }
#pragma unroll
  for (int d = G / 2; d > 0; d >>= 1) {
    cr += __shfl_xor_sync(0xffffffffu, cr, d);
    ci += __shfl_xor_sync(0xffffffffu, ci, d);
  }
  if (valid && lane_g == 0) st_round(dst + (long long)blockIdx.y * MN + o, cr, ci);
}

template <typename TO>
__global__ void reduce_partials_kernel(const double2* __restrict__ part, TO* __restrict__ C,
                                       long long MN, int ksplit) {
  long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= MN) return;
  double cr = 0.0, ci = 0.0;
  for (int s = 0; s < ksplit; s++) { double2 v = part[(long long)s * MN + o]; cr += v.x; ci += v.y; }
  st_round(C + o, cr, ci);
}

// ------------------------------------------------------------------------------------------
// K1: fused gather + DMMA ZGEMM
// ------------------------------------------------------------------------------------------
__global__ void build_tables_kernel(const __grid_constant__ LegList m, const __grid_constant__ LegList n,
                                    const __grid_constant__ LegList k, long long M, long long N, long long K,
                                    long long* __restrict__ tab) {
  const long long total = M + N + 2 * K;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (i < M) tab[i] = decomp_a(i, m);
    else if (i < M + N) tab[i] = decomp_a(i - M, n);
    else if (i < M + N + K) { long long oa, ob; decomp_ab(i - M - N, k, oa, ob); tab[i] = oa; tab[i + K] = ob; }
  }
}

__device__ __forceinline__ void cp_async16(unsigned smem_addr, const void* gptr, bool pred) {
  const int src = pred ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_addr), "l"(gptr), "r"(src));
}
// complex64 operands: 8-byte gathers (.cg only takes 16 bytes)
__device__ __forceinline__ void cp_async8(unsigned smem_addr, const void* gptr, bool pred) {
  const int src = pred ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(smem_addr), "l"(gptr), "r"(src));
}
template <typename T>
__device__ __forceinline__ void cp_async_elem(unsigned smem_addr, const T* gptr, bool pred) {
  if constexpr (sizeof(T) == 16) cp_async16(smem_addr, gptr, pred);
  else cp_async8(smem_addr, gptr, pred);
}
// volatile so that ptxas keeps the load where it is written (it otherwise sinks the prefetch to
// its first use and the latency reappears as a long_scoreboard stall in the gather issue)
__device__ __forceinline__ long long ldg_pinned(const long long* p) {
  long long v;
  asm volatile("ld.global.nc.s64 %0, [%1];\n" : "=l"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N_)); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c0), "+d"(c1)
      : "d"(a), "d"(b));
}

constexpr int K1_BK = 16;

struct K1Args {
  const void* A;        // double2 (complex128) or float2 (complex64) operands
  const void* B;
  void* C;              // complex128: double2; complex64: float2, or double2 partials when ksplit > 1
  const long long* offAm;
  const long long* offBn;
  const long long* offAk;
  const long long* offBk;
  long long M, N, K;
  int tiles_m, tiles_n;
  int ksplit;           // >1: blockIdx.x / tiles selects a K range, C points at the partial buffer
  int chunks_per_split; // BK-chunks per K range
};

// Shared-memory tiles are stored in DMMA fragment order so that every fragment load is one
// conflict-free 512-byte LDS.128 per warp:
//   row operand Bt (rows n, cols k):  slot = ((n/8)*(BK/4) + k/4)*32 + (n%8)*4 + k%4
//   col operand At (rows k, cols m):  slot = ((k/4)*(BM/8) + m/8)*32 + (m%8)*4 + k%4
//
// Loader mapping (per operand, chosen by the planner from the operand's strides):
//   KFAST  : consecutive threads walk the K index   -> thread owns kk = tid%BK, rows tid/BK + (NT/BK)*j
//   !KFAST : consecutive threads walk the free index -> warp w owns kk in [w*BK/NW, (w+1)*BK/NW),
//            lane l owns rows l + 32*j
// so a thread needs only 1 (KFAST) or BK/NW (!KFAST) K-offsets per chunk.  Those offsets are
// prefetched one chunk ahead into registers and the cp.async gathers of stage kc+STAGES-1 are
// issued in the middle of chunk kc's DMMA stream, so no table load sits on the critical path
// (ncu r01: 20 % long_scoreboard on exactly those loads before this change).
//
// complex64 (T = float2): the ring holds the 8-byte elements in the same fragment order (half the shared memory per
// stage); the fragment loads widen them to f64 before the DMMAs.
template <int BN, int BM, int WARPS_N, int WARPS_M, int STAGES, bool B_KFAST, bool A_KFAST, int MINB = 1, typename T = double2>
__global__ void __launch_bounds__(WARPS_N* WARPS_M * 32, MINB)
k1_kernel(const __grid_constant__ K1Args p) {
  constexpr int BK = K1_BK;
  constexpr int NW = WARPS_N * WARPS_M;
  constexpr int NT = NW * 32;
  constexpr int TI = BN / WARPS_N / 8; // 8-row blocks per warp
  constexpr int TJ = BM / WARPS_M / 8; // 8-col blocks per warp
  constexpr int KPW = BK / NW;         // kk per warp in !KFAST mode
  static_assert(BK % NW == 0 && BN % 32 == 0 && BM % 32 == 0 && NT % BK == 0, "tile/threads mismatch");
  constexpr int B_ROWS = B_KFAST ? BN / (NT / BK) : BN / 32; // free-index positions per thread
  constexpr int A_COLS = A_KFAST ? BM / (NT / BK) : BM / 32;
  constexpr int B_KO = B_KFAST ? 1 : KPW;                    // K positions per thread
  constexpr int A_KO = A_KFAST ? 1 : KPW;
  constexpr int STAGE_ELEMS = BN * BK + BK * BM;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* smem = reinterpret_cast<T*>(smem_raw);
  const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem);
  constexpr unsigned ES = sizeof(T);
  const T* gA = static_cast<const T*>(p.A);
  const T* gB = static_cast<const T*>(p.B);

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int wn = warp / WARPS_M;
  const int wm = warp % WARPS_M;

  // grouped rasterisation: 8 n-tiles share the same band of At columns in L2
  int tn, tm;
  const int n_tiles = p.tiles_m * p.tiles_n;
  const int split = blockIdx.x / n_tiles;
  {
    const int GROUP = 8;
    const int t = blockIdx.x - split * n_tiles;
    const int per_group = GROUP * p.tiles_m;
    const int gid = t / per_group;
    const int first_n = gid * GROUP;
    const int gsize = min(p.tiles_n - first_n, GROUP);
    const int r = t - gid * per_group;
    tn = first_n + r % gsize;
    tm = r / gsize;
  }
  const long long n0 = (long long)tn * BN;
  const long long m0 = (long long)tm * BM;

  // ---- per-thread gather geometry (constant over the K loop) ----
  long long b_off[B_ROWS]; bool b_ok[B_ROWS]; int b_rslot[B_ROWS];
  int b_kk[B_KO], b_kslot[B_KO];
#pragma unroll
  for (int j = 0; j < B_ROWS; j++) {
    const int row = B_KFAST ? (tid / BK + (NT / BK) * j) : (lane + 32 * j);
    const long long gn = n0 + row;
    b_ok[j] = gn < p.N;
    b_off[j] = __ldg(p.offBn + (b_ok[j] ? gn : 0));
    b_rslot[j] = (row >> 3) * (BK / 4) * 32 + (row & 7) * 4;
  }
#pragma unroll
  for (int q = 0; q < B_KO; q++) {
    b_kk[q] = B_KFAST ? (tid % BK) : (warp * KPW + q);
    b_kslot[q] = (b_kk[q] >> 2) * 32 + (b_kk[q] & 3);
  }
  long long a_off[A_COLS]; bool a_ok[A_COLS]; int a_cslot[A_COLS];
  int a_kk[A_KO], a_kslot[A_KO];
#pragma unroll
  for (int j = 0; j < A_COLS; j++) {
    const int col = A_KFAST ? (tid / BK + (NT / BK) * j) : (lane + 32 * j);
    const long long gm = m0 + col;
    a_ok[j] = gm < p.M;
    a_off[j] = __ldg(p.offAm + (a_ok[j] ? gm : 0));
    a_cslot[j] = BN * BK + (col >> 3) * 32 + (col & 7) * 4;
  }
#pragma unroll
  for (int q = 0; q < A_KO; q++) {
    a_kk[q] = A_KFAST ? (tid % BK) : (warp * KPW + q);
    a_kslot[q] = (a_kk[q] >> 2) * (BM / 8) * 32 + (a_kk[q] & 3);
  }

  long long b_ko[B_KO], a_ko[A_KO]; bool b_kok[B_KO], a_kok[A_KO];
  auto fetch_ko = [&](long long k0) {
#pragma unroll
    for (int q = 0; q < B_KO; q++) {
      const long long gk = k0 + b_kk[q];
      b_kok[q] = gk < p.K;
      b_ko[q] = __ldg(p.offBk + (b_kok[q] ? gk : 0));
    }
#pragma unroll
    for (int q = 0; q < A_KO; q++) {
      const long long gk = k0 + a_kk[q];
      a_kok[q] = gk < p.K;
      a_ko[q] = __ldg(p.offAk + (a_kok[q] ? gk : 0));
    }
  };
  auto issue_stage = [&](int stage) {
    const unsigned sbase = smem_base + (unsigned)(stage * STAGE_ELEMS) * ES;
#pragma unroll
    for (int q = 0; q < B_KO; q++)
#pragma unroll
      for (int j = 0; j < B_ROWS; j++)
        cp_async_elem(sbase + (unsigned)(b_rslot[j] + b_kslot[q]) * ES, gB + (b_off[j] + b_ko[q]), b_ok[j] && b_kok[q]);
#pragma unroll
    for (int q = 0; q < A_KO; q++)
#pragma unroll
      for (int j = 0; j < A_COLS; j++)
        cp_async_elem(sbase + (unsigned)(a_cslot[j] + a_kslot[q]) * ES, gA + (a_off[j] + a_ko[q]), a_ok[j] && a_kok[q]);
  };

  double cr[TI][TJ][2], ci[TI][TJ][2];
#pragma unroll
  for (int i = 0; i < TI; i++)
#pragma unroll
    for (int j = 0; j < TJ; j++) { cr[i][j][0] = cr[i][j][1] = 0.0; ci[i][j][0] = ci[i][j][1] = 0.0; }

  const int nk_total = (int)((p.K + BK - 1) / BK);
  const int kc_begin = split * p.chunks_per_split;
  const int nk = max(0, min(nk_total - kc_begin, p.chunks_per_split));
  const long long kbase = (long long)kc_begin * BK;
#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) {
    if (s < nk) { fetch_ko(kbase + (long long)s * BK); issue_stage(s); }
    cp_async_commit();
  }
  if (STAGES - 1 < nk) fetch_ko(kbase + (long long)(STAGES - 1) * BK); // offsets of the first in-loop stage

  auto compute_kb = [&](const T* sB, const T* sA, int kb) {
    double2 bf[TI], af[TJ];
#pragma unroll
    for (int i = 0; i < TI; i++) bf[i] = widen(sB[((wn * TI + i) * (BK / 4) + kb) * 32 + lane]);
#pragma unroll
    for (int j = 0; j < TJ; j++) af[j] = widen(sA[(kb * (BM / 8) + wm * TJ + j) * 32 + lane]);
    // four passes so that the two DMMAs feeding one accumulator are TI*TJ*2 issues apart
#pragma unroll
    for (int i = 0; i < TI; i++)
#pragma unroll
      for (int j = 0; j < TJ; j++) {
        dmma884(cr[i][j][0], cr[i][j][1], bf[i].x, af[j].x);
        dmma884(ci[i][j][0], ci[i][j][1], bf[i].x, af[j].y);
      }
#pragma unroll
    for (int i = 0; i < TI; i++)
#pragma unroll
      for (int j = 0; j < TJ; j++) {
        dmma884(cr[i][j][0], cr[i][j][1], -bf[i].y, af[j].y); // SASS DMMA negates the operand for free
        dmma884(ci[i][j][0], ci[i][j][1], bf[i].y, af[j].x);
      }
  };

  for (int kc = 0; kc < nk; kc++) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    const T* sB = smem + (kc % STAGES) * STAGE_ELEMS;
    const T* sA = sB + BN * BK;
#pragma unroll
    for (int kb = 0; kb < BK / 8; kb++) compute_kb(sB, sA, kb);
    {
      // stage (kc-1)%STAGES was fully consumed before this iteration's barrier
      const int nxt = kc + STAGES - 1;
      if (nxt < nk) issue_stage(nxt % STAGES);
      cp_async_commit();
      if (nxt + 1 < nk) fetch_ko(kbase + (long long)(nxt + 1) * BK); // lands during the remaining DMMAs
    }
#pragma unroll
    for (int kb = BK / 8; kb < BK / 4; kb++) compute_kb(sB, sA, kb);
  }
  cp_async_wait<0>();

  // epilogue: D fragment (row = lane/4, cols = 2*(lane%4) + {0,1}) -> C row-major [N][M]
  const int g = lane >> 2, t2 = (lane & 3) * 2;
#pragma unroll
  for (int i = 0; i < TI; i++) {
    const long long gn = n0 + (wn * TI + i) * 8 + g;
    if (gn >= p.N) continue;
#pragma unroll
    for (int j = 0; j < TJ; j++) {
      const long long gm = m0 + (wm * TJ + j) * 8 + t2;
      const long long o = (long long)split * p.M * p.N + gn * p.M + gm;
      if (sizeof(T) == sizeof(double2) || p.ksplit > 1) {   // complex128 result, or f64 partials
        double2* dst = static_cast<double2*>(p.C) + o;
        if (gm < p.M) dst[0] = make_double2(cr[i][j][0], ci[i][j][0]);
        if (gm + 1 < p.M) dst[1] = make_double2(cr[i][j][1], ci[i][j][1]);
      } else {
        float2* dst = static_cast<float2*>(p.C) + o;
        if (gm < p.M) st_round(dst, cr[i][j][0], ci[i][j][0]);
        if (gm + 1 < p.M) st_round(dst + 1, cr[i][j][1], ci[i][j][1]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// permute (Permutor::apply / tetra transpose) and conjugate
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void permute_kernel(const T* __restrict__ in, T* __restrict__ out,
                               const __grid_constant__ LegList L, long long total) {
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total;
       o += (long long)gridDim.x * blockDim.x)
    out[o] = __ldg(in + decomp_a(o, L));
}

template <typename T>
__global__ void conj_kernel(T* __restrict__ d, long long total) {
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total;
       o += (long long)gridDim.x * blockDim.x)
    d[o].y = -d[o].y;
}

// ------------------------------------------------------------------------------------------
// host launchers
// ------------------------------------------------------------------------------------------
int ensure_tab(tncb_ctx* ctx, size_t elems) {
  if (ctx->tab_elems >= elems) return TNCB_OK;
  // stream-ordered: earlier kernels still reading the old table finish before the free
  if (ctx->tab) TNCB_CUDA(cudaFreeAsync(ctx->tab, ctx->stream));
  size_t want = std::max(elems, (size_t)1 << 20);
  TNCB_CUDA(cudaMallocAsync((void**)&ctx->tab, want * sizeof(long long), ctx->stream));
  ctx->tab_elems = want;
  ctx->tab_valid = false;
  return TNCB_OK;
}

int ensure_partial(tncb_ctx* ctx, size_t elems) {
  if (ctx->partial_elems >= elems) return TNCB_OK;
  if (ctx->partial) TNCB_CUDA(cudaFreeAsync(ctx->partial, ctx->stream));
  size_t want = std::max(elems, (size_t)1 << 18);
  TNCB_CUDA(cudaMallocAsync((void**)&ctx->partial, want * sizeof(double2), ctx->stream));
  ctx->partial_elems = want;
  return TNCB_OK;
}

template <int G, typename T>
static void launch_k0_g(dim3 grid, cudaStream_t st, const T* A, const T* B, void* dst, bool split, const K0Args& a) {
  if constexpr (sizeof(T) == sizeof(double2)) k0_kernel<G, T, double2><<<grid, K0_THREADS, 0, st>>>(A, B, (double2*)dst, a);
  else if (split) k0_kernel<G, T, double2><<<grid, K0_THREADS, 0, st>>>(A, B, (double2*)dst, a);
  else k0_kernel<G, T, float2><<<grid, K0_THREADS, 0, st>>>(A, B, (float2*)dst, a);
}

// K0 launch geometry: G lanes per output, ksplit K ranges (deterministic two-pass reduction)
void k0_config(int sm_count, const PairPlan& P, int* G_out, long long* ksplit_out, long long* kchunk_out) {
  const long long MN = P.M * P.N;
  const long long target = (long long)sm_count * 1024; // lanes wanted in flight
  int G = 1;
  while (G < 32 && MN * G < target && (long long)G * 2 <= P.K) G *= 2;
  long long ksplit = 1;
  const long long per_lane = P.K / G;
  if (MN * G < target && per_lane > 64) {
    ksplit = std::min(target / std::max(1LL, MN * G), per_lane / 32);
    ksplit = std::max(1LL, std::min(ksplit, 1024LL));
  }
  const long long kchunk = (P.K + ksplit - 1) / ksplit;
  ksplit = (P.K + kchunk - 1) / kchunk;
  *G_out = G; *ksplit_out = ksplit; *kchunk_out = kchunk;
}

// elements of split-K scratch a K0 pair needs (0 = none); used by the CUDA-graph planner
size_t k0_partial_elems(int sm_count, const PairPlan& P) {
  int G; long long ksplit, kchunk;
  k0_config(sm_count, P, &G, &ksplit, &kchunk);
  return ksplit > 1 ? (size_t)(P.M * P.N * ksplit) : 0;
}

template <typename T>
static int launch_k0(tncb_ctx* ctx, const PairPlan& P, const T* A, const T* B, T* C) {
  K0Args a;
  a.m = P.m; a.n = P.n; a.k = P.k; a.M = P.M; a.N = P.N; a.K = P.K;
  const long long MN = P.M * P.N;
  int G; long long ksplit;
  k0_config(ctx->sm_count, P, &G, &ksplit, &a.kchunk);
  void* dst = C;
  if (ksplit > 1) {
    if (ctx->partial_override) {   // graph capture: plan-owned scratch with a fixed address
      if ((size_t)(MN * ksplit) > ctx->partial_override_elems) return fail(TNCB_ERR_INVALID, "graph scratch too small");
      dst = ctx->partial_override;
    } else {
      int rc = ensure_partial(ctx, (size_t)(MN * ksplit));
      if (rc) return rc;
      dst = ctx->partial;
    }
  }
  const long long per_block = K0_THREADS / G;
  const long long blocks = (MN + per_block - 1) / per_block;
  if (blocks > 0x7fffffffLL) return fail(TNCB_ERR_UNSUPPORTED, "K0 grid too large");
  dim3 grid((unsigned)blocks, (unsigned)ksplit);
  const bool split = ksplit > 1;
  switch (G) {
    case 1: launch_k0_g<1>(grid, ctx->stream, A, B, dst, split, a); break;
    case 2: launch_k0_g<2>(grid, ctx->stream, A, B, dst, split, a); break;
    case 4: launch_k0_g<4>(grid, ctx->stream, A, B, dst, split, a); break;
    case 8: launch_k0_g<8>(grid, ctx->stream, A, B, dst, split, a); break;
    case 16: launch_k0_g<16>(grid, ctx->stream, A, B, dst, split, a); break;
    default: launch_k0_g<32>(grid, ctx->stream, A, B, dst, split, a); break;
  }
  ctx->launches++;
  ctx->engine_count[ksplit > 1 ? 1 : 0]++;
  if (ksplit > 1) {
    reduce_partials_kernel<<<(unsigned)((MN + 255) / 256), 256, 0, ctx->stream>>>((const double2*)dst, C, MN, (int)ksplit);
    ctx->launches++;
  }
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

// ------------------------------------------------------------------------------------------
// K0 batch: all independent tiny pairs of one level of the contraction tree in one launch.  Block b looks its pair up
// by binary search over the prefix of block counts; arithmetic per output element is that of k0_kernel<G> with the G
// k0_config chooses for the pair (lane i sums k = i, i + G, ...; xor-butterfly over G lanes), so plans with a static
// layout give bit-identical results to the pair-by-pair executor.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ long long decomp_c(long long idx, const CompactLegs& L) {
  long long off = 0;
  for (int g = L.n - 1; g > 0; --g) {
    const long long d = L.dim[g], q = idx / d;
    off += (idx - q * d) * L.sa[g];
    idx = q;
  }
  if (L.n > 0) off += idx * L.sa[0];
  return off;
}

template <typename T>
__global__ void __launch_bounds__(K0_THREADS)
k0_batch_kernel(const K0BatchItem* __restrict__ items, const int* __restrict__ block_start, int n_items, char* __restrict__ ws) {
  int lo = 0, hi = n_items;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(block_start + mid) <= (int)blockIdx.x) lo = mid; else hi = mid;
  }
  const K0BatchItem& it = items[lo];
  const int G = it.G, tid = threadIdx.x;
  const int lane_g = tid & (G - 1);
  const long long MN = it.M * it.N;
  const long long o = (long long)((int)blockIdx.x - __ldg(block_start + lo)) * (K0_THREADS / G) + tid / G;
  const bool valid = o < MN;
  long long n = 0, m = 0;
  if (valid) { n = o / it.M; m = o - n * it.M; }
  const T* A = reinterpret_cast<const T*>(ws + it.offA) + decomp_c(m, it.m);
  const T* B = reinterpret_cast<const T*>(ws + it.offB) + decomp_c(n, it.n);
  double cr = 0.0, ci = 0.0;
  if (valid) {
    for (long long i = lane_g; i < it.K; i += G) {
      long long oa = 0, ob = 0, idx = i;
      for (int g = it.k.n - 1; g > 0; --g) {
        const long long d = it.k.dim[g], q = idx / d, r = idx - q * d;
        oa += r * it.k.sa[g]; ob += r * it.k.sb[g];
        idx = q;
      }
      if (it.k.n > 0) { oa += idx * it.k.sa[0]; ob += idx * it.k.sb[0]; }
      const double2 a = widen(A[oa]);
      const double2 b = widen(B[ob]);
      cr = fma(b.x, a.x, cr); cr = fma(-b.y, a.y, cr);
      ci = fma(b.x, a.y, ci); ci = fma(b.y, a.x, ci);
    }
  }
  for (int d = 16; d > 0; d >>= 1)
    if (d < G) {   // (G is uniform over the block)
      cr += __shfl_xor_sync(0xffffffffu, cr, d);
      ci += __shfl_xor_sync(0xffffffffu, ci, d);
    }
  if (valid && lane_g == 0) st_round(reinterpret_cast<T*>(ws + it.offC) + o, cr, ci);
}

static bool compact_ok(const LegList& L) { return L.n <= kBatchGroups; }
static void compact_fill(const LegList& L, CompactLegs& C) {
  C.n = L.n; C._pad = 0;
  for (int i = 0; i < kBatchGroups; i++) { C.dim[i] = i < L.n ? L.dim[i] : 1; C.sa[i] = i < L.n ? L.sa[i] : 0; C.sb[i] = i < L.n ? L.sb[i] : 0; }
}

bool k0_batch_eligible(int sm_count, const PairPlan& P) {
  if (P.kernel_class != 0 || P.M * P.N == 0) return false;
  if (!compact_ok(P.m) || !compact_ok(P.n) || !compact_ok(P.k)) return false;
  if (P.K > 4096 || (double)P.M * (double)P.N * (double)P.K > 4194304.0) return false;   // tiny pairs only: no offset tables in the batch kernel
  int G; long long ksplit, kchunk;
  k0_config(sm_count, P, &G, &ksplit, &kchunk);
  return ksplit == 1;
}

int k0_batch_fill(int sm_count, const PairPlan& P, K0BatchItem* it) {
  int G; long long ksplit, kchunk;
  k0_config(sm_count, P, &G, &ksplit, &kchunk);
  it->M = P.M; it->N = P.N; it->K = P.K; it->G = G; it->_pad = 0;
  compact_fill(P.m, it->m); compact_fill(P.n, it->n); compact_fill(P.k, it->k);
  const long long per_block = K0_THREADS / G;
  return (int)((P.M * P.N + per_block - 1) / per_block);
}

int launch_k0_batch(tncb_ctx* ctx, const K0BatchItem* d_items, const int* d_block_start, int n_items, int total_blocks, char* ws,
                    int dtype) {
  if (n_items <= 0 || total_blocks <= 0) return TNCB_OK;
  if (dtype == TNCB_C64) k0_batch_kernel<float2><<<(unsigned)total_blocks, K0_THREADS, 0, ctx->stream>>>(d_items, d_block_start, n_items, ws);
  else k0_batch_kernel<double2><<<(unsigned)total_blocks, K0_THREADS, 0, ctx->stream>>>(d_items, d_block_start, n_items, ws);
  ctx->launches++;
  ctx->engine_count[0] += (uint64_t)n_items;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

template <typename T, int BN, int BM, int WN, int WM, int ST, bool BKF, bool AKF, int MINB = 1>
static int launch_k1_cfg(tncb_ctx* ctx, const K1Args& a) {
  auto kern = k1_kernel<BN, BM, WN, WM, ST, BKF, AKF, MINB, T>;
  const size_t smem = (size_t)ST * (BN * K1_BK + K1_BK * BM) * sizeof(T);
  TNCB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long tiles = (long long)a.tiles_m * a.tiles_n * a.ksplit;
  if (tiles > 0x7fffffffLL) return fail(TNCB_ERR_UNSUPPORTED, "K1 grid too large");
  if (ctx->time_gemm == 1) gemm_timer_begin(ctx);       // (accumulate mode collects the tcgen05 GEMMs only)
  kern<<<(unsigned)tiles, WN * WM * 32, smem, ctx->stream>>>(a);
  if (ctx->time_gemm == 1) gemm_timer_end(ctx, 8.0 * (double)a.M * (double)a.N * (double)a.K);
  ctx->launches++;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

template <typename T, int BN, int BM, int WN, int WM, int ST, int MINB = 1>
static int launch_k1_modes(tncb_ctx* ctx, K1Args& a, bool bkf, bool akf, bool allow_split) {
  a.tiles_m = (int)((a.M + BM - 1) / BM);
  a.tiles_n = (int)((a.N + BN - 1) / BN);
  // split-K: few output tiles but a long K would leave most SMs idle (C4: M=2^8, N=2^6, K=2^20
  // ran on 4 CTAs at 0.67 TFLOP/s).  Each K range writes its own partial C, reduced in a
  // fixed order afterwards (deterministic, no atomics).
  const long long tiles = (long long)a.tiles_m * a.tiles_n;
  const int nk_total = (int)((a.K + K1_BK - 1) / K1_BK);
  T* final_c = static_cast<T*>(a.C);
  a.ksplit = 1; a.chunks_per_split = nk_total;
  const long long want_ctas = 2LL * ctx->sm_count;
  if (allow_split && tiles < want_ctas && nk_total >= 16) {
    long long ks = std::min<long long>((want_ctas + tiles - 1) / tiles, nk_total / 8);
    const long long ws_cap = ((long long)1 << 30) / 16 / std::max(1LL, a.M * a.N); // <= 1 GiB of partials
    ks = std::max(1LL, std::min(ks, ws_cap));
    if (ks > 1) {
      a.chunks_per_split = (int)((nk_total + ks - 1) / ks);
      a.ksplit = (nk_total + a.chunks_per_split - 1) / a.chunks_per_split;
      int rc = ensure_partial(ctx, (size_t)(a.M * a.N * a.ksplit));
      if (rc) return rc;
      a.C = ctx->partial;
    }
  }
  int rc;
  if (bkf && akf) rc = launch_k1_cfg<T, BN, BM, WN, WM, ST, true, true, MINB>(ctx, a);
  else if (bkf && !akf) rc = launch_k1_cfg<T, BN, BM, WN, WM, ST, true, false, MINB>(ctx, a);
  else if (!bkf && akf) rc = launch_k1_cfg<T, BN, BM, WN, WM, ST, false, true, MINB>(ctx, a);
  else rc = launch_k1_cfg<T, BN, BM, WN, WM, ST, false, false, MINB>(ctx, a);
  if (rc) return rc;
  ctx->engine_count[a.ksplit > 1 ? 3 : 2]++;
  if (a.ksplit > 1) {
    const long long MN = a.M * a.N;
    reduce_partials_kernel<<<(unsigned)((MN + 255) / 256), 256, 0, ctx->stream>>>(ctx->partial, final_c, MN, a.ksplit);
    ctx->launches++;
    TNCB_CUDA(cudaGetLastError());
  }
  return TNCB_OK;
}

template <typename T>
static int launch_k1(tncb_ctx* ctx, const PairPlan& P, const T* A, const T* B, T* C) {
  constexpr int dtype = sizeof(T) == sizeof(double2) ? TNCB_C128 : TNCB_C64;
  const size_t tab_elems = (size_t)(P.M + P.N + 2 * P.K);
  int rc = ensure_tab(ctx, tab_elems);
  if (rc) return rc;
  auto same = [](const LegList& x, const LegList& y) {
    if (x.n != y.n) return false;
    for (int i = 0; i < x.n; i++) if (x.dim[i] != y.dim[i] || x.sa[i] != y.sa[i] || x.sb[i] != y.sb[i]) return false;
    return true;
  };
  if (!(ctx->tab_valid && same(ctx->tab_m, P.m) && same(ctx->tab_n, P.n) && same(ctx->tab_k, P.k))) {
    const long long total = (long long)tab_elems;
    const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 8);
    build_tables_kernel<<<blocks, 256, 0, ctx->stream>>>(P.m, P.n, P.k, P.M, P.N, P.K, ctx->tab);
    ctx->launches++;
    ctx->tab_m = P.m; ctx->tab_n = P.n; ctx->tab_k = P.k; ctx->tab_valid = true;
  }
  K1Args a;
  a.A = A; a.B = B; a.C = C;
  a.offAm = ctx->tab; a.offBn = ctx->tab + P.M; a.offAk = ctx->tab + P.M + P.N; a.offBk = a.offAk + P.K;
  a.M = P.M; a.N = P.N; a.K = P.K;
  // K1': the same contraction on the tcgen05 int8 pipe for large GEMM-like pairs.  Default engine: modular
  // (CRT) emulation, crt.cu; the 7-bit digit-slicing engine of round 1 (ozaki.cu) stays selectable for A/B.
  if (ctx->oz_slices > 0 && P.M >= 128 && P.N >= 128) {
    static const bool force = std::getenv("TNCB_FORCE_TCGEN05") != nullptr;  // tuning aid: skip the size heuristic
    if (ctx->oz_engine == 0 || dtype == TNCB_C64) {   // (the digit-slicing engine has no complex64 path)
      const double mnk = (double)P.M * (double)P.N * (double)P.K;
      if (force || (P.K >= ctx->crt_min_k && mnk >= ctx->crt_min_mnk)) {
        int rc = launch_k1_crt(ctx, P, A, B, C, a.offAm, a.offBn, a.offAk, a.offBk, dtype);
        if (rc != TNCB_ERR_OOM && rc != TNCB_ERR_UNSUPPORTED) return rc;   // no room for the residue planes: DMMA engine
      }
    } else if (dtype == TNCB_C128 && P.M >= 256 && P.N >= 256 && P.K >= 256) {
      const long long tiles = ((P.M + 127) / 128) * ((P.N + 127) / 128);
      // crossover measured on B200 (profiles/r01_engine_sweep.txt): short K is dominated by the S
      // FP64 read-modify-write flushes per tile, few tiles leave SMs idle (1 CTA per 128x128 tile)
      if (force || (tiles >= ctx->oz_min_tiles && P.K >= ctx->oz_min_k) || (tiles >= 1024 && P.K >= 1024)) {
        int rc = launch_k1_ozaki(ctx, P, (const double2*)A, (const double2*)B, (double2*)C, ctx->oz_slices, a.offAm, a.offBn, a.offAk, a.offBk);
        if (rc == TNCB_OK) ctx->engine_count[4]++;
        if (rc != TNCB_ERR_OOM) return rc;   // no room for the digit planes: fall through to the DMMA engine
      }
    }
  }
  // Tile choice (A/B-measured on B200, C2 pair, profiles/r01_k1_tile_ab.txt): 64x64 tiles with a
  // 2-stage ring and 2 co-resident CTAs per SM reach ~90 % of the DMMA peak (independent CTAs
  // hide each other's per-chunk barrier/gather bubbles); 128x64 with 3-4 stages and 1 CTA/SM
  // stays at 75-81 %.  Skinny outputs use a 32-wide tile on the narrow side.
  static const int variant = std::getenv("TNCB_K1_VARIANT") ? atoi(std::getenv("TNCB_K1_VARIANT")) : 0;
  if (variant == 1) return launch_k1_modes<T, 128, 64, 4, 2, 4, 1>(ctx, a, P.b_kfast, P.a_kfast, true);
  if (P.N <= 32 && P.M > 32) return launch_k1_modes<T, 32, 64, 1, 2, 2, 2>(ctx, a, P.b_kfast, P.a_kfast, true);
  if (P.M <= 32 && P.N > 32) return launch_k1_modes<T, 64, 32, 2, 1, 2, 2>(ctx, a, P.b_kfast, P.a_kfast, true);
  return launch_k1_modes<T, 64, 64, 2, 2, 2, 2>(ctx, a, P.b_kfast, P.a_kfast, true);
}

// ------------------------------------------------------------------------------------------
// K2: streaming kernel for big x tiny pairs (HBM-bound).  thread <-> one index x of the big free
// side; the tiny operand sits in shared memory as S[s][k]; every thread reads its K elements of the
// big operand once and writes its NS outputs.  Algorithmic traffic 16*(BIG*K + BIG*SMALL) bytes.
// Gate-sized tiny operands (K, NS <= 4) stream at 5.8-6.1 TB/s.  With K = NS = 16 (the stem steps of the Sycamore-53 depth-12
// slices: 16 input and 16 output streams GBs apart per block) it stays at 3.2 TB/s / 35 % of the FP64 pipe although DRAM
// moves exactly the algorithmic bytes in full sectors (profiles/r02_ncu_k2_summary.txt).  Two fixes for "not enough loads
// in flight" were measured and removed again: four loads per trip (11.0 vs 10.8 ms) and a 3-stage cp.async ring in shared
// memory with 48 loads in flight per thread (11.7-13.5 ms) -- so the limit is not load latency under this access pattern.
// ------------------------------------------------------------------------------------------
struct K2Args {
  LegList big;     // free legs of the big operand (strides in the big operand)
  LegList sml;     // free legs of the tiny operand (strides in the tiny operand)
  LegList k;       // shared legs: sa = stride in the big operand, sb = stride in the tiny operand
  long long BIG, SMALL, K, M;   // M = row length of C
  int big_is_a;    // 1: x = m (C[s*M + x]),  0: x = n (C[x*M + s])
  int pow2;        // all big-side dims are powers of two -> shift/mask decomposition
  int shift[kMaxGroups];
};

__device__ __forceinline__ long long decomp_shift(long long idx, const LegList& L, const int* sh) {
  long long off = 0;
  for (int g = L.n - 1; g > 0; --g) {
    off += (idx & ((1LL << sh[g]) - 1)) * L.sa[g];
    idx >>= sh[g];
  }
  if (L.n > 0) off += idx * L.sa[0];
  return off;
}

template <int NS, typename T>
__global__ void __launch_bounds__(256)
k2_kernel(const T* __restrict__ Big, const T* __restrict__ Sml, T* __restrict__ C,
          const __grid_constant__ K2Args p) {
  __shared__ double2 s_s[16 * 64];     // S[s][k], s < NS, k < K <= 64 ... NS*K <= 256 guaranteed by the planner
  __shared__ long long s_kbig[64];
  const int K = (int)p.K;
  for (int i = threadIdx.x; i < K; i += blockDim.x) {
    long long ob, os;
    decomp_ab(i, p.k, ob, os);
    s_kbig[i] = ob;
  }
  for (int i = threadIdx.x; i < NS * K; i += blockDim.x) {
    const int sidx = i / K, k = i - sidx * K;
    double2 v = make_double2(0.0, 0.0);
    if (sidx < p.SMALL) {
      long long ob, os;
      decomp_ab(k, p.k, ob, os);
      v = ldg_wide(Sml + decomp_a(sidx, p.sml) + os);
    }
    s_s[i] = v;
  }
  __syncthreads();
  for (long long x = (long long)blockIdx.x * blockDim.x + threadIdx.x; x < p.BIG; x += (long long)gridDim.x * blockDim.x) {
    const long long off = p.pow2 ? decomp_shift(x, p.big, p.shift) : decomp_a(x, p.big);
    double ar[NS], ai[NS];
#pragma unroll
    for (int sI = 0; sI < NS; sI++) { ar[sI] = 0.0; ai[sI] = 0.0; }
    for (int k = 0; k < K; k++) {
      const double2 v = ldg_wide(Big + off + s_kbig[k]);
#pragma unroll
      for (int sI = 0; sI < NS; sI++) {
        const double2 w = s_s[sI * K + k];   // broadcast
        ar[sI] = fma(w.x, v.x, ar[sI]); ar[sI] = fma(-w.y, v.y, ar[sI]);
        ai[sI] = fma(w.x, v.y, ai[sI]); ai[sI] = fma(w.y, v.x, ai[sI]);
      }
    }
    if (p.big_is_a) {
#pragma unroll
      for (int sI = 0; sI < NS; sI++)
        if (sI < p.SMALL) st_round(C + (long long)sI * p.M + x, ar[sI], ai[sI]);
    } else {
      T* dst = C + x * p.M;
#pragma unroll
      for (int sI = 0; sI < NS; sI++)
        if (sI < p.SMALL) st_round(dst + sI, ar[sI], ai[sI]);
    }
  }
}

template <typename T>
static int launch_k2(tncb_ctx* ctx, const PairPlan& P, const T* A, const T* B, T* C) {
  K2Args a;
  const bool big_a = P.k2_big_is_a;
  a.big = big_a ? P.m : P.n;
  a.sml = big_a ? P.n : P.m;
  a.k = P.k;
  if (!big_a) for (int g = 0; g < a.k.n; g++) std::swap(a.k.sa[g], a.k.sb[g]);   // sa = big operand's stride
  a.BIG = big_a ? P.M : P.N; a.SMALL = big_a ? P.N : P.M; a.K = P.K; a.M = P.M; a.big_is_a = big_a ? 1 : 0;
  a.pow2 = 1;
  for (int g = 0; g < a.big.n; g++) {
    const long long d = a.big.dim[g];
    if (d & (d - 1)) { a.pow2 = 0; a.shift[g] = 0; } else { int sh = 0; while ((1LL << sh) < d) sh++; a.shift[g] = sh; }
  }
  const T* Big = big_a ? A : B;
  const T* Sml = big_a ? B : A;
  const int blocks = (int)std::min<long long>((a.BIG + 255) / 256, (long long)ctx->sm_count * 32);
  int ns = 1; while (ns < a.SMALL) ns *= 2;
  switch (ns) {
    case 1: k2_kernel<1, T><<<blocks, 256, 0, ctx->stream>>>(Big, Sml, C, a); break;
    case 2: k2_kernel<2, T><<<blocks, 256, 0, ctx->stream>>>(Big, Sml, C, a); break;
    case 4: k2_kernel<4, T><<<blocks, 256, 0, ctx->stream>>>(Big, Sml, C, a); break;
    case 8: k2_kernel<8, T><<<blocks, 256, 0, ctx->stream>>>(Big, Sml, C, a); break;
    default: k2_kernel<16, T><<<blocks, 256, 0, ctx->stream>>>(Big, Sml, C, a); break;
  }
  ctx->launches++;
  ctx->engine_count[5]++;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

template <typename T>
static int launch_pair_t(tncb_ctx* ctx, const PairPlan& P, const T* A, const T* B, T* C) {
  if (P.kernel_class == 2) return launch_k2(ctx, P, A, B, C);
  if (P.kernel_class == 1) return launch_k1(ctx, P, A, B, C);
  return launch_k0(ctx, P, A, B, C);
}

int launch_pair(tncb_ctx* ctx, const PairPlan& P, const void* A, const void* B, void* C, int dtype) {
  if (P.M * P.N == 0) return TNCB_OK;
  NvtxPairRange nvtx_range(P);
  if (dtype == TNCB_C64) return launch_pair_t(ctx, P, (const float2*)A, (const float2*)B, (float2*)C);
  return launch_pair_t(ctx, P, (const double2*)A, (const double2*)B, (double2*)C);
}

// ------------------------------------------------------------------------------------------
// K3: tiled transpose (Permutor::apply / tetra transpose, builders/circuit_builder.rs:86-114).
// A tile is a sub-box over a few leg groups, chosen so that it is >= 32 elements long BOTH along the input's fastest
// index and along the output's fastest index.  The CTA reads the tile in input order (coalesced 512-byte runs), parks it
// in shared memory and writes it in output order (coalesced again); a one-element pad per 32 keeps the strided
// shared-memory reads off one bank.  Bound: HBM, 32 bytes of traffic per element.
// ------------------------------------------------------------------------------------------
constexpr int K3_MAXT = 12;       // leg groups inside a tile
constexpr int K3_TILE = 2048;     // elements per tile (32 KB + pad)
struct K3Args {
  int nt;                          // tile groups
  int ext[K3_MAXT];                // tile extent per tile group
  long long dim[K3_MAXT], sin[K3_MAXT], sout[K3_MAXT];   // full dim, input stride, output stride of the tile groups
  int in_order[K3_MAXT], out_order[K3_MAXT];              // tile groups sorted by input stride / by output stride (fastest first)
  int smem_stride[K3_MAXT];        // linear index inside the tile (input order)
  int tile_elems;
  int nr;                          // block-index digits: tiles of every tile group + the remaining groups
  long long rcount[kMaxGroups + K3_MAXT], rin[kMaxGroups + K3_MAXT], rout[kMaxGroups + K3_MAXT];
  int rtile[kMaxGroups + K3_MAXT]; // >= 0: this digit walks the tiles of tile group rtile (index base += digit * ext)
};

// Per-launch tables (identical for every tile): element e of the tile in input order -> input offset and packed
// per-group indices (5 bits each, extents <= 32); element f in output order -> output offset, packed indices and the
// shared-memory slot.  Built by one tiny kernel so that the copy kernel does no division per element.
__global__ void k3_tables_kernel(const __grid_constant__ K3Args p, long long* __restrict__ tab) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.tile_elems) return;
  const int te = p.tile_elems;
  {
    int rem = e; long long off = 0; unsigned long long pk = 0;
    for (int k = 0; k < p.nt; k++) {
      const int g = p.in_order[k], x = p.ext[g], i = rem % x;
      rem /= x;
      off += (long long)i * p.sin[g];
      pk |= (unsigned long long)i << (5 * g);
    }
    tab[e] = off; tab[te + e] = (long long)pk;
  }
  {
    int rem = e, sidx = 0; long long off = 0; unsigned long long pk = 0;
    for (int k = 0; k < p.nt; k++) {
      const int g = p.out_order[k], x = p.ext[g], i = rem % x;
      rem /= x;
      off += (long long)i * p.sout[g];
      sidx += i * p.smem_stride[g];
      pk |= (unsigned long long)i << (5 * g);
    }
    tab[2 * te + e] = off; tab[3 * te + e] = (long long)pk; tab[4 * te + e] = sidx;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
k3_transpose_kernel(const T* __restrict__ in, T* __restrict__ out, const __grid_constant__ K3Args p,
                    const long long* __restrict__ tab) {
  extern __shared__ __align__(16) unsigned char k3_smem_raw[];
  T* tile = reinterpret_cast<T*>(k3_smem_raw);
  // block index -> base offsets; room left in every partially tiled group
  long long b = blockIdx.x, base_in = 0, base_out = 0;
  int room[K3_MAXT];                                  // valid indices of tile group g in this tile: i < room[g]
#pragma unroll
  for (int g = 0; g < K3_MAXT; g++) room[g] = 32;
  bool partial = false;
  for (int d = p.nr - 1; d >= 0; --d) {
    const long long c = p.rcount[d], q = b / c, r = b - q * c;
    base_in += r * p.rin[d]; base_out += r * p.rout[d];
    const int g = p.rtile[d];
    if (g >= 0) {
      const long long left = p.dim[g] - r * p.ext[g];
      if (left < p.ext[g]) { partial = true;
#pragma unroll
        for (int h = 0; h < K3_MAXT; h++) if (h == g) room[h] = (int)left;
      }
    }
    b = q;
  }
  const int te = p.tile_elems;
  auto inside = [&](unsigned long long pk) {
    bool ok = true;
#pragma unroll
    for (int g = 0; g < K3_MAXT; g++) ok &= (int)((pk >> (5 * g)) & 31) < room[g];
    return ok;
  };
  for (int e = threadIdx.x; e < te; e += 256) {
    const long long off = __ldg(tab + e);
    if (!partial || inside((unsigned long long)__ldg(tab + te + e))) tile[e + (e >> 5)] = __ldg(in + base_in + off);
  }
  __syncthreads();
  for (int f = threadIdx.x; f < te; f += 256) {
    const long long off = __ldg(tab + 2 * te + f);
    const int sidx = (int)__ldg(tab + 4 * te + f);
    if (!partial || inside((unsigned long long)__ldg(tab + 3 * te + f))) out[base_out + off] = tile[sidx + (sidx >> 5)];
  }
}

template <typename T>
static int launch_permute_t(tncb_ctx* ctx, const T* in, T* out, int rank,
                            const uint64_t* in_dims, const int* perm) {
  std::vector<long long> istr(rank);
  long long s = 1, total = 1;
  for (int i = rank - 1; i >= 0; i--) { istr[i] = s; s *= (long long)in_dims[i]; }
  total = s;
  // output leg i walks input leg perm[i]; fuse neighbours that stay adjacent in the input
  LegList L{}; int n = 0;
  for (int i = 0; i < rank; i++) {
    long long d = (long long)in_dims[perm[i]], st = istr[perm[i]];
    if (d == 1) continue;
    if (n > 0 && L.sa[n - 1] == st * d) { L.dim[n - 1] *= d; L.sa[n - 1] = st; continue; }
    if (n >= kMaxGroups) return fail(TNCB_ERR_INVALID, "too many leg groups in permute");
    L.dim[n] = d; L.sa[n] = st; L.sb[n] = 0; n++;
  }
  L.n = n;
  if (total == 0) return TNCB_OK;
  ctx->engine_count[6]++;
  static const bool no_tiled = std::getenv("TNCB_NO_K3") != nullptr;
  if (n <= 1 || no_tiled || total < 4096) {   // identity / tiny: the plain gather kernel (already coalesced or negligible)
    const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 16);
    permute_kernel<T><<<blocks, 256, 0, ctx->stream>>>(in, out, L, total);
    ctx->launches++;
    TNCB_CUDA(cudaGetLastError());
    return TNCB_OK;
  }
  // output strides of the groups
  std::vector<long long> ostr(n);
  { long long t = 1; for (int g = n - 1; g >= 0; g--) { ostr[g] = t; t *= L.dim[g]; } }
  // tile extents: walk the groups from the input's fastest index until the run is >= 32, then from the output's
  std::vector<int> by_in(n), by_out(n);
  for (int g = 0; g < n; g++) { by_in[g] = g; by_out[g] = n - 1 - g; }          // output order: last group is fastest
  std::sort(by_in.begin(), by_in.end(), [&](int x, int y) { return L.sa[x] < L.sa[y]; });
  std::vector<int> ext(n, 1);
  auto grow = [&](const std::vector<int>& order) {
    long long run = 1;
    for (int g : order) {
      if (run >= 32) break;
      if (ext[g] > 1) { run *= ext[g]; if (ext[g] < L.dim[g]) break; continue; }    // already (partly) inside the tile
      const long long want = (32 + run - 1) / run;
      ext[g] = (int)std::min<long long>(L.dim[g], want);
      run *= ext[g];
      if (ext[g] < L.dim[g]) break;        // a partial group ends the contiguous run
    }
  };
  grow(by_in); grow(by_out);
  {
    // tiles of a few dozen elements (many dim-2 legs that are fast on both sides) drown in per-CTA overhead: keep adding
    // groups, alternately from the input-fast and the output-fast side, until a tile holds >= 1024 elements
    long long te0 = 1;
    for (int g = 0; g < n; g++) te0 *= ext[g];
    size_t pi = 0, po = 0; bool turn = false; int used = 0;
    for (int g = 0; g < n; g++) used += ext[g] > 1;
    while (te0 < 1024 && used < K3_MAXT && (pi < by_in.size() || po < by_out.size())) {
      const std::vector<int>& ord = turn ? by_out : by_in;
      size_t& ptr = turn ? po : pi;
      turn = !turn;
      while (ptr < ord.size() && ext[ord[ptr]] >= L.dim[ord[ptr]]) ptr++;     // already full
      if (ptr >= ord.size()) continue;
      const int g = ord[ptr];
      const long long cur = ext[g];
      const long long factor = std::max<long long>(2, std::min<long long>((1024 + te0 - 1) / te0, K3_TILE / te0));
      const long long want = std::min<long long>({L.dim[g], (long long)32, cur * factor});
      if (want <= cur || te0 / cur * want > K3_TILE) { ptr++; continue; }
      if (cur == 1) used++;
      te0 = te0 / cur * want; ext[g] = (int)want;
      if (ext[g] >= L.dim[g] || ext[g] >= 32) ptr++;
    }
  }
  K3Args a{};
  std::vector<int> tg;                      // groups with an extent > 1 (or the fastest ones even if their dim is small)
  for (int g = 0; g < n; g++) if (ext[g] > 1) tg.push_back(g);
  bool plain = (int)tg.size() > K3_MAXT;
  a.nt = plain ? 0 : (int)tg.size();
  long long te = 1;
  for (int k = 0; k < a.nt; k++) { const int g = tg[k]; a.ext[k] = ext[g]; a.dim[k] = L.dim[g]; a.sin[k] = L.sa[g]; a.sout[k] = ostr[g]; te *= ext[g]; }
  if (plain || te > K3_TILE || te < 64) {   // degenerate tilings: the plain gather kernel
    const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)ctx->sm_count * 16);
    permute_kernel<T><<<blocks, 256, 0, ctx->stream>>>(in, out, L, total);
    ctx->launches++;
    TNCB_CUDA(cudaGetLastError());
    return TNCB_OK;
  }
  a.tile_elems = (int)te;
  std::vector<int> oi(a.nt), oo(a.nt);
  for (int k = 0; k < a.nt; k++) oi[k] = oo[k] = k;
  std::sort(oi.begin(), oi.end(), [&](int x, int y) { return a.sin[x] < a.sin[y]; });
  std::sort(oo.begin(), oo.end(), [&](int x, int y) { return a.sout[x] < a.sout[y]; });
  { int st = 1; for (int k = 0; k < a.nt; k++) { a.in_order[k] = oi[k]; a.smem_stride[oi[k]] = st; st *= a.ext[oi[k]]; } }
  for (int k = 0; k < a.nt; k++) a.out_order[k] = oo[k];
  // block digits: tiles of the tile groups, then every other group
  long long blocks = 1; a.nr = 0;
  for (int k = 0; k < a.nt; k++) {
    const long long tiles = (a.dim[k] + a.ext[k] - 1) / a.ext[k];
    if (tiles > 1) { a.rcount[a.nr] = tiles; a.rin[a.nr] = a.sin[k] * a.ext[k]; a.rout[a.nr] = a.sout[k] * a.ext[k]; a.rtile[a.nr] = k; a.nr++; blocks *= tiles; }
  }
  for (int g = 0; g < n; g++) if (ext[g] == 1) { a.rcount[a.nr] = L.dim[g]; a.rin[a.nr] = L.sa[g]; a.rout[a.nr] = ostr[g]; a.rtile[a.nr] = -1; a.nr++; blocks *= L.dim[g]; }
  if (blocks > 0x7fffffffLL) return fail(TNCB_ERR_UNSUPPORTED, "permute grid too large");
  const int smem = (int)((te + te / 32 + 1) * sizeof(T));
  static bool attr_done_dev[64] = {false};          // cudaFuncSetAttribute is per device (and per instantiation)
  bool& attr_done = attr_done_dev[ctx->device & 63];
  if (!attr_done) { TNCB_CUDA(cudaFuncSetAttribute(k3_transpose_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (K3_TILE + K3_TILE / 32 + 1) * (int)sizeof(T))); attr_done = true; }
  int rc = ensure_tab(ctx, (size_t)(5 * te));
  if (rc) return rc;
  ctx->tab_valid = false;                       // the K1 offset tables living in the same buffer are gone
  k3_tables_kernel<<<(unsigned)((te + 255) / 256), 256, 0, ctx->stream>>>(a, ctx->tab);
  k3_transpose_kernel<T><<<(unsigned)blocks, 256, smem, ctx->stream>>>(in, out, a, ctx->tab);
  ctx->launches += 2;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

int launch_permute(tncb_ctx* ctx, const void* in, void* out, int rank, const uint64_t* in_dims, const int* perm, int dtype) {
  if (dtype == TNCB_C64) return launch_permute_t(ctx, (const float2*)in, (float2*)out, rank, in_dims, perm);
  return launch_permute_t(ctx, (const double2*)in, (double2*)out, rank, in_dims, perm);
}

// complex64: the sum of two complex64 values, rounded once (numpy's complex64 addition)
template <typename T>
__global__ void add_kernel(T* __restrict__ dst, const T* __restrict__ src, long long total) {
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (long long)gridDim.x * blockDim.x) {
    T d = dst[o]; const T v = src[o];
    d.x += v.x; d.y += v.y; dst[o] = d;
  }
}

int launch_add(tncb_ctx* ctx, void* dst, const void* src, uint64_t elems, int dtype) {
  if (elems == 0) return TNCB_OK;
  const int blocks = (int)std::min<long long>(((long long)elems + 255) / 256, (long long)ctx->sm_count * 16);
  if (dtype == TNCB_C64) add_kernel<float2><<<blocks, 256, 0, ctx->stream>>>((float2*)dst, (const float2*)src, (long long)elems);
  else add_kernel<double2><<<blocks, 256, 0, ctx->stream>>>((double2*)dst, (const double2*)src, (long long)elems);
  ctx->launches++;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

int launch_conj(tncb_ctx* ctx, void* data, uint64_t elems, int dtype) {
  if (elems == 0) return TNCB_OK;
  const int blocks = (int)std::min<long long>(((long long)elems + 255) / 256, (long long)ctx->sm_count * 16);
  if (dtype == TNCB_C64) conj_kernel<float2><<<blocks, 256, 0, ctx->stream>>>((float2*)data, (long long)elems);
  else conj_kernel<double2><<<blocks, 256, 0, ctx->stream>>>((double2*)data, (long long)elems);
  ctx->launches++;
  TNCB_CUDA(cudaGetLastError());
  return TNCB_OK;
}

} // namespace tncb

// K1' -- the dense contraction on the 5th-gen tensor cores (tcgen05) through an integer modular
// (Chinese-remainder) emulation of the complex128 GEMM.
//
// tcgen05.mma has no f64 kind.  The FP64 contraction C[n,m] = sum_k Bt[n,k] * At[m,k] reaches the int8
// tensor pipe like this (all arithmetic below is exact until the last conversion):
//   1. every row of the K-major operands is scaled by a power of two and truncated to an integer,
//        X' = trunc(x * 2^(a - e_row)),   |X'| < 2^a,  a <= 53   (e_row: max(|re|,|im|) of the row < 2^e_row)
//   2. for N pairwise coprime moduli m_i <= 256 the residues X' mod m_i (symmetric, int8) are written as
//      K-major planes -- the leg permutation of the reference's TTGT is fused into this pass (gather
//      through the plan's offset tables);
//   3. per modulus ONE int8 GEMM on tcgen05.mma.kind::i8 (int32 accumulators in TMEM) gives
//      C' mod m_i for the exact integer product C' = sum_k B'[n,k] A'[m,k]; the GEMM epilogue reduces the
//      accumulator mod m_i and stores one int8 per real output;
//   4. a reconstruction pass evaluates the CRT in split double precision,
//        C'/P = frac( sum_i y_i * rho_i ),  rho_i = ((P/m_i)^-1 mod m_i) / m_i,  P = prod m_i,
//      and scales by P * 2^(e_n + e_m - 2a).
// P > 8 K 2^(2a) makes |C'| < P/4, so the representative in (-P/2, P/2) is C' itself.  With a = 53 (the
// default) that needs N = 16 moduli for K <= 2^13: 16 int8 GEMM sweeps instead of the 36 digit-pair sweeps of
// the 7-bit slicing it replaces (csrc/ozaki.cu, kept for A/B), at a provable bound
//      |C - C_exact|[n,m] <= 2^(4-a) * K * max|B[n,:]| * max|A[m,:]|      (max over re/im parts)
// (each element is truncated by < 2^(e-a); 4K products per real output; 2^e <= 2 max).  The scheme is the
// published "Ozaki scheme II" (integer modular technique for GEMM emulation); this is an independent
// implementation for complex operands with the TTGT gather fused in.
//
// GEMM kernel (crt_gemm_kernel): persistent CTA pairs (cluster 2x1, tcgen05 cta_group::2), work item =
// (modulus, K chunk, 256x128 complex tile), items ordered modulus-major with a grouped tile raster so that the
// ~74 pairs resident at any time share a few operand row bands of ONE modulus in L2.
//   warp 0  TMA producer (cp.async.bulk.tensor 2D, SWIZZLE_128B, 3 stages x 64 KB)
//   warp 1  (leader CTA) single-thread tcgen05.mma issuer: 2 UMMAs (M=256 N=256 K=32) per 32-byte K step,
//           Br x [Ar;Ai]^T and Bi x [-Ai;Ar]^T into one 256-column accumulator (cols 0-127 re, 128-255 im)
//   warps 2-9 epilogue (two per TMEM lane quarter: real / imaginary columns): tcgen05.ld -> (acc mod m_i) -> byte ->
//           shared-memory staging -> coalesced global stores; TMEM holds two accumulators, so the epilogue of item j
//           overlaps the MMAs of item j+1.
#include "internal.h"
#include <cuda.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>

namespace tncb {

constexpr int CRT_MAX_MOD = 20;
// pairwise coprime, descending; 255 is left out on purpose: with every odd modulus <= 253 the residue
// |r| <= 127 falls out of the FMA reduction without a range fix (see crt_residue_kernel)
static const int kModuli[CRT_MAX_MOD] = {256, 253, 251, 249, 247, 245, 241, 239, 233, 229,
                                         227, 223, 211, 199, 197, 193, 191, 181, 179, 173};
constexpr int CRT_BT = 128;        // tile rows per CTA (n) = tile cols (m)
constexpr int CRT_BKB = 128;       // K bytes per stage row (one 128-byte swizzle row)
constexpr int CRT_TILE = CRT_BT * CRT_BKB;      // 16 KB
// shared-memory ring of the GEMM kernel: 192 KB either way
template <bool KARA> struct CrtRing {
  static constexpr int TILES = KARA ? 2 : 4;            // four products: Br, Bi, X (Ar | Ai), Y (-Ai | Ar); three: B_p, A_p
  static constexpr int STAGE_BYTES = TILES * CRT_TILE;
  static constexpr int STAGES = KARA ? 6 : 3;
};
constexpr int CRT_RING_BYTES = 3 * 4 * CRT_TILE;
constexpr int CRT_THREADS = 320;                // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quarter)
constexpr int CRT_STG_ROW = CRT_BT;              // row of the epilogue staging tile (bytes; 16-byte chunks XOR-swizzled by row)
constexpr int CRT_STG_BYTES = 32 * CRT_STG_ROW;  // per epilogue warp: 32 rows x 128 residue bytes of one component
constexpr int CRT_KCHUNK_MAX = 32768;           // 2 * K * 128 * 128 < 2^31 for K <= 2^15
constexpr int CRT_G = 34;                       // fixed-point bits of the leading CRT weight

struct CrtTables {
  int nmod;
  int a_bits_a, a_bits_b;     // integer bits kept per operand
  int mod[CRT_MAX_MOD];
  int magic[CRT_MAX_MOD];     // round(2^32 / m)
  double inv_mod[CRT_MAX_MOD];
  double rho1[CRT_MAX_MOD];   // floor(rho * 2^G) / 2^G
  double rho2[CRT_MAX_MOD];   // rho - rho1
  double p_scaled;            // P * 2^-(a_bits_a + a_bits_b)
};

// ---- host: moduli / CRT weights ------------------------------------------------------------------
double crt_log2_product(int n) {
  double s = 0;
  for (int i = 0; i < n; i++) s += std::log2((double)kModuli[i]);
  return s;
}

// Number of moduli and operand bits for a pair with contraction length K.
//   want_bits: integer bits per operand asked for (53 = full mantissa); nmod_force > 0 pins the modulus count.
void crt_choose(long long K, int want_bits, int nmod_force, int* nmod, int* bits_a, int* bits_b) {
  const double lk = std::log2((double)std::max<long long>(K, 1));
  auto needed = [&](int bits) {
    int q = 2;
    while (q < CRT_MAX_MOD && crt_log2_product(q) - 1e-9 < 2.0 * bits + lk + 3.0) q++;
    return q;
  };
  // A forced count is clamped to what 53-bit operands need: more moduli add no accuracy (the operands have no more
  // bits) but make C'/P a tiny fraction of 1, where the absolute error of the split CRT sum (~2^-75) would show.
  int n = nmod_force > 0 ? std::min(nmod_force, needed(53)) : needed(want_bits);
  n = std::max(2, std::min(n, CRT_MAX_MOD));
  int tot = (int)std::floor(crt_log2_product(n) - lk - 3.0 - 1e-9);
  tot = std::max(tot, 2);
  int a = std::min(want_bits, tot / 2), b = std::min(want_bits, tot - a);
  *nmod = n; *bits_a = a; *bits_b = b;
}

// Operand bits that guarantee |C - C_exact|[n,m] <= tol * max|B[n,:]| * max|A[m,:]|:  2^(4-a) K <= tol.
int crt_bits_for_tolerance(long long K, double tol) {
  if (!(tol > 0.0)) return 53;
  const int a = (int)std::ceil(std::log2(16.0 * (double)std::max<long long>(K, 1) / tol));
  return std::max(8, std::min(53, a));
}

static void crt_make_tables(int nmod, int bits_a, int bits_b, CrtTables& T) {
  T.nmod = nmod; T.a_bits_a = bits_a; T.a_bits_b = bits_b;
  long double P = 1.0L;
  for (int i = 0; i < nmod; i++) P *= (long double)kModuli[i];
  for (int i = 0; i < CRT_MAX_MOD; i++) { T.mod[i] = 1; T.magic[i] = 0; T.inv_mod[i] = 1.0; T.rho1[i] = T.rho2[i] = 0.0; }
  for (int i = 0; i < nmod; i++) {
    const int m = kModuli[i];
    long long pim = 1;                               // (P / m_i) mod m_i
    for (int j = 0; j < nmod; j++) if (j != i) pim = (pim * (kModuli[j] % m)) % m;
    long long inv = 1;
    while ((pim * inv) % m != 1) inv++;              // m <= 256: brute force
    const unsigned long long num = (unsigned long long)inv << CRT_G;
    const unsigned long long q = num / (unsigned long long)m, rem = num % (unsigned long long)m;
    T.mod[i] = m;
    T.magic[i] = (int)std::llround(4294967296.0 / (double)m);
    T.inv_mod[i] = 1.0 / (double)m;
    T.rho1[i] = std::ldexp((double)q, -CRT_G);
    T.rho2[i] = std::ldexp((double)rem / (double)m, -CRT_G);
  }
  T.p_scaled = (double)std::ldexp(P, -(bits_a + bits_b));
}

int crt_export_tables(int nmod, int* moduli, double* rho1, double* rho2, double* log2_product) {
  CrtTables T;
  crt_make_tables(nmod, 0, 0, T);
  for (int i = 0; i < nmod; i++) {
    if (moduli) moduli[i] = T.mod[i];
    if (rho1) rho1[i] = T.rho1[i];
    if (rho2) rho2[i] = T.rho2[i];
  }
  if (log2_product) *log2_product = crt_log2_product(nmod);
  return TNCB_OK;
}

// ---- operand preparation ---------------------------------------------------------------------------
constexpr int RES_ROWS_C = 32, RES_K_C = 128;   // operand tile of the preparation kernels
constexpr int kExpNonFinite = 0x7fffffff;   // row contains NaN / Inf: its outputs are poisoned with NaN
constexpr int kExpMin = -1000;              // rows below 2^-1000 keep absolute accuracy 2^(-1000-a)

// Row maxima: max over k of max(|re|, |im|) as the BIT PATTERN of a non-negative double (integer max == value
// max for those; NaN / Inf patterns are the largest, so one non-finite element marks the row).  Same 32 x 128
// tiling and lane split as the residue kernel; one shared-memory atomicMax per row and warp, one global per row and CTA.
__device__ __forceinline__ int crt_exp_from_bits(unsigned long long bits) {
  const int field = (int)(bits >> 52) & 0x7ff;        // (sign bit is clear)
  if (field == 0x7ff) return kExpNonFinite;
  if (field == 0) return bits == 0ull ? 0 : kExpMin;   // zero row / denormal row
  return max(field - 1022, kExpMin);                   // ilogb(max) + 1: max * 2^-e in [0.5, 1)
}

// Element -> thread map of the 32 x 128 operand tile (shared by the row-max and the residue kernel): a warp covers
// 2^lk consecutive k times 2^(5-lk) consecutive rows, chosen on the host from the operand's strides so that a warp-wide
// load touches whole contiguous runs (lk = 5: k is the fastest index, lk = 0: the free index is; e.g. lk = 2 when four
// consecutive k are contiguous and the next-fastest index is the row).
__device__ __forceinline__ void crt_tile_coord(int e, int lk, int& r, int& k) {
  const int lane = e & 31, blk = e >> 5;               // blk in [0, 128): 2^(7-lk) k-blocks x 2^lk row-blocks
  const int kb = blk & ((128 >> lk) - 1), rb = blk >> (7 - lk);
  k = (kb << lk) + (lane & ((1 << lk) - 1));
  r = (rb << (5 - lk)) + (lane >> lk);
}

// complex64 operands (E = float2) are widened exactly to f64 as they are loaded, in this kernel and the residue kernel.
__device__ __forceinline__ double2 crt_ld(const double2* p) { return __ldg(p); }
__device__ __forceinline__ double2 crt_ld(const float2* p) { const float2 v = __ldg(p); return make_double2((double)v.x, (double)v.y); }

template <typename E>
__global__ void __launch_bounds__(256)
crt_rowmax_kernel(const E* __restrict__ src, const long long* __restrict__ off_row, const long long* __restrict__ off_k,
                  long long rows, long long K, int lk, unsigned long long* __restrict__ rowmax) {
  __shared__ unsigned long long s_max[RES_ROWS_C];
  __shared__ long long s_offr[RES_ROWS_C], s_offk[RES_K_C];
  const long long row0 = (long long)blockIdx.x * RES_ROWS_C, k0 = (long long)blockIdx.y * RES_K_C;
  const int tid = threadIdx.x;
  // the tile's offset tables first (one round trip), then 16 independent element loads per thread (a second one)
  if (tid < RES_ROWS_C) { s_max[tid] = 0ull; s_offr[tid] = row0 + tid < rows ? __ldg(off_row + row0 + tid) : -1; }
  else if (tid >= 128) { const int k = tid - 128; s_offk[k] = k0 + k < K ? __ldg(off_k + k0 + k) : -1; }
  __syncthreads();
  unsigned long long mv[RES_ROWS_C * RES_K_C / 256];
#pragma unroll
  for (int it = 0; it < RES_ROWS_C * RES_K_C / 256; it++) {
    int r, k;
    crt_tile_coord(it * 256 + tid, lk, r, k);
    const long long orow = s_offr[r], ok = s_offk[k];
    mv[it] = 0ull;
    if (orow >= 0 && ok >= 0) {
      const double2 v = crt_ld(src + orow + ok);
      mv[it] = max((unsigned long long)__double_as_longlong(fabs(v.x)), (unsigned long long)__double_as_longlong(fabs(v.y)));
    }
  }
  // a thread's row changes at most 2^lk times over the iterations (never for lk = 0), so its running maximum is flushed
  // to shared memory only when the row changes
  int cur_r = -1;
  unsigned long long cur_m = 0ull;
#pragma unroll
  for (int it = 0; it < RES_ROWS_C * RES_K_C / 256; it++) {
    int r, k;
    crt_tile_coord(it * 256 + tid, lk, r, k);
    unsigned long long m = mv[it];
    // lanes with the same row sit next to each other (2^lk of them): reduce over them, lane 0 of the group keeps the result
    for (int d = 1; d < (1 << lk); d <<= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    if (r != cur_r) {
      if (cur_m && (tid & ((1 << lk) - 1)) == 0) atomicMax(&s_max[cur_r], cur_m);
      cur_r = r; cur_m = 0ull;
    }
    cur_m = max(cur_m, m);
  }
  if (cur_m && (tid & ((1 << lk) - 1)) == 0) atomicMax(&s_max[cur_r], cur_m);
  __syncthreads();
  if (tid < RES_ROWS_C && row0 + tid < rows && s_max[tid] != 0ull) atomicMax(rowmax + row0 + tid, s_max[tid]);
}

// Tile of 32 rows x 128 k: load (coalesced along whichever index is contiguous in the source), scale +
// truncate to integer-valued doubles in shared memory, then every thread reduces 2 x 8 consecutive k of one row
// modulo every m_i and writes 8 bytes per plane and pass.
// planes: [((mod * NPL + plane) * rowsP + row) * Kp + k];
//   four-product form:  COMPS == 2 (Bt side): NPL = 2 planes (re, im);  COMPS == 3 (At side): NPL = 3 planes (-im, re, im)
//   three-product form (KARA, see crt_gemm_kernel): NPL = 3 on both sides, (re, im, re + im); plane p of Bt meets plane p
//   of At (Karatsuba: k1 = Br Ar, k2 = Bi Ai, k3 = (Br + Bi)(Ar + Ai); re = k1 - k2, im = k3 - k1 - k2).
//   The sum of two residues is brought back into a byte ([-128, 127], still the same class mod m_i) by crt_fix_byte.
__device__ __forceinline__ int crt_fix_byte(int s, int m) {
  // |s| <= 256: s > 127 -> s - m in [-125, 83], s < -128 -> s + m in [-83, 124] (173 <= m <= 256; for m = 256 the byte is unchanged)
  if (s > 127) s -= m;
  else if (s < -128) s += m;
  return s;
}
constexpr int RES_ROWS = RES_ROWS_C, RES_K = RES_K_C, RES_RS = RES_K + RES_K / 8 + 1;   // padded row stride (elements)
template <int COMPS, bool KARA, typename E>
__global__ void __launch_bounds__(256, 3)
crt_residue_kernel(const E* __restrict__ src, const long long* __restrict__ off_row, const long long* __restrict__ off_k,
                   long long rows, long long K, long long rowsP, long long Kp, const unsigned long long* __restrict__ rowmax, int bits, int lk,
                   const __grid_constant__ CrtTables T, int8_t* __restrict__ planes) {
  extern __shared__ __align__(16) unsigned char res_smem_raw[];
  double2* tile = reinterpret_cast<double2*>(res_smem_raw);
  __shared__ double s_scale[RES_ROWS];
  __shared__ long long s_offr[RES_ROWS], s_offk[RES_K];
  __shared__ double s_inv[CRT_MAX_MOD];      // the moduli tables out of the constant bank: an LDC with a register index
  __shared__ int s_mod[CRT_MAX_MOD];         // per loop trip was 35 % of this kernel's stall samples (ncu r02)
  const long long row0 = (long long)blockIdx.x * RES_ROWS, k0 = (long long)blockIdx.y * RES_K;
  const int tid = threadIdx.x;
  const double two_a = scalbn(1.0, bits);
  if (tid >= 64 && tid < 64 + CRT_MAX_MOD) { s_inv[tid - 64] = T.inv_mod[tid - 64]; s_mod[tid - 64] = T.mod[tid - 64]; }
  // the tile's offset tables and row scales first (one round trip), then 16 independent element loads per thread
  if (tid < RES_ROWS) {
    const long long r = row0 + tid;
    const int e = r < rows ? crt_exp_from_bits(rowmax[r]) : 0;
    s_scale[tid] = (e == kExpNonFinite) ? 0.0 : scalbn(1.0, -e);   // non-finite rows contribute zeros (outputs are poisoned later)
    s_offr[tid] = r < rows ? __ldg(off_row + r) : -1;
  } else if (tid >= 128) {
    const int k = tid - 128;
    s_offk[k] = k0 + k < K ? __ldg(off_k + k0 + k) : -1;
  }
  __syncthreads();
  double2 vv[RES_ROWS * RES_K / 256];
#pragma unroll
  for (int it = 0; it < RES_ROWS * RES_K / 256; it++) {
    int r, k;
    crt_tile_coord(it * 256 + tid, lk, r, k);
    const long long orow = s_offr[r], ok = s_offk[k];
    vv[it] = make_double2(0.0, 0.0);
    if (orow >= 0 && ok >= 0) vv[it] = crt_ld(src + orow + ok);
  }
#pragma unroll
  for (int it = 0; it < RES_ROWS * RES_K / 256; it++) {
    int r, k;
    crt_tile_coord(it * 256 + tid, lk, r, k);
    const double sc = s_scale[r];
    double2 v = vv[it];
    v.x = trunc(v.x * sc * two_a);    // (x * 2^-e) is exact, * 2^a is exact, |.| < 2^a <= 2^53
    v.y = trunc(v.y * sc * two_a);
    if (sc == 0.0) { v.x = 0.0; v.y = 0.0; }   // (Inf * 0 = NaN)
    tile[r * RES_RS + k + (k >> 3)] = v;
  }
  __syncthreads();
  const int r = tid >> 3;
  if (row0 + r >= rows) return;
  const double RMAGIC = 6755399441055744.0;   // 1.5 * 2^52: the low word of (x + RMAGIC) is rint(x) mod 2^32
  const long long plane_stride = rowsP * Kp;
#pragma unroll 1
  for (int pass = 0; pass < 2; pass++) {
    const int g = (tid & 7) + 8 * pass;        // group of 8 consecutive k
    double xr[8], xi[8];
    int lr[8], li[8];                           // the integers x mod 2^32
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const double2 v = tile[r * RES_RS + g * 9 + j];
      xr[j] = v.x; xi[j] = v.y;
      lr[j] = (int)__double2ll_rn(v.x); li[j] = (int)__double2ll_rn(v.y);
    }
    int8_t* dst = planes + (row0 + r) * Kp + k0 + g * 8;
    const int nmod = T.nmod;
#pragma unroll 1
    for (int i = 0; i < nmod; i++) {
      const int m = s_mod[i];
      const double inv = s_inv[i];
      uint32_t wr[2] = {0, 0}, wi[2] = {0, 0}, ws[2] = {0, 0};
#pragma unroll
      for (int j = 0; j < 8; j++) {
        // q = rint(x / m): ONE rounding (the product is exact inside the FMA, the sum has ulp 1); its low 32 bits are
        // the low word of the sum.  r = x - q m is tiny, so computing it modulo 2^32 in int32 is exact.
        // |x inv - x/m| <= 2^53/m * 2^-53 < 0.006  =>  |r| <= 0.506 m: <= 127 for every odd m <= 253, and for
        // m = 256 the byte wrap (128 -> -128) is itself a valid representative.
        const int qr = __double2loint(fma(xr[j], inv, RMAGIC));
        const int qi = __double2loint(fma(xi[j], inv, RMAGIC));
        const int rr = lr[j] - qr * m, ri = li[j] - qi * m;
        constexpr uint32_t sel[4] = {0x3214u, 0x3240u, 0x3410u, 0x4210u};   // low byte of the 2nd operand into byte j & 3
        wr[j >> 2] = __byte_perm(wr[j >> 2], (uint32_t)rr, sel[j & 3]);
        wi[j >> 2] = __byte_perm(wi[j >> 2], (uint32_t)ri, sel[j & 3]);
        if (KARA) ws[j >> 2] = __byte_perm(ws[j >> 2], (uint32_t)crt_fix_byte(rr + ri, m), sel[j & 3]);
      }
      int8_t* d = dst + (long long)i * (KARA ? 3 : COMPS) * plane_stride;
      if (KARA) {
        *reinterpret_cast<uint2*>(d) = make_uint2(wr[0], wr[1]);
        *reinterpret_cast<uint2*>(d + plane_stride) = make_uint2(wi[0], wi[1]);
        *reinterpret_cast<uint2*>(d + 2 * plane_stride) = make_uint2(ws[0], ws[1]);
      } else if (COMPS == 2) {
        *reinterpret_cast<uint2*>(d) = make_uint2(wr[0], wr[1]);
        *reinterpret_cast<uint2*>(d + plane_stride) = make_uint2(wi[0], wi[1]);
      } else {
        // byte-wise negation: |ri| <= 127 for odd m; for m = 256 the wrap -(-128) = -128 is again == 128 (mod 256)
        *reinterpret_cast<uint2*>(d) = make_uint2(__vneg4(wi[0]), __vneg4(wi[1]));
        *reinterpret_cast<uint2*>(d + plane_stride) = make_uint2(wr[0], wr[1]);
        *reinterpret_cast<uint2*>(d + 2 * plane_stride) = make_uint2(wi[0], wi[1]);
      }
    }
  }
}

// ---- tcgen05 helpers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t c_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void c_mbar_init(uint64_t* bar, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(c_smem(bar)), "r"(count)); }
__device__ __forceinline__ void c_mbar_expect_tx(uint64_t* bar, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(c_smem(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void c_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "CRT_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra CRT_DONE;\n\t"
      "bra CRT_WAIT;\n\t"
      "CRT_DONE:\n\t}" ::"r"(c_smem(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void c_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// K-major SWIZZLE_128B canonical layout (UMMA shared-memory descriptor): LBO = 1, SBO = 1024 B, version 1
__device__ __forceinline__ uint64_t c_desc(const void* smem) {
  uint64_t d = 0;
  d |= (uint64_t)((c_smem(smem) >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// both CTAs' loads signal the LEADER's barrier (peer bit of the shared::cluster address cleared)
__device__ __forceinline__ void c_tma_2d_2sm(const CUtensorMap* map, uint64_t* bar, void* smem, int c0, int c1) {
  const uint32_t leader_bar = c_smem(bar) & 0xFEFFFFFFu;
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(c_smem(smem)), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void c_umma_i8_2sm(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void c_commit_2sm(uint64_t* bar) {   // arrives on `bar` in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(c_smem(bar)), "h"((uint16_t)3) : "memory");
}
// arrive on `bar` of cluster CTA `cta`.  Default semantics (release at CTA scope), NOT .release.cluster: the only thing
// the waiter depends on is that this warp's TMEM reads are done (tcgen05.wait::ld + tcgen05.fence::before_thread_sync);
// a cluster-scope release compiles to MEMBAR.ALL.GPU + ERRBAR and stalls until every residue byte this warp just stored
// has reached L2 -- 2-3 thousand cycles per item, which paced all short-K items (ncu: top stall of the kernel).
__device__ __forceinline__ void c_mbar_arrive_cta(uint64_t* bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(c_smem(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void c_tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}

struct CrtGemmArgs {
  int8_t* R;          // residues + 128 as bytes: [((mod * nkc + kc) * NPL + plane) * Np + n] * Mp + m
                      //   four products: NPL = 2 (re, im);  three products: NPL = 3 (k1, k2, k3; re = k1 + k3, im = k1 + k2)
  int Np, Mp;         // padded plane rows of this panel (Np % 256 == 0, Mp % tile_m == 0)
  int pairs_n, tiles_m, tile_m;   // tile_m: 128 (four products: 128 re + 128 im columns) or 256 (three products)
  int nmod, nkc, kb_per_chunk, num_kb;
  int total_items;
  int group;          // n-pairs per raster band
  int negmod[CRT_MAX_MOD];   // -m_i (kept as data so that the epilogue's a - q m is ONE multiply-add)
  int magic[CRT_MAX_MOD];
};

struct CrtItem { int mod_i, prod, kc, n0, m0; };
template <bool KARA>
__device__ __forceinline__ CrtItem crt_decode(const CrtGemmArgs& p, int item) {
  const int tiles = p.pairs_n * p.tiles_m;
  const int mk = item / tiles, t = item - mk * tiles;
  CrtItem it;
  const int mp = mk / p.nkc;            // (modulus, product) major, K chunk minor
  it.kc = mk - mp * p.nkc;
  it.mod_i = KARA ? mp / 3 : mp; it.prod = KARA ? mp - it.mod_i * 3 : 0;
  // grouped raster: bands of `group` n-pairs x all m-tiles; concurrently running pairs (consecutive items)
  // share `group` Bt row bands and ~(#pairs / group) At tiles
  const int per_band = p.group * p.tiles_m;
  const int band = t / per_band, first = band * p.group;
  const int gsize = min(p.group, p.pairs_n - first);
  const int r = t - band * per_band;
  it.n0 = (first + r % gsize) * (2 * CRT_BT);
  it.m0 = (r / gsize) * p.tile_m;
  return it;
}

template <bool KARA>
__global__ void __launch_bounds__(CRT_THREADS, 1)
crt_gemm_kernel(const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapA,
                const __grid_constant__ CrtGemmArgs p) {
  constexpr int CRT_STAGES = CrtRing<KARA>::STAGES, CRT_STAGE_BYTES = CrtRing<KARA>::STAGE_BYTES;
  extern __shared__ __align__(1024) uint8_t crt_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(crt_smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ uint64_t full_bar[CRT_STAGES], empty_bar[CRT_STAGES], tfull_bar[2], tempty_bar[2];
  __shared__ uint32_t tmem_base_smem;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t crank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));   // cluster dims (2,1,1)
  const bool leader = crank == 0;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < CRT_STAGES; s++) { c_mbar_init(&full_bar[s], 1); c_mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; b++) { c_mbar_init(&tfull_bar[b], 1); c_mbar_init(&tempty_bar[b], 16); }   // 8 epilogue warps x 2 CTAs
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // both CTAs, same warp id, same smem destination
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(c_smem(&tmem_base_smem)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  c_cluster_sync();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_smem;

  if (warp == 0 && lane == 0) {
    // ================= TMA producer (both CTAs) =================
    int it = 0;
    for (int item = cluster_id; item < p.total_items; item += n_clusters) {
      const CrtItem w = crt_decode<KARA>(p, item);
      const int kb0 = w.kc * p.kb_per_chunk, kb1 = min(p.num_kb, kb0 + p.kb_per_chunk);
      // own 128 of the pair's 256 Bt rows; three products: plane `prod` of both operands, own 128 of the 256 At rows
      const int rowB = (KARA ? w.mod_i * 3 + w.prod : w.mod_i * 2) * p.Np + w.n0 + (int)crank * CRT_BT;
      const int rowA = (KARA ? (w.mod_i * 3 + w.prod) * p.Mp + w.m0 + (int)crank * CRT_BT : (w.mod_i * 3) * p.Mp + w.m0);
      for (int kb = kb0; kb < kb1; kb++, it++) {
        const int s = it % CRT_STAGES;
        if (it >= CRT_STAGES) c_mbar_wait(&empty_bar[s], ((it / CRT_STAGES) - 1) & 1);
        uint8_t* st = smem + s * CRT_STAGE_BYTES;
        if (leader) c_mbar_expect_tx(&full_bar[s], 2 * CRT_STAGE_BYTES);   // bytes of both CTAs land on the leader's barrier
        const int kx = kb * CRT_BKB;
        if (KARA) {
          c_tma_2d_2sm(&mapB, &full_bar[s], st + 0 * CRT_TILE, kx, rowB);           // B_p
          c_tma_2d_2sm(&mapA, &full_bar[s], st + 1 * CRT_TILE, kx, rowA);           // A_p (N rows 128 crank ...)
          continue;
        }
        c_tma_2d_2sm(&mapB, &full_bar[s], st + 0 * CRT_TILE, kx, rowB);             // Br
        c_tma_2d_2sm(&mapB, &full_bar[s], st + 1 * CRT_TILE, kx, rowB + p.Np);      // Bi
        if (leader) {
          c_tma_2d_2sm(&mapA, &full_bar[s], st + 2 * CRT_TILE, kx, rowA + p.Mp);    // X: Ar   (N rows   0..127)
          c_tma_2d_2sm(&mapA, &full_bar[s], st + 3 * CRT_TILE, kx, rowA);           // Y: -Ai
        } else {
          c_tma_2d_2sm(&mapA, &full_bar[s], st + 2 * CRT_TILE, kx, rowA + 2 * p.Mp);// X: Ai   (N rows 128..255)
          c_tma_2d_2sm(&mapA, &full_bar[s], st + 3 * CRT_TILE, kx, rowA + p.Mp);    // Y: Ar
        }
      }
    }
  } else if (warp == 1 && lane == 0 && leader) {
    // ================= MMA issuer (leader CTA only) =================
    // idesc: D = S32 (2)@4, A/B signed int8 (1)@7,@10, both K-major, N = 256 (>>3)@17, M = 256 (>>4)@24
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((256u >> 4) << 24);
    int it = 0, f = 0;
    for (int item = cluster_id; item < p.total_items; item += n_clusters, f++) {
      const CrtItem w = crt_decode<KARA>(p, item);
      const int kb0 = w.kc * p.kb_per_chunk, kb1 = min(p.num_kb, kb0 + p.kb_per_chunk);
      const int buf = f & 1;
      if (f >= 2) { c_mbar_wait(&tempty_bar[buf], ((f >> 1) - 1) & 1); asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
      const uint32_t acc = tmem_base + (uint32_t)(buf * 256);
      bool first = true;
      for (int kb = kb0; kb < kb1; kb++, it++) {
        const int s = it % CRT_STAGES;
        c_mbar_wait(&full_bar[s], (it / CRT_STAGES) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint8_t* st = smem + s * CRT_STAGE_BYTES;
        if (KARA) {
          const uint64_t d_b = c_desc(st), d_a = c_desc(st + CRT_TILE);
#pragma unroll
          for (int k = 0; k < CRT_BKB / 32; k++) {
            c_umma_i8_2sm(acc, d_b + (uint64_t)(k * 32 >> 4), d_a + (uint64_t)(k * 32 >> 4), idesc, first ? 0u : 1u);   // B_p x A_p (256 At rows)
            first = false;
          }
        } else {
          const uint64_t d_br = c_desc(st), d_bi = c_desc(st + CRT_TILE), d_x = c_desc(st + 2 * CRT_TILE), d_y = c_desc(st + 3 * CRT_TILE);
#pragma unroll
          for (int k = 0; k < CRT_BKB / 32; k++) {
            const uint64_t ko = (uint64_t)(k * 32 >> 4);
            c_umma_i8_2sm(acc, d_br + ko, d_x + ko, idesc, first ? 0u : 1u);   // Br x [Ar ; Ai]
            first = false;
            c_umma_i8_2sm(acc, d_bi + ko, d_y + ko, idesc, 1u);               // Bi x [-Ai ; Ar]
          }
        }
        c_commit_2sm(&empty_bar[s]);
      }
      c_commit_2sm(&tfull_bar[buf]);
    }
  } else if (warp >= 2) {
    // ================= epilogue (both CTAs; own 128 rows): acc mod m_i -> one (offset) byte =================
    // Eight warps: warp w reads TMEM lanes 32 (w % 4) ..., warps 2-5 take the real columns 0-127, warps 6-9 the imaginary
    // columns 128-255.  Two warps per scheduler hide each other's dependency stalls and keep all four TMEM read ports busy
    // (ncu r02 with four warps: issue slots 35 % busy, the epilogue -- not the MMA -- paced every item with K <= 1024).
    const int q = warp & 3;              // TMEM lane quarter this warp may read
    const int comp = (warp - 2) >> 2;    // 0: real, 1: imaginary (three products: At rows 0-127 / 128-255 of the tile)
    int f = 0;
    for (int item = cluster_id; item < p.total_items; item += n_clusters, f++) {
      const CrtItem w = crt_decode<KARA>(p, item);
      const int buf = f & 1;
      const int negm = p.negmod[w.mod_i], magic = p.magic[w.mod_i];
      const long long row0 = (long long)w.n0 + (int)crank * CRT_BT + q * 32;     // first of this warp's 32 rows
      int8_t* dst = KARA ? p.R + ((long long)((w.mod_i * p.nkc + w.kc) * 3 + w.prod) * p.Np + row0) * p.Mp + w.m0 + comp * CRT_BT
                         : p.R + ((long long)((w.mod_i * p.nkc + w.kc) * 2 + comp) * p.Np + row0) * p.Mp + w.m0;
      c_mbar_wait(&tfull_bar[buf], (f >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 256 + comp * CRT_BT);
      // 32 columns at a time; the TMEM load of chunk c+1 is in flight while chunk c is reduced (tcgen05.wait::ld waits for
      // every outstanding load of the thread, so it sits before the NEXT issue).  A thread owns a ROW of the accumulator,
      // so direct stores would scatter 32 x 16 bytes over 32 lines per instruction: the 32 x 128 bytes are parked in a
      // per-warp shared-memory tile (16-byte chunks XOR-swizzled by row) and written out 4 full 128-byte rows at a time.
      uint8_t* stg = smem + CRT_STAGES * CRT_STAGE_BYTES + (warp - 2) * CRT_STG_BYTES;
      uint32_t va[32], vb[32];
      c_tmem_ld32(tbase, va);
#pragma unroll
      for (int ch = 0; ch < 4; ch++) {
        uint32_t (&v)[32] = (ch & 1) == 0 ? va : vb;
        uint32_t (&nx)[32] = (ch & 1) == 0 ? vb : va;
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (ch < 3) c_tmem_ld32(tbase + (uint32_t)(32 * (ch + 1)), nx);
        uint32_t wds[8];
#pragma unroll
        for (int j = 0; j < 32; j++) {
          const int a = (int)v[j];
          // q = floor(a * magic / 2^32) in [a/m - 1.25, a/m + 0.25] (|a| < 2^31, |magic / 2^32 - 1/m| <= 2^-33), so
          // t = a - q m lies in [-0.25 m, 1.25 m] = [-64, 320]: one conditional subtraction of m leaves a representative in
          // [-128, 127]; its low byte, with the top bit flipped (once per packed word), is the OFFSET byte residue + 128.
          // (-m is passed in, the condition is a predicate: IMAD.HI + IMAD are the only multiplier-pipe instructions --
          // ncu r02, K = 512: that pipe was 68 % busy and paced the item, see profiles/r02_ncu_crt_gemm_k512.txt)
          int t = __mulhi(a, magic) * negm + a;
          if (t > 127) t += negm;
          constexpr uint32_t sel[4] = {0x3214u, 0x3240u, 0x3410u, 0x4210u};
          if ((j & 3) == 0) wds[j >> 2] = 0;
          wds[j >> 2] = __byte_perm(wds[j >> 2], (uint32_t)t, sel[j & 3]);
        }
#pragma unroll
        for (int j = 0; j < 8; j++) wds[j] ^= 0x80808080u;
        uint8_t* srow = stg + lane * CRT_STG_ROW;
        *reinterpret_cast<uint4*>(srow + (((2 * ch) ^ (lane & 7)) << 4)) = make_uint4(wds[0], wds[1], wds[2], wds[3]);
        *reinterpret_cast<uint4*>(srow + (((2 * ch + 1) ^ (lane & 7)) << 4)) = make_uint4(wds[4], wds[5], wds[6], wds[7]);
      }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int r = i * 4 + (lane >> 3), c16 = lane & 7;
        *reinterpret_cast<uint4*>(dst + (long long)r * p.Mp + c16 * 16) = *reinterpret_cast<const uint4*>(stg + r * CRT_STG_ROW + ((c16 ^ (r & 7)) << 4));
      }
      __syncwarp();
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) c_mbar_arrive_cta(&tempty_bar[buf], 0);   // the leader's MMA issuer waits for all 8 epilogue warps
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  c_cluster_sync();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
}

// ---- CRT reconstruction -------------------------------------------------------------------------------
struct CrtReconArgs {
  const int8_t* R;
  void* C;             // &C[n_begin * ldc + m_begin]: double2, or float2 for complex64 pairs
  const unsigned long long* max_n;   // row maxima (bit patterns) of this panel's Bt rows
  const unsigned long long* max_m;   // ... of this panel's At rows
  long long rows, cols, ldc;   // valid panel extent, row stride of C
  long long Np, Mp;
  int nkc;
};

// one thread: 4 consecutive m of one row n (56 registers -> 4 resident CTAs per SM: the kernel is bound by the latency of
// its residue loads, ncu r02: 52 % long_scoreboard at 25 % occupancy with 8 m per thread).  No conversion-pipe
// instruction in the inner loop: a residue byte u = y + 128 becomes the double 2^52 + u by a byte permute into the low
// mantissa word, one DADD removes 2^52 + 128 nkc.
// KARA (three products): the planes hold k1, k2, k3 (+128 each); re = k1 - k2 and im = k3 - k1 - k2 are formed here from the
// bytes (the CRT sum is linear, no reduction mod m_i needed: |y| <= 3 * 128 * 32 < 2^13.6 keeps S1 exact, 13.6 + 34 + 4.4 bits).
template <bool ONE_CHUNK, bool KARA, typename TO>
__global__ void __launch_bounds__(256, 4)
crt_reconstruct_kernel(const __grid_constant__ CrtReconArgs a, const __grid_constant__ CrtTables T) {
  const long long cols4 = a.Mp >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n = idx / cols4, m4 = (idx - n * cols4) * 4;
  if (n >= a.rows || m4 >= a.cols) return;
  double s1r[4], s2r[4], s1i[4], s2i[4];
#pragma unroll
  for (int j = 0; j < 4; j++) { s1r[j] = s2r[j] = s1i[j] = s2i[j] = 0.0; }
  const long long plane = a.Np * a.Mp;
  const int8_t* base = a.R + n * a.Mp + m4;
  // a byte is u = y + 128; four products: sum of u over chunks - 128 nkc.  Three: re = (u1 - u2 + 256) - 256 per chunk,
  // im = (u3 - u1 - u2 + 512) - 384 per chunk (the +256 / +512 keep the running sums non-negative for the conversion below)
  const double bias = 4503599627370496.0 + (KARA ? 256.0 : 128.0) * (double)a.nkc;   // 2^52 + ...
  const double bias_i = 4503599627370496.0 + (KARA ? 384.0 : 128.0) * (double)a.nkc;
#pragma unroll 8
  for (int i = 0; i < T.nmod; i++) {
    uint32_t ur[4], ui[4];     // byte sums over the K chunks (still == C' + 128 nkc mod m_i)
    if (KARA) {
#pragma unroll
      for (int j = 0; j < 4; j++) { ur[j] = 0; ui[j] = 0; }
      for (int c = 0; c < (ONE_CHUNK ? 1 : a.nkc); c++) {
        const int8_t* pk = base + (long long)((i * a.nkc + c) * 3) * plane;
        const uint32_t w1 = __ldg(reinterpret_cast<const uint32_t*>(pk));
        const uint32_t w2 = __ldg(reinterpret_cast<const uint32_t*>(pk + plane));
        const uint32_t w3 = __ldg(reinterpret_cast<const uint32_t*>(pk + 2 * plane));
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const uint32_t k1 = __byte_perm(w1, 0, 0x4440 + j), k2 = __byte_perm(w2, 0, 0x4440 + j);
          ur[j] += 256u + k1 - k2;
          ui[j] += 512u + __byte_perm(w3, 0, 0x4440 + j) - k1 - k2;
        }
      }
    } else if (ONE_CHUNK) {
      const uint32_t wr = __ldg(reinterpret_cast<const uint32_t*>(base + (long long)(i * 2) * plane));
      const uint32_t wi = __ldg(reinterpret_cast<const uint32_t*>(base + (long long)(i * 2 + 1) * plane));
#pragma unroll
      for (int j = 0; j < 4; j++) { ur[j] = __byte_perm(wr, 0, 0x4440 + j); ui[j] = __byte_perm(wi, 0, 0x4440 + j); }
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++) { ur[j] = 0; ui[j] = 0; }
      for (int c = 0; c < a.nkc; c++) {
        const int8_t* pr = base + (long long)((i * a.nkc + c) * 2) * plane;
        const uint32_t wr = __ldg(reinterpret_cast<const uint32_t*>(pr));
        const uint32_t wi = __ldg(reinterpret_cast<const uint32_t*>(pr + plane));
#pragma unroll
        for (int j = 0; j < 4; j++) { ur[j] += __byte_perm(wr, 0, 0x4440 + j); ui[j] += __byte_perm(wi, 0, 0x4440 + j); }
      }
    }
    const double r1 = T.rho1[i], r2 = T.rho2[i];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      // y * rho1 is exact (|y| <= 2^13, rho1 on a 2^-34 grid) and so is the sum over <= 20 moduli (|S1| < 2^18)
      const double dr = __hiloint2double(0x43300000, (int)ur[j]) - bias;
      const double di = __hiloint2double(0x43300000, (int)ui[j]) - bias_i;
      s1r[j] = fma(dr, r1, s1r[j]); s2r[j] = fma(dr, r2, s2r[j]);
      s1i[j] = fma(di, r1, s1i[j]); s2i[j] = fma(di, r2, s2i[j]);
    }
  }
  const int en = crt_exp_from_bits(a.max_n[n]);
  TO* dst = static_cast<TO*>(a.C) + n * a.ldc + m4;
  const double RMAGIC = 6755399441055744.0;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    if (m4 + j >= a.cols) break;
    const int em = crt_exp_from_bits(a.max_m[m4 + j]);
    double2 out;
    if (en == kExpNonFinite || em == kExpNonFinite) {
      out = make_double2(__longlong_as_double(0x7ff8000000000000LL), __longlong_as_double(0x7ff8000000000000LL));
    } else {
      // C'/P = S - round(S), |C'/P| <= 1/4; (S1 - Q) is exact, the rest rounds relative to the result itself
      const double qr = ((s1r[j] + s2r[j]) + RMAGIC) - RMAGIC;
      const double qi = ((s1i[j] + s2i[j]) + RMAGIC) - RMAGIC;
      const double fr = (s1r[j] - qr) + s2r[j], fi = (s1i[j] - qi) + s2i[j];
      out = make_double2(scalbn(fr * T.p_scaled, en + em), scalbn(fi * T.p_scaled, en + em));
    }
    if constexpr (sizeof(TO) == sizeof(double2)) dst[j] = out;
    else dst[j] = make_float2((float)out.x, (float)out.y);   // the one rounding of a complex64 result
  }
}

// ---- host side ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn crt_get_encode() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    cudaDriverEntryPointQueryResult q;
    void* p = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess) fn = (EncodeTiledFn)p;
  }
  return fn;
}
static int crt_make_map(CUtensorMap* m, void* ptr, uint64_t rows, uint64_t kbytes) {
  EncodeTiledFn enc = crt_get_encode();
  if (!enc) return fail(TNCB_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
  cuuint64_t dims[2] = {kbytes, rows};
  cuuint64_t strides[1] = {kbytes};
  cuuint32_t box[2] = {(cuuint32_t)CRT_BKB, (cuuint32_t)CRT_BT};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TNCB_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return TNCB_OK;
}

static inline long long round_up_ll(long long x, long long a) { return (x + a - 1) / a * a; }


// tables: offAm[M], offBn[N], offAk[K], offBk[K] (built by the caller, see kernels.cu)
template <typename E>
static int launch_k1_crt_t(tncb_ctx* ctx, const PairPlan& P, const E* A, const E* B, E* C,
                           const long long* offAm, const long long* offBn, const long long* offAk, const long long* offBk) {
  int nmod, bits_a, bits_b;
  // complex64 operands carry 24-bit mantissas: a = 28 bits keep the bound at 2^-24 K max|b| max|a|, the worst case of an
  // FP32 dot product, with about 9 instead of 16 moduli at K = 4096.  A tolerance set on the context still decides.
  const int dflt = sizeof(E) == sizeof(double2) ? ctx->crt_bits : kCrtBitsC64;
  const int want = ctx->crt_tol > 0.0 ? crt_bits_for_tolerance(P.K, ctx->crt_tol) : dflt;
  crt_choose(P.K, want, ctx->crt_nmod_force, &nmod, &bits_a, &bits_b);
  CrtTables T;
  crt_make_tables(nmod, bits_a, bits_b, T);
  cudaStream_t st = ctx->stream;
  const long long Kp = round_up_ll(P.K, CRT_BKB);
  const int num_kb = (int)(Kp / CRT_BKB);
  const int n_clusters_max = std::max(1, ctx->sm_count / 2);
  // three real products per complex product (Karatsuba; sums of residues are exact mod m_i) instead of four: 25 % fewer int8
  // operations for one more operand plane per side and one more residue plane.  An item then carries half the MMA work per
  // accumulator, so short K (where the epilogue paces the item) keeps the four-product form: measured break-even K ~ 4096.
  const bool kara = ctx->crt_products == 3 || (ctx->crt_products == 0 && Kp >= ctx->crt_kara_min_k);
  const int TM = kara ? 2 * CRT_BT : CRT_BT;        // At rows per tile
  const int NPB = kara ? 3 : 2, NPR = kara ? 3 : 2;  // Bt operand planes, residue planes per modulus
  // K chunks: int32-safe length, and more chunks when there are too few tiles to fill the machine (split-K:
  // the reconstruction adds the chunk residues)
  const long long tiles_total = round_up_ll(P.N, 2 * CRT_BT) / (2 * CRT_BT) * (round_up_ll(P.M, TM) / TM);
  int nkc = (int)((Kp + CRT_KCHUNK_MAX - 1) / CRT_KCHUNK_MAX);
  {
    const long long items = tiles_total * nmod * (kara ? 3 : 1);
    const long long want = 2LL * n_clusters_max;
    if (items * nkc < want) nkc = (int)std::min<long long>((want + items - 1) / items, std::max(1, num_kb / 8));
    nkc = std::max(1, std::min(nkc, 32));      // exactness of the reconstruction: sum of <= 32 chunk residues
  }
  int kb_per_chunk = (num_kb + nkc - 1) / nkc;
  nkc = (num_kb + kb_per_chunk - 1) / kb_per_chunk;
  if ((long long)kb_per_chunk * CRT_BKB > CRT_KCHUNK_MAX) return fail(TNCB_ERR_UNSUPPORTED, "K too long for the int8 engine");

  // ---- panels: bound the workspace (planes + residues) ----
  const size_t budget = ctx->crt_ws_bytes;
  long long pn = round_up_ll(P.N, 2 * CRT_BT), pm = round_up_ll(P.M, TM);   // panel extents (padded)
  auto ws_bytes = [&](long long n_, long long m_) {
    return (size_t)nmod * (size_t)Kp * (size_t)(NPB * n_ + 3 * m_) + (size_t)nmod * nkc * NPR * (size_t)n_ * (size_t)m_;
  };
  while (ws_bytes(pn, pm) > budget && (pm > TM || pn > 2 * CRT_BT)) {
    if (pm >= pn && pm > TM) pm = round_up_ll(pm / 2, TM);
    else if (pn > 2 * CRT_BT) pn = round_up_ll(pn / 2, 2 * CRT_BT);
    else pm = round_up_ll(pm / 2, TM);
  }
  const size_t bytesB = (size_t)nmod * NPB * pn * Kp, bytesA = (size_t)nmod * 3 * pm * Kp;
  const size_t bytesR = (size_t)nmod * nkc * NPR * pn * pm;
  const size_t bytesE = (size_t)(pn + pm) * sizeof(unsigned long long);
  void *pb = nullptr, *pa = nullptr, *pr = nullptr, *pe = nullptr;
  int rc;
  if ((rc = ctx->arena.alloc(bytesB, &pb))) return rc;
  if ((rc = ctx->arena.alloc(bytesA, &pa))) { ctx->arena.free(pb, bytesB); return rc; }
  if ((rc = ctx->arena.alloc(bytesR, &pr))) { ctx->arena.free(pb, bytesB); ctx->arena.free(pa, bytesA); return rc; }
  if ((rc = ctx->arena.alloc(bytesE, &pe))) { ctx->arena.free(pb, bytesB); ctx->arena.free(pa, bytesA); ctx->arena.free(pr, bytesR); return rc; }
  auto cleanup = [&]() { ctx->arena.free(pb, bytesB); ctx->arena.free(pa, bytesA); ctx->arena.free(pr, bytesR); ctx->arena.free(pe, bytesE); };
  unsigned long long* max_n = (unsigned long long*)pe;
  unsigned long long* max_m = max_n + pn;

  static bool attr_done_dev[64] = {false};          // cudaFuncSetAttribute is per device
  bool& attr_done = attr_done_dev[ctx->device & 63];
  const int smem_gemm = CRT_RING_BYTES + 8 * CRT_STG_BYTES + 1024;
  const int smem_res = RES_ROWS * RES_RS * (int)sizeof(double2);   // (the tile holds widened, truncated values)
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(crt_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_gemm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crt_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_gemm);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crt_residue_kernel<2, false, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_res);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crt_residue_kernel<3, false, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_res);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crt_residue_kernel<2, true, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_res);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crt_residue_kernel<3, true, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_res);
    if (e != cudaSuccess) { cleanup(); return fail(TNCB_ERR_CUDA, cudaGetErrorString(e)); }
    attr_done = true;
  }
  // lanes of a warp: 2^lk along k, the rest along rows -- as many k lanes as the operand's fastest K leg is long when k is
  // the fastest index (stride 1), otherwise as many row lanes as the fastest free leg is long
  auto lane_split = [](const LegList& kl, bool k_is_b, const LegList& fl) {
    auto p2 = [](long long d) { int b = 0; while ((2LL << b) <= d && b < 5) b++; return b; };
    const long long ks = kl.n ? (k_is_b ? kl.sb[kl.n - 1] : kl.sa[kl.n - 1]) : (1LL << 62);
    const long long fs = fl.n ? fl.sa[fl.n - 1] : (1LL << 62);
    if (ks <= fs) return kl.n ? p2(kl.dim[kl.n - 1]) : 0;          // k fastest: as many k lanes as that leg is long
    return 0;   // rows fastest: all lanes along rows (the K list's last group need not be this operand's fastest K leg,
                // so lanes along k could land on far-apart addresses)
  };
  const int lk_b = lane_split(P.k, true, P.n), lk_a = lane_split(P.k, false, P.m);
  ctx->last_int8_ops = 0.0; ctx->last_nmod = nmod; ctx->last_products = kara ? 3 : 4;
  bool timed = false;

  for (long long n0 = 0; n0 < P.N; n0 += pn) {
    const long long nrows = std::min(pn, P.N - n0);
    const long long Np = round_up_ll(nrows, 2 * CRT_BT);
    // ---- Bt panel: exponents + residues (padding rows / K tail must be zero residues) ----
    if (Np != nrows) cudaMemsetAsync(pb, 0, (size_t)nmod * NPB * Np * Kp, st);
    cudaMemsetAsync(max_n, 0, (size_t)nrows * sizeof(unsigned long long), st);
    {
      dim3 g((unsigned)((nrows + RES_ROWS - 1) / RES_ROWS), (unsigned)(Kp / RES_K));
      crt_rowmax_kernel<<<g, 256, 0, st>>>(B, offBn + n0, offBk, nrows, P.K, lk_b, max_n);
      if (kara) crt_residue_kernel<2, true, E><<<g, 256, smem_res, st>>>(B, offBn + n0, offBk, nrows, P.K, Np, Kp, max_n, bits_b, lk_b, T, (int8_t*)pb);
      else crt_residue_kernel<2, false, E><<<g, 256, smem_res, st>>>(B, offBn + n0, offBk, nrows, P.K, Np, Kp, max_n, bits_b, lk_b, T, (int8_t*)pb);
    }
    ctx->launches += 2;
    CUtensorMap mapB;
    if ((rc = crt_make_map(&mapB, pb, (uint64_t)nmod * NPB * Np, (uint64_t)Kp))) { cleanup(); return rc; }
    for (long long m0 = 0; m0 < P.M; m0 += pm) {
      const long long mcols = std::min(pm, P.M - m0);
      const long long Mp = round_up_ll(mcols, TM);
      if (Mp != mcols) cudaMemsetAsync(pa, 0, (size_t)nmod * 3 * Mp * Kp, st);
      cudaMemsetAsync(max_m, 0, (size_t)mcols * sizeof(unsigned long long), st);
      {
        dim3 g((unsigned)((mcols + RES_ROWS - 1) / RES_ROWS), (unsigned)(Kp / RES_K));
        crt_rowmax_kernel<<<g, 256, 0, st>>>(A, offAm + m0, offAk, mcols, P.K, lk_a, max_m);
        if (kara) crt_residue_kernel<3, true, E><<<g, 256, smem_res, st>>>(A, offAm + m0, offAk, mcols, P.K, Mp, Kp, max_m, bits_a, lk_a, T, (int8_t*)pa);
        else crt_residue_kernel<3, false, E><<<g, 256, smem_res, st>>>(A, offAm + m0, offAk, mcols, P.K, Mp, Kp, max_m, bits_a, lk_a, T, (int8_t*)pa);
      }
      ctx->launches += 2;
      CUtensorMap mapA;
      if ((rc = crt_make_map(&mapA, pa, (uint64_t)nmod * 3 * Mp, (uint64_t)Kp))) { cleanup(); return rc; }
      CrtGemmArgs g;
      g.R = (int8_t*)pr; g.Np = (int)Np; g.Mp = (int)Mp;
      g.pairs_n = (int)(Np / (2 * CRT_BT)); g.tiles_m = (int)(Mp / TM); g.tile_m = TM;
      g.nmod = nmod; g.nkc = nkc; g.kb_per_chunk = kb_per_chunk; g.num_kb = num_kb;
      const long long items = (long long)g.pairs_n * g.tiles_m * nmod * nkc * (kara ? 3 : 1);
      if (items > 0x7fffffffLL) { cleanup(); return fail(TNCB_ERR_UNSUPPORTED, "too many work items"); }
      g.total_items = (int)items;
      g.group = ctx->crt_group;
      for (int i = 0; i < CRT_MAX_MOD; i++) { g.negmod[i] = -T.mod[i]; g.magic[i] = T.magic[i]; }
      const int n_clusters = (int)std::min<long long>(n_clusters_max, items);
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3((unsigned)(2 * n_clusters)); cfg.blockDim = dim3(CRT_THREADS);
      cfg.dynamicSmemBytes = smem_gemm; cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      const double ops = 2.0 * (kara ? 3.0 : 4.0) * (double)nmod * (double)Np * (double)Mp * (double)Kp;
      const bool time_this = ctx->time_gemm == 2 || (ctx->time_gemm == 1 && !timed);
      if (time_this) gemm_timer_begin(ctx);
      cudaError_t e = kara ? cudaLaunchKernelEx(&cfg, crt_gemm_kernel<true>, mapB, mapA, g)
                           : cudaLaunchKernelEx(&cfg, crt_gemm_kernel<false>, mapB, mapA, g);
      if (time_this) { gemm_timer_end(ctx, ops); timed = true; }
      if (e != cudaSuccess) { cleanup(); return fail(TNCB_ERR_CUDA, std::string("crt_gemm_kernel launch: ") + cudaGetErrorString(e)); }
      ctx->last_int8_ops += ops;
      CrtReconArgs r;
      r.R = (const int8_t*)pr; r.C = C + n0 * P.M + m0; r.max_n = max_n; r.max_m = max_m;
      r.rows = nrows; r.cols = mcols; r.ldc = P.M; r.Np = Np; r.Mp = Mp; r.nkc = nkc;
      const long long threads = nrows * (Mp / 4);
      const unsigned rg = (unsigned)((threads + 255) / 256);
      if (kara) {
        if (nkc == 1) crt_reconstruct_kernel<true, true, E><<<rg, 256, 0, st>>>(r, T);
        else crt_reconstruct_kernel<false, true, E><<<rg, 256, 0, st>>>(r, T);
      } else {
        if (nkc == 1) crt_reconstruct_kernel<true, false, E><<<rg, 256, 0, st>>>(r, T);
        else crt_reconstruct_kernel<false, false, E><<<rg, 256, 0, st>>>(r, T);
      }
      ctx->launches += 2;
    }
  }
  ctx->engine_count[4]++;
  cudaError_t e = cudaGetLastError();
  cleanup();   // stream-ordered reuse: later allocations are only touched by later kernels
  if (e != cudaSuccess) return fail(TNCB_ERR_CUDA, std::string("K1' (CRT) launch: ") + cudaGetErrorString(e));
  return TNCB_OK;
}

int launch_k1_crt(tncb_ctx* ctx, const PairPlan& P, const void* A, const void* B, void* C,
                  const long long* offAm, const long long* offBn, const long long* offAk, const long long* offBk, int dtype) {
  if (dtype == TNCB_C64)
    return launch_k1_crt_t(ctx, P, (const float2*)A, (const float2*)B, (float2*)C, offAm, offBn, offAk, offBk);
  return launch_k1_crt_t(ctx, P, (const double2*)A, (const double2*)B, (double2*)C, offAm, offBn, offAk, offBk);
}

} // namespace tncb

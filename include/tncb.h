/*
 * tncb.h -- C ABI of libtncb200: the B200-native pairwise tensor-contraction hot
 * path of qc-tum/TNC (tnc v1.0.0 @ 5dd62b3).
 *
 * This is the drop-in boundary.  TNC reaches its numeric kernel through plain
 * Rust calls into the un-vendored crate `tetra` (tnc/src/tensornetwork/
 * contraction.rs:3,78-84); a maintainer replaces those calls by the entry
 * points below through an `extern "C"` block (see INTEGRATION.md for the Rust
 * binding).  Every entry point cites the reference interface it replaces
 * (paths relative to the reference checkout).
 *
 * Conventions (identical to the reference, SURVEY.md A.1):
 *   - elements are complex128, passed as interleaved (re, im) doubles;
 *   - data is row-major (C order) over the tensor's leg order;
 *   - the result of contracting a and b has legs (b \ a) ++ (a \ b)
 *     (tnc/src/tensornetwork/tensor.rs:463-479 via contraction.rs:64);
 *   - paths are "replace-left": (i, j) stores the result in slot i
 *     (tnc/src/contractionpath.rs:29-35).
 *
 * Errors: every function returns 0 (TNCB_OK) or a negative tncb_status; nothing
 * aborts.  The reference panics instead (tensordata.rs:42, contraction.rs:50);
 * the language shim maps non-zero to panic!/exception.
 * Threading: a tncb_ctx is single-threaded like the reference's driver loop;
 * distinct contexts (devices) may be driven from distinct threads.
 * There is NO CPU fallback: without a CUDA device tncb_ctx_create fails with
 * TNCB_ERR_CUDA.
 */
#ifndef TNCB_H
#define TNCB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum tncb_status {
  TNCB_OK = 0,
  TNCB_ERR_INVALID = -1,      /* bad argument / malformed network or path            */
  TNCB_ERR_SHAPE = -2,        /* bond dimensions of a shared leg disagree            */
  TNCB_ERR_UNCONTRACTED = -3, /* slot already consumed / no data (tensordata.rs:42)  */
  TNCB_ERR_NOT_CONTRACTED = -4, /* >1 tensor left ("Not fully contracted", contraction.rs:50) */
  TNCB_ERR_OOM = -5,          /* device arena exhausted (peak live bytes > capacity) */
  TNCB_ERR_CUDA = -6,         /* CUDA runtime error (tncb_last_error has the text)   */
  TNCB_ERR_GATE = -7,         /* unknown gate / wrong angle count (gates.rs:54,103)  */
  TNCB_ERR_NCCL = -8,         /* NCCL error or libnccl not loadable                  */
  TNCB_ERR_UNSUPPORTED = -9,  /* e.g. an HDF5 feature outside the supported subset     */
  TNCB_ERR_IO = -10           /* file missing / unreadable / not (well-formed) HDF5    */
} tncb_status;

/* Element type of a tensor, a network run or a plan.  complex128 is the default of every entry point without a
 * dtype argument.  complex64 is always explicit (the *_dt entry points) and follows one precision contract:
 * operands are read as complex64 and widened exactly to f64, products and sums run in f64 (in the order of the
 * complex128 kernel), the result is rounded to complex64 once, at the store.  K0, K0-batch, K1 (DMMA) and K2 make
 * the same kernel and configuration choices for both types, so their complex64 result equals, bit for bit,
 * complex64(complex128 kernel(widen(a), widen(b))).  K1' (CRT) keeps a = 28 operand bits for complex64 pairs unless
 * a tolerance is set: the bound below becomes 2^-24 K max|b[n,:]| max|a[m,:]|, the classical worst case of an FP32 dot
 * product, with about 9 moduli at K = 4096.  complex64 pairs that qualify for K1' always use the CRT engine, also
 * when tncb_ctx_set_tcgen05_engine(1) selected digit slicing (which has no complex64 path).
 * Operands of different dtypes are refused with TNCB_ERR_INVALID (no implicit promotion). */
typedef enum tncb_dtype { TNCB_C128 = 0, TNCB_C64 = 1 } tncb_dtype;

typedef struct tncb_ctx tncb_ctx;       /* one device + stream + arena              */
typedef struct tncb_tensor tncb_tensor; /* a device-resident complex128 or complex64 tensor */
typedef struct tncb_plan tncb_plan;     /* a compiled (network, path) schedule      */
typedef struct tncb_h5file tncb_h5file; /* an opened HDF5 tensor file (host only)   */

const char* tncb_strerror(int status);
/* Text of the last error raised on this thread (CUDA/NCCL message, offending pair). */
const char* tncb_last_error(void);
/* Library version / build info (arch list) -- cheap, needs no GPU. */
const char* tncb_version(void);

/* ---- context ------------------------------------------------------------------ */
/* arena_bytes = 0: grow on demand up to the device's free memory. */
int tncb_ctx_create(int device, size_t arena_bytes, tncb_ctx** out);
void tncb_ctx_destroy(tncb_ctx* ctx);
int tncb_ctx_synchronize(tncb_ctx* ctx);
/* The CUDA stream every kernel of this ctx is enqueued on (a cudaStream_t). */
void* tncb_ctx_stream(tncb_ctx* ctx);
/* Counters since creation / last reset: kernels launched by this library, arena peak. */
/* Give device memory back to the driver: synchronises, then cudaFree's every arena slab that holds no live block (the
 * arena otherwise keeps what it reserved for reuse).  For processes that switch between workloads of very different
 * footprints (e.g. a flat network, then a sliced one with a 64 GiB workspace).  The internal plan cache of
 * tncb_contract_tensor_network is dropped as well; plans created with tncb_plan_create keep their workspaces until they
 * are destroyed. */
int tncb_ctx_trim(tncb_ctx* ctx, uint64_t* freed_bytes, uint64_t* reserved_bytes);
int tncb_ctx_stats(tncb_ctx* ctx, uint64_t* kernel_launches, uint64_t* arena_peak_bytes,
                   uint64_t* arena_live_bytes);
int tncb_ctx_reset_stats(tncb_ctx* ctx);
/* Dense-GEMM engine for large GEMM-like pairs (M, N >= 128, K >= 256, M*N*K >= 2^28): K1', the tcgen05 int8
 * tensor pipe (tcgen05.mma has no f64 kind).  Default engine = integer modular (CRT) emulation: every operand row
 * is scaled by a power of two and truncated to an `a`-bit integer (a = 53 by default = the whole mantissa of the
 * row's largest element), one int8 GEMM per coprime modulus (16 moduli for a = 53, K <= 2^13), exact CRT
 * reconstruction.  GUARANTEED bound (not "exact"):
 *     |C - C_exact|[n,m] <= 2^(4-a) * K * max|b[n,:]| * max|a[m,:]|     (max over real and imaginary parts)
 * i.e. normwise per output row/column, FP64-GEMM-equivalent for a = 53 (measured 3e-16..1e-15 of max|C|).
 * Elements far below their row maximum lose relative precision; a row whose maximum is below 2^-1000 keeps absolute
 * accuracy 2^(-1000-a); a row containing NaN/Inf poisons its outputs with NaN.
 * slices = 0 -> FP64 tensor pipe (DMMA) for every pair; non-zero -> K1' enabled (the value is the digit count of the
 * legacy 7-bit digit-slicing engine, see tncb_ctx_set_tcgen05_engine).  Smaller pairs always use DMMA / K0 / K2.
 * Environment: TNCB_OZAKI_SLICES, TNCB_TCGEN05_ENGINE, TNCB_CRT_MODULI override the defaults. */
int tncb_ctx_set_tcgen05_slices(tncb_ctx* ctx, int slices);
/* 0 = modular / CRT engine (default), 1 = 7-bit digit slicing of round 1 (S(S+1)/2 int8 GEMMs, drops digit
 * products p+q >= S: error <= (S+1) K 2^(-7S) of the same scale; kept for A/B measurements). */
int tncb_ctx_set_tcgen05_engine(tncb_ctx* ctx, int engine);
/* Requested normwise tolerance of K1': the engine keeps a = min(53, ceil(log2(16 K / rel))) bits per operand so that
 * |C - C_exact|[n,m] <= rel * max|b[n,:]| * max|a[m,:]| holds for every pair; rel = 0 (default) = full mantissa.
 * Fewer bits need fewer moduli (= int8 GEMM sweeps): see tncb_tcgen05_bound. */
int tncb_ctx_set_tolerance(tncb_ctx* ctx, double rel);
/* Pin the number of moduli (2..20; 0 = derive from the tolerance).  The operand bits then follow from
 * log2(prod m_i) >= a + b + log2(K) + 3; counts above what 53-bit operands need for the pair's K are clamped to that
 * (more moduli cannot add accuracy).  Measurement / test aid. */
int tncb_ctx_set_tcgen05_moduli(tncb_ctx* ctx, int n_moduli);
/* Real int8 GEMMs per modulus behind one complex product: 4 (re = ArBr - AiBi, im = ArBi + AiBr) or 3 (Karatsuba:
 * k1 = ArBr, k2 = AiBi, k3 = (Ar+Ai)(Br+Bi); re = k1 - k2, im = k3 - k1 - k2 -- the operand sums are taken on the residues,
 * i.e. exactly, so both forms reconstruct the same integers and differ only in the last rounding of the reconstruction).
 * 25 % fewer int8 operations for one more operand plane per side and one more residue plane, which pays from K ~ 4096
 * (profiles/r02_engine_sweep.jsonl): 0 (default) = 3 when K >= min_k3 (default 4096), else 4; min_k3 <= 0 keeps the
 * current threshold. */
int tncb_ctx_set_tcgen05_products(tncb_ctx* ctx, int products, long long min_k3);
/* What K1' would do for contraction length k (no GPU): modulus count, operand bits and the guaranteed factor
 * `bound` with |C - C_exact|[n,m] <= bound * max|b[n,:]| * max|a[m,:]|. */
int tncb_tcgen05_bound(uint64_t k, double rel, int n_moduli_force, int* n_moduli, int* bits_a, int* bits_b, double* bound);
/* The moduli and the split CRT weights rho_i = rho1_i + rho2_i = ((P/m_i)^-1 mod m_i) / m_i the engine uses for
 * `n_moduli` moduli (host-only; arrays of n_moduli entries): C'/P = frac(sum_i y_i rho_i) for residues y_i. */
int tncb_tcgen05_tables(int n_moduli, int* moduli, double* rho1, double* rho2, double* log2_product);
/* Workspace budget of K1' (residue planes + residues, default 12 GiB): larger pairs are processed in panels. */
int tncb_ctx_set_tcgen05_workspace(tncb_ctx* ctx, size_t bytes);
/* Size thresholds: (min_tiles, min_k) of the digit-slicing engine; for the modular engine min_k is the K threshold
 * and min_tiles == 1 drops the M*N*K >= 2^28 requirement (used by the parity tests). */
int tncb_ctx_set_tcgen05_threshold(tncb_ctx* ctx, long long min_tiles, long long min_k);
/* Pairs executed per engine since the last tncb_ctx_reset_stats: [0] K0, [1] K0 split-K, [2] K1 (DMMA),
 * [3] K1 split-K, [4] K1' (tcgen05), [5] K2, [6] permute, [7] reserved. */
int tncb_ctx_engine_counts(tncb_ctx* ctx, uint64_t counts[8]);
/* int8 operations (2 x MAC) executed by the GEMM kernels of the last K1' pair and its modulus count. */
int tncb_ctx_last_tcgen05_info(tncb_ctx* ctx, double* int8_ops, int* n_moduli);
/* ... and whether it used the 3- or the 4-product form. */
int tncb_ctx_last_tcgen05_products(tncb_ctx* ctx, int* products);
/* Measurement aid: bracket the dominant GEMM kernel of every large pair (k1_kernel / oz_gemm_kernel)
 * with CUDA events on the ctx stream; tncb_ctx_last_gemm_ms synchronises and returns the last one. */
int tncb_ctx_time_gemm(tncb_ctx* ctx, int enable);
int tncb_ctx_last_gemm_ms(tncb_ctx* ctx, float* ms);
/* enable = 2: every launch of the tcgen05 GEMM kernel is bracketed; tncb_ctx_gemm_totals synchronises, returns the
 * summed device time, the executed int8 operations (2 x MAC, padded tiles) and the launch count, and resets. */
int tncb_ctx_gemm_totals(tncb_ctx* ctx, double* ms, double* int8_ops, uint64_t* launches);

/* ---- tensors: replaces tetra::Tensor::{new_from_flat, elements, shape, ndim}
 *      (tnc/src/tensornetwork/tensordata.rs:31-37, tnc/src/io/hdf5.rs:105-106) ---- */
int tncb_tensor_upload(tncb_ctx* ctx, int rank, const uint64_t* dims,
                       const double* host_re_im, tncb_tensor** out);
int tncb_tensor_alloc(tncb_ctx* ctx, int rank, const uint64_t* dims, tncb_tensor** out);
/* Same with an element type: host_re_im holds interleaved float pairs for TNCB_C64, double pairs for TNCB_C128. */
int tncb_tensor_upload_dt(tncb_ctx* ctx, int rank, const uint64_t* dims, int dtype, const void* host_re_im, tncb_tensor** out);
int tncb_tensor_alloc_dt(tncb_ctx* ctx, int rank, const uint64_t* dims, int dtype, tncb_tensor** out);
/* tncb_dtype of t (TNCB_ERR_INVALID for NULL). */
int tncb_tensor_dtype(const tncb_tensor* t);
/* download / write / read copy raw data in the tensor's own dtype: for a complex64 tensor the host buffer holds
 * interleaved float pairs (8 bytes per element) although the pointer is declared double*. */
int tncb_tensor_download(tncb_ctx* ctx, const tncb_tensor* t, double* host_re_im);
/* Asynchronous variants on the ctx stream (host buffer should be pinned; the caller
 * synchronises with tncb_ctx_synchronize before touching it). */
int tncb_tensor_write(tncb_ctx* ctx, tncb_tensor* t, const double* host_re_im);
int tncb_tensor_read(tncb_ctx* ctx, const tncb_tensor* t, double* host_re_im);
int tncb_tensor_free(tncb_ctx* ctx, tncb_tensor* t);
int tncb_tensor_rank(const tncb_tensor* t);
int tncb_tensor_dims(const tncb_tensor* t, uint64_t* dims_out);
uint64_t tncb_tensor_elements(const tncb_tensor* t);
void* tncb_tensor_device_ptr(const tncb_tensor* t); /* double2* (complex128) or float2* (complex64), row-major */

/* ---- one pairwise contraction: replaces
 *      tetra::contract(out_legs, a_legs, a, b_legs, b) as called at
 *      tnc/src/tensornetwork/contraction.rs:78-84.  Consumes a and b (the Rust
 *      call moves them), returns a new tensor whose legs are out_legs, which must
 *      equal (b \ a) ++ (a \ b).  Pass out_legs = NULL to skip that check and
 *      read the legs back with tncb_pair_out_legs.
 *      The pair entry points, tncb_permute, tncb_conjugate and tncb_tensor_add follow their operands' dtype (the
 *      result has it too); operands (and the output of _into) of different dtypes -> TNCB_ERR_INVALID.
 *      tncb_contract_pair_host is complex128 only. ---- */
int tncb_contract_pair(tncb_ctx* ctx, int n_out, const uint64_t* out_legs,
                       int n_a, const uint64_t* a_legs, tncb_tensor* a,
                       int n_b, const uint64_t* b_legs, tncb_tensor* b,
                       tncb_tensor** out);
/* Same, but a and b stay alive (for benchmarking a single pair repeatedly). */
int tncb_contract_pair_keep(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const tncb_tensor* a,
                            int n_b, const uint64_t* b_legs, const tncb_tensor* b,
                            tncb_tensor** out);
/* Into a caller-provided output tensor (no allocation inside the timed region). */
int tncb_contract_pair_into(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const tncb_tensor* a,
                            int n_b, const uint64_t* b_legs, const tncb_tensor* b,
                            tncb_tensor* out);
/* tetra::contract for HOST operands (interleaved complex128, row-major), pipelined and asynchronous: the call enqueues
 * H2D(a, b) on a copy stream, the pair kernels on the ctx stream and D2H(result) on a second copy stream, then
 * returns.  Back-to-back calls overlap the upload of pair j+1, the kernels of pair j and the download of pair j-1
 * (three private sets of device buffers).  host_c receives (b \ a) ++ (a \ b) in row-major order
 * (tncb_pair_out_legs gives legs and dims).  Pinned host memory is required for the overlap; buffers are valid /
 * reusable after tncb_ctx_synchronize. */
int tncb_contract_pair_host(tncb_ctx* ctx, int n_a, const uint64_t* a_legs, const uint64_t* a_dims, const double* host_a,
                            int n_b, const uint64_t* b_legs, const uint64_t* b_dims, const double* host_b, double* host_c);
/* Leg algebra only (no GPU): Tensor::symmetric_difference, tensor.rs:463-479.
 * Writes (b\a)++(a\b) and the GEMM view M=|a\b|, N=|b\a|, K=|a&b|. */
int tncb_pair_out_legs(int n_a, const uint64_t* a_legs, const uint64_t* a_dims,
                       int n_b, const uint64_t* b_legs, const uint64_t* b_dims,
                       int* n_out, uint64_t* out_legs, uint64_t* out_dims,
                       uint64_t* m, uint64_t* n, uint64_t* k);
/* Which kernel class the planner would pick for that pair (no GPU):
 * 0 = K0 strided/warp-reduce kernel, 1 = K1 fused gather ZGEMM (DMMA, or tcgen05 K1' above the size
 * threshold), 2 = K2 streaming kernel (big tensor x tiny tensor, HBM-bound). */
int tncb_pair_kernel_class(int n_a, const uint64_t* a_legs, const uint64_t* a_dims,
                           int n_b, const uint64_t* b_legs, const uint64_t* b_dims);

/* ---- tetra::Tensor::transpose / conjugate
 *      (tnc/src/builders/circuit_builder.rs:106 Permutor::apply; gates.rs:87,98) ---- */
/* out dims[i] = in dims[perm[i]] (numpy.transpose semantics); consumes `t`. */
int tncb_permute(tncb_ctx* ctx, tncb_tensor* t, const int* perm, tncb_tensor** out);
int tncb_conjugate(tncb_ctx* ctx, tncb_tensor* t); /* in place */
/* dst += src (same element count): accumulation of sliced contractions (the reference's declared
 * future work, book/src/future_work.md:9-11). */
int tncb_tensor_add(tncb_ctx* ctx, tncb_tensor* dst, const tncb_tensor* src);

/* ---- gate table: replaces load_gate / load_gate_adjoint (tnc/src/gates.rs:50-66).
 *      Host-side; writes 4 or 16 interleaved complex values, *rank = 2 or 4. ---- */
int tncb_gate_matrix(const char* name, const double* angles, int n_angles, int adjoint,
                     double* out_re_im, int* rank);

/* ---- networks: mirrors tnc::tensornetwork::tensor::Tensor (tensor.rs:21-37) and
 *      tnc::contractionpath::ContractionPath (contractionpath.rs:29-35) as plain
 *      C trees so that cgo / Rust repr(C) / ctypes can build them. ---- */
typedef enum tncb_data_kind {
  TNCB_DATA_UNCONTRACTED = 0, /* TensorData::Uncontracted (composite or empty slot) */
  TNCB_DATA_MATRIX = 1,       /* TensorData::Matrix: host_re_im, row-major          */
  TNCB_DATA_GATE = 2,         /* TensorData::Gate((name, angles, adjoint))          */
  TNCB_DATA_DEVICE = 3,       /* already on the device (consumed by the call)       */
  TNCB_DATA_FILE = 4          /* TensorData::File((path, adjoint)): HDF5, see below */
} tncb_data_kind;

typedef struct tncb_tn {
  /* composite: n_children > 0, legs ignored.  leaf: n_children == 0. */
  size_t n_children;
  const struct tncb_tn* children;
  int rank;
  const uint64_t* legs;
  const uint64_t* dims;
  int kind; /* tncb_data_kind */
  const double* host_re_im;
  const char* gate_name;
  const double* gate_angles;
  int n_gate_angles;
  int gate_adjoint;
  tncb_tensor* device;
  /* TNCB_DATA_FILE (tensordata.rs:43-49): the first member of the file's /tensors group is loaded while the leaves are
   * staged (load_data, io/hdf5.rs:37-43), adjointed when file_adjoint != 0 (halves of the dims swapped + conjugated,
   * gates.rs:82-99; the rank must then be a power of two) and must have exactly this leaf's dims -> TNCB_ERR_SHAPE. */
  const char* file_path;
  int file_adjoint;
} tncb_tn;

typedef struct tncb_path {
  size_t n_pairs;
  const uint64_t* pairs; /* i0, j0, i1, j1, ... replace-left */
  size_t n_nested;
  const uint64_t* nested_index; /* child indices that have their own path */
  const struct tncb_path* nested;
} tncb_path;

/* contract_tensor_network(tn, path) (tnc/src/tensornetwork/contraction.rs:30-52):
 * nested paths first (ascending child index), then the top-level pairs in order.
 * Leaves are materialised (gates.rs tables) and uploaded in ONE host->device
 * copy, every pair runs on the device without host round trips, and the result
 * stays on the device.  out_legs must have room for *n_out legs (<= 64).
 * TNCB_DATA_DEVICE leaves are consumed atomically: on TNCB_OK every one of them has been freed
 * (the Rust call moves them); on ANY error none has been touched and the caller still owns all of
 * them.  Their storage stays allocated until the whole schedule has been enqueued.
 * The second and later calls with the same STRUCTURE (tree, legs, dims, payload kinds, path -- payload values are free)
 * run through a compiled plan kept in a small per-context cache (at most 4 plans / a quarter of the device memory,
 * least recently used evicted; TNCB_PLAN_CACHE=0 disables): no schedule construction, tiny pairs batched per level. */
int tncb_contract_tensor_network(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path,
                                 tncb_tensor** out, int* n_out, uint64_t* out_legs);
/* The same in a chosen element type (tncb_contract_tensor_network == dtype TNCB_C128).  tncb_tn is unchanged: host
 * payloads (Matrix, Gate, File) stay complex128 and are narrowed to complex64 while they are written into the pinned
 * staging block (one H2D copy of half the size).  TNCB_DATA_DEVICE leaves must already have `dtype`
 * (TNCB_ERR_INVALID otherwise).  The plan cache keys on the dtype as well. */
int tncb_contract_tensor_network_dt(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, int dtype,
                                    tncb_tensor** out, int* n_out, uint64_t* out_legs);

/* Legs and bond dimensions of the result of tncb_contract_tensor_network(tn, path), from metadata alone (host only, no
 * GPU work; the same validation and the same errors as the real call).  The fan-in needs it: only the raw buffer of a
 * contracted partition travels (tncb_comm_send), so the receiver derives the leg order of what arrives from the sender's
 * partition and local path (the reference ships legs inside the serialised tensor, serialization.rs:43-67).
 * out_legs / out_dims need room for 64 entries; either may be NULL. */
int tncb_network_out_legs(const tncb_tn* tn, const tncb_path* path, int* n_out, uint64_t* out_legs, uint64_t* out_dims);

/* Compile once / execute many: the same circuit with different payloads
 * (e.g. other bitstrings or angles) re-uses the schedule, arena layout and the
 * captured CUDA graph. */
int tncb_plan_create(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, tncb_plan** out);
/* A plan in a chosen element type: execute / stage / run / stage_slices / run_slices then work in that type (the static
 * layout, batch descriptors and workspace limits use its element size; tncb_plan_info reports bytes at it). */
int tncb_plan_create_dt(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, int dtype, tncb_plan** out);
/* `tn` must have the structure the plan was compiled from: every leaf is re-validated (kind, rank,
 * dims, non-null payload, live device handle) -> TNCB_ERR_INVALID / TNCB_ERR_SHAPE /
 * TNCB_ERR_UNCONTRACTED before any copy.  Device leaves: same atomic rule as above.  A plan may be
 * destroyed before or after its context. */
int tncb_plan_execute(tncb_ctx* ctx, tncb_plan* plan, const tncb_tn* tn,
                      tncb_tensor** out, int* n_out, uint64_t* out_legs);
/* Keep the materialised leaves of `tn` on the device (one H2D), then execute the schedule any number of times with no
 * host work besides the kernel launches: the "inputs already resident in HBM" mode.  Not for plans with
 * TNCB_DATA_DEVICE leaves (consumed per call) -> TNCB_ERR_UNSUPPORTED. */
int tncb_plan_stage(tncb_ctx* ctx, tncb_plan* plan, const tncb_tn* tn);
int tncb_plan_run(tncb_ctx* ctx, tncb_plan* plan, tncb_tensor** out, int* n_out, uint64_t* out_legs);
/* Sliced execution (fixing the value of summed legs splits one contraction into independent contractions whose results
 * add up; the reference's declared future work, book/src/future_work.md:9-11): `plan` is compiled for the sliced
 * structure, the leaf payloads of all n_slices slice networks are materialised and uploaded ONCE, then
 * tncb_plan_run_slices contracts slices first, first + stride, ... with no host work per slice and returns their sum
 * (zeros if the range is empty) -- ranks of a multi-GPU job pass (rank, world) and combine with tncb_comm_allreduce_sum. */
int tncb_plan_stage_slices(tncb_ctx* ctx, tncb_plan* plan, size_t n_slices, const tncb_tn* const* slice_tns);
int tncb_plan_run_slices(tncb_ctx* ctx, tncb_plan* plan, size_t first, size_t stride,
                         tncb_tensor** out_sum, int* n_out, uint64_t* out_legs);
/* Schedule facts: #pairs, sum 8MNK, sum s(MK+KN+MN), peak arena bytes, #kernels (s = 16 B per element for complex128,
 * 8 B for complex64 plans). */
int tncb_plan_info(const tncb_plan* plan, uint64_t* n_pairs, double* flops, double* bytes,
                   uint64_t* peak_bytes, uint64_t* n_kernels);
void tncb_plan_destroy(tncb_plan* plan);

/* ---- HDF5 tensor files: replaces tnc::io::hdf5 (tnc/src/io/hdf5.rs), which binds libhdf5 through hdf5-metno.
 *      Neither is available here; csrc/hdf5io.cpp restates the published file format for the subset those calls produce
 *      and read (old- and new-style groups, object headers 1/2, contiguous / compact / chunked data with deflate and
 *      shuffle, Complex = compound of two floats, integer attributes).  Host only, no GPU needed.  Layout (hdf5.rs:1-15):
 *      one group `tensors`, one dataset per tensor (its shape = the bond dimensions), integer attribute `bids` = the
 *      bond ids; the dataset named "-1" carries the network's open bonds in `bids` and no data. ---- */
/* File::open + group(`group`), NULL = "/tensors".  Members are listed in ascending name order (strcmp), the order of
 * Group::member_names (H5Literate by name), so "-1" < "0" < "1" < "10" < "2". */
int tncb_hdf5_open(const char* path, const char* group, tncb_h5file** out);
void tncb_hdf5_close(tncb_h5file* file);
size_t tncb_hdf5_count(const tncb_h5file* file);
const char* tncb_hdf5_name(const tncb_h5file* file, size_t i);      /* NULL when i is out of range */
/* Shape of member i (dims needs room for 32 entries); any of rank / dims / elems may be NULL. */
int tncb_hdf5_shape(const tncb_h5file* file, size_t i, int* rank, uint64_t* dims, uint64_t* elems);
/* Integer attribute (`bids`, `tids`) of member i, widened to int64 (Attribute::read_1d, hdf5.rs:61,70).
 * out == NULL: only *n is set. */
int tncb_hdf5_attr(const tncb_h5file* file, size_t i, const char* name, size_t cap, int64_t* out, size_t* n);
/* read_dyn::<Complex64> (hdf5.rs:71,96): row-major interleaved re/im doubles.  Compounds of two f32 / big-endian floats
 * are converted; a real floating-point dataset is widened with zero imaginary parts (extension). */
int tncb_hdf5_read(const tncb_h5file* file, size_t i, double* out_re_im);
/* TensorData::File((path, adjoint)).into_data() (tensordata.rs:43-49) on the host: load_data(path) = the first member of
 * /tensors, then matrix_adjoint_inplace when adjoint != 0; the result must have exactly rank / dims (-> TNCB_ERR_SHAPE).
 * This is the routine the network executors call for TNCB_DATA_FILE leaves. */
int tncb_hdf5_load_leaf(const char* path, int adjoint, int rank, const uint64_t* dims, double* out_re_im);
/* store_data (hdf5.rs:46-52,105-113): a new file with /tensors/-1 = the tensor. */
int tncb_hdf5_store_data(const char* path, int rank, const uint64_t* dims, const double* data_re_im);
/* A whole network file in the layout read_tensor expects (the reference builds such files only in its tests,
 * hdf5.rs:141-170): n datasets, data_re_im[i] == NULL declares a dataset without data, n_bids[i] < 0 (or n_bids == NULL)
 * omits the attribute. */
int tncb_hdf5_store(const char* path, size_t n, const char* const* names, const int* ranks, const uint64_t* const* dims,
                    const double* const* data_re_im, const int64_t* n_bids, const uint64_t* const* bids);

/* ---- partitioned fan-in: replaces tnc::mpi::communication
 *      (scatter_tensor_network :125-195, intermediate_reduce_tensor_network :199-249).
 *      One process per GPU; boundary tensors move GPU->GPU with ncclSend/ncclRecv
 *      on the ctx stream (no serialisation: legs/dims are derived on every rank). ---- */
/* 128-byte NCCL unique id; create on rank 0, broadcast out of band. */
int tncb_comm_unique_id(uint8_t id_out[128]);
int tncb_comm_init(tncb_ctx* ctx, int world_size, int rank, const uint8_t id[128]);
/* send / recv / allreduce_sum move complex128 tensors only: a complex64 tensor -> TNCB_ERR_UNSUPPORTED. */
int tncb_comm_send(tncb_ctx* ctx, const tncb_tensor* t, int peer);
int tncb_comm_recv(tncb_ctx* ctx, int rank_dims, const uint64_t* dims, int peer, tncb_tensor** out);
/* In-place sum over all ranks (ncclAllReduce on the ctx stream): combines sliced contractions. */
int tncb_comm_allreduce_sum(tncb_ctx* ctx, tncb_tensor* t);
int tncb_comm_destroy(tncb_ctx* ctx);
/* get_tensor_mapping (mpi/communication.rs:89-115): partition -> rank, the
 * partition on the left of the last top-level pair goes to rank 0, the others
 * to 1, 2, ... in the order the reference walks `path.nested.keys()`: the
 * iteration order of FxHashMap<usize,_>::from_iter(partition_index) (rustc-hash
 * 2.1.1 on hashbrown), reproduced bit-exactly and pinned by the reference KAT
 * communication.rs:257-279 (0 -> 0, 1 -> 2, 2 -> 1).  rank_of[p] for p < n_partitions. */
int tncb_fanin_mapping(size_t n_partitions, const uint64_t* partition_index,
                       size_t n_pairs, const uint64_t* toplevel_pairs, int world_size,
                       int* rank_of_partition);

/* ---- planning aids (host only, no GPU work) ---------------------------------------------------------------
 * Subtree reconfiguration of a contraction tree -- what the reference gets from cotengra via rustengra
 * (tnc/src/contractionpath/paths/tree_reconfiguration.rs:54-58).  Legs are relabelled by the caller to bit positions
 * 0 .. 64*n_words-1; leaf_legs holds n_leaves bitsets of n_words words; leg_log2[l] = log2(dim of leg l); a leg joins at
 * most two leaves (the reference's tensor model).  ssa_pairs (n_leaves-1 pairs, SSA ids) is refined in place:
 * pieces of the tree with at most subtree_size (2..15) frontier nodes are re-ordered optimally (subset DP) while that lowers
 *   sum over pair steps of  prod dims(legs(a) | legs(b)) + size_weight * prod dims(legs(a) ^ legs(b)),
 * for at most max_sweeps sweeps.  With time_model != NULL (8 doubles: int8-engine flop/s, its K half-rate constant, FP64
 * flop/s, HBM byte/s, seconds per launch, the FP64 kernels' K half-rate constant, the int8 engine's largest K, its operand
 * conversion bytes per element -- contraction_cost.GPU_RATES) the objective is the modelled device time
 *   sum over pair steps of  max(8 mnk / rate(m, n, k), 16 (mk + nk + mn) / hbm) + launch       (gpu_time_mnk)
 * instead.  flops = sum of prod dims(legs(a) | legs(b)), max_size = the largest tensor, objective = the minimised sum. */
int tncb_path_reconfigure(int n_leaves, int n_words, const uint64_t* leaf_legs, const double* leg_log2, int32_t* ssa_pairs,
                          int subtree_size, int max_sweeps, double size_weight, const double* time_model, uint64_t seed,
                          double* flops, double* max_size, double* objective);
/* Slicing scores of a tree, per leg l (arrays of 64*n_words): cost_without[l] = the objective of ONE slice once l is fixed,
 * size_without[l] = the largest tensor then; cost / max_size = the unsliced tree's. */
int tncb_path_leg_scores(int n_leaves, int n_words, const uint64_t* leaf_legs, const double* leg_log2, const int32_t* ssa_pairs,
                         double size_weight, const double* time_model,
                         double* cost_without, double* size_without, double* cost, double* max_size);

#ifdef __cplusplus
}
#endif
#endif /* TNCB_H */

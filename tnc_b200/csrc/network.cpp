// contract_tensor_network on the device: replaces tnc/src/tensornetwork/contraction.rs:30-88.
//
// The reference walks the path sequentially and, per pair, materialises the payloads
// (tensordata.rs:40-59), allocates a result and calls tetra::contract.  Here the (nested)
// path is first compiled from metadata alone into a flat schedule of pair plans (leg algebra
// of tensor.rs:463-479); execution stages every leaf payload (gate tables, host matrices)
// into pinned memory, ships them in ONE host->device copy and then enqueues all pair kernels
// on the context stream without host round trips.  Arena memory of consumed operands is
// recycled in stream order.
#include "internal.h"
#include <algorithm>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>

namespace tncb {

int gate_matrix(const char* name, const double* ang, int n_ang, bool adjoint, std::complex<double>* out);

struct SlotMeta {
  std::vector<uint64_t> legs, dims;
  uint64_t elems = 1;
  int leaf_index = -1;      // >= 0: payload comes from the leaf block / a device handle
};

struct Step { int a, b, out; PairPlan plan; };

struct Schedule {
  std::vector<SlotMeta> slots;
  std::vector<size_t> leaf_offset; // element offset of leaf i in the leaf block
  std::vector<int> leaf_kind;
  size_t leaf_block_elems = 0;
  std::vector<Step> steps;
  int result_slot = -1;
  double flops = 0, bytes = 0;      // bytes at 16 B per element (PairPlan::bytes); scaled by esz() / 16 where reported
  size_t n_leaves_total = 0;
  int dtype = TNCB_C128;            // element type of every device tensor of the run (host payloads stay complex128)
  size_t esz() const { return dtype_size(dtype); }
};

static const tncb_path* find_nested(const tncb_path* path, size_t idx) {
  if (!path) return nullptr;
  for (size_t q = 0; q < path->n_nested; q++)
    if (path->nested_index[q] == idx) return &path->nested[q];
  return nullptr;
}

static size_t count_leaves(const tncb_tn* tn) {
  if (tn->n_children == 0) return 1;
  size_t c = 0;
  for (size_t i = 0; i < tn->n_children; i++) c += count_leaves(&tn->children[i]);
  return c;
}

static int add_leaf(const tncb_tn* leaf, Schedule& S, size_t leaf_idx, int* slot_out) {
  S.leaf_kind[leaf_idx] = leaf->kind;
  if (leaf->kind == TNCB_DATA_UNCONTRACTED) { *slot_out = -1; return TNCB_OK; }
  if (leaf->rank < 0 || leaf->rank > kMaxLegs) return fail(TNCB_ERR_INVALID, "leaf rank out of range");
  SlotMeta m;
  m.legs.assign(leaf->legs, leaf->legs + leaf->rank);
  m.dims.assign(leaf->dims, leaf->dims + leaf->rank);
  for (int i = 0; i < leaf->rank; i++) m.elems *= leaf->dims[i];
  m.leaf_index = (int)leaf_idx;
  if (leaf->kind == TNCB_DATA_GATE) {
    if (!leaf->gate_name) return fail(TNCB_ERR_GATE, "gate leaf without a name");
    std::complex<double> tmp[16];
    int cnt = gate_matrix(leaf->gate_name, leaf->gate_angles, leaf->n_gate_angles, leaf->gate_adjoint != 0, tmp);
    if (cnt < 0) return cnt;
    if ((uint64_t)cnt != m.elems) return fail(TNCB_ERR_SHAPE, std::string("gate '") + leaf->gate_name + "' does not match the leaf's bond dimensions");
  } else if (leaf->kind == TNCB_DATA_MATRIX) {
    if (!leaf->host_re_im) return fail(TNCB_ERR_INVALID, "matrix leaf without host data");
  } else if (leaf->kind == TNCB_DATA_DEVICE) {
    if (!leaf->device) return fail(TNCB_ERR_INVALID, "device leaf without a tensor handle");
    if (leaf->device->dtype != S.dtype) return fail(TNCB_ERR_INVALID, "device leaf: dtype differs from the network's");
    if (leaf->device->elems != m.elems) return fail(TNCB_ERR_SHAPE, "device leaf: element count mismatch");
  } else if (leaf->kind == TNCB_DATA_FILE) {
    if (!leaf->file_path) return fail(TNCB_ERR_INVALID, "file leaf without a path");
  } else {
    return fail(TNCB_ERR_INVALID, "unknown TensorData kind " + std::to_string(leaf->kind));
  }
  if (leaf->kind != TNCB_DATA_DEVICE) {
    S.leaf_offset[leaf_idx] = S.leaf_block_elems;
    S.leaf_block_elems += std::max<uint64_t>(m.elems, 1);
  }
  S.slots.push_back(std::move(m));
  *slot_out = (int)S.slots.size() - 1;
  return TNCB_OK;
}

// Returns the slot id that holds the contraction result of `tn` (-1: nothing / empty tensor).
static int build(const tncb_tn* tn, const tncb_path* path, Schedule& S, size_t& leaf_counter, int* result) {
  if (tn->n_children == 0) { // a leaf handed to contract_tensor_network: only an empty path is legal
    if (path && (path->n_pairs || path->n_nested)) return fail(TNCB_ERR_INVALID, "path given for a leaf tensor");
    return add_leaf(tn, S, leaf_counter++, result);
  }
  const size_t nc = tn->n_children;
  std::vector<int> slot(nc, -1);
  std::vector<char> uncontracted_composite(nc, 0);
  if (path) for (size_t q = 0; q < path->n_nested; q++)
    if (path->nested_index[q] >= nc) return fail(TNCB_ERR_INVALID, "nested path index out of range");
  // nested paths first (contraction.rs:34-38); ascending child order
  for (size_t i = 0; i < nc; i++) {
    const tncb_tn* c = &tn->children[i];
    const tncb_path* np = find_nested(path, i);
    int rc;
    if (c->n_children == 0) {
      if (np && (np->n_pairs || np->n_nested)) return fail(TNCB_ERR_INVALID, "nested path given for a leaf child");
      if ((rc = add_leaf(c, S, leaf_counter++, &slot[i]))) return rc;
    } else if (np) {
      if ((rc = build(c, np, S, leaf_counter, &slot[i]))) return rc;
    } else {
      uncontracted_composite[i] = 1; // stays TensorData::Uncontracted
      size_t n = count_leaves(c);
      for (size_t q = 0; q < n; q++) S.leaf_kind[leaf_counter + q] = TNCB_DATA_UNCONTRACTED;
      leaf_counter += n;
    }
  }
  const size_t np_ = path ? path->n_pairs : 0;
  for (size_t q = 0; q < np_; q++) {
    const uint64_t i = path->pairs[2 * q], j = path->pairs[2 * q + 1];
    if (i >= nc || j >= nc) return fail(TNCB_ERR_INVALID, "pair (" + std::to_string(i) + "," + std::to_string(j) + ") indexes past the tensor list");
    if (i == j || slot[i] < 0 || slot[j] < 0)
      return fail(TNCB_ERR_UNCONTRACTED, "pair (" + std::to_string(i) + "," + std::to_string(j) + "): Cannot convert uncontracted tensor to data");
    const SlotMeta& a = S.slots[slot[i]];
    const SlotMeta& b = S.slots[slot[j]];
    Step st; st.a = slot[i]; st.b = slot[j];
    int rc = plan_pair((int)a.legs.size(), a.legs.data(), a.dims.data(), (int)b.legs.size(), b.legs.data(), b.dims.data(), st.plan);
    if (rc) return rc;
    SlotMeta o; o.legs = st.plan.out_legs; o.dims = st.plan.out_dims;
    for (uint64_t d : o.dims) o.elems *= d;
    S.slots.push_back(std::move(o));
    st.out = (int)S.slots.size() - 1;
    S.flops += st.plan.flops(); S.bytes += st.plan.bytes();
    S.steps.push_back(std::move(st));
    slot[i] = S.steps.back().out; slot[j] = -1; uncontracted_composite[j] = 0;
  }
  // retain(non-empty leaf or composite); at most one may remain (contraction.rs:48-51)
  int remaining = 0, last = -1;
  for (size_t i = 0; i < nc; i++) {
    if (slot[i] >= 0) { remaining++; last = slot[i]; }
    else if (uncontracted_composite[i]) { remaining++; last = -2; }
  }
  if (remaining > 1 || last == -2) return fail(TNCB_ERR_NOT_CONTRACTED, "Not fully contracted");
  *result = last;
  return TNCB_OK;
}

static int build_schedule(const tncb_tn* tn, const tncb_path* path, Schedule& S, int dtype = TNCB_C128) {
  if (!tn) return fail(TNCB_ERR_INVALID, "tn is null");
  if (!dtype_size(dtype)) return fail(TNCB_ERR_INVALID, "dtype must be TNCB_C128 or TNCB_C64");
  S.dtype = dtype;
  S.n_leaves_total = count_leaves(tn);
  S.leaf_offset.assign(S.n_leaves_total, 0);
  S.leaf_kind.assign(S.n_leaves_total, TNCB_DATA_UNCONTRACTED);
  size_t counter = 0;
  return build(tn, path, S, counter, &S.result_slot);
}

static void collect_leaf_nodes(const tncb_tn* tn, std::vector<const tncb_tn*>& v) {
  if (tn->n_children == 0) { v.push_back(tn); return; }
  for (size_t i = 0; i < tn->n_children; i++) collect_leaf_nodes(&tn->children[i], v);
}

// A schedule may be executed on a network other than the one it was compiled from (tncb_plan_execute):
// every leaf must still have the kind, rank, dims and a payload that the plan's offsets were sized for.
static int validate_leaves(const Schedule& S, const std::vector<const tncb_tn*>& leaves) {
  if (leaves.size() != S.n_leaves_total) return fail(TNCB_ERR_INVALID, "network does not match the plan (leaf count)");
  std::vector<const SlotMeta*> meta(leaves.size(), nullptr);
  for (const SlotMeta& m : S.slots) if (m.leaf_index >= 0) meta[m.leaf_index] = &m;
  for (size_t li = 0; li < leaves.size(); li++) {
    const tncb_tn* lf = leaves[li];
    if (S.leaf_kind[li] != lf->kind) return fail(TNCB_ERR_INVALID, "network payload kinds do not match the plan (leaf " + std::to_string(li) + ")");
    if (lf->kind == TNCB_DATA_UNCONTRACTED) continue;
    const SlotMeta* m = meta[li];
    if (!m) return fail(TNCB_ERR_INVALID, "plan has no slot for leaf " + std::to_string(li));
    if (lf->rank != (int)m->dims.size() || (lf->rank > 0 && !lf->dims))
      return fail(TNCB_ERR_SHAPE, "leaf " + std::to_string(li) + ": rank differs from the plan");
    for (int i = 0; i < lf->rank; i++)
      if (lf->dims[i] != m->dims[i]) return fail(TNCB_ERR_SHAPE, "leaf " + std::to_string(li) + ": bond dimensions differ from the plan");
    if (lf->kind == TNCB_DATA_MATRIX && !lf->host_re_im) return fail(TNCB_ERR_INVALID, "matrix leaf " + std::to_string(li) + " without host data");
    if (lf->kind == TNCB_DATA_GATE && !lf->gate_name) return fail(TNCB_ERR_GATE, "gate leaf " + std::to_string(li) + " without a name");
    if (lf->kind == TNCB_DATA_FILE && !lf->file_path) return fail(TNCB_ERR_INVALID, "file leaf " + std::to_string(li) + " without a path");
    if (lf->kind == TNCB_DATA_DEVICE) {
      if (!lf->device || !lf->device->ptr) return fail(TNCB_ERR_UNCONTRACTED, "device leaf " + std::to_string(li) + " without a tensor handle (already consumed?)");
      if (lf->device->dtype != S.dtype) return fail(TNCB_ERR_INVALID, "device leaf " + std::to_string(li) + ": dtype differs from the plan's");
      if (lf->device->elems != m->elems) return fail(TNCB_ERR_SHAPE, "device leaf " + std::to_string(li) + ": element count mismatch");
    }
  }
  for (size_t x = 0; x < leaves.size(); x++)       // the same device handle twice would be freed twice
    if (leaves[x]->kind == TNCB_DATA_DEVICE)
      for (size_t y = x + 1; y < leaves.size(); y++)
        if (leaves[y]->kind == TNCB_DATA_DEVICE && leaves[y]->device == leaves[x]->device)
          return fail(TNCB_ERR_INVALID, "the same device tensor is passed as two leaves");
  return TNCB_OK;
}

static int stage_leaves(const Schedule& S, const std::vector<const tncb_tn*>& leaves, void* stage);

// `resident` != nullptr: the leaf block already sits on the device (tncb_plan_stage); `tn` may then be null.
static int execute(tncb_ctx* ctx, const Schedule& S, const tncb_tn* tn, tncb_tensor** out, int* n_out, uint64_t* out_legs,
                   const void* resident = nullptr) {
  const size_t esz = S.esz();
  TNCB_CUDA(cudaSetDevice(ctx->device));
  std::vector<const tncb_tn*> leaves;
  if (tn) collect_leaf_nodes(tn, leaves);
  if (!resident) { int vrc = validate_leaves(S, leaves); if (vrc) return vrc; }
  // ---- stage all host payloads, one H2D copy ----
  const size_t block_bytes = resident ? 0 : S.leaf_block_elems * esz;
  void* leaf_block = nullptr;
  if (block_bytes) {
    if (ctx->stage_bytes < block_bytes) {
      if (ctx->stage_host) { TNCB_CUDA(cudaStreamSynchronize(ctx->stream)); cudaFreeHost(ctx->stage_host); ctx->stage_host = nullptr; }
      size_t want = std::max(block_bytes, (size_t)1 << 20);
      TNCB_CUDA(cudaMallocHost(&ctx->stage_host, want));
      ctx->stage_bytes = want;
    } else {
      // the previous network's upload may still be reading the staging buffer
      TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    { int src = stage_leaves(S, leaves, ctx->stage_host); if (src) return src; }
    int rc = ctx->arena.alloc(block_bytes, &leaf_block);
    if (rc) return rc;
    TNCB_CUDA(cudaMemcpyAsync(leaf_block, ctx->stage_host, block_bytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  // ---- run the schedule ----
  struct Live { char* ptr = nullptr; size_t bytes = 0; tncb_tensor* handle = nullptr; };
  std::vector<Live> live(S.slots.size());
  for (size_t s = 0; s < S.slots.size(); s++) {
    const int li = S.slots[s].leaf_index;
    if (li < 0) continue;
    if (S.leaf_kind[li] == TNCB_DATA_DEVICE) { live[s].ptr = (char*)leaves[li]->device->ptr; live[s].handle = leaves[li]->device; }
    else live[s].ptr = (resident ? (char*)const_cast<void*>(resident) : (char*)leaf_block) + S.leaf_offset[li] * esz;
  }
  int rc = TNCB_OK;
  std::vector<tncb_tensor*> consumed;
  // TNCB_TRACE=1: per-step device times on stderr (tuning aid; adds two events per pair)
  const bool trace = std::getenv("TNCB_TRACE") != nullptr;
  std::vector<cudaEvent_t> tev;
  if (trace) { tev.resize(S.steps.size() + 1); for (auto& e : tev) cudaEventCreate(&e); cudaEventRecord(tev[0], ctx->stream); }
  size_t step_no = 0;
  for (const Step& st : S.steps) {
    const SlotMeta& om = S.slots[st.out];
    size_t bytes = std::max<size_t>(om.elems * esz, 16);
    void* p = nullptr;
    if ((rc = ctx->arena.alloc(bytes, &p))) break;
    live[st.out].ptr = (char*)p; live[st.out].bytes = bytes;
    if ((rc = launch_pair(ctx, st.plan, live[st.a].ptr, live[st.b].ptr, live[st.out].ptr, S.dtype))) break;
    for (int s : {st.a, st.b}) { // operands are consumed (mem::take, contraction.rs:61-62)
      // caller-owned device leaves are released only after the WHOLE schedule was enqueued (atomic consumption:
      // on any error every device input is still alive and owned by the caller, see tncb.h)
      if (live[s].handle) consumed.push_back(live[s].handle);
      else if (live[s].bytes) ctx->arena.free(live[s].ptr, live[s].bytes);
      live[s].ptr = nullptr; live[s].bytes = 0; live[s].handle = nullptr;
    }
    if (trace) cudaEventRecord(tev[++step_no], ctx->stream);
  }
  if (trace) {
    cudaStreamSynchronize(ctx->stream);
    for (size_t q = 0; q < step_no; q++) {
      float ms = 0; cudaEventElapsedTime(&ms, tev[q], tev[q + 1]);
      const PairPlan& P = S.steps[q].plan;
      fprintf(stderr, "TNCB_TRACE step %zu class K%d M %lld N %lld K %lld groups m%d n%d k%d akf %d bkf %d ms %.4f tflops %.2f gbs %.1f\n",
              q, P.kernel_class, P.M, P.N, P.K, P.m.n, P.n.n, P.k.n, (int)P.a_kfast, (int)P.b_kfast, ms,
              P.flops() / (ms * 1e-3) * 1e-12, P.bytes() * (double)esz / 16.0 / (ms * 1e-3) * 1e-9);
    }
    for (auto& e : tev) cudaEventDestroy(e);
  }
  tncb_tensor* result = nullptr;
  if (!rc && S.result_slot >= 0) {
    const SlotMeta& rm = S.slots[S.result_slot];
    Live& rl = live[S.result_slot];
    result = new tncb_tensor();
    result->rank = (int)rm.dims.size(); result->elems = rm.elems; result->dtype = S.dtype;
    for (size_t i = 0; i < rm.dims.size(); i++) result->dims[i] = rm.dims[i];
    if (rl.bytes) { // produced by a pair: hand the arena block over
      result->ptr = (double2*)rl.ptr; result->bytes = rl.bytes; rl.bytes = 0;
    } else if (rl.handle) { // a device leaf that was never contracted: the result takes its storage over
      *result = *rl.handle; rl.handle->ptr = nullptr; rl.handle->bytes = 0; consumed.push_back(rl.handle); rl.handle = nullptr;
    } else { // an uploaded leaf that was never contracted: copy it out of the leaf block
      result->bytes = std::max<size_t>(rm.elems * esz, 16);
      void* p = nullptr;
      rc = ctx->arena.alloc(result->bytes, &p);
      if (!rc) {
        result->ptr = (double2*)p;
        cudaMemcpyAsync(p, rl.ptr, rm.elems * esz, cudaMemcpyDeviceToDevice, ctx->stream);
      } else { delete result; result = nullptr; }
    }
  }
  // anything still live was not consumed because of an error
  for (size_t s = 0; s < live.size(); s++)
    if (live[s].bytes) ctx->arena.free(live[s].ptr, live[s].bytes);
  if (leaf_block) ctx->arena.free(leaf_block, block_bytes);
  if (rc) return rc;                                 // nothing in `consumed` was touched
  for (tncb_tensor* h : consumed) tncb_tensor_free(ctx, h);
  if (out) *out = result; else if (result) tncb_tensor_free(ctx, result);
  if (n_out) *n_out = S.result_slot >= 0 ? (int)S.slots[S.result_slot].legs.size() : 0;
  if (out_legs && S.result_slot >= 0)
    for (size_t i = 0; i < S.slots[S.result_slot].legs.size(); i++) out_legs[i] = S.slots[S.result_slot].legs[i];
  return TNCB_OK;
}

} // namespace tncb

// Compile once / execute many.  A plan gets a STATIC memory layout (every slot at a fixed offset of one workspace,
// blocks recycled level by level) unless it has caller-owned device leaves.  Its steps are re-ordered by the level of
// the contraction tree; all independent tiny (K0) pairs of a level run as ONE batched launch (k0_batch_kernel), the
// other pairs one by one.  Plans without K1 steps (the launch-bound regime) are additionally captured into a CUDA
// graph (H2D of the staged leaves + every kernel) and replayed.
struct tncb_plan {
  tncb::Schedule S;
  bool is_static = false;            // static layout + level batches available
  bool graphable = false;
  std::vector<size_t> slot_off;      // byte offset of every slot in the workspace
  size_t ws_bytes = 0, scratch_off = 0, scratch_elems = 0, leaf_off = 0;
  // level structure: steps [level_begin[l], level_begin[l+1]) of S.steps form level l; the batched ones come first
  std::vector<int> level_begin, level_batched;
  std::vector<tncb::K0BatchItem> items;            // batched steps of all levels, level by level
  std::vector<int> block_start;                    // per level: n_batched + 1 prefix entries
  std::vector<size_t> item_first, bs_first;        // per level: first index into items / block_start
  void* batch_dev = nullptr; size_t batch_bytes = 0;   // device copy of items + block_start
  tncb_ctx* ctx = nullptr;           // device state is tied to this context (stream, device)
  void* ws = nullptr;                // arena block
  void* stage = nullptr;             // plan-owned pinned staging of the leaf block
  cudaEvent_t stage_ev = nullptr;    // recorded after the last eager upload out of `stage` (re-staging waits for it)
  bool stage_busy = false;
  bool leaves_resident = false;      // tncb_plan_stage put the leaf block into ws
  cudaGraphExec_t exec[2] = {nullptr, nullptr};    // [0]: with the H2D of the staged leaves, [1]: leaves resident
  uint64_t kernels_per_run = 0;
  void* resident = nullptr;          // non-static plans: device copy of the leaf block (tncb_plan_stage)
  size_t resident_bytes = 0;
  void* slices_dev = nullptr;        // tncb_plan_stage_slices: n_slices leaf blocks, back to back
  size_t n_slices = 0, slices_bytes = 0;
};

namespace tncb {

// first-fit offset allocator with coalescing (same policy as the arena) for the static layout
struct OffsetAlloc {
  std::map<size_t, size_t> free_by_off; size_t top = 0;
  static size_t up(size_t b) { return (std::max<size_t>(b, 256) + 255) / 256 * 256; }
  size_t alloc(size_t bytes) {
    bytes = up(bytes);
    for (auto it = free_by_off.begin(); it != free_by_off.end(); ++it)
      if (it->second >= bytes) {
        size_t off = it->first, sz = it->second;
        free_by_off.erase(it);
        if (sz > bytes) free_by_off[off + bytes] = sz - bytes;
        return off;
      }
    size_t off = top; top += bytes; return off;
  }
  void free(size_t off, size_t bytes) {
    bytes = up(bytes);
    auto it = free_by_off.emplace(off, bytes).first;
    auto nx = std::next(it);
    if (nx != free_by_off.end() && it->first + it->second == nx->first) { it->second += nx->second; free_by_off.erase(nx); }
    if (it != free_by_off.begin()) { auto pv = std::prev(it); if (pv->first + pv->second == it->first) { pv->second += it->second; free_by_off.erase(it); } }
  }
};

static void plan_static_layout(tncb_plan* P, int sm_count, size_t device_bytes) {
  Schedule& S = P->S;
  P->is_static = !S.steps.empty() && std::getenv("TNCB_NO_STATIC") == nullptr;
  for (int k : S.leaf_kind) if (k == TNCB_DATA_DEVICE) P->is_static = false;   // addresses change per call
  if (!P->is_static) return;
  // ---- levels: a step's level is 1 + the deepest level among its operands' producers (leaves: 0) ----
  std::vector<int> slot_level(S.slots.size(), 0), step_level(S.steps.size(), 0);
  int n_levels = 0;
  for (size_t q = 0; q < S.steps.size(); q++) {
    const Step& st = S.steps[q];
    step_level[q] = std::max(slot_level[st.a], slot_level[st.b]) + 1;
    slot_level[st.out] = step_level[q];
    n_levels = std::max(n_levels, step_level[q]);
  }
  static const bool no_batch = std::getenv("TNCB_NO_BATCH") != nullptr;
  std::vector<size_t> order(S.steps.size());
  for (size_t q = 0; q < order.size(); q++) order[q] = q;
  std::vector<char> batchable(S.steps.size(), 0);
  for (size_t q = 0; q < S.steps.size(); q++) batchable[q] = !no_batch && k0_batch_eligible(sm_count, S.steps[q].plan);
  std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) {
    if (step_level[x] != step_level[y]) return step_level[x] < step_level[y];
    return batchable[x] > batchable[y];                  // batched pairs first inside a level
  });
  std::vector<Step> sorted; sorted.reserve(S.steps.size());
  std::vector<int> lv; std::vector<char> bt;
  for (size_t q : order) { sorted.push_back(std::move(S.steps[q])); lv.push_back(step_level[q]); bt.push_back(batchable[q]); }
  S.steps.swap(sorted);
  // steps [level_begin[l], level_begin[l+1]) form level l (0-based); step_level counts from 1
  P->level_begin.assign(n_levels + 1, 0); P->level_batched.assign(n_levels, 0);
  for (size_t q = 0; q < S.steps.size(); q++) { P->level_begin[lv[q]]++; if (bt[q]) P->level_batched[lv[q] - 1]++; }
  for (int l = 1; l <= n_levels; l++) P->level_begin[l] += P->level_begin[l - 1];
  for (int l = 0; l < n_levels; l++) if (P->level_batched[l] < 2) P->level_batched[l] = 0;   // a batch of one is just a launch
  // ---- layout: outputs of a level are allocated before any operand of that level is released ----
  size_t scratch = 0;
  for (const Step& st : S.steps) if (st.plan.kernel_class == 0) scratch = std::max(scratch, k0_partial_elems(sm_count, st.plan));
  OffsetAlloc A;
  const size_t esz = S.esz();
  P->leaf_off = A.alloc(std::max<size_t>(S.leaf_block_elems * esz, 16));
  P->scratch_elems = scratch;
  P->scratch_off = scratch ? A.alloc(scratch * sizeof(double2)) : 0;   // split-K partials are f64 for both dtypes
  P->slot_off.assign(S.slots.size(), 0);
  std::vector<size_t> sz(S.slots.size(), 0);
  for (size_t s2 = 0; s2 < S.slots.size(); s2++)
    if (S.slots[s2].leaf_index >= 0) P->slot_off[s2] = P->leaf_off + S.leaf_offset[S.slots[s2].leaf_index] * esz;
  for (int l = 0; l < n_levels; l++) {
    for (int q = P->level_begin[l]; q < P->level_begin[l + 1]; q++) {
      const Step& st = S.steps[q];
      sz[st.out] = std::max<size_t>(S.slots[st.out].elems * esz, 16);
      P->slot_off[st.out] = A.alloc(sz[st.out]);
    }
    for (int q = P->level_begin[l]; q < P->level_begin[l + 1]; q++) {
      const Step& st = S.steps[q];
      for (int s2 : {st.a, st.b}) if (sz[s2]) { A.free(P->slot_off[s2], sz[s2]); sz[s2] = 0; }
    }
  }
  P->ws_bytes = A.top;
  // one workspace for all intermediates of a run: at most 64 GiB or 0.62 of the device (B200: ~110 GiB; leaves room for the
  // int8 engine's 12 GiB of planes and the staged leaves), whichever is larger; TNCB_PLAN_WS_GB overrides
  size_t limit = std::max((size_t)64 << 30, (size_t)(0.62 * (double)device_bytes));
  if (const char* e = std::getenv("TNCB_PLAN_WS_GB")) limit = (size_t)std::max(1, atoi(e)) << 30;
  if (P->ws_bytes > limit) { P->is_static = false; return; }
  // ---- batch descriptors ----
  P->item_first.assign(n_levels, 0); P->bs_first.assign(n_levels, 0);
  for (int l = 0; l < n_levels; l++) {
    P->item_first[l] = P->items.size(); P->bs_first[l] = P->block_start.size();
    const int nb = P->level_batched[l];
    if (!nb) continue;
    int blocks = 0;
    for (int q = P->level_begin[l]; q < P->level_begin[l] + nb; q++) {
      const Step& st = S.steps[q];
      K0BatchItem it{};
      const int nblk = k0_batch_fill(sm_count, st.plan, &it);
      it.offA = (long long)P->slot_off[st.a]; it.offB = (long long)P->slot_off[st.b]; it.offC = (long long)P->slot_off[st.out];
      P->items.push_back(it);
      P->block_start.push_back(blocks);
      blocks += nblk;
    }
    P->block_start.push_back(blocks);
  }
  P->graphable = std::getenv("TNCB_NO_GRAPH") == nullptr && P->ws_bytes <= ((size_t)1 << 30);   // graphs are for small networks
  for (const Step& st : S.steps) if (st.plan.kernel_class == 1) { P->graphable = false; break; }   // K1/K1' use ctx-owned tables / arena scratch
}

// Host payloads are complex128; a complex64 run narrows them (one rounding per part) as they go into the staging block.
static int stage_leaves(const Schedule& S, const std::vector<const tncb_tn*>& leaves, void* stage_v) {
  const bool c64 = S.dtype == TNCB_C64;
  std::complex<double>* stage = (std::complex<double>*)stage_v;
  std::vector<std::complex<double>> wide;   // complex64 runs: gate / file payloads before narrowing
  for (size_t li = 0; li < leaves.size(); li++) {
    const tncb_tn* lf = leaves[li];
    if (S.leaf_kind[li] != lf->kind) return fail(TNCB_ERR_INVALID, "network payload kinds do not match the plan");
    if (lf->kind != TNCB_DATA_GATE && lf->kind != TNCB_DATA_MATRIX && lf->kind != TNCB_DATA_FILE) continue;
    uint64_t e = 1; for (int i = 0; i < lf->rank; i++) e *= lf->dims[i];
    const double* src = nullptr;
    if (c64 && lf->kind != TNCB_DATA_MATRIX) wide.resize(std::max<uint64_t>(e, 16));
    std::complex<double>* dst = c64 ? wide.data() : stage + S.leaf_offset[li];
    if (lf->kind == TNCB_DATA_GATE) {
      int cnt = gate_matrix(lf->gate_name, lf->gate_angles, lf->n_gate_angles, lf->gate_adjoint != 0, dst);
      if (cnt < 0) return cnt;
      e = (uint64_t)cnt;
      src = (const double*)dst;
    } else if (lf->kind == TNCB_DATA_MATRIX) {
      if (!c64) std::memcpy(stage + S.leaf_offset[li], lf->host_re_im, e * sizeof(double2));
      src = lf->host_re_im;
    } else {      // into_data for TensorData::File (tensordata.rs:43-49)
      int rc = h5::load_file_leaf(lf->file_path, lf->file_adjoint != 0, lf->rank, lf->dims, (double*)dst);
      if (rc) return rc;
      src = (const double*)dst;
    }
    if (c64) {
      float* d = (float*)stage_v + 2 * S.leaf_offset[li];
      for (uint64_t i = 0; i < 2 * e; i++) d[i] = (float)src[i];
    }
  }
  return TNCB_OK;
}

// workspace, pinned staging and the device copy of the batch descriptors (once per plan and context)
static int plan_device_state(tncb_ctx* ctx, tncb_plan* P) {
  if (P->ctx && P->ctx != ctx) return fail(TNCB_ERR_INVALID, "plan belongs to another context");
  if (!P->ctx) { P->ctx = ctx; ctx->plans.push_back(P); }
  int rc;
  if (!P->ws && (rc = ctx->arena.alloc(P->ws_bytes, &P->ws))) return rc;
  const size_t block_bytes = std::max<size_t>(P->S.leaf_block_elems * P->S.esz(), 16);
  if (!P->stage) TNCB_CUDA(cudaMallocHost(&P->stage, block_bytes));
  if (!P->batch_dev && !P->items.empty()) {
    const size_t ib = P->items.size() * sizeof(K0BatchItem), bb = P->block_start.size() * sizeof(int);
    P->batch_bytes = ib + bb;
    if ((rc = ctx->arena.alloc(P->batch_bytes, &P->batch_dev))) return rc;
    TNCB_CUDA(cudaMemcpyAsync(P->batch_dev, P->items.data(), ib, cudaMemcpyHostToDevice, ctx->stream));
    TNCB_CUDA(cudaMemcpyAsync((char*)P->batch_dev + ib, P->block_start.data(), bb, cudaMemcpyHostToDevice, ctx->stream));
    TNCB_CUDA(cudaStreamSynchronize(ctx->stream));   // (pageable sources)
  }
  return TNCB_OK;
}

// every kernel of the plan on the ctx stream, level by level
static int enqueue_static(tncb_ctx* ctx, tncb_plan* P) {
  const Schedule& S = P->S;
  char* ws = (char*)P->ws;
  ctx->partial_override = P->scratch_elems ? (double2*)(ws + P->scratch_off) : nullptr;
  ctx->partial_override_elems = P->scratch_elems;
  int rc = TNCB_OK;
  const K0BatchItem* d_items = (const K0BatchItem*)P->batch_dev;
  const int* d_bs = (const int*)((char*)P->batch_dev + P->items.size() * sizeof(K0BatchItem));
  const int n_levels = (int)P->level_batched.size();
  for (int l = 0; l < n_levels && !rc; l++) {
    const int nb = P->level_batched[l];
    if (nb) {
      const int total_blocks = P->block_start[P->bs_first[l] + nb];
      rc = launch_k0_batch(ctx, d_items + P->item_first[l], d_bs + P->bs_first[l], nb, total_blocks, ws, S.dtype);
    }
    for (int q = P->level_begin[l] + nb; q < P->level_begin[l + 1] && !rc; q++) {
      const Step& st = S.steps[q];
      rc = launch_pair(ctx, st.plan, ws + P->slot_off[st.a], ws + P->slot_off[st.b], ws + P->slot_off[st.out], S.dtype);
    }
  }
  ctx->partial_override = nullptr; ctx->partial_override_elems = 0;
  return rc;
}

// `tn` == nullptr: run on the leaves that tncb_plan_stage left in the workspace
static int execute_static(tncb_ctx* ctx, tncb_plan* P, const tncb_tn* tn, tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  const Schedule& S = P->S;
  TNCB_CUDA(cudaSetDevice(ctx->device));
  int rc;
  std::vector<const tncb_tn*> leaves;
  if (tn) {
    collect_leaf_nodes(tn, leaves);
    if ((rc = validate_leaves(S, leaves))) return rc;
  } else if (!P->leaves_resident) return fail(TNCB_ERR_INVALID, "tncb_plan_stage has not been called on this plan");
  if ((rc = plan_device_state(ctx, P))) return rc;
  const size_t block_bytes = std::max<size_t>(S.leaf_block_elems * S.esz(), 16);
  char* ws = (char*)P->ws;
  const int which = tn ? 0 : 1;
  if (tn) {
    // an earlier upload may still read the staging buffer (it waits behind the previous network's kernels on the stream)
    if (P->exec[0] || P->leaves_resident) TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
    else if (P->stage_busy) TNCB_CUDA(cudaEventSynchronize(P->stage_ev));
    if ((rc = stage_leaves(S, leaves, P->stage))) return rc;
    P->leaves_resident = false;     // the workspace copy is about to be overwritten with this call's payloads
  }
  if (P->graphable) {
    if (!P->exec[which]) {
      cudaGraph_t graph = nullptr;
      const uint64_t launches_before = ctx->launches;
      uint64_t ec_before[8]; for (int i = 0; i < 8; i++) ec_before[i] = ctx->engine_count[i];
      TNCB_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
      if (tn) cudaMemcpyAsync(ws + P->leaf_off, P->stage, block_bytes, cudaMemcpyHostToDevice, ctx->stream);
      rc = enqueue_static(ctx, P);
      cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
      P->kernels_per_run = ctx->launches - launches_before;
      ctx->launches = launches_before;
      for (int i = 0; i < 8; i++) ctx->engine_count[i] = ec_before[i];
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ce != cudaSuccess) { P->graphable = false; return fail(TNCB_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce)); }
      ce = cudaGraphInstantiate(&P->exec[which], graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) {   // the plan runs eagerly from now on
        P->exec[which] = nullptr; P->graphable = false;
        return fail(TNCB_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(ce));
      }
    }
    TNCB_CUDA(cudaGraphLaunch(P->exec[which], ctx->stream));
    ctx->launches += P->kernels_per_run;
    ctx->engine_count[0] += S.steps.size();   // (graphable plans hold K0 / K2 pairs only; counted as tiny pairs)
  } else {
    if (tn) {
      TNCB_CUDA(cudaMemcpyAsync(ws + P->leaf_off, P->stage, block_bytes, cudaMemcpyHostToDevice, ctx->stream));
      if (!P->stage_ev) TNCB_CUDA(cudaEventCreateWithFlags(&P->stage_ev, cudaEventDisableTiming));
      TNCB_CUDA(cudaEventRecord(P->stage_ev, ctx->stream));
      P->stage_busy = true;
    }
    if ((rc = enqueue_static(ctx, P))) return rc;
  }
  tncb_tensor* result = nullptr;
  if (S.result_slot >= 0) {
    const SlotMeta& rm = S.slots[S.result_slot];
    if ((rc = tensor_new(ctx, (int)rm.dims.size(), rm.dims.data(), &result, S.dtype))) return rc;
    TNCB_CUDA(cudaMemcpyAsync(result->ptr, ws + P->slot_off[S.result_slot], rm.elems * S.esz(), cudaMemcpyDeviceToDevice, ctx->stream));
  }
  if (out) *out = result; else if (result) tncb_tensor_free(ctx, result);
  if (n_out) *n_out = S.result_slot >= 0 ? (int)S.slots[S.result_slot].legs.size() : 0;
  if (out_legs && S.result_slot >= 0)
    for (size_t i = 0; i < S.slots[S.result_slot].legs.size(); i++) out_legs[i] = S.slots[S.result_slot].legs[i];
  return TNCB_OK;
}

} // namespace tncb

extern "C" {

// Structure key of a (network, path): everything the schedule depends on (tree shape, legs, dims, payload kinds, pairs)
// and nothing it does not (payload values).  Two calls with equal keys share one compiled plan.
static void key_tn(const tncb_tn* t, std::vector<uint64_t>& k, bool* cacheable) {
  k.push_back(0x7e00000000000000ull | (uint64_t)t->n_children);
  if (t->n_children == 0) {
    k.push_back(((uint64_t)(uint32_t)t->kind << 32) | (uint32_t)t->rank);
    if (t->kind == TNCB_DATA_DEVICE) *cacheable = false;       // consumed per call, addresses differ
    if (t->rank < 0 || t->rank > tncb::kMaxLegs || (t->rank > 0 && (!t->legs || !t->dims))) { *cacheable = false; return; }
    for (int i = 0; i < t->rank; i++) { k.push_back(t->legs[i]); k.push_back(t->dims[i]); }
    return;
  }
  for (size_t i = 0; i < t->n_children; i++) key_tn(&t->children[i], k, cacheable);
}
static void key_path(const tncb_path* p, std::vector<uint64_t>& k) {
  if (!p) { k.push_back(0x7f00000000000000ull); return; }
  k.push_back(0x7d00000000000000ull | (uint64_t)p->n_pairs);
  for (size_t i = 0; i < 2 * p->n_pairs; i++) k.push_back(p->pairs[i]);
  k.push_back(0x7c00000000000000ull | (uint64_t)p->n_nested);
  for (size_t i = 0; i < p->n_nested; i++) { k.push_back(p->nested_index[i]); key_path(&p->nested[i], k); }
}

int tncb_contract_tensor_network(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path,
                                 tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  return tncb_contract_tensor_network_dt(ctx, tn, path, TNCB_C128, out, n_out, out_legs);
}

int tncb_contract_tensor_network_dt(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, int dtype,
                                    tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  if (!ctx || !tn) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  if (!tncb::dtype_size(dtype)) return tncb::fail(TNCB_ERR_INVALID, "dtype must be TNCB_C128 or TNCB_C64");
  // Repeated contractions of the same circuit (other bitstrings, angles, or simply again) hit a small per-context cache
  // of compiled plans: no schedule construction, static layout, batched tiny pairs.  TNCB_PLAN_CACHE=0 disables it.
  static const bool cache_on = !(std::getenv("TNCB_PLAN_CACHE") && atoi(std::getenv("TNCB_PLAN_CACHE")) == 0) && std::getenv("TNCB_TRACE") == nullptr;
  if (cache_on) {
    std::vector<uint64_t> key;
    bool cacheable = true;
    key.push_back(0x7b00000000000000ull | (uint64_t)dtype);
    key_tn(tn, key, &cacheable);
    key_path(path, key);
    if (cacheable) {
      auto& cache = ctx->plan_cache;
      for (size_t i = 0; i < cache.size(); i++)
        if (cache[i].key == key) {
          tncb_ctx::CachedPlan hit = std::move(cache[i]);
          cache.erase(cache.begin() + i);
          cache.push_back(std::move(hit));                       // most recently used last
          tncb_plan* pl = cache.back().plan;
          int rc = tncb::execute_static(ctx, pl, tn, out, n_out, out_legs);
          if (rc != TNCB_ERR_OOM) return rc;
          tncb_plan_destroy(pl); cache.pop_back();               // no room for its workspace any more: pair-by-pair path
          break;
        }
      // a second sighting is what earns a plan: remember the key of a miss, compile on the next call with the same key
      static thread_local std::vector<uint64_t> last_miss;
      if (last_miss == key) {
        tncb_plan* pl = nullptr;
        if (tncb_plan_create_dt(ctx, tn, path, dtype, &pl) == TNCB_OK && pl->is_static) {
          size_t total = 0, free_b = 0, total_b = 0;
          for (auto& c : cache) total += c.plan->ws_bytes;
          cudaMemGetInfo(&free_b, &total_b);
          while (!cache.empty() && (cache.size() >= 4 || total + pl->ws_bytes > total_b / 4)) {   // at most 4 plans / a quarter of the device
            total -= cache.front().plan->ws_bytes;
            tncb_plan_destroy(cache.front().plan); cache.erase(cache.begin());
          }
          if (pl->ws_bytes <= total_b / 4) {
            int rc = tncb::execute_static(ctx, pl, tn, out, n_out, out_legs);
            if (rc == TNCB_OK) { cache.push_back({std::move(key), pl}); last_miss.clear(); return rc; }
            tncb_plan_destroy(pl);
            if (rc != TNCB_ERR_OOM) return rc;
          } else tncb_plan_destroy(pl);
        } else if (pl) tncb_plan_destroy(pl);
      } else last_miss = key;
    }
  }
  tncb::Schedule S;
  int rc = tncb::build_schedule(tn, path, S, dtype);
  if (rc) return rc;
  return tncb::execute(ctx, S, tn, out, n_out, out_legs);
}

int tncb_plan_create(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, tncb_plan** out) {
  return tncb_plan_create_dt(ctx, tn, path, TNCB_C128, out);
}

int tncb_plan_create_dt(tncb_ctx* ctx, const tncb_tn* tn, const tncb_path* path, int dtype, tncb_plan** out) {
  if (!tn || !out) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  tncb_plan* p = new tncb_plan();
  int rc = tncb::build_schedule(tn, path, p->S, dtype);
  if (rc) { delete p; return rc; }
  size_t dev_free = 0, dev_total = 0;
  if (ctx) { cudaSetDevice(ctx->device); if (cudaMemGetInfo(&dev_free, &dev_total) != cudaSuccess) { dev_total = 0; cudaGetLastError(); } }
  tncb::plan_static_layout(p, ctx ? ctx->sm_count : 148, dev_total);
  *out = p;
  return TNCB_OK;
}

int tncb_plan_execute(tncb_ctx* ctx, tncb_plan* plan, const tncb_tn* tn, tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  if (!ctx || !plan || !tn) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  static const bool trace = std::getenv("TNCB_TRACE") != nullptr;   // per-step times come from the pair-by-pair executor
  if (plan->is_static && !trace && (plan->ctx == nullptr || plan->ctx == ctx)) {
    int rc = tncb::execute_static(ctx, plan, tn, out, n_out, out_legs);
    if (rc != TNCB_ERR_OOM || plan->ws) return rc;
    plan->is_static = false;        // no room for the static workspace (it keeps a whole tree level alive): pair-by-pair executor
  }
  return tncb::execute(ctx, plan->S, tn, out, n_out, out_legs);
}

// Materialise the leaves of `tn` once and keep them on the device; tncb_plan_run then executes the schedule without
// any host work besides the kernel launches (the "inputs already resident in HBM" measurement, and the shared leaf
// block of sliced execution).
int tncb_plan_stage(tncb_ctx* ctx, tncb_plan* plan, const tncb_tn* tn) {
  if (!ctx || !plan || !tn) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  const tncb::Schedule& S = plan->S;
  for (int k : S.leaf_kind) if (k == TNCB_DATA_DEVICE) return tncb::fail(TNCB_ERR_UNSUPPORTED, "plans with device leaves cannot be staged (they are consumed per call)");
  if (plan->ctx && plan->ctx != ctx) return tncb::fail(TNCB_ERR_INVALID, "plan belongs to another context");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  std::vector<const tncb_tn*> leaves;
  tncb::collect_leaf_nodes(tn, leaves);
  int rc = tncb::validate_leaves(S, leaves);
  if (rc) return rc;
  const size_t bytes = std::max<size_t>(S.leaf_block_elems * S.esz(), 16);
  std::vector<std::complex<double>> host(std::max<size_t>(S.leaf_block_elems, 1));   // (complex64 plans use the first half)
  if (plan->is_static && (rc = tncb::plan_device_state(ctx, plan))) {
    if (rc != TNCB_ERR_OOM || plan->ws) return rc;
    plan->is_static = false;    // the static workspace does not fit: resident leaf block + pair-by-pair executor
  }
  if (plan->is_static) {      // the leaf block lives inside the plan workspace
    TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
    if ((rc = tncb::stage_leaves(S, leaves, plan->stage))) return rc;
    TNCB_CUDA(cudaMemcpyAsync((char*)plan->ws + plan->leaf_off, plan->stage, bytes, cudaMemcpyHostToDevice, ctx->stream));
    TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
    plan->leaves_resident = true;
    return TNCB_OK;
  }
  if ((rc = tncb::stage_leaves(S, leaves, host.data()))) return rc;
  if (!plan->ctx) { plan->ctx = ctx; ctx->plans.push_back(plan); }
  if (!plan->resident) {
    if ((rc = ctx->arena.alloc(bytes, &plan->resident))) return rc;
    plan->resident_bytes = bytes;
  }
  TNCB_CUDA(cudaMemcpyAsync(plan->resident, host.data(), S.leaf_block_elems * S.esz(), cudaMemcpyHostToDevice, ctx->stream));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));   // `host` dies with this frame
  return TNCB_OK;
}

int tncb_plan_run(tncb_ctx* ctx, tncb_plan* plan, tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  if (!ctx || !plan) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  static const bool trace = std::getenv("TNCB_TRACE") != nullptr;
  if (plan->is_static && plan->leaves_resident && plan->ctx == ctx) {
    if (!trace) return tncb::execute_static(ctx, plan, nullptr, out, n_out, out_legs);
    return tncb::execute(ctx, plan->S, nullptr, out, n_out, out_legs, (char*)plan->ws + plan->leaf_off);
  }
  if (!plan->resident || plan->ctx != ctx) return tncb::fail(TNCB_ERR_INVALID, "tncb_plan_stage has not been called on this context");
  return tncb::execute(ctx, plan->S, nullptr, out, n_out, out_legs, plan->resident);
}

// Sliced execution (the reference's declared future work, book/src/future_work.md:9-11) without host work per slice:
// `plan` is compiled for the SLICED structure; the leaf blocks of all slice networks are materialised and uploaded
// once, then tncb_plan_run_slices walks slices first, first+stride, ... : one device-to-device copy of the slice's leaf
// block (KBs), the plan's kernels (batched / graph as usual), one accumulation kernel.
int tncb_plan_stage_slices(tncb_ctx* ctx, tncb_plan* plan, size_t n_slices, const tncb_tn* const* slice_tns) {
  if (!ctx || !plan || !slice_tns || n_slices == 0) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  if (!plan->is_static) return tncb::fail(TNCB_ERR_UNSUPPORTED, "sliced execution needs a plan with a static layout (no device leaves)");
  const tncb::Schedule& S = plan->S;
  TNCB_CUDA(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = tncb::plan_device_state(ctx, plan))) return rc;
  const size_t block = std::max<size_t>(S.leaf_block_elems, 1) * S.esz();   // bytes per slice
  std::vector<char> host(block * n_slices);
  for (size_t q = 0; q < n_slices; q++) {
    if (!slice_tns[q]) return tncb::fail(TNCB_ERR_INVALID, "slice network is null");
    std::vector<const tncb_tn*> leaves;
    tncb::collect_leaf_nodes(slice_tns[q], leaves);
    if ((rc = tncb::validate_leaves(S, leaves))) return rc;
    if ((rc = tncb::stage_leaves(S, leaves, host.data() + q * block))) return rc;
  }
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (plan->slices_dev) { ctx->arena.free(plan->slices_dev, plan->slices_bytes); plan->slices_dev = nullptr; }
  plan->slices_bytes = host.size();
  if ((rc = ctx->arena.alloc(plan->slices_bytes, &plan->slices_dev))) return rc;
  TNCB_CUDA(cudaMemcpyAsync(plan->slices_dev, host.data(), plan->slices_bytes, cudaMemcpyHostToDevice, ctx->stream));
  TNCB_CUDA(cudaStreamSynchronize(ctx->stream));
  plan->n_slices = n_slices;
  return TNCB_OK;
}

int tncb_plan_run_slices(tncb_ctx* ctx, tncb_plan* plan, size_t first, size_t stride, tncb_tensor** out, int* n_out, uint64_t* out_legs) {
  if (!ctx || !plan || stride == 0) return tncb::fail(TNCB_ERR_INVALID, "bad argument");
  if (!plan->slices_dev || plan->ctx != ctx) return tncb::fail(TNCB_ERR_INVALID, "tncb_plan_stage_slices has not been called on this context");
  const tncb::Schedule& S = plan->S;
  if (S.result_slot < 0) return tncb::fail(TNCB_ERR_INVALID, "plan has no result");
  TNCB_CUDA(cudaSetDevice(ctx->device));
  const tncb::SlotMeta& rm = S.slots[S.result_slot];
  tncb_tensor* sum = nullptr;
  int rc = tncb::tensor_new(ctx, (int)rm.dims.size(), rm.dims.data(), &sum, S.dtype);
  if (rc) return rc;
  const size_t esz = S.esz();
  const size_t block_bytes = std::max<size_t>(S.leaf_block_elems, 1) * esz;
  char* ws = (char*)plan->ws;
  bool any = false;
  for (size_t q = first; q < plan->n_slices; q += stride) {
    TNCB_CUDA(cudaMemcpyAsync(ws + plan->leaf_off, (char*)plan->slices_dev + q * block_bytes, block_bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    plan->leaves_resident = true;
    tncb_tensor* part = nullptr;
    if ((rc = tncb::execute_static(ctx, plan, nullptr, &part, nullptr, nullptr))) { tncb_tensor_free(ctx, sum); return rc; }
    if (!any) {
      TNCB_CUDA(cudaMemcpyAsync(sum->ptr, part->ptr, rm.elems * esz, cudaMemcpyDeviceToDevice, ctx->stream));
      any = true;
    } else if ((rc = tncb::launch_add(ctx, sum->ptr, part->ptr, rm.elems, S.dtype))) { tncb_tensor_free(ctx, part); tncb_tensor_free(ctx, sum); return rc; }
    tncb_tensor_free(ctx, part);
  }
  if (!any) TNCB_CUDA(cudaMemsetAsync(sum->ptr, 0, std::max<size_t>(rm.elems, 1) * esz, ctx->stream));   // more ranks than slices
  if (out) *out = sum; else tncb_tensor_free(ctx, sum);
  if (n_out) *n_out = (int)rm.legs.size();
  if (out_legs) for (size_t i = 0; i < rm.legs.size(); i++) out_legs[i] = rm.legs[i];
  return TNCB_OK;
}

// Legs and bond dimensions of contract_tensor_network(tn, path) from metadata alone (no GPU work): what a receiver of the
// fan-in needs to know about a raw buffer it is about to get (communication.rs:221-226; the reference ships the legs inside
// the serialised tensor instead).
int tncb_network_out_legs(const tncb_tn* tn, const tncb_path* path, int* n_out, uint64_t* out_legs, uint64_t* out_dims) {
  if (!tn || !n_out) return tncb::fail(TNCB_ERR_INVALID, "null argument");
  tncb::Schedule S;
  int rc = tncb::build_schedule(tn, path, S);
  if (rc) return rc;
  if (S.result_slot < 0) { *n_out = 0; return TNCB_OK; }
  const tncb::SlotMeta& m = S.slots[S.result_slot];
  *n_out = (int)m.legs.size();
  for (size_t i = 0; i < m.legs.size(); i++) {
    if (out_legs) out_legs[i] = m.legs[i];
    if (out_dims) out_dims[i] = m.dims[i];
  }
  return TNCB_OK;
}

int tncb_plan_info(const tncb_plan* plan, uint64_t* n_pairs, double* flops, double* bytes, uint64_t* peak_bytes, uint64_t* n_kernels) {
  if (!plan) return tncb::fail(TNCB_ERR_INVALID, "plan is null");
  const tncb::Schedule& S = plan->S;
  if (n_pairs) *n_pairs = S.steps.size();
  const size_t esz = S.esz();
  if (flops) *flops = S.flops;
  if (bytes) *bytes = S.bytes * (double)esz / 16.0;
  if (peak_bytes) { // replay the liveness: leaves + live intermediates
    size_t live = S.leaf_block_elems * esz, peak = live;
    std::vector<size_t> sz(S.slots.size(), 0);
    for (const tncb::Step& st : S.steps) {
      sz[st.out] = std::max<size_t>(S.slots[st.out].elems * esz, 256);
      live += sz[st.out]; peak = std::max(peak, live);
      live -= sz[st.a] + sz[st.b]; sz[st.a] = sz[st.b] = 0;
    }
    *peak_bytes = peak;
  }
  if (n_kernels) {
    uint64_t k = 0;
    for (const tncb::Step& st : S.steps) k += st.plan.kernel_class == 1 ? 2 : 1;  // (K1: table build + GEMM)
    for (int nb : plan->level_batched) if (nb) k -= (uint64_t)(nb - 1);            // a batch is one launch
    *n_kernels = k;
  }
  return TNCB_OK;
}

// Releases everything a plan holds on its context (graph, workspace, staging) and detaches it.  Called by
// tncb_plan_destroy and by tncb_ctx_destroy for plans that outlive their context (either order is safe).
void tncb_plan_release_device_state(tncb_plan* plan) {
  tncb_ctx* ctx = plan->ctx;
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < 2; i++) if (plan->exec[i]) { cudaGraphExecDestroy(plan->exec[i]); plan->exec[i] = nullptr; }
  if (plan->batch_dev) { ctx->arena.free(plan->batch_dev, plan->batch_bytes); plan->batch_dev = nullptr; }
  if (plan->slices_dev) { ctx->arena.free(plan->slices_dev, plan->slices_bytes); plan->slices_dev = nullptr; plan->n_slices = 0; }
  plan->leaves_resident = false;
  if (plan->ws) { ctx->arena.free(plan->ws, plan->ws_bytes); plan->ws = nullptr; }
  if (plan->stage) { cudaFreeHost(plan->stage); plan->stage = nullptr; }
  if (plan->stage_ev) { cudaEventDestroy(plan->stage_ev); plan->stage_ev = nullptr; plan->stage_busy = false; }
  if (plan->resident) { ctx->arena.free(plan->resident, plan->resident_bytes); plan->resident = nullptr; }
  for (size_t i = 0; i < ctx->plans.size(); i++)
    if (ctx->plans[i] == plan) { ctx->plans.erase(ctx->plans.begin() + i); break; }
  plan->ctx = nullptr;
}

void tncb_plan_destroy(tncb_plan* plan) {
  if (!plan) return;
  tncb_plan_release_device_state(plan);
  delete plan;
}

} // extern "C"

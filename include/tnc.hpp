// tnc.hpp -- header-only C++ host-side mirror of the reference's interface for the hot path,
// written above the C ABI of include/tncb.h (the Rust toolchain is absent in this image, the
// reference is compiled code, so the compiled host side is C++).
//
//   tnc::Tensor            <- tnc::tensornetwork::tensor::Tensor        (tensor.rs:21-37)
//   tnc::TensorData        <- tnc::tensornetwork::tensordata::TensorData (tensordata.rs:15-26)
//   tnc::ContractionPath   <- tnc::contractionpath::ContractionPath     (contractionpath.rs:29-35)
//   tnc::contract_tensor_network(Tensor, const ContractionPath&) -> Tensor   (contraction.rs:30)
//
// Errors: the reference panics; here every non-zero tncb_status becomes a tnc::Error exception.
#pragma once
#include <complex>
#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "tncb.h"

namespace tnc {

using Complex64 = std::complex<double>;

struct Error : std::runtime_error {
  int status;
  Error(int s, const std::string& m) : std::runtime_error(m), status(s) {}
};
inline void check(int rc) {
  if (rc != TNCB_OK) {
    std::string m = tncb_last_error();
    throw Error(rc, m.empty() ? tncb_strerror(rc) : m);
  }
}

class Context {
 public:
  explicit Context(int device = 0, size_t arena_bytes = 0) { check(tncb_ctx_create(device, arena_bytes, &h_)); }
  ~Context() { tncb_ctx_destroy(h_); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  tncb_ctx* get() const { return h_; }
  // requested normwise tolerance of the tcgen05 engine (0 = full FP64 mantissa), see tncb_ctx_set_tolerance
  void set_tolerance(double rel) { check(tncb_ctx_set_tolerance(h_, rel)); }
  void synchronize() { check(tncb_ctx_synchronize(h_)); }
 private:
  tncb_ctx* h_ = nullptr;
};

// Device payload with shared ownership ("clone does not clone the data", like tetra::Tensor).
struct DeviceData {
  tncb_ctx* ctx = nullptr;
  tncb_tensor* t = nullptr;
  ~DeviceData() { if (t) tncb_tensor_free(ctx, t); }
};

struct TensorData {
  enum Kind { Uncontracted, Gate, Matrix, Device, File } kind = Uncontracted;
  std::string file_path;                                                     // File((path, adjoint)), HDF5 (io::hdf5)
  std::string gate_name; std::vector<double> angles; bool adjoint = false;   // Gate((name, angles, adjoint))
  std::vector<Complex64> matrix;                                             // Matrix (host, row-major)
  std::shared_ptr<DeviceData> device;                                        // Matrix resident on the GPU

  static TensorData gate(std::string name, std::vector<double> ang = {}, bool adj = false) {
    TensorData d; d.kind = Gate; d.gate_name = std::move(name); d.angles = std::move(ang); d.adjoint = adj; return d;
  }
  static TensorData file(std::string path, bool adj = false) {
    TensorData d; d.kind = File; d.file_path = std::move(path); d.adjoint = adj; return d;
  }
  // TensorData::new_from_data(dimensions, data, None)  (tensordata.rs:31-37)
  static TensorData new_from_data(const std::vector<uint64_t>&, std::vector<Complex64> data) {
    TensorData d; d.kind = Matrix; d.matrix = std::move(data); return d;
  }
};

struct Tensor {
  std::vector<Tensor> tensors;
  std::vector<uint64_t> legs, bond_dims;
  TensorData tensordata;

  Tensor() = default;
  Tensor(std::vector<uint64_t> l, std::vector<uint64_t> d) : legs(std::move(l)), bond_dims(std::move(d)) {}
  static Tensor new_from_const(std::vector<uint64_t> l, uint64_t dim) {
    std::vector<uint64_t> d(l.size(), dim); return Tensor(std::move(l), std::move(d));
  }
  static Tensor new_composite(std::vector<Tensor> ts) { Tensor t; t.tensors = std::move(ts); return t; }
  bool is_leaf() const { return tensors.empty(); }
  bool is_composite() const { return !tensors.empty(); }
  void set_tensor_data(TensorData d) { tensordata = std::move(d); }
  void push_tensor(Tensor t) { tensors.push_back(std::move(t)); }
  const Tensor& tensor(size_t i) const { return tensors.at(i); }

  // `elements()`: row-major data of a contracted leaf (downloads from the device; complex64 results are widened)
  std::vector<Complex64> elements() const {
    if (tensordata.kind == TensorData::Matrix) return tensordata.matrix;
    if (tensordata.kind != TensorData::Device) throw Error(TNCB_ERR_UNCONTRACTED, "Cannot convert uncontracted tensor to data");
    const tncb_tensor* t = tensordata.device->t;
    std::vector<Complex64> out(tncb_tensor_elements(t));
    if (tncb_tensor_dtype(t) == TNCB_C64) {
      std::vector<std::complex<float>> narrow(out.size());
      check(tncb_tensor_download(tensordata.device->ctx, t, reinterpret_cast<double*>(narrow.data())));
      for (size_t i = 0; i < out.size(); i++) out[i] = Complex64(narrow[i].real(), narrow[i].imag());
      return out;
    }
    check(tncb_tensor_download(tensordata.device->ctx, t, reinterpret_cast<double*>(out.data())));
    return out;
  }
};

struct ContractionPath {
  std::map<size_t, ContractionPath> nested;
  std::vector<std::pair<size_t, size_t>> toplevel;
  static ContractionPath simple(std::vector<std::pair<size_t, size_t>> p) { ContractionPath c; c.toplevel = std::move(p); return c; }
  static ContractionPath single(size_t a, size_t b) { return simple({{a, b}}); }
};

namespace detail {
struct Marshal {  // owns every buffer the C structs point into
  std::vector<std::unique_ptr<std::vector<tncb_tn>>> tn_arrays;
  std::vector<std::unique_ptr<std::vector<tncb_path>>> path_arrays;
  std::vector<std::unique_ptr<std::vector<uint64_t>>> u64s;

  tncb_tn tn(const Tensor& t) {
    tncb_tn n{};
    if (t.is_composite()) {
      auto arr = std::make_unique<std::vector<tncb_tn>>();
      for (const Tensor& c : t.tensors) arr->push_back(tn(c));
      n.n_children = arr->size(); n.children = arr->data();
      tn_arrays.push_back(std::move(arr));
      return n;
    }
    n.rank = (int)t.legs.size(); n.legs = t.legs.data(); n.dims = t.bond_dims.data();
    switch (t.tensordata.kind) {
      case TensorData::Gate:
        n.kind = TNCB_DATA_GATE; n.gate_name = t.tensordata.gate_name.c_str();
        n.gate_angles = t.tensordata.angles.data(); n.n_gate_angles = (int)t.tensordata.angles.size();
        n.gate_adjoint = t.tensordata.adjoint; break;
      case TensorData::Matrix:
        n.kind = TNCB_DATA_MATRIX; n.host_re_im = reinterpret_cast<const double*>(t.tensordata.matrix.data()); break;
      case TensorData::Device:
        n.kind = TNCB_DATA_DEVICE; n.device = t.tensordata.device->t; break;
      case TensorData::File:
        n.kind = TNCB_DATA_FILE; n.file_path = t.tensordata.file_path.c_str(); n.file_adjoint = t.tensordata.adjoint; break;
      default: n.kind = TNCB_DATA_UNCONTRACTED;
    }
    return n;
  }
  tncb_path path(const ContractionPath& p) {
    tncb_path o{};
    auto pairs = std::make_unique<std::vector<uint64_t>>();
    for (auto& q : p.toplevel) { pairs->push_back(q.first); pairs->push_back(q.second); }
    o.n_pairs = p.toplevel.size(); o.pairs = pairs->data();
    u64s.push_back(std::move(pairs));
    if (!p.nested.empty()) {
      auto idx = std::make_unique<std::vector<uint64_t>>();
      auto arr = std::make_unique<std::vector<tncb_path>>();
      for (auto& kv : p.nested) { idx->push_back(kv.first); arr->push_back(path(kv.second)); }
      o.n_nested = idx->size(); o.nested_index = idx->data(); o.nested = arr->data();
      u64s.push_back(std::move(idx)); path_arrays.push_back(std::move(arr));
    }
    return o;
  }
};
inline void release_device_inputs(Tensor& t) {  // the call consumed them (mem::take)
  if (t.is_composite()) { for (Tensor& c : t.tensors) release_device_inputs(c); return; }
  if (t.tensordata.kind == TensorData::Device && t.tensordata.device) t.tensordata.device->t = nullptr;
}
}  // namespace detail

// Fully contracts `tn` (moved in, as in the reference) with the replace-left `path`.  dtype = TNCB_C64 runs every kernel
// in complex64 (f64 accumulation, one rounding per result); host payloads stay complex128 and are narrowed on upload.
inline Tensor contract_tensor_network(Context& ctx, Tensor tn, const ContractionPath& path, tncb_dtype dtype = TNCB_C128) {
  detail::Marshal m;
  tncb_tn c_tn = m.tn(tn);
  tncb_path c_path = m.path(path);
  tncb_tensor* out = nullptr; int n_out = 0; uint64_t legs[64];
  check(tncb_contract_tensor_network_dt(ctx.get(), &c_tn, &c_path, dtype, &out, &n_out, legs));
  detail::release_device_inputs(tn);
  Tensor res;
  if (!out) return res;
  res.legs.assign(legs, legs + n_out);
  res.bond_dims.resize(n_out);
  if (n_out) check(tncb_tensor_dims(out, res.bond_dims.data()));
  res.tensordata.kind = TensorData::Device;
  res.tensordata.device = std::make_shared<DeviceData>();
  res.tensordata.device->ctx = ctx.get(); res.tensordata.device->t = out;
  return res;
}

// Compile once / execute many (tncb_plan_*): the same circuit with other payloads (bitstrings, angles) re-uses the
// schedule, the static memory layout, the batched tiny pairs and (for launch-bound networks) the CUDA graph.
class NetworkPlan {
 public:
  NetworkPlan(Context& ctx, const Tensor& tn, const ContractionPath& path, tncb_dtype dtype = TNCB_C128) : ctx_(ctx) {
    detail::Marshal m;
    tncb_tn c_tn = m.tn(tn);
    tncb_path c_path = m.path(path);
    check(tncb_plan_create_dt(ctx.get(), &c_tn, &c_path, dtype, &h_));
  }
  ~NetworkPlan() { tncb_plan_destroy(h_); }
  NetworkPlan(const NetworkPlan&) = delete;
  NetworkPlan& operator=(const NetworkPlan&) = delete;
  Tensor execute(const Tensor& tn) {                 // host leaves -> one H2D -> all kernels
    detail::Marshal m;
    tncb_tn c_tn = m.tn(tn);
    tncb_tensor* out = nullptr; int n_out = 0; uint64_t legs[64];
    check(tncb_plan_execute(ctx_.get(), h_, &c_tn, &out, &n_out, legs));
    return wrap(out, n_out, legs);
  }
  void stage(const Tensor& tn) { detail::Marshal m; tncb_tn c_tn = m.tn(tn); check(tncb_plan_stage(ctx_.get(), h_, &c_tn)); }
  Tensor run() {                                     // leaves resident on the device: no host data movement
    tncb_tensor* out = nullptr; int n_out = 0; uint64_t legs[64];
    check(tncb_plan_run(ctx_.get(), h_, &out, &n_out, legs));
    return wrap(out, n_out, legs);
  }
 private:
  Tensor wrap(tncb_tensor* out, int n_out, const uint64_t* legs) {
    Tensor res;
    if (!out) return res;
    res.legs.assign(legs, legs + n_out);
    res.bond_dims.resize(n_out);
    if (n_out) check(tncb_tensor_dims(out, res.bond_dims.data()));
    res.tensordata.kind = TensorData::Device;
    res.tensordata.device = std::make_shared<DeviceData>();
    res.tensordata.device->ctx = ctx_.get(); res.tensordata.device->t = out;
    return res;
  }
  Context& ctx_;
  tncb_plan* h_ = nullptr;
};

// tnc::builders (tnc/src/builders/circuit_builder.rs): Permutor (:72-129) and Circuit (:135-335).
namespace builders {

// TensorData::adjoint (tensordata.rs:62-72) for the payload kinds a circuit holds
inline TensorData adjoint(const TensorData& d, const std::vector<uint64_t>& dims) {
  TensorData a = d;
  if (d.kind == TensorData::Gate || d.kind == TensorData::File) { a.adjoint = !d.adjoint; return a; }
  if (d.kind != TensorData::Matrix) return a;
  const size_t r = dims.size(), half = r / 2;
  size_t rows = 1, cols = 1;
  for (size_t i = 0; i < half; i++) rows *= dims[i];
  for (size_t i = half; i < r; i++) cols *= dims[i];
  for (size_t i = 0; i < rows; i++)
    for (size_t j = 0; j < cols; j++) a.matrix[j * rows + i] = std::conj(d.matrix[i * cols + j]);
  return a;
}

class Permutor {
 public:
  explicit Permutor(std::vector<uint64_t> target) : target_leg_order(std::move(target)) {}
  bool is_identity() const { return target_leg_order.empty(); }
  // permutation p with given[p[i]] == target[i] (circuit_builder.rs:125-129)
  static std::vector<int> permutation_between(const std::vector<uint64_t>& given, const std::vector<uint64_t>& target) {
    if (given.size() != target.size()) throw Error(TNCB_ERR_INVALID, "given and target must be permutations of each other");
    std::vector<int> p;
    for (uint64_t l : target) {
      size_t q = 0;
      while (q < given.size() && given[q] != l) q++;
      if (q == given.size()) throw Error(TNCB_ERR_INVALID, "given and target must be permutations of each other");
      p.push_back((int)q);
    }
    return p;
  }
  // Permutor::apply (:86-114): transposes the device data into the target leg order (one tncb_permute launch)
  Tensor apply(Context& ctx, Tensor t) const {
    if (is_identity()) return t;
    if (t.tensordata.kind != TensorData::Device) throw Error(TNCB_ERR_UNCONTRACTED, "Permutor::apply needs a contracted (device) tensor");
    std::vector<int> perm = permutation_between(t.legs, target_leg_order);
    tncb_tensor* out = nullptr;
    check(tncb_permute(ctx.get(), t.tensordata.device->t, perm.data(), &out));
    t.tensordata.device->t = nullptr;                 // consumed
    Tensor res(target_leg_order, {});
    for (int q : perm) res.bond_dims.push_back(t.bond_dims[q]);
    res.tensordata.kind = TensorData::Device;
    res.tensordata.device = std::make_shared<DeviceData>();
    res.tensordata.device->ctx = ctx.get(); res.tensordata.device->t = out;
    return res;
  }
  std::vector<uint64_t> target_leg_order;
};

class Circuit {
 public:
  size_t num_qubits() const { return open_edges_.size(); }
  // allocate_register (:184-203): returns the indices of the new qubits
  std::vector<size_t> allocate_register(size_t size) {
    std::vector<size_t> reg;
    for (size_t i = 0; i < size; i++) {
      reg.push_back(num_qubits());
      const uint64_t e = next_edge_++;
      open_edges_.push_back(e);
      Tensor ket = Tensor::new_from_const({e}, 2);
      ket.set_tensor_data(ket_data(0));
      tensors_.push_back(std::move(ket));
    }
    return reg;
  }
  // append_gate (:205-241): legs = [old edges ..., new edges ...]
  void append_gate(TensorData gate, const std::vector<size_t>& qubits) {
    for (size_t i = 0; i < qubits.size(); i++)
      for (size_t j = i + 1; j < qubits.size(); j++)
        if (qubits[i] == qubits[j]) throw Error(TNCB_ERR_INVALID, "Qubit arguments must be unique");
    std::vector<uint64_t> edges;
    for (size_t q : qubits) edges.push_back(open_edges_.at(q));
    for (size_t i = 0; i < qubits.size(); i++) { edges.push_back(next_edge_ + i); open_edges_[qubits[i]] = next_edge_ + i; }
    next_edge_ += qubits.size();
    Tensor t = Tensor::new_from_const(std::move(edges), 2);
    t.set_tensor_data(std::move(gate));
    tensors_.push_back(std::move(t));
  }
  // into_amplitude_network (:243-277): '0' / '1' close a qubit with a bra, '*' leaves it open
  std::pair<Tensor, Permutor> into_amplitude_network(const std::string& bitstring) && {
    if (bitstring.size() != num_qubits()) throw Error(TNCB_ERR_INVALID, "bitstring length differs from the number of qubits");
    std::vector<uint64_t> final_legs;
    for (size_t q = 0; q < bitstring.size(); q++) {
      const char c = bitstring[q];
      if (c == '*') { final_legs.push_back(open_edges_[q]); continue; }
      if (c != '0' && c != '1') throw Error(TNCB_ERR_INVALID, "Only 0, 1 and * are allowed in bitstring");
      Tensor bra = Tensor::new_from_const({open_edges_[q]}, 2);
      bra.set_tensor_data(ket_data(c - '0'));
      tensors_.push_back(std::move(bra));
    }
    return {Tensor::new_composite(std::move(tensors_)), Permutor(std::move(final_legs))};
  }
  std::pair<Tensor, Permutor> into_statevector_network() && { return std::move(*this).into_amplitude_network(std::string(num_qubits(), '*')); }
  // into_expectation_value_network (:315-335): the circuit, its adjoint mirror image (legs + offset) and a layer of Z
  Tensor into_expectation_value_network() && {
    const uint64_t offset = next_edge_;
    const size_t n = tensors_.size();
    for (size_t i = 0; i < n; i++) {
      const Tensor& t = tensors_[i];
      const size_t half = t.legs.size() / 2;
      Tensor a;
      for (size_t q = half; q < t.legs.size(); q++) { a.legs.push_back(t.legs[q] + offset); a.bond_dims.push_back(t.bond_dims[q]); }
      for (size_t q = 0; q < half; q++) { a.legs.push_back(t.legs[q] + offset); a.bond_dims.push_back(t.bond_dims[q]); }
      a.set_tensor_data(adjoint(t.tensordata, t.bond_dims));
      tensors_.push_back(std::move(a));
    }
    for (uint64_t e : open_edges_) {
      Tensor z = Tensor::new_from_const({e, e + offset}, 2);
      z.set_tensor_data(TensorData::gate("z"));
      tensors_.push_back(std::move(z));
    }
    return Tensor::new_composite(std::move(tensors_));
  }

 private:
  static TensorData ket_data(int bit) {
    return TensorData::new_from_data({2}, bit == 0 ? std::vector<Complex64>{{1, 0}, {0, 0}} : std::vector<Complex64>{{0, 0}, {1, 0}});
  }
  std::vector<uint64_t> open_edges_;
  uint64_t next_edge_ = 0;
  std::vector<Tensor> tensors_;
};

}  // namespace builders

// tnc::io::hdf5 (tnc/src/io/hdf5.rs): /tensors/<name> datasets with `bids` attributes, "-1" = the output tensor.
namespace io { namespace hdf5 {
namespace detail {
struct File {
  tncb_h5file* h = nullptr;
  explicit File(const std::string& path) { check(tncb_hdf5_open(path.c_str(), nullptr, &h)); }
  ~File() { tncb_hdf5_close(h); }
  File(const File&) = delete;
  File& operator=(const File&) = delete;
  std::vector<uint64_t> bids(size_t i) const {
    size_t n = 0;
    check(tncb_hdf5_attr(h, i, "bids", 0, nullptr, &n));
    std::vector<int64_t> v(n ? n : 1);
    check(tncb_hdf5_attr(h, i, "bids", n, v.data(), &n));
    std::vector<uint64_t> out;
    for (size_t q = 0; q < n; q++) { if (v[q] < 0) throw Error(TNCB_ERR_INVALID, "negative bond id"); out.push_back((uint64_t)v[q]); }
    return out;
  }
  std::vector<Complex64> read(size_t i, std::vector<uint64_t>* shape) const {
    int rank = 0; uint64_t dims[32], elems = 0;
    check(tncb_hdf5_shape(h, i, &rank, dims, &elems));
    shape->assign(dims, dims + rank);
    std::vector<Complex64> data(elems);
    if (elems) check(tncb_hdf5_read(h, i, reinterpret_cast<double*>(data.data())));
    return data;
  }
};
}  // namespace detail

// load_tensor (hdf5.rs:28-34, 54-88): a composite of Matrix leaves in member order; legs = the `bids` of "-1"
inline Tensor load_tensor(const std::string& filename) {
  detail::File f(filename);
  Tensor tn;
  bool have_out = false;
  for (size_t i = 0; i < tncb_hdf5_count(f.h); i++) {
    if (std::string(tncb_hdf5_name(f.h, i)) == "-1") { tn.legs = f.bids(i); have_out = true; continue; }
    std::vector<uint64_t> shape;
    std::vector<Complex64> data = f.read(i, &shape);
    Tensor t(f.bids(i), shape);
    t.set_tensor_data(TensorData::new_from_data(shape, std::move(data)));
    tn.push_tensor(std::move(t));
  }
  if (!have_out) throw Error(TNCB_ERR_IO, "no output tensor '-1' in /tensors");
  return tn;
}
// load_data (hdf5.rs:37-43, 90-103): the first member of /tensors
inline std::vector<Complex64> load_data(const std::string& filename, std::vector<uint64_t>* shape) {
  detail::File f(filename);
  if (tncb_hdf5_count(f.h) == 0) throw Error(TNCB_ERR_IO, "no member in /tensors");
  return f.read(0, shape);
}
// store_data (hdf5.rs:46-52, 105-113)
inline void store_data(const std::string& filename, const std::vector<uint64_t>& shape, const std::vector<Complex64>& data) {
  check(tncb_hdf5_store_data(filename.c_str(), (int)shape.size(), shape.data(), reinterpret_cast<const double*>(data.data())));
}
}}  // namespace io::hdf5

}  // namespace tnc

// b200fft.hpp — header-only C++ host layer over the C ABI (b200fft.h), with the names and argument
// meaning of the reference's `fft` package (fft/fft/fft.mojo): `plan_fft` builds a reusable plan,
// `fft(output, x, stream, plan)` enqueues the transform asynchronously and the caller synchronises.
//
// The reference's compile-time parameters (dtypes, layouts incl. batch, inverse, bases —
// fft/fft/fft.mojo:160-176) are runtime values of `Layout` / `PlanOptions` here; its compile-time
// asserts (`_check_layout_conditions_nd`, fft.mojo:20-46; base asserts, _utils.mojo:205-220) come
// back as `b200fft::Error` with the C ABI's status code. No torch, no CUDA headers: device buffers
// are plain pointers and the stream is an opaque `void*` (a `cudaStream_t` / `CUstream`).
//
//   b200fft::Layout in{{100, 640, 480, 2}}, out = in;                   // (batches, d0, d1, 2)
//   auto plan = b200fft::plan_fft(b200fft::f32, b200fft::f32, in, out); // reference: plan_fft[...](ctx=ctx)
//   b200fft::fft(d_out, d_x, stream, plan);                             // reference: fft(output, x, ctx, plan=plan)
//
// Link with -lb200fft (hackathon-fft_b200/lib). There is no CPU path: plan_fft throws status 5
// (B200FFT_ERR_CUDA) without an sm_100 device; `dry_run` and the base rules work anywhere.
#ifndef B200FFT_HPP
#define B200FFT_HPP

#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "b200fft.h"

namespace b200fft {

enum DType : int32_t { u8 = B200FFT_U8, f32 = B200FFT_F32, f64 = B200FFT_F64 };
enum RealMode : int32_t { real_full = B200FFT_REAL_FULL, real_half = B200FFT_REAL_HALF };

// Non-zero status of a C ABI call, with the library's thread-local detail message.
class Error : public std::runtime_error {
 public:
  Error(int status, const std::string& detail)
      : std::runtime_error("b200fft status " + std::to_string(status) + ": " + detail), status_(status) {}
  int status() const { return status_; }

 private:
  int status_;
};

inline void check(int rc) {
  if (rc == B200FFT_OK) return;
  const char* detail = b200fft_last_error();
  throw Error(rc, (detail && *detail) ? detail : b200fft_strerror(rc));
}

// The reference's `Layout.row_major(batches, d0[, d1...], 1|2)` as a shape list.
struct Layout {
  std::vector<int64_t> shape;
  size_t rank() const { return shape.size(); }
  int64_t size() const {
    int64_t n = 1;
    for (int64_t v : shape) n *= v;
    return n;
  }
};

// The keyword parameters of the reference's GPU `plan_fft` (fft.mojo:160-176) plus what is new here.
struct PlanOptions {
  std::vector<std::vector<uint32_t>> bases;  // one list per axis; empty = the reference's default rule
  bool inverse = false;
  bool runtime_twfs = true;        // accepted for signature compatibility, ignored
  unsigned max_cluster_size = 8;   // accepted for signature compatibility, ignored
  bool test_generic = false;       // the role of `_test: _GPUTest`: force the generic kernel
  RealMode real_mode = real_full;  // real_half: cuFFT-style n/2+1 bins (new)
  uint32_t axis_mask = 0;          // 0 = all axes (reference)
  int device = -1;                 // -1 = current device
  uint32_t flags = 0;
  // strided buffers (b200fft_plan_create_strided): one stride per dimension of the layout but the last, in ELEMENTS
  // (complex pairs or real scalars) of that buffer; empty = dense
  std::vector<int64_t> in_strides, out_strides;
};

namespace detail {
struct Marshalled {
  b200fft_desc desc{};
  std::vector<uint32_t> flat;
  std::vector<int32_t> counts;
};

// Layout rules that need both layouts (the rest is validated by the library, same messages as
// `_check_layout_conditions_nd`), then the runtime descriptor.
inline void marshal(DType in_dtype, DType out_dtype, const Layout& in, const Layout& out, const PlanOptions& o,
                    Marshalled* m) {
  if (out.rank() <= 2)
    throw Error(B200FFT_ERR_LAYOUT, "The rank should be bigger than 2. The first dimension represents the amount of "
                                    "batches, and the last the complex dimension.");
  if (in.rank() != out.rank()) throw Error(B200FFT_ERR_LAYOUT, "in_layout and out_layout must have equal rank");
  const size_t r = out.rank();
  const bool half = o.real_mode == real_half;
  const Layout& logical = (half && !o.inverse) ? in : out;  // half spectrum: the REAL side carries the lengths
  if (!half) {
    if (out.shape[r - 1] != 2) throw Error(B200FFT_ERR_LAYOUT, "out_layout must have the last dimension equal to 2");
    for (size_t i = 0; i + 1 < r; ++i)
      if (in.shape[i] != out.shape[i])
        throw Error(B200FFT_ERR_LAYOUT, "out_layout and in_layout should have the same shape before the last dimension");
  } else {
    const Layout& cplx = o.inverse ? in : out;
    bool ok = logical.shape[r - 1] == 1 && cplx.shape[r - 1] == 2 && cplx.shape[r - 2] == logical.shape[r - 2] / 2 + 1;
    for (size_t i = 0; i + 2 < r; ++i) ok = ok && cplx.shape[i] == logical.shape[i];
    if (!ok)
      throw Error(B200FFT_ERR_LAYOUT, "REAL_HALF layouts must be real (B, dims..., 1) and complex (B, dims[:-1]..., n/2+1, 2)");
  }
  if (r - 2 > B200FFT_MAX_RANK) throw Error(B200FFT_ERR_LAYOUT, "at most 8 transformed axes");
  b200fft_desc& d = m->desc;
  d.rank = (int32_t)(r - 2);
  for (size_t i = 0; i + 2 < r; ++i) d.dims[i] = logical.shape[i + 1];
  d.batch = out.shape[0];
  d.in_components = (int32_t)in.shape[r - 1];
  d.in_dtype = in_dtype;
  d.out_dtype = out_dtype;
  d.inverse = o.inverse ? 1 : 0;
  d.real_mode = o.real_mode;
  d.axis_mask = o.axis_mask;
  d.device = o.device;
  d.flags = o.flags | (o.test_generic ? (uint32_t)B200FFT_FLAG_FORCE_GENERIC : 0u);
  if (!o.bases.empty()) {
    if (o.bases.size() != r - 2)
      throw Error(B200FFT_ERR_BASES, "The bases list should have the same outer size as the amount of internal "
                                     "dimensions. e.g. (batches, dim_0, dim_1, dim_2, 2) -> len(bases) == 3");
    for (const auto& axis : o.bases) {
      m->counts.push_back((int32_t)axis.size());
      m->flat.insert(m->flat.end(), axis.begin(), axis.end());
    }
    if (m->flat.empty()) m->flat.push_back(0);  // non-null pointer for all-default lists
    d.bases = m->flat.data();
    d.bases_count = m->counts.data();
  }
}
}  // namespace detail

// Runtime analogue of the reference's `_GPUPlan` (fft/fft/_ndim_fft_gpu.mojo:153-207): owns the device
// twiddle tables and the kernel choice, built once and reused; move-only; not re-entrant (one exec at a time).
class Plan {
 public:
  Plan() = default;
  Plan(b200fft_plan* h, Layout in, Layout out) : h_(h), in_(std::move(in)), out_(std::move(out)) {}
  Plan(Plan&& o) noexcept : h_(o.h_), in_(std::move(o.in_)), out_(std::move(o.out_)) { o.h_ = nullptr; }
  Plan& operator=(Plan&& o) noexcept {
    if (this != &o) {
      reset();
      h_ = o.h_;
      in_ = std::move(o.in_);
      out_ = std::move(o.out_);
      o.h_ = nullptr;
    }
    return *this;
  }
  Plan(const Plan&) = delete;
  Plan& operator=(const Plan&) = delete;
  ~Plan() { reset(); }

  void exec(void* d_out, const void* d_in, void* stream = nullptr) const { check(b200fft_exec(h_, d_out, d_in, stream)); }
  // host buffers: chunked H2D -> kernels -> D2H pipeline, returns when h_out is complete
  void exec_host(void* h_out, const void* h_in) const { check(b200fft_exec_host(h_, h_out, h_in)); }

  std::vector<uint32_t> bases(int axis) const {
    uint32_t buf[64];
    const int n = b200fft_plan_get_bases(h_, axis, buf, 64);
    return n < 0 ? std::vector<uint32_t>() : std::vector<uint32_t>(buf, buf + n);
  }
  std::string describe() const {
    std::string s(b200fft_plan_describe(h_, nullptr, 0), '\0');
    if (!s.empty()) b200fft_plan_describe(h_, &s[0], s.size());
    while (!s.empty() && s.back() == '\0') s.pop_back();
    return s;
  }
  int launches() const { return b200fft_plan_launches(h_); }
  size_t in_bytes() const { return b200fft_plan_in_bytes(h_); }
  size_t out_bytes() const { return b200fft_plan_out_bytes(h_); }
  size_t workspace_bytes() const { return b200fft_plan_workspace_bytes(h_); }
  const Layout& in_layout() const { return in_; }
  const Layout& out_layout() const { return out_; }
  b200fft_plan* handle() const { return h_; }
  explicit operator bool() const { return h_ != nullptr; }

 private:
  void reset() {
    if (h_) b200fft_plan_destroy(h_);
    h_ = nullptr;
  }
  b200fft_plan* h_ = nullptr;
  Layout in_, out_;
};

// Plan the FFT on GPU — the reference's `plan_fft[in_dtype, out_dtype, in_layout, out_layout, bases=..., inverse=...](ctx=ctx)`
// (fft/fft/fft.mojo:160-210).
inline Plan plan_fft(DType in_dtype, DType out_dtype, const Layout& in_layout, const Layout& out_layout,
                     const PlanOptions& options = PlanOptions()) {
  detail::Marshalled m;
  detail::marshal(in_dtype, out_dtype, in_layout, out_layout, options, &m);
  b200fft_plan* h = nullptr;
  if (options.in_strides.empty() && options.out_strides.empty()) {
    check(b200fft_plan_create(&h, &m.desc));
  } else {
    const size_t want = out_layout.rank() - 1;
    if ((!options.in_strides.empty() && options.in_strides.size() != want) || (!options.out_strides.empty() && options.out_strides.size() != want))
      throw Error(B200FFT_ERR_LAYOUT, "in_strides / out_strides need one stride per dimension of the layout but the last");
    check(b200fft_plan_create_strided(&h, &m.desc, options.in_strides.empty() ? nullptr : options.in_strides.data(),
                                      options.out_strides.empty() ? nullptr : options.out_strides.data()));
  }
  return Plan(h, in_layout, out_layout);
}

// Calculate the FFT on GPU — the reference's `fft(output, x, ctx, plan=plan)` (fft/fft/fft.mojo:262-323):
// asynchronous on `stream`, device pointers with the plan's layouts, caller synchronises (fft/bench.mojo:51-52).
inline void fft(void* output, const void* x, void* stream, const Plan& plan) { plan.exec(output, x, stream); }

// One host process, several GPUs (b200fft_mgpu_*): batch sharding without communication, or the slab decomposition of ONE
// 3-D complex fp32 / fp64 transform (dims (Z, Y, X); slot g holds z planes [g Z/G, (g+1) Z/G), the result is Y-slab
// distributed), or of a real one with options.real_mode = half spectrum: R2C forward as above over X/2+1 bins, C2R inverse
// from those Y-slabs back to z planes (include/b200fft.h, B200FFT_MGPU_SLAB).
enum class MultiGpuMode { batch_shard = B200FFT_MGPU_BATCH_SHARD, slab = B200FFT_MGPU_SLAB };

class MultiGpuPlan {
 public:
  MultiGpuPlan() = default;
  MultiGpuPlan(DType in_dtype, DType out_dtype, const Layout& in_layout, const Layout& out_layout, const std::vector<int>& devices,
               MultiGpuMode mode = MultiGpuMode::batch_shard, const PlanOptions& options = PlanOptions()) {
    detail::Marshalled m;
    detail::marshal(in_dtype, out_dtype, in_layout, out_layout, options, &m);
    check(b200fft_mgpu_plan_create(&h_, &m.desc, (int)devices.size(), devices.data(), (int)mode));
  }
  MultiGpuPlan(MultiGpuPlan&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  MultiGpuPlan& operator=(MultiGpuPlan&& o) noexcept {
    if (this != &o) {
      reset();
      h_ = o.h_;
      o.h_ = nullptr;
    }
    return *this;
  }
  MultiGpuPlan(const MultiGpuPlan&) = delete;
  MultiGpuPlan& operator=(const MultiGpuPlan&) = delete;
  ~MultiGpuPlan() { reset(); }

  int ngpu() const { return b200fft_mgpu_ngpu(h_); }
  // (first, count) of the batch items (batch shard) / z planes (slab) device slot g holds
  std::pair<int64_t, int64_t> shard(int g) const {
    int64_t first = 0, count = 0;
    check(b200fft_mgpu_shard(h_, g, &first, &count));
    return {first, count};
  }
  size_t in_bytes(int g) const { return b200fft_mgpu_in_bytes(h_, g); }
  size_t out_bytes(int g) const { return b200fft_mgpu_out_bytes(h_, g); }
  // enqueue on every slot's plan-owned stream (d_out[g] / d_in[g] live on slot g's device); synchronize() before reading
  void exec(void* const* d_out, const void* const* d_in) const { check(b200fft_mgpu_exec(h_, d_out, d_in)); }
  void synchronize() const { check(b200fft_mgpu_synchronize(h_)); }
  void* stream(int g) const { return b200fft_mgpu_stream(h_, g); }
  // the whole job from / to host memory in natural order; returns when h_out is complete
  void exec_host(void* h_out, const void* h_in) const { check(b200fft_mgpu_exec_host(h_, h_out, h_in)); }
  std::string describe() const {
    std::string s(b200fft_mgpu_describe(h_, nullptr, 0), '\0');
    if (!s.empty()) b200fft_mgpu_describe(h_, &s[0], s.size());
    while (!s.empty() && s.back() == '\0') s.pop_back();
    return s;
  }
  explicit operator bool() const { return h_ != nullptr; }

 private:
  void reset() {
    if (h_) b200fft_mgpu_plan_destroy(h_);
    h_ = nullptr;
  }
  b200fft_mgpu_plan* h_ = nullptr;
};

// Validate a request and return the pass list it would produce, without touching CUDA.
inline std::string dry_run(DType in_dtype, DType out_dtype, const Layout& in_layout, const Layout& out_layout,
                           const PlanOptions& options = PlanOptions()) {
  detail::Marshalled m;
  detail::marshal(in_dtype, out_dtype, in_layout, out_layout, options, &m);
  std::string buf(4096, '\0');
  check(b200fft_plan_dry_run(&m.desc, &buf[0], buf.size()));
  buf.resize(buf.find('\0') == std::string::npos ? buf.size() : buf.find('\0'));
  return buf;
}

// `_build_ordered_bases` + validity (fft/fft/_utils.mojo:163-221); empty when the reference rejects the bases.
inline std::vector<uint32_t> ordered_bases(uint64_t length, const std::vector<uint32_t>& bases) {
  uint32_t out[64];
  const int n = b200fft_ordered_bases(length, bases.data(), (int)bases.size(), out, 64);
  return n < 0 ? std::vector<uint32_t>() : std::vector<uint32_t>(out, out + n);
}

// `_estimate_best_bases` (fft/fft/fft.mojo:49-104).
inline std::vector<uint32_t> default_bases(uint64_t length, bool gpu_target = true) {
  uint32_t out[64];
  const int n = b200fft_default_bases(length, gpu_target ? 1 : 0, out, 64);
  return n < 0 ? std::vector<uint32_t>() : std::vector<uint32_t>(out, out + n);
}

}  // namespace b200fft
#endif  // B200FFT_HPP

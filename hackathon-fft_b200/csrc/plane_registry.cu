// Plane kernels (plane.cuh): the two innermost axes of a half-spectrum inverse in one tile per (y, x) plane.
// Registered for the plane sizes of the BASELINE 3-D shapes; the planner (api.cu: build_passes) puts the pass in place of
// the strided pass over the second-to-last axis + the C2R row pass when the stage lists can be grouped into it.
#define B200FFT_PACKED 1  // packed FADD2 complex adds (dft.cuh): strided / shared-memory-resident kernels
#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "fast_registry.hpp"
#include "plan.hpp"
#include "plane.cuh"

namespace b200fft {

namespace {

struct PlaneVariant {
  int ny, h;  // NY rows, H = n / 2 complex points per row
  std::vector<int> ry, rx;
  int threads;
  size_t smem;
  void (*launch)(const PlaneArgs&, unsigned, size_t, cudaStream_t);
  const void* func;
  std::string name;
  bool by_default = true;  // false: only with B200FFT_PLANE_C2R=1 (registered, tested, measured slower than the per-axis passes)
};

template <int NY, int H, class RLY, class RLX, int NT>
void launch_plane(const PlaneArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  c2r_plane_kernel<NY, H, RLY, RLX, NT><<<grid, NT, smem, st>>>(a);
}

template <int NY, int H, class RLY, class RLX, int NT>
PlaneVariant make_variant() {
  PlaneVariant v;
  v.ny = NY;
  v.h = H;
  v.ry = radix_vec<RLY>();
  v.rx = radix_vec<RLX>();
  v.threads = NT;
  v.smem = c2r_plane_smem_bytes<NY, H, RLY, RLX>();
  v.launch = &launch_plane<NY, H, RLY, RLX, NT>;
  v.func = (const void*)c2r_plane_kernel<NY, H, RLY, RLX, NT>;
  v.name = "c2rplane" + std::to_string(NY) + "x" + std::to_string(2 * H) + "(" + radix_name(v.ry) + ";" + radix_name(v.rx) + ";2)_t" +
           std::to_string(NT);
  return v;
}

template <int NY, int H, class RLY, class RLX, int NT>
void launch_plane_ip(const PlaneArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  c2r_plane_ip_kernel<NY, H, RLY, RLX, NT><<<grid, NT, smem, st>>>(a);
}
template <int NY, int H, class RLY, class RLX, int NT>
PlaneVariant make_ip_variant() {
  PlaneVariant v;
  v.ny = NY;
  v.h = H;
  v.ry = radix_vec<RLY>();
  v.rx = radix_vec<RLX>();
  v.threads = NT;
  v.smem = r2c_plane_ip_smem_bytes<NY, H, RLX>();
  v.launch = &launch_plane_ip<NY, H, RLY, RLX, NT>;
  v.func = (const void*)c2r_plane_ip_kernel<NY, H, RLY, RLX, NT>;
  v.name = "c2rplane" + std::to_string(NY) + "x" + std::to_string(2 * H) + "(" + radix_name(v.ry) + ";" + radix_name(v.rx) + ";2)_inplace_t" +
           std::to_string(NT);
  return v;
}

const std::vector<PlaneVariant>& plane_registry() {
  static const std::vector<PlaneVariant> r = [] {
    std::vector<PlaneVariant> v;
    // 128 x 128 in ONE 74 KB buffer (three stages exchanged in place): 10 x 128^3 C2R 0.1155 ms vs 0.0951 ms per axis — opt-in
    // like the two-buffer 133 KB variant below (B200FFT_PLANE_C2R=1), unlike its forward twin, which wins (r2_plane.md)
    v.push_back(make_ip_variant<128, 64, Radices<8, 16>, Radices<8, 8>, 512>());
    v.back().by_default = false;
    v.push_back(make_variant<64, 32, Radices<8, 8>, Radices<8, 4>, 128>());
    // 128 x 128: 133 KB of shared memory = one CTA per SM: 10 x 128^3 C2R 0.132 ms vs 0.096 ms per axis (profiles/r2_c2r.md)
    v.push_back(make_variant<128, 64, Radices<16, 8>, Radices<8, 8>, 256>());
    v.back().by_default = false;
    return v;
  }();
  return r;
}

struct PlaneC2RPass : Pass {
  const PlaneVariant* v = nullptr;
  long long planes_per_batch = 1;
  float scale = 1.f;
  float2 *twy = nullptr, *twx = nullptr, *tw2 = nullptr;
  std::string text;
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    PlaneArgs a;
    a.in = reinterpret_cast<const float2*>(src);
    a.out = reinterpret_cast<float2*>(dst);
    a.twy = twy;
    a.twx = twx;
    a.tw2 = tw2;
    a.planes = nbatch * planes_per_batch;
    a.scale = scale;
    if (a.planes <= 0) return B200FFT_OK;
    if (a.planes > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many planes");
    v->launch(a, (unsigned)a.planes, v->smem, stream);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override { return src ? 0 : 8; }  // the real rows are stored as float2 pairs
};

// ---- forward / complex plane kernels
struct PlaneFwdVariant {
  bool r2c;   // half-spectrum forward (ny x 2h reals -> ny x (h+1) bins) or complex / real-input full spectrum (ny x nx)
  int ny, nx; // r2c: nx = h = n / 2
  std::vector<int> ry, rx;
  int threads;
  size_t smem;
  void (*launch)(bool inv, bool real, const PlaneFwdArgs&, unsigned, size_t, cudaStream_t);
  cudaError_t (*prepare)(size_t);
  std::string name;
};

template <int NY, int NX, class RLY, class RLX, int NT>
struct C2CPlaneV {
  static void launch(bool inv, bool real, const PlaneFwdArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
    if (inv) c2c_plane_kernel<NY, NX, RLY, RLX, NT, true, false><<<grid, NT, smem, st>>>(a);
    else if (real) c2c_plane_kernel<NY, NX, RLY, RLX, NT, false, true><<<grid, NT, smem, st>>>(a);
    else c2c_plane_kernel<NY, NX, RLY, RLX, NT, false, false><<<grid, NT, smem, st>>>(a);
  }
  static cudaError_t prepare(size_t smem) {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    cudaError_t e = cudaFuncSetAttribute(c2c_plane_kernel<NY, NX, RLY, RLX, NT, true, false>, attr, (int)smem);
    if (!e) e = cudaFuncSetAttribute(c2c_plane_kernel<NY, NX, RLY, RLX, NT, false, true>, attr, (int)smem);
    if (!e) e = cudaFuncSetAttribute(c2c_plane_kernel<NY, NX, RLY, RLX, NT, false, false>, attr, (int)smem);
    return e;
  }
};
template <int NY, int NX, class RLY, class RLX, int NT>
struct C2CPlaneIpV {
  static void launch(bool inv, bool real, const PlaneFwdArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
    if (inv) c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, true, false><<<grid, NT, smem, st>>>(a);
    else if (real) c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, false, true><<<grid, NT, smem, st>>>(a);
    else c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, false, false><<<grid, NT, smem, st>>>(a);
  }
  static cudaError_t prepare(size_t smem) {
    const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
    cudaError_t e = cudaFuncSetAttribute(c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, true, false>, attr, (int)smem);
    if (!e) e = cudaFuncSetAttribute(c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, false, true>, attr, (int)smem);
    if (!e) e = cudaFuncSetAttribute(c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, false, false>, attr, (int)smem);
    return e;
  }
};
template <int NY, int H, class RLY, class RLX, int NT>
struct R2CPlaneV {
  static void launch(bool, bool, const PlaneFwdArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
    r2c_plane_kernel<NY, H, RLY, RLX, NT><<<grid, NT, smem, st>>>(a);
  }
  static cudaError_t prepare(size_t smem) {
    return cudaFuncSetAttribute(r2c_plane_kernel<NY, H, RLY, RLX, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
};

template <int NT>
PlaneFwdVariant c2c64_variant() {
  using RY = Radices<8, 8>;
  using RX = Radices<8, 8>;
  PlaneFwdVariant c;
  c.r2c = false; c.ny = 64; c.nx = 64; c.ry = radix_vec<RY>(); c.rx = radix_vec<RX>(); c.threads = NT;
  c.smem = c2c_plane_smem_bytes<64, 64, RY, RX>();
  c.launch = &C2CPlaneV<64, 64, RY, RX, NT>::launch;
  c.prepare = &C2CPlaneV<64, 64, RY, RX, NT>::prepare;
  c.name = "plane64x64(8x8;8x8)_t" + std::to_string(NT);
  return c;
}
template <int NT>
PlaneFwdVariant c2c64_ip_variant() {
  using RY = Radices<8, 8>;
  using RX = Radices<8, 8>;
  PlaneFwdVariant c;
  c.r2c = false; c.ny = 64; c.nx = 64; c.ry = radix_vec<RY>(); c.rx = radix_vec<RX>(); c.threads = NT;
  c.smem = c2c_plane_ip_smem_bytes<64, 64, RX>();
  c.launch = &C2CPlaneIpV<64, 64, RY, RX, NT>::launch;
  c.prepare = &C2CPlaneIpV<64, 64, RY, RX, NT>::prepare;
  c.name = "plane64x64(8x8;8x8)_inplace_t" + std::to_string(NT);
  return c;
}
// 128 x 128 planes only fit as ONE shared buffer (139 KB, one CTA per SM): stages exchanged in place through registers
template <int NT>
PlaneFwdVariant c2c128_ip_variant() {
  using RY = Radices<16, 8>;
  using RX = Radices<16, 8>;
  PlaneFwdVariant c;
  c.r2c = false; c.ny = 128; c.nx = 128; c.ry = radix_vec<RY>(); c.rx = radix_vec<RX>(); c.threads = NT;
  c.smem = c2c_plane_ip_smem_bytes<128, 128, RX>();
  c.launch = &C2CPlaneIpV<128, 128, RY, RX, NT>::launch;
  c.prepare = &C2CPlaneIpV<128, 128, RY, RX, NT>::prepare;
  c.name = "plane128x128(16x8;16x8)_inplace_t" + std::to_string(NT);
  return c;
}
template <int NT>
PlaneFwdVariant r2c64_variant() {
  using RY = Radices<8, 8>;
  using RX = Radices<8, 4>;
  PlaneFwdVariant c;
  c.r2c = true; c.ny = 64; c.nx = 32; c.ry = radix_vec<RY>(); c.rx = radix_vec<RX>(); c.threads = NT;
  c.smem = r2c_plane_smem_bytes<64, 32, RY, RX>();
  c.launch = &R2CPlaneV<64, 32, RY, RX, NT>::launch;
  c.prepare = &R2CPlaneV<64, 32, RY, RX, NT>::prepare;
  c.name = "r2cplane64x64(8x8;2;8x4)_t" + std::to_string(NT);
  return c;
}

// order = preference; B200FFT_PLANE_PREFER=<substr> moves matching names to the front (tuning aid)
template <int NY, int H, class RLY, class RLX, int NT>
struct R2CPlaneIpV {
  static void launch(bool, bool, const PlaneFwdArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
    r2c_plane_ip_kernel<NY, H, RLY, RLX, NT><<<grid, NT, smem, st>>>(a);
  }
  static cudaError_t prepare(size_t smem) {
    return cudaFuncSetAttribute(r2c_plane_ip_kernel<NY, H, RLY, RLX, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  }
};
template <int NT, class RY>
PlaneFwdVariant r2c128_ip_variant(const char* tag) {
  using RX = Radices<8, 8>;
  PlaneFwdVariant c;
  c.r2c = true; c.ny = 128; c.nx = 64; c.ry = radix_vec<RY>(); c.rx = radix_vec<RX>(); c.threads = NT;
  c.smem = r2c_plane_ip_smem_bytes<128, 64, RX>();
  c.launch = &R2CPlaneIpV<128, 64, RY, RX, NT>::launch;
  c.prepare = &R2CPlaneIpV<128, 64, RY, RX, NT>::prepare;
  c.name = "r2cplane128x128(" + radix_name(c.ry) + ";2;8x8)_inplace_t" + std::to_string(NT) + tag;
  return c;
}

const std::vector<PlaneFwdVariant>& plane_fwd_registry() {
  static const std::vector<PlaneFwdVariant> r = [] {
    std::vector<PlaneFwdVariant> v;
    v.push_back(c2c64_variant<256>());  // 6400 x 64 x 64 C2C: t256 0.0904, t512 0.0986, t128 0.1129 ms (per-axis: 0.1188)
    v.push_back(c2c64_variant<128>());
    v.push_back(c2c64_variant<512>());
    // one shared-memory buffer, stages exchanged in place through registers (37 KB, 4-6 CTAs per SM): 0.0945 / 0.0984 ms —
    // occupancy was not the limit: ncu shows the LSU data pipe 81 % busy in the two-buffer kernel, 85 % here (r2_plane.md)
    v.push_back(c2c64_ip_variant<256>());
    v.push_back(c2c64_ip_variant<512>());
    v.push_back(c2c128_ip_variant<512>());
    v.push_back(c2c128_ip_variant<1024>());
    v.push_back(r2c128_ip_variant<512, Radices<8, 16>>(""));
    v.push_back(r2c128_ip_variant<512, Radices<16, 8>>("_y16x8"));
    v.push_back(r2c128_ip_variant<256, Radices<8, 16>>(""));
    v.push_back(r2c64_variant<256>());  // 6400 x 64 x 64 R2C: t256 0.0618, t128 0.0647, t64 0.0712 ms
    v.push_back(r2c64_variant<128>());
    v.push_back(r2c64_variant<64>());
    return v;
  }();
  return r;
}

struct PlaneFwdPass : Pass {
  const PlaneFwdVariant* v = nullptr;
  long long planes_per_batch = 1;
  bool inverse = false, real_in = false;
  float scale = 1.f;
  float2 *twy = nullptr, *twx = nullptr, *tw2 = nullptr;
  std::string text;
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    PlaneFwdArgs a;
    a.in = src;
    a.out = reinterpret_cast<float2*>(dst);
    a.twx = twx;
    a.twy = twy;
    a.tw2 = tw2;
    a.planes = nbatch * planes_per_batch;
    a.scale = scale;
    a.do_scale = inverse ? 1 : 0;
    if (a.planes <= 0) return B200FFT_OK;
    if (a.planes > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many planes");
    v->launch(inverse, real_in, a, (unsigned)a.planes, v->smem, stream);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override { return src && v->r2c ? 8 : 0; }  // R2C: real rows read as float2 pairs
};

}  // namespace

// The two innermost axes of a forward half-spectrum / complex / real-input transform as one plane pass (input -> output),
// or nullptr. `default_only`: only where it was measured to beat the alternatives (B200FFT_PLANE=1 lifts that, =0 disables).
std::unique_ptr<Pass> make_plane_fwd_pass(b200fft_plan& plan) {
  const Problem& p = plan.prob;
  if (p.rank < 2 || (p.half && p.desc.inverse)) return nullptr;
  if (p.desc.out_dtype != B200FFT_F32 || p.desc.in_dtype != B200FFT_F32) return nullptr;
  if (p.desc.flags & (B200FFT_FLAG_FORCE_GENERIC | B200FFT_FLAG_FORCE_RT | B200FFT_FLAG_NO_FUSED | B200FFT_FLAG_PREFER_FUSED)) return nullptr;
  if (const char* e = getenv("B200FFT_PLANE"))
    if (atoi(e) == 0) return nullptr;
  const int last = p.rank - 1;
  if (!p.axes[last].transformed || !p.axes[last - 1].transformed) return nullptr;
  const bool real_in = !p.half && p.desc.in_components == 1;
  if (real_in && p.desc.inverse) return nullptr;
  std::vector<const PlaneFwdVariant*> order;
  for (const PlaneFwdVariant& v : plane_fwd_registry()) order.push_back(&v);
  if (const char* pref = getenv("B200FFT_PLANE_PREFER")) {
    const std::string key(pref);
    std::stable_sort(order.begin(), order.end(), [&](const PlaneFwdVariant* a, const PlaneFwdVariant* b) {
      return (a->name.find(key) != std::string::npos) > (b->name.find(key) != std::string::npos);
    });
  }
  for (const PlaneFwdVariant* vp : order) {
    const PlaneFwdVariant& v = *vp;
    if (v.r2c != p.half || p.axes[last - 1].n != v.ny) continue;
    if (!can_group(p.axes[last - 1].ordered, v.ry)) continue;
    if (v.r2c) {
      if (p.axes[last].n != 2 * v.nx) continue;
      bool okx = false;
      for (const auto& o : drop_factor_two(p.axes[last].ordered)) okx = okx || can_group(o, v.rx);
      if (!okx) continue;
    } else if (p.axes[last].n != v.nx || !can_group(p.axes[last].ordered, v.rx)) {
      continue;
    }
    if (v.smem > 48 * 1024 && v.prepare(v.smem) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    auto pass = std::make_unique<PlaneFwdPass>();
    pass->v = &v;
    pass->inverse = p.desc.inverse != 0;
    pass->real_in = real_in;
    pass->planes_per_batch = 1;
    for (int a = 0; a < last - 1; ++a) pass->planes_per_batch *= p.axes[a].n;
    pass->scale = pass->inverse ? (float)(1.0 / ((double)v.ny * v.nx)) : 1.f;
    if (!(pass->twy = plan_upload(plan, build_twiddles(v.ry, pass->inverse))) ||
        !(pass->twx = plan_upload(plan, build_twiddles(v.rx, pass->inverse))))
      return nullptr;
    if (v.r2c && !(pass->tw2 = plan_upload(plan, build_half_twiddles(2 * v.nx, false)))) return nullptr;
    char buf[320];
    snprintf(buf, sizeof buf, "axes %d,%d: %s: one tile per (y, x) plane (x transform%s, y transform in shared memory)%s, smem=%zuB", last - 1,
             last, v.name.c_str(), v.r2c ? " of the real rows, Hermitian unpack on the fly" : "", real_in ? " real-in" : "", v.smem);
    pass->text = buf;
    return pass;
  }
  return make_jit_plane_pass(plan);  // no registered plane size: specialise one at plan time when the plane fits
}

// the two innermost axes of a half-spectrum inverse as one pass, or nullptr when no variant covers them
std::unique_ptr<Pass> make_plane_c2r_pass(b200fft_plan& plan) {
  const Problem& p = plan.prob;
  if (!p.half || !p.desc.inverse || p.rank < 2) return nullptr;
  if (p.desc.out_dtype != B200FFT_F32 || p.desc.in_dtype != B200FFT_F32) return nullptr;
  if (p.desc.flags & (B200FFT_FLAG_FORCE_GENERIC | B200FFT_FLAG_FORCE_RT | B200FFT_FLAG_NO_FUSED)) return nullptr;
  bool force = false;
  if (const char* e = getenv("B200FFT_PLANE_C2R")) {
    if (atoi(e) == 0) return nullptr;
    force = true;
  }
  const int last = p.rank - 1;
  if (!p.axes[last].transformed || !p.axes[last - 1].transformed || p.axes[last].n % 2) return nullptr;
  for (const PlaneVariant& v : plane_registry()) {
    if (p.axes[last - 1].n != v.ny || p.axes[last].n != 2 * v.h || (!v.by_default && !force)) continue;
    if (!can_group(p.axes[last - 1].ordered, v.ry)) continue;
    bool okx = false;
    for (const auto& o : drop_factor_two(p.axes[last].ordered)) okx = okx || can_group(o, v.rx);
    if (!okx) continue;
    if (v.smem > 48 * 1024 &&
        cudaFuncSetAttribute(v.func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v.smem) != cudaSuccess) {
      cudaGetLastError();
      continue;
    }
    auto pass = std::make_unique<PlaneC2RPass>();
    pass->v = &v;
    pass->planes_per_batch = 1;
    for (int a = 0; a < last - 1; ++a) pass->planes_per_batch *= p.axes[a].n;
    pass->scale = (float)(1.0 / ((double)v.ny * 2.0 * v.h));
    if (!(pass->twy = plan_upload(plan, build_twiddles(v.ry, true))) || !(pass->twx = plan_upload(plan, build_twiddles(v.rx, true))) ||
        !(pass->tw2 = plan_upload(plan, build_half_twiddles(2 * v.h, true))))
      return nullptr;
    char buf[320];
    snprintf(buf, sizeof buf, "axes %d,%d: %s: (y, x) plane of %d x %d bins -> %d x %d reals in one tile (y inverse, Hermitian pack, "
             "x inverse), smem=%zuB", last - 1, last, v.name.c_str(), v.ny, v.h + 1, v.ny, 2 * v.h, v.smem);
    pass->text = buf;
    return pass;
  }
  return nullptr;
}

}  // namespace b200fft

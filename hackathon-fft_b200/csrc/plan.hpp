// Plan = validated problem + device twiddle tables + an ordered list of kernel passes.
#pragma once
#include <cuda_runtime.h>

#include <memory>
#include <string>
#include <vector>

#include "planner.hpp"

namespace b200fft {

// The 1-D sub-transforms of one axis inside a dense row-major (batch, dims...) array:
// element (o, n, i) lives at (o*N + n)*inner + i, with outer = batch * prod(dims before
// the axis) and inner = prod(dims after it). inner == 1 is the contiguous-row case.
struct AxisView {
  int64_t outer_per_batch = 1;  // prod(dims before axis)
  int64_t n = 0;                // axis length
  int64_t inner = 1;            // prod(dims after axis) = element stride along the axis
};

// Where a pass reads from: the user's input (any dtype, real or complex) or the
// working complex buffer (out dtype).
struct IoSpec {
  int dtype = B200FFT_F32;  // scalar type
  int comps = 2;            // 1 real, 2 interleaved complex
};

// Peer scatter for the slab exchange fused into the last pass's store.
struct Scatter {
  void* const* peer_out = nullptr;  // HOST array of npeers device pointers (copied into the kernel's arguments)
  int npeers = 0;
  int my_rank = 0;
  long long zbase = -1;  // first z plane of this call inside the peers' slabs; -1 = my_rank * (planes of this call)
};

// which buffer a pass reads / writes
enum BufSel { BUF_INPUT = 0, BUF_OUTPUT = 1, BUF_WORK = 2 };

// Half-spectrum handling of the last axis (B200FFT_REAL_HALF)
enum HalfMode { HALF_NONE = 0, HALF_R2C = 1, HALF_C2R = 2 };

struct Pass {
  virtual ~Pass() {}
  // Run this pass for `nbatch` batch items. src/dst already point at the first item.
  virtual int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) = 0;
  virtual std::string describe() const = 0;
  virtual int launches() const { return 1; }
  // Byte alignment the pass's kernels need of the buffer they read (src) or write (!src). 0 = the alignment of one
  // element of that buffer, which any access needs; passes whose kernels move wider units (128-bit, TMA or bulk-async
  // copies, real rows read or written as pairs) return it. b200fft_exec refuses user pointers less aligned than the
  // maximum over the plan's passes (b200fft_plan::in_align / out_align).
  virtual size_t min_align(bool /*src*/) const { return 0; }
  // Same pass, but output row i of the transformed axis goes to sc.peer_out[i / rows_per_peer]
  // (slab exchange fused into the store). Only strided fast passes implement it.
  virtual int launch_scatter(const void*, const Scatter&, int64_t, cudaStream_t) {
    return fail(B200FFT_ERR_UNSUPPORTED, "this pass has no scattering store (%s)", describe().c_str());
  }
  // Whether launch_scatter can run, with whatever kernel it needs built now rather than on its first call.
  virtual int prepare_scatter() {
    return fail(B200FFT_ERR_UNSUPPORTED, "this pass has no scattering store (%s)", describe().c_str());
  }
  int axis = -1;
  BufSel src_sel = BUF_OUTPUT, dst_sel = BUF_OUTPUT;
  // Serpentine pass order: every second pass of a per-axis plan walks its tiles back to front, starting on the part
  // of the array the previous pass wrote last (still in L2) instead of the part it wrote first (long evicted).
  bool reverse_order = false;
  // A pass that stands for ALL axes (the fused N-d kernel) carries the per-axis passes of the same plan: they run
  // in its place when its launch is refused (cooperative launch cannot be satisfied on this context).
  std::vector<std::unique_ptr<Pass>> fallback;
};

// The longest axis the two-pass split serves (two tiles of at most 8192 points would reach 2^26; its W_n table of n
// entries is the limit). api.cu uploads that table only for axes up to this length; longer contiguous axes take the
// three-pass split (jit.cu), whose twiddles are two tables of about sqrt(n) entries.
constexpr int64_t SPLIT2_MAX_N = 1 << 24;

struct DeviceTwiddles {
  void* ptr = nullptr;  // out-dtype complex W_N^n, n in [0, N)
  int64_t n = 0;
};

}  // namespace b200fft

struct b200fft_plan {
  b200fft::Problem prob;
  int device = 0;
  int sm_count = 148;
  std::vector<b200fft::DeviceTwiddles> tw;  // one per axis (null for skipped axes)
  std::vector<std::unique_ptr<b200fft::Pass>> passes;
  std::vector<void*> owned_device;          // misc device allocations freed at destroy
  bool building_fallback = false;           // build_passes is collecting the per-axis passes behind a fused pass
  void* workspace = nullptr;
  size_t workspace_bytes = 0;
  size_t work_stride = 0;     // workspace bytes per batch item
  size_t in_align = 1, out_align = 1;  // least byte alignment of the input / output pointers the passes accept
  // strided layouts (b200fft_plan_create_strided): per-buffer element strides over (batch, dims...), the bytes each buffer
  // spans, and whether d_out == d_in maps every element onto itself (the only in-place call such a plan accepts)
  bool strided = false;
  std::vector<int64_t> in_strides, out_strides;
  size_t in_span = 0, out_span = 0;
  bool inplace_exact = false;
  // the Z pass of a half-spectrum slab inverse (scatter_z_plan_create): one pass that only runs through exec_scatter
  bool scatter_z = false;
  // exec_host resources (lazily created)
  cudaStream_t hs[3] = {nullptr, nullptr, nullptr};
  void* h_dev_in[2] = {nullptr, nullptr};
  void* h_dev_out[2] = {nullptr, nullptr};
  cudaEvent_t h_ev[8] = {};
  int64_t host_chunk = 0;
  bool host_ready = false;
};

namespace b200fft {

// Copies `t` into a new device allocation that the plan owns from before the copy (so a failed copy does not leak it).
// nullptr, with the CUDA error cleared, when the allocation or the copy fails.
template <class T>
T* plan_upload(b200fft_plan& plan, const std::vector<T>& t) {
  void* d = nullptr;
  if (cudaMalloc(&d, t.size() * sizeof(T)) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  plan.owned_device.push_back(d);
  if (cudaMemcpy(d, t.data(), t.size() * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return static_cast<T*>(d);
}

// kernel families (each returns nullptr when it does not cover the request)
// `half`: HALF_R2C = rows of n reals -> n/2+1 complex bins; HALF_C2R = the inverse (rows only).
std::unique_ptr<Pass> make_generic_pass(const b200fft_plan& plan, int axis, const AxisView& view,
                                        const IoSpec& src, bool scale_inverse, HalfMode half = HALF_NONE);
// compile-time kernels (fast_registry.cu); uploads its twiddle tables with plan_upload
std::unique_ptr<Pass> make_fast_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                     bool scale_inverse, HalfMode half = HALF_NONE);

// long axes as two passes (split_registry.cu); nullptr when no (N1, N2) pair of kernels covers the length
std::unique_ptr<Pass> make_split_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                      bool scale_inverse, HalfMode half = HALF_NONE);
// runtime-length pass with compile-time codelets (rt.cu): any stage list with radices <= 32, f32 output
std::unique_ptr<Pass> make_rt_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                   bool scale_inverse, HalfMode half = HALF_NONE);
// strided layouts (strided.cu). strided_check: validate the strides of a validated problem and record them in `plan`, no
// CUDA call (status 2 overlapping output / negative input strides, 1 offsets beyond int64, 4 a layout or axis this build does
// not serve); *dense = both layouts are the dense ones, for which b200fft_plan_create's plan is built instead.
// build_strided_passes: the passes of such a plan, one per transformed axis.
int strided_check(b200fft_plan* plan, const int64_t* in_strides, const int64_t* out_strides, bool* dense);
int build_strided_passes(b200fft_plan* plan);
// fused N-d kernel (fused_registry.cu): one pass object that replaces ALL per-axis passes, or nullptr
std::unique_ptr<Pass> make_fused_pass(b200fft_plan& plan);
// half-spectrum inverse: the two innermost axes in one tile per plane (plane_registry.cu), or nullptr
std::unique_ptr<Pass> make_plane_c2r_pass(b200fft_plan& plan);
// forward half spectrum / complex / real input: the two innermost axes in one tile per plane, or nullptr
std::unique_ptr<Pass> make_plane_fwd_pass(b200fft_plan& plan);
// ... the same for plane sizes without a registered variant, specialised at plan time (jit.cu)
std::unique_ptr<Pass> make_jit_plane_pass(b200fft_plan& plan);
// plan-time specialisation (jit.cu): the compile-time kernels instantiated through NVRTC for unregistered lengths
// *status becomes B200FFT_ERR_ALLOC when an axis it would serve cannot get its device memory (stays as given otherwise)
std::unique_ptr<Pass> make_jit_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src, bool scale_inverse,
                                    HalfMode half, int* status);
// the Z pass of a half-spectrum slab inverse with the reverse exchange in its stores (TILE_SCATTER_Z), always through NVRTC;
// nullptr with *status = B200FFT_ERR_UNSUPPORTED when the axis does not fit one column tile (B200FFT_ERR_ALLOC: no memory)
std::unique_ptr<Pass> make_jit_scatter_z_pass(b200fft_plan& plan, int axis, const AxisView& view, int* status);
int jit_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
              int in_dtype, int out_dtype, std::string* report);
// the StrLay form of that kernel, for strided layouts (same arguments; inner > 1: column tiles over `inner` columns)
int jit_probe_strided(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
                      int in_dtype, int out_dtype, std::string* report);
// the two passes the plan-time tier builds for an axis too long for one tile (same arguments)
int jit_split_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
                    int in_dtype, int out_dtype, std::string* report);
// the three passes it builds for a contiguous axis longer than SPLIT2_MAX_N points (same arguments)
int jit_split3_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
                     int in_dtype, int out_dtype, std::string* report);
// Multi-device slab plumbing (mgpu.cu).
// scatter_z_plan_create: a plan over (Z, Y/G, X/2+1) complex in the working precision, axis_mask 1, whose single pass is the
// Z pass of a half-spectrum slab inverse with the reverse exchange in its stores; b200fft_exec_scatter(plan, peer_out, G, g,
// d_in, d_in, stream) runs it, storing output z into the [Z/G][Y][X/2+1] buffer peer_out[z / (Z/G)]. Status 4 when Z does
// not fit one column tile.
int scatter_z_plan_create(b200fft_plan** out, const b200fft_desc* desc);
// Whether b200fft_exec_scatter can run `plan`, with its scattering kernel built now: status 4 when the plan's last pass
// (the split axis) is not one column tile with a scattering store.
int plan_prepare_scatter(b200fft_plan* plan);
// number of registered kernel variants per tier (host-only; triggers the one-time registration)
size_t fast_variant_count();
size_t fused_variant_count();
size_t split_variant_count();
// one line per variant for b200fft_variant_info (host-only); empty for an index past the end
std::string fast_variant_info(size_t index);
std::string fused_variant_info(size_t index);
std::string split_variant_info(size_t index);

}  // namespace b200fft

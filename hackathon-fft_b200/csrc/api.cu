// extern "C" surface of libb200fft.so (include/b200fft.h): plan construction,
// kernel selection, execution on device or host buffers.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "plan.hpp"

using namespace b200fft;

namespace {

struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = cudaSetDevice(dev) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};

// W_N^n = exp(-/+ 2*pi*i*n/N) evaluated in double, stored in the working dtype.
// (The reference forms theta in the working dtype, _utils.mojo:63-104; evaluating in
// double first is strictly more accurate, and the parity tolerance covers the
// reference's fp32-theta error, not ours.)
int upload_twiddles(int64_t n, bool inverse, bool f64, DeviceTwiddles* out) {
  const double sgn = inverse ? 1.0 : -1.0;
  void* d = nullptr;
  if (f64) {
    std::vector<double2> h((size_t)n);
    for (int64_t k = 0; k < n; ++k) {
      const double th = 2.0 * M_PI * (double)k / (double)n;
      h[(size_t)k] = make_double2(std::cos(th), sgn * std::sin(th));
    }
    B200_CUDA_CHECK(cudaMalloc(&d, sizeof(double2) * (size_t)n));
    out->ptr = d;  // owned by the plan from here on: a failed copy is freed by b200fft_plan_destroy
    B200_CUDA_CHECK(cudaMemcpy(d, h.data(), sizeof(double2) * (size_t)n, cudaMemcpyHostToDevice));
  } else {
    std::vector<float2> h((size_t)n);
    for (int64_t k = 0; k < n; ++k) {
      const double th = 2.0 * M_PI * (double)k / (double)n;
      h[(size_t)k] = make_float2((float)std::cos(th), (float)(sgn * std::sin(th)));
    }
    B200_CUDA_CHECK(cudaMalloc(&d, sizeof(float2) * (size_t)n));
    out->ptr = d;
    B200_CUDA_CHECK(cudaMemcpy(d, h.data(), sizeof(float2) * (size_t)n, cudaMemcpyHostToDevice));
  }
  out->ptr = d;
  out->n = n;
  return B200FFT_OK;
}

AxisView view_of(const Problem& p, int axis) {
  AxisView v;
  v.n = p.axes[axis].n;
  for (int a = 0; a < axis; ++a) v.outer_per_batch *= p.axes[a].n;
  for (int a = axis + 1; a < p.rank; ++a) v.inner *= p.axes[a].n;
  return v;
}

// nullptr with *status = why no kernel family serves the axis (B200FFT_ERR_UNSUPPORTED or B200FFT_ERR_ALLOC)
std::unique_ptr<Pass> make_pass(b200fft_plan* plan, int axis, const AxisView& view, const IoSpec& src, HalfMode half, int* status) {
  const Problem& p = plan->prob;
  *status = B200FFT_ERR_UNSUPPORTED;
  // an axis longer than SPLIT2_MAX_N points: only the three-pass split of the specialisation tier can serve it, so its
  // reason for refusing is the one reported (the runtime-length and generic kernels refuse any such axis)
  std::string long_why = "FORCE_GENERIC and FORCE_RT leave out the plan-time three-pass split that axes longer than 2^24 "
                         "points need";
  std::unique_ptr<Pass> pass;
  if (!(p.desc.flags & B200FFT_FLAG_FORCE_GENERIC)) {
    if (!(p.desc.flags & B200FFT_FLAG_FORCE_RT)) {
      pass = make_fast_pass(*plan, axis, view, src, p.desc.inverse != 0, half);
      if (!pass) pass = make_split_pass(*plan, axis, view, src, p.desc.inverse != 0, half);
      if (!pass) pass = make_jit_pass(*plan, axis, view, src, p.desc.inverse != 0, half, status);
      if (!pass && *status != B200FFT_ERR_UNSUPPORTED) return nullptr;
      if (!pass) long_why = last_error();
    }
    if (!pass) pass = make_rt_pass(*plan, axis, view, src, p.desc.inverse != 0, half);
  }
  if (!pass) pass = make_generic_pass(*plan, axis, view, src, p.desc.inverse != 0, half);
  if (!pass && view.n > SPLIT2_MAX_N) fail(B200FFT_ERR_UNSUPPORTED, "axis %d: %s", axis, long_why.c_str());
  return pass;
}

std::string stage_text(const Problem& p, int axis) {
  std::string radices;
  for (uint32_t r : p.axes[axis].ordered) radices += (radices.empty() ? "" : ",") + std::to_string(r);
  return radices;
}

// Kernel selection. Axes run right to left like the reference (_ndim_fft_gpu.mojo:635-642);
// the first pass reads the user's input (cast / real -> complex), the rest run in
// place on the output. `dry` builds only the description.
//
// B200FFT_REAL_HALF: forward = R2C rows pass on the last axis (input -> output), then the
// other axes as strided passes over the (.., n/2+1) half spectrum in place. Inverse = the
// other axes first (input -> workspace, in place on the workspace), then the C2R rows pass
// (workspace -> output); rank 1 needs no workspace.
int build_passes(b200fft_plan* plan, bool dry, std::string* text) {
  const Problem& p = plan->prob;
  const int last = p.rank - 1;
  const IoSpec in_spec{p.desc.in_dtype, p.desc.in_components};
  const IoSpec work_spec{p.desc.out_dtype, 2};
  auto add = [&](int axis, AxisView view, IoSpec src, HalfMode half, BufSel ssel, BufSel dsel) -> int {
    if (dry) {
      char buf[256];
      snprintf(buf, sizeof buf, "axis %d: n=%lld inner=%lld stages=[%s]%s%s\n", axis, (long long)view.n,
               (long long)view.inner, stage_text(p, axis).c_str(),
               half == HALF_R2C ? " r2c" : half == HALF_C2R ? " c2r" : "",
               ssel == BUF_INPUT ? " (reads input)" : " (in place)");
      *text += buf;
      return B200FFT_OK;
    }
    int status;
    std::unique_ptr<Pass> pass = make_pass(plan, axis, view, src, half, &status);
    if (!pass) return status;
    pass->src_sel = ssel;
    pass->dst_sel = dsel;
    pass->axis = axis;
    {  // B200FFT_SERPENTINE=0 switches the alternating tile order off (A/B knob; profiles/r2_serpentine.md)
      const char* e = getenv("B200FFT_SERPENTINE");
      pass->reverse_order = !(e && atoi(e) == 0) && (plan->passes.size() % 2 == 1);
    }
    plan->passes.push_back(std::move(pass));
    return B200FFT_OK;
  };

  // Forward half spectrum / complex / real input: the two innermost axes as ONE plane pass where a plane kernel covers them
  // (plane_registry.cu), strided passes for the outer axes. It ties the fused persistent kernel on 100 x 64^3 (0.147 vs
  // 0.149 ms C2C, 0.090 vs 0.092 ms R2C; profiles/r2_plane.md) with two plain launches — no cooperative grid, no
  // dependency spinning — so it goes first; B200FFT_FUSED=1, B200FFT_FUSED_PREFER, the PREFER_FUSED flag or B200FFT_PLANE=0
  // put the fused kernel back in front.
  std::unique_ptr<Pass> plane;
  if (!dry && !(p.half && p.desc.inverse)) {
    bool fused_wanted = (p.desc.flags & B200FFT_FLAG_PREFER_FUSED) != 0 || getenv("B200FFT_FUSED_PREFER") != nullptr;
    if (const char* e = getenv("B200FFT_FUSED")) fused_wanted = fused_wanted || atoi(e) != 0;
    if (!fused_wanted || plan->building_fallback) plane = make_plane_fwd_pass(*plan);
  }

  // one persistent kernel for all axes when a fused variant covers the problem (fused_registry.cu); the other passes
  // are still built and kept behind it as its fallback (a refused cooperative launch)
  if (!dry && !plan->building_fallback && !plane) {
    std::unique_ptr<Pass> fused = make_fused_pass(*plan);
    if (fused) {
      plan->building_fallback = true;
      const int rc = build_passes(plan, false, nullptr);
      plan->building_fallback = false;
      if (rc == B200FFT_OK) fused->fallback = std::move(plan->passes);
      plan->passes.clear();
      plan->passes.push_back(std::move(fused));
      return B200FFT_OK;
    }
  }

  if (plane) {
    plane->src_sel = BUF_INPUT;
    plane->dst_sel = BUF_OUTPUT;
    plane->axis = last;
    plan->passes.push_back(std::move(plane));
    const int64_t hb2 = p.axes[last].n / 2 + 1;
    for (int axis = last - 2; axis >= 0; --axis) {
      if (!p.axes[axis].transformed) continue;
      AxisView v = view_of(p, axis);
      if (p.half) {  // strided passes see the last axis as n/2+1 bins
        v.inner = hb2;
        for (int a = axis + 1; a < last; ++a) v.inner *= p.axes[a].n;
      }
      int rc = add(axis, v, work_spec, HALF_NONE, BUF_OUTPUT, BUF_OUTPUT);
      if (rc) return rc;
    }
    return B200FFT_OK;
  }

  if (!p.half) {
    bool first = true;
    for (int axis = last; axis >= 0; --axis) {
      if (!p.axes[axis].transformed) continue;
      int rc = add(axis, view_of(p, axis), first ? in_spec : work_spec, HALF_NONE, first ? BUF_INPUT : BUF_OUTPUT,
                   BUF_OUTPUT);
      if (rc) return rc;
      first = false;
    }
    return B200FFT_OK;
  }

  // ---- half spectrum: strided passes see the last axis as n/2+1 complex bins
  const int64_t hb = p.axes[last].n / 2 + 1;
  auto half_view = [&](int axis) {
    AxisView v;
    v.n = p.axes[axis].n;
    for (int a = 0; a < axis; ++a) v.outer_per_batch *= p.axes[a].n;
    for (int a = axis + 1; a < last; ++a) v.inner *= p.axes[a].n;
    v.inner *= hb;
    return v;
  };
  AxisView rows = view_of(p, last);  // outer_per_batch = prod(dims[:-1]), n = real length
  if (!p.desc.inverse) {
    int rc = add(last, rows, in_spec, HALF_R2C, BUF_INPUT, BUF_OUTPUT);
    if (rc) return rc;
    for (int axis = last - 1; axis >= 0; --axis) {
      if (!p.axes[axis].transformed) continue;
      if ((rc = add(axis, half_view(axis), work_spec, HALF_NONE, BUF_OUTPUT, BUF_OUTPUT))) return rc;
    }
    return B200FFT_OK;
  }
  // the two innermost axes in one tile per (y, x) plane when a plane kernel covers them (plane_registry.cu): the outer
  // axes' strided passes first (input -> workspace), then the plane pass (-> output)
  std::unique_ptr<Pass> plane_inv = dry ? nullptr : make_plane_c2r_pass(*plan);
  const int first_cols_axis = plane_inv ? last - 2 : last - 1;
  bool any = false;
  for (int axis = first_cols_axis; axis >= 0; --axis) {
    if (!p.axes[axis].transformed) continue;
    int rc = add(axis, half_view(axis), any ? work_spec : in_spec, HALF_NONE, any ? BUF_WORK : BUF_INPUT, BUF_WORK);
    if (rc) return rc;
    any = true;
  }
  if (any && !dry) {
    plan->work_stride = (size_t)(rows.outer_per_batch * hb) * 2 * p.out_elem;
    plan->workspace_bytes = plan->work_stride * (size_t)p.batch;
    if (cudaMalloc(&plan->workspace, plan->workspace_bytes) != cudaSuccess) {
      cudaGetLastError();
      return fail(B200FFT_ERR_ALLOC, "cannot allocate %zu B of C2R workspace", plan->workspace_bytes);
    }
  }
  if (plane_inv) {
    plane_inv->src_sel = any ? BUF_WORK : BUF_INPUT;
    plane_inv->dst_sel = BUF_OUTPUT;
    plane_inv->axis = last;
    plan->passes.push_back(std::move(plane_inv));
    return B200FFT_OK;
  }
  return add(last, rows, any ? work_spec : in_spec, HALF_C2R, any ? BUF_WORK : BUF_INPUT, BUF_OUTPUT);
}

// the one pass of a scatter_z_plan_create plan: axis 0 of the user's input, stored into the peers' buffers
int build_scatter_z_pass(b200fft_plan* plan) {
  int status;
  std::unique_ptr<Pass> pass = make_jit_scatter_z_pass(*plan, 0, view_of(plan->prob, 0), &status);
  if (!pass) return status;
  pass->src_sel = BUF_INPUT;
  pass->dst_sel = BUF_OUTPUT;
  pass->axis = 0;
  plan->passes.push_back(std::move(pass));
  return B200FFT_OK;
}

// The alignment b200fft_exec requires of the input and output pointers: one element of each buffer, raised to what the
// kernels of every pass that touches it need (Pass::min_align), fallback passes included.
void record_alignment(b200fft_plan* plan) {
  const Problem& p = plan->prob;
  const bool real_out = p.half && p.desc.inverse;
  plan->in_align = p.in_elem * (p.desc.in_components == 2 ? 2 : 1);
  plan->out_align = p.out_elem * (real_out ? 1 : 2);
  auto user_buffer = [&](BufSel sel) -> size_t* {  // the plan-owned workspace is cudaMalloc'ed: no requirement to record
    return sel == BUF_INPUT ? &plan->in_align : sel == BUF_OUTPUT ? &plan->out_align : nullptr;
  };
  auto visit = [&](const Pass& pass, auto& self) -> void {
    if (size_t* a = user_buffer(pass.src_sel)) *a = std::max(*a, pass.min_align(true));
    if (size_t* a = user_buffer(pass.dst_sel)) *a = std::max(*a, pass.min_align(false));
    for (const auto& f : pass.fallback) self(*f, self);
  };
  for (const auto& pass : plan->passes) visit(*pass, visit);
}

int check_alignment(const b200fft_plan* plan, const void* in, const char* in_name, const void* out, const char* out_name) {
  if ((uintptr_t)in % plan->in_align)
    return fail(B200FFT_ERR_INVALID_ARG, "%s %p is not aligned to %zu bytes, which this plan's kernels need", in_name, in,
                plan->in_align);
  if ((uintptr_t)out % plan->out_align)
    return fail(B200FFT_ERR_INVALID_ARG, "%s %p is not aligned to %zu bytes, which this plan's kernels need", out_name, out,
                plan->out_align);
  return B200FFT_OK;
}

int copy_bases(const std::vector<uint32_t>& v, uint32_t* out, int cap) {
  if (!out || (int)v.size() > cap) return -1;
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  return (int)v.size();
}

}  // namespace

extern "C" {

int b200fft_version(void) { return 100; }

uint64_t b200fft_launch_count(void) { return g_launch_count.load(); }

int b200fft_variant_count(int tier) {
  switch (tier) {
    case 0: return (int)fast_variant_count();
    case 1: return (int)fused_variant_count();
    case 2: return (int)split_variant_count();
    default: return -1;
  }
}

int b200fft_variant_info(int tier, int index, char* buf, size_t cap) {
  if (index < 0) return -1;
  std::string line;
  switch (tier) {
    case 0: line = fast_variant_info((size_t)index); break;
    case 1: line = fused_variant_info((size_t)index); break;
    case 2: line = split_variant_info((size_t)index); break;
    default: return -1;
  }
  if (line.empty()) return -1;
  if (buf && cap) {
    strncpy(buf, line.c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  return (int)line.size() + 1;
}

const char* b200fft_last_error(void) { return last_error().c_str(); }

const char* b200fft_strerror(int status) {
  switch (status) {
    case B200FFT_OK: return "ok";
    case B200FFT_ERR_INVALID_ARG: return "invalid argument";
    case B200FFT_ERR_LAYOUT: return "layout violates the reference's layout conditions";
    case B200FFT_ERR_BASES: return "bases do not factor the axis length";
    case B200FFT_ERR_UNSUPPORTED: return "valid for the reference but not supported by this build";
    case B200FFT_ERR_CUDA: return "CUDA error";
    case B200FFT_ERR_ALLOC: return "allocation failed";
    default: return "unknown status";
  }
}

int b200fft_ordered_bases(uint64_t length, const uint32_t* bases, int nbases, uint32_t* out, int cap) {
  if (!bases || nbases <= 0) return -1;
  std::vector<uint32_t> user(bases, bases + nbases);
  for (uint32_t b : user)
    if (b < 2) return -1;
  std::vector<uint32_t> o = build_ordered_bases(length, user);
  if (!ordered_bases_valid(length, o)) return -1;
  return copy_bases(o, out, cap);
}

int b200fft_default_bases(uint64_t length, int gpu_target, uint32_t* out, int cap) {
  return copy_bases(estimate_best_bases(length, gpu_target != 0), out, cap);
}

}  // extern "C"

namespace {
// b200fft_jit_probe / b200fft_jit_split_probe / b200fft_jit_split3_probe: validate, order the bases, run the host-only probe
using ProbeFn = int (*)(int64_t, int64_t, const std::vector<uint32_t>&, bool, bool, int, int, int, std::string*);
int probe_entry(ProbeFn probe, int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in, int half,
                int in_dtype, int out_dtype, char* buf, size_t cap, int max_half = 2) {
  if (in_dtype < B200FFT_U8 || in_dtype > B200FFT_F64 || (out_dtype != B200FFT_F32 && out_dtype != B200FFT_F64))
    return fail(B200FFT_ERR_INVALID_ARG, "dtypes %d -> %d", in_dtype, out_dtype);
  if (half < 0 || half > max_half)  // 3, the scattering Z pass of a half-spectrum slab inverse: b200fft_jit_probe only
    return fail(B200FFT_ERR_INVALID_ARG, "half = %d (0 complex, 1 R2C, 2 C2R%s)", half, max_half > 2 ? ", 3 slab Z scatter" : "");
  if (n < 2 || inner < 1) return fail(B200FFT_ERR_INVALID_ARG, "axis length %lld, inner %lld", (long long)n, (long long)inner);
  std::vector<uint32_t> ordered;
  if (bases && nbases > 0) {
    ordered = build_ordered_bases((uint64_t)n, std::vector<uint32_t>(bases, bases + nbases));
  } else {
    ordered = build_ordered_bases((uint64_t)n, estimate_best_bases((uint64_t)n, true));
  }
  if (!ordered_bases_valid((uint64_t)n, ordered)) return fail(B200FFT_ERR_BASES, "bases do not factor %lld", (long long)n);
  std::string report;
  const int rc = probe(n, inner, ordered, inverse != 0, real_in != 0, half, in_dtype, out_dtype, &report);
  if (rc != B200FFT_OK) return rc;
  if (buf && cap) {
    strncpy(buf, report.c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  return B200FFT_OK;
}
}  // namespace

extern "C" {

int b200fft_jit_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in, int half,
                      int in_dtype, int out_dtype, char* buf, size_t cap) {
  return probe_entry(jit_probe, n, inner, bases, nbases, inverse, real_in, half, in_dtype, out_dtype, buf, cap, 3);
}

int b200fft_jit_probe_strided(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in, int half,
                              int in_dtype, int out_dtype, char* buf, size_t cap) {
  return probe_entry(jit_probe_strided, n, inner, bases, nbases, inverse, real_in, half, in_dtype, out_dtype, buf, cap);
}

int b200fft_jit_split_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in, int half,
                            int in_dtype, int out_dtype, char* buf, size_t cap) {
  return probe_entry(jit_split_probe, n, inner, bases, nbases, inverse, real_in, half, in_dtype, out_dtype, buf, cap);
}

int b200fft_jit_split3_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in, int half,
                             int in_dtype, int out_dtype, char* buf, size_t cap) {
  return probe_entry(jit_split3_probe, n, inner, bases, nbases, inverse, real_in, half, in_dtype, out_dtype, buf, cap);
}

int b200fft_schedule_dry_run(int nphases, const int64_t* phases, int64_t batch, int64_t* segments, int cap) {
  if (nphases < 1 || nphases > 8 || !phases || batch < 0) return -1;
  std::vector<SchedPhase> ph((size_t)nphases);
  for (int p = 0; p < nphases; ++p) {
    ph[p].tiles_per_transform = phases[4 * p];
    ph[p].tiles_per_group = phases[4 * p + 1];
    ph[p].dep_div = phases[4 * p + 2];
    ph[p].quota = phases[4 * p + 3];
    if (ph[p].tiles_per_transform < 1 || ph[p].tiles_per_group < 1 || ph[p].dep_div < 1) return -1;
  }
  const std::vector<NdSegment> segs = build_schedule(nphases, ph.data(), batch);
  if (segments)
    for (size_t i = 0; i < segs.size() && (int)i < cap; ++i) {
      segments[4 * i] = segs[i].phase;
      segments[4 * i + 1] = segs[i].first_item;
      segments[4 * i + 2] = segs[i].first_tile;
      segments[4 * i + 3] = segs[i].count;
    }
  return (int)segs.size();
}

int b200fft_plan_dry_run(const b200fft_desc* desc, char* buf, size_t cap) {
  b200fft_plan tmp;
  int rc = validate(desc, &tmp.prob);
  if (rc != B200FFT_OK) return rc;
  std::string text;
  rc = build_passes(&tmp, /*dry=*/true, &text);
  if (rc != B200FFT_OK) return rc;
  if (buf && cap) {
    strncpy(buf, text.c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  return B200FFT_OK;
}

}  // extern "C"

// the device part of plan creation: twiddle tables (dense plans), passes, alignment; *out only on success
static int finish_plan(std::unique_ptr<b200fft_plan> plan, const b200fft_desc* desc, b200fft_plan** out) {
  int rc;
  int dev = desc->device;
  if (dev < 0) B200_CUDA_CHECK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  B200_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10)
    return fail(B200FFT_ERR_CUDA, "device %d is sm_%d%d; this library only carries sm_100a code (no fallback)", dev,
                prop.major, prop.minor);
  plan->device = dev;
  plan->sm_count = prop.multiProcessorCount;
  DeviceGuard guard(dev);

  const bool f64 = desc->out_dtype == B200FFT_F64;
  plan->tw.resize(plan->prob.rank);
  for (int a = 0; a < plan->prob.rank; ++a) {
    // the n-entry W_n table serves passes of at most SPLIT2_MAX_N points; a longer axis has twiddle tables of its own, and
    // the single-tile passes of a strided plan upload their own stage tables
    if (plan->strided || plan->scatter_z || !plan->prob.axes[a].transformed || plan->prob.axes[a].n > SPLIT2_MAX_N) continue;
    rc = upload_twiddles(plan->prob.axes[a].n, desc->inverse != 0, f64, &plan->tw[a]);
    if (rc != B200FFT_OK) { b200fft_plan_destroy(plan.release()); return rc; }
  }
  rc = plan->strided     ? build_strided_passes(plan.get())
       : plan->scatter_z ? build_scatter_z_pass(plan.get())
                         : build_passes(plan.get(), /*dry=*/false, nullptr);
  if (rc != B200FFT_OK) { b200fft_plan_destroy(plan.release()); return rc; }
  record_alignment(plan.get());
  // The tables were uploaded with cudaMemcpy from pageable memory on the legacy stream: make sure they have landed
  // before the caller launches on a non-blocking stream of its own (which is not ordered after the legacy stream).
  if (cudaError_t e = cudaDeviceSynchronize(); e != cudaSuccess) {
    b200fft_plan_destroy(plan.release());
    return fail(B200FFT_ERR_CUDA, "plan upload: %s", cudaGetErrorString(e));
  }
  *out = plan.release();
  return B200FFT_OK;
}

int b200fft::scatter_z_plan_create(b200fft_plan** out, const b200fft_desc* desc) {
  if (!out) return fail(B200FFT_ERR_INVALID_ARG, "null plan pointer");
  *out = nullptr;
  std::unique_ptr<b200fft_plan> plan(new b200fft_plan());
  int rc = validate(desc, &plan->prob);
  if (rc != B200FFT_OK) return rc;
  if (plan->prob.half || plan->prob.batch != 1 || plan->prob.rank < 2 || desc->axis_mask != 1)
    return fail(B200FFT_ERR_INVALID_ARG, "the scattering Z pass takes one complex volume, axis 0 only");
  plan->scatter_z = true;
  return finish_plan(std::move(plan), desc, out);
}

int b200fft::plan_prepare_scatter(b200fft_plan* plan) {
  if (plan->passes.empty() || plan->passes.back()->axis != 0)
    return fail(B200FFT_ERR_UNSUPPORTED, "the last pass of the plan does not transform the split axis 0");
  return plan->passes.back()->prepare_scatter();
}

extern "C" {

int b200fft_plan_create(b200fft_plan** out, const b200fft_desc* desc) {
  if (!out) return fail(B200FFT_ERR_INVALID_ARG, "null plan pointer");
  *out = nullptr;
  std::unique_ptr<b200fft_plan> plan(new b200fft_plan());
  int rc = validate(desc, &plan->prob);
  if (rc != B200FFT_OK) return rc;
  return finish_plan(std::move(plan), desc, out);
}

int b200fft_plan_create_strided(b200fft_plan** out, const b200fft_desc* desc, const int64_t* in_strides, const int64_t* out_strides) {
  if (!out) return fail(B200FFT_ERR_INVALID_ARG, "null plan pointer");
  *out = nullptr;
  std::unique_ptr<b200fft_plan> plan(new b200fft_plan());
  int rc = validate(desc, &plan->prob);
  if (rc != B200FFT_OK) return rc;
  bool dense = false;
  if ((rc = strided_check(plan.get(), in_strides, out_strides, &dense)) != B200FFT_OK) return rc;
  if (dense) return b200fft_plan_create(out, desc);
  return finish_plan(std::move(plan), desc, out);
}

int b200fft_plan_destroy(b200fft_plan* plan) {
  if (!plan) return B200FFT_OK;
  DeviceGuard guard(plan->device);
  for (auto& t : plan->tw)
    if (t.ptr) cudaFree(t.ptr);
  for (void* p : plan->owned_device)
    if (p) cudaFree(p);
  if (plan->workspace) cudaFree(plan->workspace);
  for (int i = 0; i < 2; ++i) {
    if (plan->h_dev_in[i]) cudaFree(plan->h_dev_in[i]);
    if (plan->h_dev_out[i]) cudaFree(plan->h_dev_out[i]);
  }
  for (int i = 0; i < 3; ++i)
    if (plan->hs[i]) cudaStreamDestroy(plan->hs[i]);
  for (auto& e : plan->h_ev)
    if (e) cudaEventDestroy(e);
  delete plan;
  return B200FFT_OK;
}

// work_batch0: first batch item of this call inside the plan-wide workspace (exec_host chunks)
static int run_passes(b200fft_plan* plan, void* d_out, const void* d_in, int64_t nbatch, cudaStream_t st,
                      int64_t work_batch0 = 0) {
  char* work = (char*)plan->workspace + (size_t)work_batch0 * plan->work_stride;
  for (auto& pass : plan->passes) {
    const void* src = pass->src_sel == BUF_INPUT ? d_in : pass->src_sel == BUF_WORK ? (const void*)work : (const void*)d_out;
    void* dst = pass->dst_sel == BUF_WORK ? (void*)work : d_out;
    int rc = pass->launch(src, dst, nbatch, st);
    if (rc != B200FFT_OK) return rc;
  }
  return B200FFT_OK;
}

int b200fft_exec(b200fft_plan* plan, void* d_out, const void* d_in, void* cu_stream) {
  if (!plan || !d_out || !d_in) return fail(B200FFT_ERR_INVALID_ARG, "null plan or buffer");
  if (int rc = check_alignment(plan, d_in, "d_in", d_out, "d_out")) return rc;
  if (plan->strided && d_out == d_in && !plan->inplace_exact)
    return fail(B200FFT_ERR_INVALID_ARG, "this strided plan cannot run in place: its input and output layouts do not map every "
                                         "element onto itself (equal strides and element types, or the padded real layout of "
                                         "twice the complex strides)");
  DeviceGuard guard(plan->device);
  return run_passes(plan, d_out, d_in, plan->prob.batch, (cudaStream_t)cu_stream);
}

static int exec_scatter_impl(b200fft_plan* plan, void* const* peer_out, int npeers, int my_rank, long long zbase, const void* d_in,
                             void* d_work, void* cu_stream) {
  if (!plan || !peer_out || !d_in || !d_work) return fail(B200FFT_ERR_INVALID_ARG, "null plan or buffer");
  if (plan->prob.half && plan->prob.desc.inverse)
    return fail(B200FFT_ERR_UNSUPPORTED, "exec_scatter takes complex or forward half-spectrum (R2C) plans; this one is C2R");
  if (plan->prob.half && d_work == d_in)
    return fail(B200FFT_ERR_INVALID_ARG, "exec_scatter of an R2C plan: d_work holds the half spectrum and cannot be the real "
                                         "input d_in");
  if (plan->strided) return fail(B200FFT_ERR_UNSUPPORTED, "exec_scatter takes dense layouts; this plan is strided");
  if (my_rank < 0 || my_rank >= npeers) return fail(B200FFT_ERR_INVALID_ARG, "my_rank %d outside 0..%d", my_rank, npeers);
  if (plan->passes.empty() || plan->passes.back()->axis != 0)
    return fail(B200FFT_ERR_INVALID_ARG, "exec_scatter: the plan's last pass must transform axis 0 (the split axis); "
                                         "create the plan with B200FFT_FLAG_NO_FUSED");
  if (int rc = check_alignment(plan, d_in, "d_in", d_work, "d_work")) return rc;
  for (int i = 0; i < npeers && i < 16; ++i)
    if (!peer_out[i] || (uintptr_t)peer_out[i] % plan->out_align)
      return fail(B200FFT_ERR_INVALID_ARG, "peer_out[%d] %p is null or not aligned to %zu bytes", i, peer_out[i], plan->out_align);
  DeviceGuard guard(plan->device);
  cudaStream_t st = (cudaStream_t)cu_stream;
  const size_t n = plan->passes.size();
  for (size_t i = 0; i + 1 < n; ++i) {
    Pass& pass = *plan->passes[i];
    int rc = pass.launch(pass.src_sel == BUF_INPUT ? d_in : (const void*)d_work, d_work, plan->prob.batch, st);
    if (rc != B200FFT_OK) return rc;
  }
  Pass& last = *plan->passes.back();
  Scatter sc;
  sc.peer_out = peer_out;
  sc.npeers = npeers;
  sc.my_rank = my_rank;
  sc.zbase = zbase;
  // a one-pass plan (only the split axis transformed) scatters straight from d_in
  return last.launch_scatter(n == 1 || last.src_sel == BUF_INPUT ? d_in : (const void*)d_work, sc, plan->prob.batch, st);
}

int b200fft_exec_scatter(b200fft_plan* plan, void* const* peer_out, int npeers, int my_rank, const void* d_in,
                         void* d_work, void* cu_stream) {
  return exec_scatter_impl(plan, peer_out, npeers, my_rank, -1, d_in, d_work, cu_stream);
}

int b200fft_exec_scatter_at(b200fft_plan* plan, void* const* peer_out, int npeers, int64_t z_first, const void* d_in,
                            void* d_work, void* cu_stream) {
  if (z_first < 0) return fail(B200FFT_ERR_INVALID_ARG, "negative plane offset");
  return exec_scatter_impl(plan, peer_out, npeers, 0, (long long)z_first, d_in, d_work, cu_stream);
}

int b200fft_stream_synchronize(void* cu_stream) {
  B200_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)cu_stream));
  return B200FFT_OK;
}

int b200fft_host_register(void* h_ptr, size_t bytes) {
  if (!h_ptr || !bytes) return fail(B200FFT_ERR_INVALID_ARG, "null host range");
  B200_CUDA_CHECK(cudaHostRegister(h_ptr, bytes, cudaHostRegisterPortable));
  return B200FFT_OK;
}
int b200fft_host_unregister(void* h_ptr) {
  B200_CUDA_CHECK(cudaHostUnregister(h_ptr));
  return B200FFT_OK;
}

int b200fft_malloc(void** d_ptr, size_t bytes) {
  if (!d_ptr) return fail(B200FFT_ERR_INVALID_ARG, "null pointer");
  B200_CUDA_CHECK(cudaMalloc(d_ptr, bytes));
  return B200FFT_OK;
}
int b200fft_free(void* d_ptr) {
  B200_CUDA_CHECK(cudaFree(d_ptr));
  return B200FFT_OK;
}
int b200fft_ipc_export(void* d_ptr, unsigned char handle[B200FFT_IPC_HANDLE_BYTES]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == B200FFT_IPC_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  B200_CUDA_CHECK(cudaIpcGetMemHandle(&h, d_ptr));
  memcpy(handle, &h, sizeof h);
  return B200FFT_OK;
}
int b200fft_ipc_open(const unsigned char handle[B200FFT_IPC_HANDLE_BYTES], void** d_ptr) {
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  B200_CUDA_CHECK(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return B200FFT_OK;
}
int b200fft_ipc_close(void* d_ptr) {
  B200_CUDA_CHECK(cudaIpcCloseMemHandle(d_ptr));
  return B200FFT_OK;
}

// Host-buffer execution: the batch is cut into chunks that flow through
// H2D (stream 0) -> kernels (stream 1) -> D2H (stream 2) with two device buffers
// per direction, so PCIe transfers in both directions overlap the kernels.
int b200fft_exec_host(b200fft_plan* plan, void* h_out, const void* h_in) {
  if (!plan || !h_out || !h_in) return fail(B200FFT_ERR_INVALID_ARG, "null plan or buffer");
  if (plan->strided) return fail(B200FFT_ERR_UNSUPPORTED, "exec_host takes dense layouts; this plan is strided");
  DeviceGuard guard(plan->device);
  const Problem& p = plan->prob;
  const size_t in_stride = (size_t)p.in_scalars_per_batch * p.in_elem;
  const size_t out_stride = (size_t)p.out_scalars_per_batch * p.out_elem;
  if (!plan->host_ready) {
    // chunks of ~24 MiB (fill / drain of the 3-stage pipeline costs one chunk each way), at least 4 and
    // at most 64 of them, at least 1 batch item each
    const size_t per = std::max(in_stride, out_stride);
    size_t chunk_mb = 24;  // B200FFT_HOST_CHUNK_MB: tuning knob (profiles/r1_e2e.md)
    if (const char* e = getenv("B200FFT_HOST_CHUNK_MB")) chunk_mb = (size_t)std::max(1, atoi(e));
    int64_t nchunks = (int64_t)(((size_t)p.batch * per + (chunk_mb << 20) - 1) / (chunk_mb << 20));
    nchunks = std::min<int64_t>(64, std::max<int64_t>(4, nchunks));
    int64_t chunk = std::max<int64_t>(1, (p.batch + nchunks - 1) / nchunks);
    plan->host_chunk = chunk;
    // each resource is created only while still null, so a call that failed half way through can be retried
    // without leaking what it had already made (b200fft_plan_destroy frees whatever exists)
    for (int i = 0; i < 3; ++i)
      if (!plan->hs[i]) B200_CUDA_CHECK(cudaStreamCreateWithFlags(&plan->hs[i], cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      if (!plan->h_dev_in[i]) B200_CUDA_CHECK(cudaMalloc(&plan->h_dev_in[i], (size_t)chunk * in_stride));
      if (!plan->h_dev_out[i]) B200_CUDA_CHECK(cudaMalloc(&plan->h_dev_out[i], (size_t)chunk * out_stride));
    }
    for (auto& e : plan->h_ev)
      if (!e) B200_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    plan->host_ready = true;
  }
  cudaEvent_t* ev_in = &plan->h_ev[0];    // [2] H2D done
  cudaEvent_t* ev_k = &plan->h_ev[2];     // [2] kernels done
  cudaEvent_t* ev_out = &plan->h_ev[4];   // [2] D2H done
  const int64_t chunk = plan->host_chunk;
  auto pipeline = [&]() -> int {
    int64_t k = 0;
    for (int64_t b0 = 0; b0 < p.batch; b0 += chunk, ++k) {
      const int slot = (int)(k & 1);
      const int64_t nb = std::min<int64_t>(chunk, p.batch - b0);
      if (k >= 2) B200_CUDA_CHECK(cudaStreamWaitEvent(plan->hs[0], ev_k[slot], 0));  // input slot consumed
      B200_CUDA_CHECK(cudaMemcpyAsync(plan->h_dev_in[slot], (const char*)h_in + (size_t)b0 * in_stride,
                                      (size_t)nb * in_stride, cudaMemcpyHostToDevice, plan->hs[0]));
      B200_CUDA_CHECK(cudaEventRecord(ev_in[slot], plan->hs[0]));
      B200_CUDA_CHECK(cudaStreamWaitEvent(plan->hs[1], ev_in[slot], 0));
      if (k >= 2) B200_CUDA_CHECK(cudaStreamWaitEvent(plan->hs[1], ev_out[slot], 0));  // output slot drained
      int rc = run_passes(plan, plan->h_dev_out[slot], plan->h_dev_in[slot], nb, plan->hs[1], b0);
      if (rc != B200FFT_OK) return rc;
      B200_CUDA_CHECK(cudaEventRecord(ev_k[slot], plan->hs[1]));
      B200_CUDA_CHECK(cudaStreamWaitEvent(plan->hs[2], ev_k[slot], 0));
      B200_CUDA_CHECK(cudaMemcpyAsync((char*)h_out + (size_t)b0 * out_stride, plan->h_dev_out[slot],
                                      (size_t)nb * out_stride, cudaMemcpyDeviceToHost, plan->hs[2]));
      B200_CUDA_CHECK(cudaEventRecord(ev_out[slot], plan->hs[2]));
    }
    B200_CUDA_CHECK(cudaStreamSynchronize(plan->hs[2]));
    return B200FFT_OK;
  };
  const int rc = pipeline();
  if (rc != B200FFT_OK)  // the caller may free its host buffers once we return: no copy may still be in flight
    for (int i = 0; i < 3; ++i) cudaStreamSynchronize(plan->hs[i]);
  return rc;
}

size_t b200fft_plan_workspace_bytes(const b200fft_plan* plan) { return plan ? plan->workspace_bytes : 0; }

int b200fft_plan_get_bases(const b200fft_plan* plan, int axis, uint32_t* out, int cap) {
  if (!plan || axis < 0 || axis >= plan->prob.rank) return -1;
  return copy_bases(plan->prob.axes[axis].ordered, out, cap);
}

size_t b200fft_plan_describe(const b200fft_plan* plan, char* buf, size_t cap) {
  if (!plan) return 0;
  std::string text;
  for (auto& pass : plan->passes) text += pass->describe() + "\n";
  if (buf && cap) {
    strncpy(buf, text.c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  return text.size() + 1;
}

int b200fft_plan_launches(const b200fft_plan* plan) {
  if (!plan) return 0;
  int n = 0;
  for (auto& pass : plan->passes) n += pass->launches();
  return n;
}

size_t b200fft_plan_in_bytes(const b200fft_plan* plan) {
  if (plan && plan->strided) return plan->in_span;
  return plan ? (size_t)plan->prob.batch * plan->prob.in_scalars_per_batch * plan->prob.in_elem : 0;
}
size_t b200fft_plan_out_bytes(const b200fft_plan* plan) {
  if (plan && plan->strided) return plan->out_span;
  return plan ? (size_t)plan->prob.batch * plan->prob.out_scalars_per_batch * plan->prob.out_elem : 0;
}

}  // extern "C"

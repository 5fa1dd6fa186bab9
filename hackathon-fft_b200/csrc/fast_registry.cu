// Registry of compile-time kernel variants (fast.cuh) and the passes that launch them.
//
// A variant is (axis length N, super-stage list, tile size, threads). The planner picks, for
// an axis, the first registered variant whose super-stages can be formed by grouping the
// axis's ordered base list (the reference's stage list, _utils.mojo:163-221): e.g. user
// bases [2] on 128 -> stages [2]x7 -> fused as (16)(8). Bases that cannot be grouped into any
// registered variant (say [32,4] with only (16,8) registered) run on the generic kernel.
// B200FFT_PREFER="substr[,substr...]" moves matching variant names to the front (tuning aid).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include <cudaTypedefs.h>

#include "fast_registry.hpp"
#include "plan.hpp"

namespace b200fft {

std::vector<Variant>& registry() {
  static std::vector<Variant> r;
  return r;
}
void register_rows_pow2();
void register_rows_mixed();
void register_cols_pow2();
void register_cols_mixed();
void register_cols_tma();

namespace {

void register_all() {
  // function-local static: initialised exactly once even when two threads create their first plans concurrently
  // (include/b200fft.h promises that distinct plans may be used from distinct threads)
  static const bool done = [] {
    register_rows_pow2();
    register_rows_mixed();
    register_cols_pow2();
    register_cols_mixed();
    register_cols_tma();
    return true;
  }();
  (void)done;
}

}  // namespace

// can `target` (super-stage radices) be formed by partitioning `ordered` (the user's stage
// list) into groups with exactly those products?
bool can_group(std::vector<uint32_t> ordered, std::vector<int> target) {
  if (target.empty()) return ordered.empty();
  const int want = target.back();
  target.pop_back();
  // choose a sub-multiset of `ordered` with product `want`
  const size_t n = ordered.size();
  if (n > 24) return false;
  std::function<bool(size_t, int, std::vector<uint32_t>&)> rec = [&](size_t i, int prod, std::vector<uint32_t>& rest) {
    if (prod == want) {
      std::vector<uint32_t> remaining(rest);
      remaining.insert(remaining.end(), ordered.begin() + i, ordered.end());
      return can_group(remaining, target);
    }
    if (i >= n || prod > want) return false;
    // take ordered[i]
    if (want % (prod * (int)ordered[i]) == 0) {
      if (rec(i + 1, prod * (int)ordered[i], rest)) return true;
    }
    // skip ordered[i] (and equal values, to avoid re-trying the same choice)
    size_t k = i;
    while (k < n && ordered[k] == ordered[i]) { rest.push_back(ordered[k]); ++k; }
    const bool ok = rec(k, prod, rest);
    for (size_t t = i; t < k; ++t) rest.pop_back();
    return ok;
  };
  std::vector<uint32_t> rest;
  return rec(0, 1, rest);
}

// per-stage twiddle table: stage s >= 1 holds tw[(j-1)*P + p] = W_{P*R}^{j*p}
std::vector<float2> build_twiddles(const std::vector<int>& radices, bool inverse) {
  std::vector<float2> t;
  long long P = 1;
  for (size_t s = 0; s < radices.size(); ++s) {
    const int R = radices[s];
    if (s > 0) {
      const long long Q = P * R;
      for (int j = 1; j < R; ++j)
        for (long long p = 0; p < P; ++p) {
          const double th = 2.0 * M_PI * (double)((j * p) % Q) / (double)Q;
          t.push_back(make_float2((float)std::cos(th), (float)((inverse ? 1.0 : -1.0) * std::sin(th))));
        }
    }
    P *= R;
  }
  if (t.empty()) t.push_back(make_float2(1.f, 0.f));
  return t;
}

// W_n^{+-k}, k = 0..n/2, for the R2C unpack / C2R pack
std::vector<float2> build_half_twiddles(long long n, bool inverse) {
  std::vector<float2> t;
  for (long long k = 0; k <= n / 2; ++k) {
    const double th = 2.0 * M_PI * (double)k / (double)n;
    t.push_back(make_float2((float)std::cos(th), (float)((inverse ? 1.0 : -1.0) * std::sin(th))));
  }
  return t;
}

// stage list of length n with one factor 2 removed (the even/odd split the real transform uses)
std::vector<std::vector<uint32_t>> drop_factor_two(const std::vector<uint32_t>& ordered) {
  std::vector<std::vector<uint32_t>> out;
  for (size_t i = 0; i < ordered.size(); ++i) {
    if (ordered[i] % 2) continue;
    if (i > 0 && ordered[i] == ordered[i - 1]) continue;
    std::vector<uint32_t> o(ordered);
    if (o[i] == 2) o.erase(o.begin() + i);
    else o[i] /= 2;
    out.push_back(o);
  }
  return out;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
PFN_cuTensorMapEncodeTiled_v12000 tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (PFN_cuTensorMapEncodeTiled_v12000)p;
  }();
  return fn;
}

bool tensor_maps_available() { return tensor_map_encoder() != nullptr; }

// tensor map over the (inner, N, outer) view of a dense complex64 array; box = (CW, box_rows, 1)
bool encode_axis_map(CUtensorMap* map, const void* base, long long inner, long long n, long long outer, int cw,
                     int box_rows) {
  auto enc = tensor_map_encoder();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)inner, (cuuint64_t)n, (cuuint64_t)outer};
  cuuint64_t strides[2] = {(cuuint64_t)inner * 8, (cuuint64_t)inner * (cuuint64_t)n * 8};
  cuuint32_t box[3] = {(cuuint32_t)cw, (cuuint32_t)box_rows, 1};
  cuuint32_t es[3] = {1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, const_cast<void*>(base), dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

namespace {

struct FastPass : Pass {
  const Variant* v = nullptr;
  HalfMode half = HALF_NONE;
  enum R2CMode { R2C_SMEM = 0, R2C_REG = 1, R2C_ODD = 2 } r2c_mode = R2C_SMEM;  // which R2C kernel (fast.cuh); R2C_ODD also
                                                                                // marks the odd-length C2R
  float2* d_tw2 = nullptr;
  AxisView view;
  bool inverse = false, real_in = false, do_scale = false;
  float scale = 1.f;
  float2* d_tw = nullptr;
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    return launch_outer(src, dst, nbatch * view.outer_per_batch, stream);
  }
  // `outer` consecutive outer slabs (rows passes: rows) starting at src / dst
  int launch_outer(const void* src, void* dst, int64_t outer, cudaStream_t stream) {
    if (half != HALF_NONE) {
      HalfArgs a;
      a.in = src;
      a.out = dst;
      a.tw = d_tw;
      a.tw2 = d_tw2;
      a.nrows = outer;
      a.scale = scale;
      const long long grid = (a.nrows + v->tile - 1) / v->tile;
      if (grid <= 0) return B200FFT_OK;
      if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many row tiles");
      if (half == HALF_R2C && r2c_mode == R2C_REG) v->launch_r2c_reg(a, (unsigned)grid, stream);
      else if (half == HALF_R2C && r2c_mode == R2C_ODD) v->launch_r2c_odd(a, (unsigned)grid, v->smem, stream);
      else if (half == HALF_C2R && r2c_mode == R2C_ODD) v->launch_c2r_odd(a, (unsigned)grid, v->smem, stream);
      else v->launch_half(half == HALF_C2R, a, (unsigned)grid, stream);
    } else if (v->kind == ROWS) {
      RowsArgs a;
      a.in = src;
      a.out = reinterpret_cast<float2*>(dst);
      a.tw = d_tw;
      a.nrows = outer;
      a.scale = scale;
      a.do_scale = do_scale;
      const long long grid = (a.nrows + v->tile - 1) / v->tile;
      if (grid <= 0) return B200FFT_OK;
      if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many row tiles");
      v->launch_rows(inverse, real_in, a, (unsigned)grid, v->smem, stream);
    } else if (v->kind == COLS_TMA) {
      CUtensorMap mi, mo;
      if (!encode_axis_map(&mi, src, view.inner, view.n, outer, v->tile, v->box_rows) ||
          !encode_axis_map(&mo, dst, view.inner, view.n, outer, v->tile, v->box_rows))
        return fail(B200FFT_ERR_CUDA, "cuTensorMapEncodeTiled failed for the strided-axis pass");
      ColsTmaArgs a;
      a.tw = d_tw;
      a.tiles_per_outer = (int)((view.inner + v->tile - 1) / v->tile);
      a.scale = scale;
      a.do_scale = do_scale;
      const long long grid = outer * a.tiles_per_outer;
      if (grid <= 0) return B200FFT_OK;
      if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many column tiles");
      v->launch_cols_tma(inverse, mi, mo, a, (unsigned)grid, v->smem, stream);
    } else {
      ColsArgs a;
      a.in = src;
      a.out = reinterpret_cast<float2*>(dst);
      a.tw = d_tw;
      a.inner = view.inner;
      a.tiles_per_outer = (int)((view.inner + v->tile - 1) / v->tile);
      a.scale = scale;
      a.do_scale = do_scale;
      a.reverse = reverse_order ? 1 : 0;
      const long long grid = outer * a.tiles_per_outer;
      if (grid <= 0) return B200FFT_OK;
      if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many column tiles");
      v->launch_cols(inverse, real_in, a, (unsigned)grid, v->smem, stream);
    }
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  int launch_scatter(const void* src, const Scatter& sc, int64_t nbatch, cudaStream_t stream) override {
    if (v->kind != COLS || !v->launch_scatter || half != HALF_NONE || real_in)
      return fail(B200FFT_ERR_UNSUPPORTED, "no scattering store for %s", text.c_str());
    if (sc.npeers < 1 || sc.npeers > 16 || view.n % sc.npeers)
      return fail(B200FFT_ERR_INVALID_ARG, "split axis length %lld is not divisible by %d peers", (long long)view.n, sc.npeers);
    ColsArgs a;
    a.in = src;
    a.out = nullptr;
    a.tw = d_tw;
    a.inner = view.inner;
    a.tiles_per_outer = (int)((view.inner + v->tile - 1) / v->tile);
    a.scale = scale;
    a.do_scale = do_scale;
    a.reverse = reverse_order ? 1 : 0;
    ScatterArgs sa;
    for (int i = 0; i < 16; ++i) sa.peer[i] = i < sc.npeers ? reinterpret_cast<float2*>(sc.peer_out[i]) : nullptr;
    sa.yl = (int)(view.n / sc.npeers);
    const long long outer = nbatch * view.outer_per_batch;
    sa.zbase = sc.zbase >= 0 ? sc.zbase : (long long)sc.my_rank * outer;
    const long long grid = outer * a.tiles_per_outer;
    if (grid <= 0) return B200FFT_OK;
    if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many column tiles");
    v->launch_scatter(inverse, a, sa, (unsigned)grid, v->smem, stream);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override {
    if (v->kind == COLS_TMA) return 16;  // tensor maps need 16-byte global addresses
    // rowsV: complex-input instantiations load and store through float4 (GlobalSrcV4 / GlobalDstV4)
    if (half == HALF_NONE && v->kind == ROWS && !real_in && v->name.compare(0, 5, "rowsV") == 0) return 16;
    // even half spectrum: R2C reads the real row as float2 pairs, C2R stores it as float2 pairs
    if (r2c_mode != R2C_ODD && half == (src ? HALF_R2C : HALF_C2R)) return 8;
    return 0;
  }
};

}  // namespace

size_t fast_variant_count() {
  register_all();
  return registry().size();
}

std::string fast_variant_info(size_t i) {
  register_all();
  if (i >= registry().size()) return "";
  const Variant& v = registry()[i];
  std::string kind, forms;
  auto add = [&](const char* f) { forms += (forms.empty() ? "" : ",") + std::string(f); };
  if (v.kind == ROWS) {
    kind = v.inv_ok ? "rowsIP" : "rows";
    add("fwd");
    if (v.full || v.inv_ok) { add("inv"); add("real"); }
    if (v.launch_half) { add("r2c"); add("c2r"); }
    if (v.launch_r2c_reg) add("r2c-reg");
    if (v.launch_r2c_odd) add("r2c-odd");
    if (v.launch_c2r_odd) add("c2r-odd");
  } else if (v.kind == COLS) {
    kind = "cols";
    add("fwd");
    if (v.full) { add("inv"); add("real"); }
    if (v.launch_scatter) add("scatter");
  } else {
    kind = "colsT";  // complex input only: the tensor maps describe complex64 elements
    add("fwd");
    add("inv");
  }
  return "name=" + v.name + " kind=" + kind + " n=" + std::to_string(v.n) + " radices=" + radix_name(v.radices) +
         " tile=" + std::to_string(v.tile) + " threads=" + std::to_string(v.threads) + " full=" + (v.full ? "1" : "0") +
         " smem=" + std::to_string(v.smem) + " smem_r2c=" + std::to_string(v.smem_r2c) +
         " smem_c2r=" + std::to_string(v.smem_c2r) + " forms=" + forms;
}

std::unique_ptr<Pass> make_fast_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                     bool scale_inverse, HalfMode half) {
  register_all();
  const Problem& p = plan.prob;
  if (p.desc.out_dtype != B200FFT_F32 || src.dtype != B200FFT_F32) return nullptr;
  if (view.n > 0x7fffffff) return nullptr;
  const Kind kind = view.inner == 1 ? ROWS : COLS;
  const AxisSpec& ax = p.axes[axis];

  std::vector<const Variant*> cands;
  const bool odd_r2c = half != HALF_NONE && kind == ROWS && view.n % 2 == 1;  // (both directions of an odd half-spectrum axis)
  if (odd_r2c) {
    // odd n: the n-point row variant itself — R2C on real input storing bins 0..n/2, C2R on the Hermitian-extended row
    if (src.dtype != B200FFT_F32) return nullptr;
    for (const Variant& v : registry())
      if (v.kind == ROWS && v.n == (int)view.n && v.launch_r2c_odd && v.launch_c2r_odd && can_group(ax.ordered, v.radices))
        cands.push_back(&v);
  } else if (half != HALF_NONE) {
    if (kind != ROWS || view.n % 2) return nullptr;
    const auto reduced = drop_factor_two(ax.ordered);
    for (const Variant& v : registry()) {
      if (v.kind != ROWS || v.n != (int)(view.n / 2) || !v.launch_half) continue;
      for (const auto& o : reduced)
        if (can_group(o, v.radices)) { cands.push_back(&v); break; }
    }
  } else {
    // TMA tiles need 16-byte global strides (even inner), complex fp32 source, a usable encoder
    const bool tma_ok = kind == COLS && src.comps == 2 && view.inner % 2 == 0 && tensor_map_encoder() != nullptr &&
                        (unsigned long long)view.inner * view.n * 8 < (1ull << 40);
    const char* ip_env = std::getenv("B200FFT_ROWS_INPLACE");  // =0: long rows as two split passes again (A/B, tests)
    const bool ip_ok = !(ip_env && ip_env[0] == '0');
    for (const Variant& v : registry()) {
      const bool kind_ok = (v.kind == kind || (v.kind == COLS_TMA && tma_ok)) && (ip_ok || !v.inv_ok);
      if (kind_ok && v.n == (int)view.n && (v.full || v.inv_ok || (!p.desc.inverse && src.comps == 2)) &&
          can_group(ax.ordered, v.radices))
        cands.push_back(&v);
    }
  }
  if (cands.empty()) return nullptr;
  if (kind == COLS && half == HALF_NONE) {
    // a tile wider than the axis's inner extent would leave lanes idle: prefer variants that fit
    std::vector<const Variant*> fit;
    for (const Variant* v : cands)
      if (v->tile <= view.inner) fit.push_back(v);
    if (!fit.empty()) cands.swap(fit);
  }
  if (const char* pref = getenv("B200FFT_PREFER")) {
    std::string s(pref);
    size_t pos = 0;
    std::vector<std::string> keys;
    while (pos <= s.size()) {
      size_t e = s.find(',', pos);
      if (e == std::string::npos) e = s.size();
      if (e > pos) keys.push_back(s.substr(pos, e - pos));
      pos = e + 1;
    }
    std::stable_sort(cands.begin(), cands.end(), [&](const Variant* a, const Variant* b) {
      auto rank = [&](const Variant* v) {
        for (size_t i = 0; i < keys.size(); ++i)
          if (v->name.find(keys[i]) != std::string::npos) return (int)i;
        return (int)keys.size();
      };
      return rank(a) < rank(b);
    });
  }
  const Variant* v = cands[0];
  // B200FFT_R2C_SMEM=1: keep the shared-memory Hermitian unpack (A/B knob for the register unpack)
  const char* r2c_env = getenv("B200FFT_R2C_SMEM");
  const bool r2c_reg = half == HALF_R2C && !odd_r2c && v->launch_r2c_reg && !(r2c_env && atoi(r2c_env) != 0);
  cudaError_t prep = odd_r2c ? v->prepare_r2c_odd(v->smem) : half != HALF_NONE ? v->prepare_half() : v->prepare(v->smem);
  if (prep == cudaSuccess && r2c_reg) prep = v->prepare_r2c_reg();
  if (prep != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  auto pass = std::make_unique<FastPass>();
  pass->v = v;
  pass->view = view;
  pass->inverse = p.desc.inverse != 0;
  pass->real_in = src.comps == 1;
  pass->do_scale = scale_inverse;
  pass->scale = scale_inverse ? (float)(1.0 / (double)view.n) : 1.f;
  pass->half = half;
  pass->r2c_mode = odd_r2c ? FastPass::R2C_ODD : r2c_reg ? FastPass::R2C_REG : FastPass::R2C_SMEM;
  if (odd_r2c) pass->real_in = half == HALF_R2C;
  if (odd_r2c && half == HALF_C2R) pass->scale = (float)(1.0 / (double)view.n);
  if (half != HALF_NONE && !odd_r2c) {
    if (half == HALF_C2R) pass->scale = (float)(1.0 / (double)view.n);  // 1/(2H): the inverse is always normalised
    std::vector<float2> tw2 = build_half_twiddles(view.n, half == HALF_C2R);
    if (cudaMalloc(&pass->d_tw2, tw2.size() * sizeof(float2)) != cudaSuccess) return nullptr;
    plan.owned_device.push_back(pass->d_tw2);
    if (cudaMemcpy(pass->d_tw2, tw2.data(), tw2.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
  }
  std::vector<float2> tw = build_twiddles(v->radices, half == HALF_NONE ? pass->inverse : half == HALF_C2R);  // (C2R: inverse tables)
  if (cudaMalloc(&pass->d_tw, tw.size() * sizeof(float2)) != cudaSuccess) return nullptr;
  plan.owned_device.push_back(pass->d_tw);  // owned by the plan BEFORE the copy: a failed copy must not leak it
  if (cudaMemcpy(pass->d_tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
  std::string stages;
  for (uint32_t r : ax.ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  char buf[320];
  if (odd_r2c)
    snprintf(buf, sizeof buf, "axis %d: %s[%s] n=%lld (%s) smem=%zuB user stages=[%s] fused as (%s)", axis,
             half == HALF_R2C ? "r2c-odd" : "c2r-odd", v->name.c_str(), (long long)view.n,
             half == HALF_R2C ? "real rows, bins 0..n/2 stored" : "Hermitian-extended load, real rows stored", v->smem, stages.c_str(),
             radix_name(v->radices).c_str());
  else if (half != HALF_NONE)
    snprintf(buf, sizeof buf, "axis %d: %s[%s] n=%lld (as %d complex) smem=%zuB user stages=[%s] fused as (2)(%s)", axis,
             half == HALF_R2C ? (r2c_reg ? "r2c-reg" : "r2c") : "c2r", v->name.c_str(), (long long)view.n, v->n,
             half == HALF_R2C ? (r2c_reg ? v->smem_r2c_reg : v->smem_r2c) : v->smem_c2r, stages.c_str(),
             radix_name(v->radices).c_str());
  else
    snprintf(buf, sizeof buf, "axis %d: %s n=%lld inner=%lld smem=%zuB user stages=[%s] fused as (%s)%s", axis,
             v->name.c_str(), (long long)view.n, (long long)view.inner, v->smem, stages.c_str(),
             radix_name(v->radices).c_str(), pass->real_in ? " real-in" : "");
  pass->text = buf;
  return pass;
}

}  // namespace b200fft

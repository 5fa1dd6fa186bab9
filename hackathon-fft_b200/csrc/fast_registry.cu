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

size_t fast_variant_count() {
  register_all();
  return registry().size();
}

std::string fast_variant_info(size_t i) {
  register_all();
  if (i >= registry().size()) return "";
  const Variant& v = registry()[i];
  static const struct { Form form; const char* name; } forms[] = {
      {FORM_FWD, "fwd"}, {FORM_INV, "inv"}, {FORM_FWD_REAL, "real"}, {FORM_R2C, "r2c"}, {FORM_C2R, "c2r"},
      {FORM_R2C_REG, "r2c-reg"}, {FORM_R2C_ODD, "r2c-odd"}, {FORM_C2R_ODD, "c2r-odd"}, {FORM_SCATTER_FWD, "scatter"}};
  std::string list;
  for (const auto& f : forms)
    if (v.sym[f.form]) list += (list.empty() ? "" : ",") + std::string(f.name);
  const char* kind = v.kind == TILE_ROWS ? "rows" : v.kind == TILE_ROWS_IP ? "rowsIP" : v.kind == TILE_COLS ? "cols" : "colsT";
  return "name=" + v.name + " kind=" + kind + " n=" + std::to_string(v.n) + " radices=" + radix_name(v.radices) +
         " tile=" + std::to_string(v.tile) + " threads=" + std::to_string(v.threads) + " full=" + (v.full ? "1" : "0") +
         " smem=" + std::to_string(v.smem) + " smem_r2c=" + std::to_string(v.smem_r2c) +
         " smem_c2r=" + std::to_string(v.smem_c2r) + " forms=" + list;
}

std::unique_ptr<Pass> make_fast_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                     bool scale_inverse, HalfMode half) {
  register_all();
  const Problem& p = plan.prob;
  if (p.desc.out_dtype != B200FFT_F32 || src.dtype != B200FFT_F32) return nullptr;
  if (view.n > 0x7fffffff) return nullptr;
  const TileKind kind = view.inner == 1 ? TILE_ROWS : TILE_COLS;
  const AxisSpec& ax = p.axes[axis];

  std::vector<const Variant*> cands;
  const bool odd_r2c = half != HALF_NONE && kind == TILE_ROWS && view.n % 2 == 1;  // (both directions of an odd half-spectrum axis)
  if (odd_r2c) {
    // odd n: the n-point row variant itself — R2C on real input storing bins 0..n/2, C2R on the Hermitian-extended row
    if (src.dtype != B200FFT_F32) return nullptr;
    for (const Variant& v : registry())
      if (v.kind == TILE_ROWS && v.n == (int)view.n && v.sym[FORM_R2C_ODD] && v.sym[FORM_C2R_ODD] && can_group(ax.ordered, v.radices))
        cands.push_back(&v);
  } else if (half != HALF_NONE) {
    if (kind != TILE_ROWS || view.n % 2) return nullptr;
    const auto reduced = drop_factor_two(ax.ordered);
    for (const Variant& v : registry()) {
      if (v.kind != TILE_ROWS || v.n != (int)(view.n / 2) || !v.sym[FORM_R2C]) continue;
      for (const auto& o : reduced)
        if (can_group(o, v.radices)) { cands.push_back(&v); break; }
    }
  } else {
    // TMA tiles need 16-byte global strides (even inner), complex fp32 source, a usable encoder
    const bool tma_ok = kind == TILE_COLS && src.comps == 2 && view.inner % 2 == 0 && tensor_map_encoder() != nullptr &&
                        (unsigned long long)view.inner * view.n * 8 < (1ull << 40);
    const char* ip_env = std::getenv("B200FFT_ROWS_INPLACE");  // =0: long rows as two split passes again (A/B, tests)
    const bool ip_ok = !(ip_env && ip_env[0] == '0');
    const Form form = p.desc.inverse ? (src.comps == 1 ? FORM_INV_REAL : FORM_INV) : (src.comps == 1 ? FORM_FWD_REAL : FORM_FWD);
    for (const Variant& v : registry()) {
      const bool kind_ok =
          v.kind == kind || (v.kind == TILE_ROWS_IP && kind == TILE_ROWS && ip_ok) || (v.kind == TILE_COLS_TMA && tma_ok);
      if (kind_ok && v.n == (int)view.n && v.sym[form] && can_group(ax.ordered, v.radices))
        cands.push_back(&v);
    }
  }
  if (cands.empty()) return nullptr;
  if (kind == TILE_COLS && half == HALF_NONE) {
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
  const bool r2c_reg = half == HALF_R2C && !odd_r2c && v->sym[FORM_R2C_REG] && !(r2c_env && atoi(r2c_env) != 0);
  auto pass = std::make_unique<TilePass>();
  TileSpec& s = pass->spec;
  s.n = v->n;
  s.radices = v->radices;
  s.tile = v->tile;
  s.threads = v->threads;
  s.vec = v->vec;
  s.inverse = half == HALF_NONE ? p.desc.inverse != 0 : half == HALF_C2R;  // (C2R: inverse tables)
  s.real_in = half == HALF_NONE && src.comps == 1;
  Form form;
  pass->smem = v->smem;
  if (odd_r2c) {
    s.kind = half == HALF_R2C ? TILE_R2C_ODD : TILE_C2R_ODD;
    form = half == HALF_R2C ? FORM_R2C_ODD : FORM_C2R_ODD;
  } else if (half == HALF_R2C) {
    s.kind = r2c_reg ? TILE_R2C_REG : TILE_R2C;
    form = r2c_reg ? FORM_R2C_REG : FORM_R2C;
    pass->smem = r2c_reg ? v->smem_r2c_reg : v->smem_r2c;
  } else if (half == HALF_C2R) {
    s.kind = TILE_C2R;
    form = FORM_C2R;
    pass->smem = v->smem_c2r;
  } else {
    s.kind = v->kind;
    form = s.inverse ? (s.real_in ? FORM_INV_REAL : FORM_INV) : (s.real_in ? FORM_FWD_REAL : FORM_FWD);
  }
  pass->k = {v->sym[form], nullptr, v->name};
  if (s.kind == TILE_COLS) pass->k_scatter = {v->sym[s.inverse ? FORM_SCATTER_INV : FORM_SCATTER_FWD], nullptr, v->name};
  cudaError_t prep = prepare_tile(pass->k.sym, pass->smem);
  if (prep == cudaSuccess && pass->k_scatter.sym) prep = prepare_tile(pass->k_scatter.sym, pass->smem);
  if (prep != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  pass->view = view;
  pass->device = plan.device;
  pass->do_scale = scale_inverse;
  pass->scale = (scale_inverse || half == HALF_C2R) ? 1.0 / (double)view.n : 1.0;  // the half-spectrum inverse is always normalised
  if (half != HALF_NONE && !odd_r2c && !(pass->tw2 = plan_upload(plan, build_half_twiddles(view.n, half == HALF_C2R)))) return nullptr;
  if (!(pass->tw = plan_upload(plan, build_twiddles(v->radices, s.inverse)))) return nullptr;
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
             radix_name(v->radices).c_str(), s.real_in ? " real-in" : "");
  pass->text = buf;
  return pass;
}

}  // namespace b200fft

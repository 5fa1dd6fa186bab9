// Two-pass ("four-step") treatment of axes that are too long for one tile: N = N1 * N2,
//   pass A  N1-point strided transforms with the W_N^{k1*n2} twiddle fused into the store  (src -> temp)
//   pass B  N2-point transforms whose store puts output k2 at axis index k1 + N1*k2        (temp -> dst)
// so a long axis costs two tile passes and one plan-owned temporary, never a transpose kernel. Used when no
// single-tile variant exists for the axis length (the reference's published shapes (100, 16384), 1920x1080,
// 3840x2160, 7680x4320: fft/bench.mojo:107-122). The user's stage list must be groupable into the two
// variants' super-stages, as for every other fast kernel.
#define B200FFT_PACKED 1  // packed FADD2 complex adds (dft.cuh): strided / mixed-radix kernels
#include "split_registry.hpp"

#include <cstring>

#include "plan.hpp"

namespace b200fft {

std::vector<SplitKernel>& split_registry() {
  static std::vector<SplitKernel> r;
  return r;
}

namespace {

void register_split() {
  static const bool done = [] {  // thread-safe one-time initialisation (see register_all, fast_registry.cu)
    // pass A candidates (N1): <role, N, columns per tile, threads, super-stages...>
    reg_split<TILE_SPLIT_A, 128, 16, 128, 16, 8>();
    reg_split<TILE_SPLIT_A, 256, 16, 256, 16, 16>();
    reg_split<TILE_SPLIT_A, 512, 16, 256, 32, 16>();
    reg_split<TILE_SPLIT_A, 512, 16, 256, 8, 8, 8>();  // the reference's default bases for 7680 are [15, 8, 8, 8]
    reg_split<TILE_SPLIT_A, 64, 16, 128, 8, 8>();
    // pass B candidates (N2)
    reg_split<TILE_SPLIT_B_COLS, 15, 128, 128, 15>();
    reg_split<TILE_SPLIT_B_COLS, 30, 64, 64, 30>();
    reg_split<TILE_SPLIT_B_COLS, 16, 128, 128, 16>();
    reg_split<TILE_SPLIT_B_ROWS, 128, 32, 256, 16, 8>();
    reg_split<TILE_SPLIT_B_ROWS, 64, 32, 256, 8, 8>();
    reg_split<TILE_SPLIT_B_ROWS, 256, 16, 256, 16, 16>();
    return true;
  }();
  (void)done;
}

}  // namespace

size_t split_variant_count() {
  register_split();
  return split_registry().size();
}

std::string split_variant_info(size_t i) {
  register_split();
  if (i >= split_registry().size()) return "";
  const SplitKernel& k = split_registry()[i];
  const char* kind = k.kind == TILE_SPLIT_A ? "splitA" : k.kind == TILE_SPLIT_B_COLS ? "splitB_cols" : "splitB_rows";
  return "name=" + k.name + " kind=" + kind + " n=" + std::to_string(k.n) + " radices=" + radix_name(k.radices) +
         " tile=" + std::to_string(k.tile) + " threads=" + std::to_string(k.threads) + " smem=" + std::to_string(k.smem) +
         " forms=fwd,inv";
}

std::unique_ptr<Pass> make_split_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                      bool scale_inverse, HalfMode half) {
  register_split();
  const Problem& p = plan.prob;
  if (half != HALF_NONE || p.desc.out_dtype != B200FFT_F32 || src.dtype != B200FFT_F32 || src.comps != 2) return nullptr;
  if (view.n > (1 << 24) || !plan.tw[axis].ptr) return nullptr;
  const AxisSpec& ax = p.axes[axis];
  const SplitKernel *best_a = nullptr, *best_b = nullptr;
  for (const SplitKernel& ka : split_registry()) {
    if (ka.kind != TILE_SPLIT_A || view.n % ka.n) continue;
    const long long n2 = view.n / ka.n;
    for (const SplitKernel& kb : split_registry()) {
      if (kb.n != n2) continue;
      if (kb.kind != (view.inner == 1 ? TILE_SPLIT_B_ROWS : TILE_SPLIT_B_COLS)) continue;
      if (kb.kind == TILE_SPLIT_B_ROWS && ka.n % kb.tile) continue;  // row tiles must not straddle transforms
      std::vector<int> all(ka.radices);
      all.insert(all.end(), kb.radices.begin(), kb.radices.end());
      if (!can_group(ax.ordered, all)) continue;
      if (!best_a) { best_a = &ka; best_b = &kb; }
    }
  }
  if (!best_a) return nullptr;
  const bool inv = p.desc.inverse != 0;
  auto pass = std::make_unique<SplitPass>();
  const void* twN = plan.tw[axis].ptr;
  int i = 0;
  for (const SplitKernel* k : {best_a, best_b}) {
    SplitPass::Stage& st = pass->st[i];
    st.spec.kind = k->kind;
    st.spec.n = k->n;
    st.spec.radices = k->radices;
    st.spec.tile = k->tile;
    st.spec.threads = k->threads;
    st.spec.inverse = inv;
    st.k = {k->sym[inv], nullptr, k->name};
    st.smem = k->smem;
    st.twN = twN;
    st.n2 = best_b->n;
    pass->len[i++] = k->n;
    if (prepare_tile(st.k.sym, st.smem) != cudaSuccess) {
      cudaGetLastError();
      return nullptr;
    }
  }
  pass->view = view;
  pass->do_scale = scale_inverse;
  pass->scale = scale_inverse ? 1.0 / (double)view.n : 1.0;
  if (!(pass->st[0].tw = plan_upload(plan, build_twiddles(best_a->radices, inv))) ||
      !(pass->st[1].tw = plan_upload(plan, build_twiddles(best_b->radices, inv))))
    return nullptr;
  const size_t tmp_bytes = (size_t)p.batch * view.outer_per_batch * view.n * view.inner * sizeof(float2);
  if (cudaMalloc(&pass->tmp, tmp_bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  plan.owned_device.push_back(pass->tmp);
  plan.workspace_bytes += tmp_bytes;
  std::string stages;
  for (uint32_t r : ax.ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  char buf[400];
  snprintf(buf, sizeof buf, "axis %d: split n=%lld = %d x %d inner=%lld: %s (+W_n twiddle) -> %s (natural-order store); temp=%zuB user stages=[%s]",
           axis, (long long)view.n, best_a->n, best_b->n, (long long)view.inner, best_a->name.c_str(), best_b->name.c_str(),
           tmp_bytes, stages.c_str());
  pass->text = buf;
  return pass;
}

}  // namespace b200fft

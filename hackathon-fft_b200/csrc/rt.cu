// Runtime-length axis pass with compile-time codelets: the fast tier for every axis length that has no
// hand-registered variant.
//
// The registered variants (fast_reg_*.cu) fix the axis length at compile time. Everything else used to fall to
// the generic kernel, which follows the reference's per-output-point formula (O(sum r) complex FMAs per point,
// generic.cu) and is 15-25x slower. This kernel keeps the tile structure of fast.cuh — stage 0 reads global
// memory, the last stage writes it, the exchanges in between go through padded shared memory, each butterfly is a
// register codelet Dft<R> — but takes the axis length, the tile shape and the list of super-stage radices at run
// time; only the codelet is selected by a switch over R = 2..32 (all compiled into one kernel). The user's
// ordered stage list (any primes up to 31, any composites, the reference's rules) is grouped into super-stages
// of product <= 32; a stage list with a radix above 32 stays on the generic kernel.
// Serves f32 output with f32 / f64 / u8, real or complex input; rows and strided axes.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "fast_registry.hpp"
#include "rt_kernel.cuh"
#include "plan.hpp"

namespace b200fft {

namespace {

// Group the ordered stage list (a multiset of bases whose product is N) into the fewest super-stages of product
// <= RT_MAX_RADIX, balanced: bases in descending order, each to the currently smallest group that still has room
// (longest-processing-time rule). 100 = [5,5,2,2] -> (10)(10); 1000 -> (10)(10)(10); 243 = [3]x5 -> (27)(9).
bool group_stages(const std::vector<uint32_t>& ordered, std::vector<int>* out) {
  for (uint32_t r : ordered)
    if (r > (uint32_t)RT_MAX_RADIX) return false;
  std::vector<uint32_t> bases(ordered);
  std::sort(bases.begin(), bases.end(), [](uint32_t x, uint32_t y) { return x > y; });
  for (int want = 1; want <= RT_MAX_STAGES; ++want) {
    std::vector<long long> g((size_t)want, 1);
    bool ok = true;
    for (uint32_t b : bases) {
      int best = -1;
      for (int i = 0; i < want; ++i)
        if (g[i] * b <= RT_MAX_RADIX && (best < 0 || g[i] < g[best])) best = i;
      if (best < 0) { ok = false; break; }
      g[best] *= b;
    }
    if (!ok) continue;
    std::sort(g.begin(), g.end(), [](long long x, long long y) { return x > y; });  // largest radix first
    out->clear();
    for (long long v : g)
      if (v > 1) out->push_back((int)v);
    if (out->empty()) out->push_back(1);
    return true;
  }
  return false;
}

struct RtPass : Pass {
  RtArgs base;
  AxisView view;
  bool inverse = false, small = false;
  size_t smem = 0;
  int sm_count = 148;
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    return launch_outer(src, dst, nbatch * view.outer_per_batch, stream);
  }
  int launch_outer(const void* src, void* dst, long long outer, cudaStream_t stream) {
    RtArgs a = base;
    a.in = src;
    a.out = reinterpret_cast<float2*>(dst);
    if (a.row) {
      a.outer = outer;
      a.ntiles = (outer + a.tile - 1) / a.tile;
    } else {
      a.outer = outer;
      a.ntiles = outer * a.tiles_per_outer;
    }
    if (a.ntiles <= 0) return B200FFT_OK;
    const unsigned grid = (unsigned)std::min<long long>(a.ntiles, (long long)sm_count * 32);
    rt_launch(inverse, small, a, grid, smem, stream);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
};

}  // namespace

std::unique_ptr<Pass> make_rt_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src,
                                   bool scale_inverse, HalfMode half) {
  const Problem& p = plan.prob;
  if (p.desc.out_dtype != B200FFT_F32 || view.n > (1 << 20)) return nullptr;
  if (half != HALF_NONE && view.inner != 1) return nullptr;  // half-spectrum handling is a row pass
  const AxisSpec& ax = p.axes[axis];
  std::vector<int> radices;
  if (!group_stages(ax.ordered, &radices)) return nullptr;
  const int S = (int)radices.size();
  const int n = (int)view.n;

  auto pass = std::make_unique<RtPass>();
  RtArgs& a = pass->base;
  memset(&a, 0, sizeof a);
  a.n = n;
  a.nstages = S;
  a.row = view.inner == 1;
  a.inner = view.inner;
  a.in_dtype = src.dtype;
  a.in_comps = src.comps;
  a.half = (int)half;
  a.do_scale = (scale_inverse || half == HALF_C2R) ? 1 : 0;  // the half-spectrum inverse is always normalised
  a.scale = a.do_scale ? (float)(1.0 / (double)n) : 1.f;
  // tile: ~4096 points per CTA for rows (at least enough butterflies for the threads), 16 columns for strided axes
  // tile: enough sub-transforms that the stage with the largest radix (fewest butterflies) still gives every
  // thread about two butterflies; strided axes take at least 16 columns (128 contiguous bytes per row)
  const int rmax = *std::max_element(radices.begin(), radices.end());
  int tile = (int)((2LL * RT_THREADS * rmax + n - 1) / n);
  if (a.row) {
    tile = std::max(1, tile);
  } else {
    tile = std::max(16, (tile + 7) / 8 * 8);
    tile = (int)std::min<long long>(tile, (view.inner + 7) / 8 * 8);
    tile = std::max(1, tile);
  }
  // exchange geometry
  long long P = 1;
  int max_stride = n;
  int off = 0;
  for (int s = 0; s < S; ++s) {
    const int R = radices[s];
    a.radix[s] = R;
    a.tw_off[s] = off;
    if (s > 0) off += (R - 1) * (int)P;
    const long long Q = P * R;
    const bool padded = a.row && P < 16 && Q % 2 == 0 && Q < n;
    a.padP[s] = padded ? (int)P : 0;
    a.stride[s] = n + (padded ? (int)(n / Q * P) : 0);
    if (s + 1 < S) max_stride = std::max(max_stride, a.stride[s]);
    P = Q;
  }
  const size_t nbuf = S > 2 ? 2 : (S > 1 ? 1 : 0);
  auto smem_for = [&](int t) { return nbuf * (size_t)(a.row ? (size_t)t * max_stride : (size_t)n * t) * sizeof(float2); };
  // two CTAs per SM when possible, but a strided tile keeps at least 8 columns (64 contiguous bytes per row)
  const int min_tile = a.row ? 1 : (int)std::min<long long>(8, view.inner);
  while (tile > min_tile && smem_for(tile) > 112 * 1024) tile = std::max(min_tile, (tile + 1) / 2);
  if (smem_for(tile) > 227 * 1024) return nullptr;  // too long for one tile: split_registry / generic decide
  a.tile = tile;
  a.tiles_per_outer = a.row ? 1 : (int)((view.inner + tile - 1) / tile);
  a.buf_elems = (int)(a.row ? (size_t)tile * max_stride : (size_t)n * tile);
  {
    long long PP = 1;
    for (int s2 = 0; s2 < S; ++s2) {
      a.div_nb[s2].set((unsigned)(n / radices[s2]));
      a.div_p[s2].set((unsigned)PP);
      PP *= radices[s2];
    }
    a.div_cn.set((unsigned)(a.row ? 1 : tile));
  }
  pass->smem = smem_for(tile);
  pass->view = view;
  pass->inverse = p.desc.inverse != 0;
  pass->sm_count = plan.sm_count;
  pass->small = rmax <= 16;
  if (rt_prepare(pass->inverse, pass->small, 227 * 1024) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (!(a.tw = plan_upload(plan, build_twiddles(radices, pass->inverse)))) return nullptr;
  std::string stages;
  for (uint32_t r : ax.ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  char buf[320];
  snprintf(buf, sizeof buf, "axis %d: rt_%s n=%d inner=%lld tile=%d smem=%zuB user stages=[%s] fused as (%s)%s", axis,
           a.row ? "rows" : "cols", n, (long long)view.inner, tile, pass->smem, stages.c_str(), radix_name(radices).c_str(),
           half == HALF_R2C ? " r2c (n-point, bins 0..n/2 stored)" : half == HALF_C2R ? " c2r (Hermitian load)"
                                                                                       : src.comps == 1 ? " real-in" : "");
  pass->text = buf;
  return pass;
}

}  // namespace b200fft

// Registry + pass object of the fused N-d kernel (fused.cuh): which shapes have a fused variant, how
// a validated problem is mapped onto its phases, the tile schedule upload, and the launch.
//
// A fused variant replaces ALL per-axis passes of a plan (api.cu: build_passes tries it first). It is
// used when every axis is transformed, the data is fp32, and the user's stage lists can be grouped
// into the variant's super-stages (same rule as the per-axis variants, fast_registry.cu).
//   B200FFT_FUSED=1 / 0    use every matching fused variant / none; unset = only the variants measured to win
//                          (see make_fused_pass; plan flag B200FFT_FLAG_NO_FUSED always wins)
//   B200FFT_CHUNK_MB=<n>   pipeline chunk size (default 8): how much phase-0 output is produced per
//                          round; ~2-3 chunks are live in L2 at any time
//   B200FFT_FUSED_PREFER=substr   prefer variants whose name contains substr (tuning aid; "substr:" = name ENDS with it)
// The v2 kernels (static work assignment) are launched COOPERATIVELY: the driver guarantees the whole grid is
// co-resident or refuses the launch, in which case the pass runs the plan's per-axis kernels instead (Pass::fallback).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "fast_registry.hpp"
#include "fused.cuh"
#include "fused_registry.hpp"
#include "plan.hpp"

namespace b200fft {

std::vector<FusedVariant>& fused_registry() {
  static std::vector<FusedVariant> r;
  return r;
}
void register_fused_3d();
void register_fused_2d();
void register_fused_async_3d();
void register_fused_async_2d();

namespace {

void register_all_fused() {
  static const bool done = [] {  // thread-safe one-time initialisation (see register_all, fast_registry.cu)
    register_fused_async_3d();  // v2 first: preferred when applicable
    register_fused_async_2d();
    register_fused_3d();
    register_fused_2d();
    return true;
  }();
  (void)done;
}

long long prod(const std::vector<long long>& v, size_t a, size_t b) {
  long long p = 1;
  for (size_t i = a; i < b && i < v.size(); ++i) p *= v[i];
  return p;
}

struct FusedPass : Pass {
  const FusedVariant* v = nullptr;
  NdArgs base;                 // everything but the per-launch pointers / schedule
  SchedPhase sched[ND_MAX_PHASES];
  int groups[ND_MAX_PHASES] = {0, 0, 0};
  int max_grid = 148;
  struct MapGeom { long long inner = 0, n = 0, outer_per_batch = 0; int cw = 0, box_rows = 0; } geom[ND_MAX_PHASES];
  std::string text;
  struct PerBatch {
    NdSegment* d_segs = nullptr;
    unsigned* d_ctrl = nullptr;
    int nsegs = 0;
    unsigned total_items = 0;
    int cnt_off[ND_MAX_PHASES] = {0, 0, 0};
    int nwords = 0;
  };
  std::map<int64_t, PerBatch> per_batch;  // schedules are built per batch count (exec_host runs chunks)
  b200fft_plan* plan = nullptr;

  int prepare(int64_t nbatch, PerBatch** out) {
    auto it = per_batch.find(nbatch);
    if (it != per_batch.end()) { *out = &it->second; return B200FFT_OK; }
    PerBatch pb;
    std::vector<NdSegment> segs = build_schedule(v->nphases, sched, nbatch);
    long long items = 0;
    for (auto& s : segs) items += s.count;
    if (items >= 0xffffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many tiles for the fused kernel");
    pb.total_items = (unsigned)items;
    pb.nsegs = (int)segs.size();
    int off = 2;
    for (int p = 0; p + 1 < v->nphases; ++p) {
      pb.cnt_off[p] = off;
      off += (int)(nbatch * groups[p]);
    }
    pb.nwords = off;
    B200_CUDA_CHECK(cudaMalloc(&pb.d_segs, sizeof(NdSegment) * segs.size()));
    plan->owned_device.push_back(pb.d_segs);
    B200_CUDA_CHECK(cudaMalloc(&pb.d_ctrl, sizeof(unsigned) * (size_t)pb.nwords));
    plan->owned_device.push_back(pb.d_ctrl);
    B200_CUDA_CHECK(cudaMemcpy(pb.d_segs, segs.data(), sizeof(NdSegment) * segs.size(), cudaMemcpyHostToDevice));
    B200_CUDA_CHECK(cudaMemset(pb.d_ctrl, 0, sizeof(unsigned) * (size_t)pb.nwords));
    // one-time, per batch count: the schedule and the zeroed counters must be in place before the kernel runs on
    // the caller's stream, which need not be ordered after the legacy stream used above
    B200_CUDA_CHECK(cudaDeviceSynchronize());
    auto ins = per_batch.emplace(nbatch, pb);
    *out = &ins.first->second;
    return B200FFT_OK;
  }

  unsigned* h_err = nullptr;  // mapped host word the kernels raise when a dependency wait gives up
  unsigned* d_err = nullptr;
  bool use_fallback = false;  // a cooperative launch was refused once: stay on the per-axis kernels

  int run_fallback(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) {
    if (fallback.empty()) return fail(B200FFT_ERR_CUDA, "%s cannot be launched and the plan has no per-axis passes", v->name.c_str());
    for (auto& p : fallback) {
      int rc = p->launch(p->src_sel == BUF_INPUT ? src : (const void*)dst, dst, nbatch, stream);
      if (rc != B200FFT_OK) return rc;
    }
    return B200FFT_OK;
  }

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    if (nbatch <= 0) return B200FFT_OK;
    if (use_fallback) return run_fallback(src, dst, nbatch, stream);
    if (h_err && *reinterpret_cast<volatile unsigned*>(h_err)) {
      // a previous launch of this plan gave up waiting for a dependency: its output was invalid and its counters are
      // stale. Report it once, reset, and leave the statically scheduled kernel for good.
      *h_err = 0;
      use_fallback = !fallback.empty();
      for (auto& kv : per_batch) cudaMemsetAsync(kv.second.d_ctrl, 0, sizeof(unsigned) * (size_t)kv.second.nwords, stream);
      return fail(B200FFT_ERR_CUDA, "%s: a dependency wait timed out in an earlier launch (its result was invalid)", v->name.c_str());
    }
    PerBatch* pb = nullptr;
    int rc = prepare(nbatch, &pb);
    if (rc != B200FFT_OK) return rc;
    NdArgs a = base;
    a.in = src;
    a.out = reinterpret_cast<float2*>(dst);
    a.segs = pb->d_segs;
    a.nsegs = pb->nsegs;
    a.total_items = pb->total_items;
    a.ctrl = pb->d_ctrl;
    a.err = d_err;
    for (int p = 0; p < ND_MAX_PHASES; ++p) a.cnt_off[p] = pb->cnt_off[p];
    a.nwords = pb->nwords;
    const unsigned grid = (unsigned)std::min<long long>(pb->total_items, max_grid);
    if (v->async) {
      CUtensorMap maps[ND_MAX_PHASES];
      memset(maps, 0, sizeof maps);
      for (int q = 1; q < v->nphases; ++q)
        if (!encode_axis_map(&maps[q], dst, geom[q].inner, geom[q].n, geom[q].outer_per_batch * nbatch, geom[q].cw,
                             geom[q].box_rows))
          return fail(B200FFT_ERR_CUDA, "cuTensorMapEncodeTiled failed for phase %d of %s", q, v->name.c_str());
      // B200FFT_TEST_REFUSE_COOP=1 (tests): behave as if the driver had refused the cooperative launch
      const char* refuse = getenv("B200FFT_TEST_REFUSE_COOP");
      const cudaError_t e = (refuse && atoi(refuse)) ? cudaErrorCooperativeLaunchTooLarge
                                                     : v->launch_async(a, maps[1], maps[2], grid, v->smem, stream);
      if (e != cudaSuccess) {
        // refused (the grid cannot be co-resident on this context: fewer SMs than at plan time, MPS / green-context
        // partition, cooperative launch unsupported): nothing was launched; run the per-axis kernels from now on
        cudaGetLastError();
        use_fallback = true;
        return run_fallback(src, dst, nbatch, stream);
      }
    } else {
      v->launch(a, grid, v->smem, stream);
    }
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  ~FusedPass() override {
    if (h_err) cudaFreeHost(h_err);
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override {
    if (v->async) return 16;  // bulk-async copies of the input tiles, tensor maps over the output
    // half spectrum: the real rows are read as float2 pairs
    if (src && v->mode == 2) return 8;
    return 0;
  }
};

}  // namespace

size_t fused_variant_count() {
  register_all_fused();
  return fused_registry().size();
}

std::string fused_variant_info(size_t i) {
  register_all_fused();
  if (i >= fused_registry().size()) return "";
  const FusedVariant& v = fused_registry()[i];
  std::string dims, radices;
  for (size_t a = 0; a < v.dims.size(); ++a) dims += (a ? "x" : "") + std::to_string(v.dims[a]);
  for (int q = 0; q < v.nphases; ++q) {  // phases in order; a plane phase lists its y stages, then ';', then its x stages
    const FusedPhaseInfo& ph = v.ph[q];
    radices += (q ? "|" : "") + (ph.radices2.empty() ? "" : radix_name(ph.radices2) + ";") + radix_name(ph.radices);
  }
  return "name=" + v.name + " kind=fused n=" + dims + " radices=" + radices + " tile=" + std::to_string(v.ph[0].tile) +
         " threads=" + std::to_string(v.threads) + " smem=" + std::to_string(v.smem) + " async=" + (v.async ? "1" : "0") +
         " mode=" + (v.mode == 0 ? "c2c" : v.mode == 1 ? "real" : "r2c") + " forms=" + (v.inverse ? "inv" : "fwd");
}

std::unique_ptr<Pass> make_fused_pass(b200fft_plan& plan) {
  register_all_fused();
  const Problem& p = plan.prob;
  // B200FFT_FUSED=1: any matching fused variant; =0: none; unset: only the variants measured to beat the
  // per-axis kernels (default_min_batch > 0: 64^3 at every batch, 128^3 from batch 4; profiles/r1_fused_v1.md)
  int mode_env = -1;
  if (const char* e = getenv("B200FFT_FUSED")) mode_env = atoi(e) != 0;
  if (p.desc.flags & (B200FFT_FLAG_FORCE_GENERIC | B200FFT_FLAG_NO_FUSED | B200FFT_FLAG_FORCE_RT)) return nullptr;
  if (p.desc.flags & B200FFT_FLAG_PREFER_FUSED) mode_env = 1;
  if (mode_env == 0) return nullptr;
  if (p.desc.out_dtype != B200FFT_F32 || p.desc.in_dtype != B200FFT_F32) return nullptr;
  if (p.rank < 2 || p.rank > 3) return nullptr;
  for (auto& ax : p.axes)
    if (!ax.transformed) return nullptr;
  const int mode = p.half ? 2 : (p.desc.in_components == 1 ? 1 : 0);
  if (p.half && p.desc.inverse) return nullptr;
  const int last = p.rank - 1;

  std::vector<long long> dims;
  for (auto& ax : p.axes) dims.push_back(ax.n);
  // the complex extents the strided phases see (half spectrum: last axis has n/2+1 bins)
  std::vector<long long> cdims(dims);
  if (p.half) cdims[last] = dims[last] / 2 + 1;

  const char* prefer = getenv("B200FFT_FUSED_PREFER");
  const FusedVariant* pick = nullptr;
  std::vector<int> pick_axes;
  for (int round = prefer ? 0 : 1; round < 2 && !pick; ++round) {  // round 0: preferred names only
    for (const FusedVariant& v : fused_registry()) {
      if (round == 0) {  // substring of the variant name; a trailing ':' anchors it at the END of the name
        std::string want(prefer);
        const bool anchored = !want.empty() && want.back() == ':';
        if (anchored) want.pop_back();
        const size_t at = anchored ? v.name.rfind(want) : v.name.find(want);
        if (at == std::string::npos || (anchored && at + want.size() != v.name.size())) continue;
      }
      if (mode_env < 0 && (v.default_min_batch <= 0 || p.batch < v.default_min_batch)) continue;
      if ((int)v.dims.size() != p.rank || v.inverse != (p.desc.inverse != 0) || v.mode != mode) continue;
      bool ok = true;
      for (int a = 0; a < p.rank; ++a) ok = ok && v.dims[a] == dims[a];
      if (!ok) continue;
      // axes of the phases: phase 0 takes the last axis (rows / r2c) or the last two (plane), the
      // strided phases walk the remaining axes right to left
      std::vector<int> axes;
      int next_axis = last;
      for (int q = 0; q < v.nphases && ok; ++q) {
        const FusedPhaseInfo& ph = v.ph[q];
        if (q == 0 && (ph.kind == ND_PLANE || ph.kind == ND_R2C_PLANE)) { axes.push_back(last); next_axis = last - 2; }
        else if (q == 0 && (ph.kind == ND_ROWS || ph.kind == ND_R2C)) { axes.push_back(last); next_axis = last - 1; }
        else if (q > 0 && ph.kind == ND_COLS && next_axis >= 0) { axes.push_back(next_axis); --next_axis; }
        else ok = false;
      }
      if (!ok || next_axis != -1) continue;
      // the user's stage lists must be groupable into the variant's super-stages
      for (int q = 0; q < v.nphases && ok; ++q) {
        const FusedPhaseInfo& ph = v.ph[q];
        const int a = axes[q];
        if (ph.kind == ND_R2C || ph.kind == ND_R2C_PLANE) {
          bool any = false;
          for (const auto& o : drop_factor_two(p.axes[a].ordered)) any = any || can_group(o, ph.radices);
          ok = any && dims[a] == ph.n;
          if (ok && ph.kind == ND_R2C_PLANE) ok = a >= 1 && dims[a - 1] == ph.n2 && can_group(p.axes[a - 1].ordered, ph.radices2);
        } else {
          ok = dims[a] == ph.n && can_group(p.axes[a].ordered, ph.radices);
          if (ok && ph.kind == ND_PLANE) ok = dims[a - 1] == ph.n2 && can_group(p.axes[a - 1].ordered, ph.radices2);
        }
      }
      if (!ok) continue;
      // group structure: rows tiles must not straddle the next phase's outer slabs
      if ((v.ph[0].kind == ND_ROWS || v.ph[0].kind == ND_R2C) && p.rank == 3 && dims[1] % v.ph[0].tile) continue;
      if (v.async) {
        // bulk-async staging: TMA boxes need whole tiles and 16-byte strides on every strided phase
        if (!tensor_maps_available()) continue;
        for (int q = 1; q < v.nphases && ok; ++q) {
          long long inner = 1;
          for (int a = axes[q] + 1; a < p.rank; ++a) inner *= cdims[a];
          ok = inner % v.ph[q].tile == 0 && inner % 2 == 0;
        }
        if (!ok) continue;
      }
      pick = &v;
      pick_axes = axes;
      break;
    }
  }
  if (!pick) return nullptr;
  const FusedVariant& v = *pick;

  auto pass = std::make_unique<FusedPass>();
  pass->v = &v;
  pass->plan = &plan;
  NdArgs& A = pass->base;
  memset(&A, 0, sizeof A);
  A.nphases = v.nphases;
  long long in_scalars = 1, out_pts = 1;
  for (int a = 0; a < p.rank; ++a) { in_scalars *= dims[a]; out_pts *= cdims[a]; }
  A.in_stride_bytes = in_scalars * (p.desc.in_components == 1 ? 4 : 8);
  A.out_stride = out_pts;

  const bool inv = p.desc.inverse != 0;
  double total_scale = 1.0;
  for (int a = 0; a < p.rank; ++a) total_scale *= (double)dims[a];
  // 64^3 x100: 8 -> 0.1472, 12 -> 0.1464, 16 -> 0.1483 ms; 128^3 x10: 8 -> 0.1457, 12 -> 0.1474;
  // half spectrum 64^3 x100 (tiles half the size): 8 -> 0.1012, 16 -> 0.0982, 24 -> 0.0944 (t160)
  long long chunk_mb = p.half ? 16 : 8;
  if (const char* e = getenv("B200FFT_CHUNK_MB")) chunk_mb = std::max(1, atoi(e));
  std::string desc;
  for (int q = 0; q < v.nphases; ++q) {
    const FusedPhaseInfo& ph = v.ph[q];
    NdPhase& P = A.ph[q];
    SchedPhase& S = pass->sched[q];
    const int a = pick_axes[q];
    const bool lastp = q == v.nphases - 1;
    {
      std::vector<float2> table = build_twiddles(ph.radices, inv);
      if (ph.kind == ND_R2C_PLANE) {  // [x stage twiddles | W_n^k, k = 0..n/2]: one table, staged once per CTA
        const std::vector<float2> half = build_half_twiddles(dims[last], false);
        table.insert(table.end(), half.begin(), half.end());
      }
      if (!(P.tw = plan_upload(plan, table))) return nullptr;
    }
    P.scale = 1.f;
    P.do_scale = 0;
    long long tile_bytes = 0;
    if (ph.kind == ND_ROWS || ph.kind == ND_R2C) {
      P.units_per_transform = prod(dims, 0, last);
      P.tiles_per_transform = (int)((P.units_per_transform + ph.tile - 1) / ph.tile);
      P.tiles_per_outer = 1;
      if (ph.kind == ND_R2C && !(P.tw2 = plan_upload(plan, build_half_twiddles(dims[last], false)))) return nullptr;
      tile_bytes = (long long)ph.tile * cdims[last] * 8;
    } else if (ph.kind == ND_PLANE || ph.kind == ND_R2C_PLANE) {
      P.units_per_transform = prod(dims, 0, last - 1);
      P.tiles_per_transform = (int)P.units_per_transform;
      P.tiles_per_outer = 1;
      if (!(P.tw2 = plan_upload(plan, build_twiddles(ph.radices2, inv)))) return nullptr;
      tile_bytes = cdims[last] * dims[last - 1] * 8;
    } else {  // ND_COLS on axis a
      P.inner = prod(cdims, a + 1, cdims.size());
      P.tiles_per_outer = (int)((P.inner + ph.tile - 1) / ph.tile);
      P.tiles_per_transform = (int)(prod(dims, 0, a) * P.tiles_per_outer);
      P.dep_div = P.tiles_per_outer;
      tile_bytes = (long long)ph.tile * dims[a] * 8;
      pass->geom[q].inner = P.inner;
      pass->geom[q].n = dims[a];
      pass->geom[q].outer_per_batch = prod(dims, 0, a);
      pass->geom[q].cw = ph.tile;
      pass->geom[q].box_rows = tma_box_rows((int)dims[a]);
    }
    if (!lastp) {
      // the next phase is a strided pass over axis a' (= the axis left of everything done so far);
      // its outer slabs are this phase's dependency groups
      const int an = pick_axes[q + 1];
      const long long outer_next = prod(dims, 0, an);
      P.groups_per_transform = (int)outer_next;
      if (P.tiles_per_transform % outer_next) return nullptr;
      P.tiles_per_group = (int)(P.tiles_per_transform / outer_next);
      pass->groups[q] = P.groups_per_transform;
    } else {
      P.groups_per_transform = 1;
      P.tiles_per_group = P.tiles_per_transform;
      if (inv) { P.scale = (float)(1.0 / total_scale); P.do_scale = 1; }
    }
    S.tiles_per_transform = P.tiles_per_transform;
    S.tiles_per_group = P.tiles_per_group;
    S.dep_div = q > 0 ? P.dep_div : 1;
    S.quota = 0;
    if (q == 0) {
      long long q0 = std::max<long long>(1, (chunk_mb << 20) / std::max<long long>(1, tile_bytes));
      q0 = ((q0 + P.tiles_per_group - 1) / P.tiles_per_group) * P.tiles_per_group;
      S.quota = q0;
    }
    char buf[256];
    snprintf(buf, sizeof buf, "%s%s", q ? " -> " : "", ph.text.c_str());
    desc += buf;
  }
  // a plane phase scales nothing itself unless it is last (it never is); an inverse with the scale on
  // the last phase covers all axes at once (1/prod(dims))

  if (v.smem > 48 * 1024 &&
      cudaFuncSetAttribute(v.func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)v.smem) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, v.func, v.threads, v.smem) != cudaSuccess || occ < 1) {
    cudaGetLastError();
    return nullptr;
  }
  pass->max_grid = occ * plan.sm_count;
  if (v.async) {
    int coop = 0;
    if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, plan.device) != cudaSuccess || !coop) {
      cudaGetLastError();
      return nullptr;  // the per-axis kernels run instead
    }
  }
  if (cudaHostAlloc(&pass->h_err, sizeof(unsigned), cudaHostAllocMapped) != cudaSuccess ||
      cudaHostGetDevicePointer(&pass->d_err, pass->h_err, 0) != cudaSuccess) {
    cudaGetLastError();
    if (pass->h_err) cudaFreeHost(pass->h_err);
    pass->h_err = pass->d_err = nullptr;  // no error word: the kernels then only lose the time-out report
  } else {
    *pass->h_err = 0;
  }
  // schedule + counters for the plan's own batch are built NOW, so that b200fft_exec itself never allocates or
  // synchronises (graph capture, asynchronous callers); other batch counts (exec_host chunks) are prepared on first use
  {
    FusedPass::PerBatch* pb = nullptr;
    if (pass->prepare(p.batch, &pb) != B200FFT_OK) return nullptr;
  }
  std::string stages;
  for (int a = 0; a < p.rank; ++a) {
    stages += a ? " | " : "";
    for (size_t i = 0; i < p.axes[a].ordered.size(); ++i)
      stages += (i ? "," : "") + std::to_string(p.axes[a].ordered[i]);
  }
  char buf[640];
  snprintf(buf, sizeof buf, "fused %s: %s; persistent grid %d x %d threads, smem=%zuB, chunk=%lldMB, user stages=[%s]",
           v.name.c_str(), desc.c_str(), pass->max_grid, v.threads, v.smem, chunk_mb, stages.c_str());
  pass->text = buf;
  pass->src_sel = BUF_INPUT;
  pass->dst_sel = BUF_OUTPUT;
  pass->axis = -1;
  return pass;
}

}  // namespace b200fft

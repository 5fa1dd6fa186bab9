// The passes that run the tile kernels of fast.cuh, the launch path they share, and the tables they upload.
#include "tile.hpp"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "fast_registry.hpp"

namespace b200fft {

size_t in_scalar_bytes(int dtype) { return dtype == B200FFT_U8 ? 1 : dtype == B200FFT_F64 ? 8 : 4; }

size_t tile_min_align(const std::vector<const TileSpec*>& stages, bool src) {
  size_t a = 0;
  for (const TileSpec* s : stages) {
    // tensor maps need 16-byte global addresses; rowsV complex rows load and store through float4 (GlobalSrcV4 / GlobalDstV4)
    if (s->kind == TILE_COLS_TMA || (s->kind == TILE_ROWS && s->vec && !s->real_in)) a = std::max<size_t>(a, 16);
    // even half spectrum: R2C reads the real rows as pairs of input scalars (single tile, split pass B's unpack, R2C
    // planes), C2R stores them as complex pairs (single tile, split pass A's pack)
    const bool r2c = s->kind == TILE_R2C || s->kind == TILE_R2C_REG || s->kind == TILE_SPLIT_B_R2C || s->kind == TILE_PLANE_R2C;
    if (src && r2c) a = std::max(a, 2 * in_scalar_bytes(stages[0]->in_dtype));
    if (!src && (s->kind == TILE_C2R || s->kind == TILE_SPLIT_A_C2R)) a = std::max(a, s->esz());
  }
  return a;
}

// Programmatic dependent launch for the passes that FOLLOW another pass of a plan (strided passes, the C2R row pass).
// Measured (profiles/r2_pdl.md): 256^3 0.126 -> 0.122 ms, its R2C 0.071 -> 0.066, 2-D 640 x 480 0.161 -> 0.158,
// 100 x 64^3 0.149 -> 0.146.
static bool pdl_enabled() {
  const char* e = getenv("B200FFT_PDL");  // read per launch (~50 ns): lets one process A/B the two launch modes
  return !(e && atoi(e) == 0);
}

int launch_tile(const TileKernel& k, long long grid, int threads, size_t smem, bool dependent, void** params, cudaStream_t stream) {
  if (grid <= 0) return B200FFT_OK;
  if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many tiles for %s", k.name.c_str());
  const bool pdl = dependent && pdl_enabled();
  if (k.sym) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelExC(&cfg, k.sym, params);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(B200FFT_ERR_CUDA, "launch of %s failed: %s", k.name.c_str(), cudaGetErrorString(e));
    }
  } else {
    CUlaunchConfig cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDimX = (unsigned)grid;
    cfg.gridDimY = cfg.gridDimZ = 1;
    cfg.blockDimX = (unsigned)threads;
    cfg.blockDimY = cfg.blockDimZ = 1;
    cfg.sharedMemBytes = (unsigned)smem;
    cfg.hStream = (CUstream)stream;
    CUlaunchAttribute attr;
    memset(&attr, 0, sizeof attr);
    attr.id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
    attr.value.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = pdl ? 1 : 0;
    const CUresult r = driver().LaunchKernelEx(&cfg, k.fn, params, nullptr);
    if (r != CUDA_SUCCESS) return fail(B200FFT_ERR_CUDA, "launch of %s failed (CUresult %d)", k.name.c_str(), (int)r);
  }
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return B200FFT_OK;
}

cudaError_t prepare_tile(const void* sym, size_t smem) {
  if (smem <= 48 * 1024) return cudaSuccess;
  return cudaFuncSetAttribute(sym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// float2 tables are evaluated in double, double2 tables in long double
template <class T2>
using TwiddleReal = std::conditional_t<std::is_same<T2, float2>::value, double, long double>;

template <class T2>
static T2 unit(TwiddleReal<T2> th, bool inverse) {
  using S = decltype(T2::x);
  T2 v;
  v.x = (S)std::cos(th);
  v.y = (S)((inverse ? TwiddleReal<T2>(1) : TwiddleReal<T2>(-1)) * std::sin(th));
  return v;
}

template <class T2>
std::vector<T2> build_twiddles(const std::vector<int>& radices, bool inverse) {
  using R = TwiddleReal<T2>;
  const R two_pi = std::is_same<T2, float2>::value ? R(2.0 * M_PI) : 2.0L * 3.14159265358979323846264338327950288L;
  std::vector<T2> t;
  long long P = 1;
  for (size_t s = 0; s < radices.size(); ++s) {
    const int r = radices[s];
    if (s > 0) {
      const long long Q = P * r;
      for (int j = 1; j < r; ++j)
        for (long long p = 0; p < P; ++p) t.push_back(unit<T2>(two_pi * (R)((j * p) % Q) / (R)Q, inverse));
    }
    P *= r;
  }
  if (t.empty()) {
    T2 one;
    one.x = 1;
    one.y = 0;
    t.push_back(one);
  }
  return t;
}

template <class T2>
std::vector<T2> build_half_twiddles(long long n, bool inverse) {
  using R = TwiddleReal<T2>;
  const R two_pi = std::is_same<T2, float2>::value ? R(2.0 * M_PI) : 2.0L * 3.14159265358979323846264338327950288L;
  std::vector<T2> t;
  for (long long k = 0; k <= n / 2; ++k) t.push_back(unit<T2>(two_pi * (R)k / (R)n, inverse));
  return t;
}

template std::vector<float2> build_twiddles<float2>(const std::vector<int>&, bool);
template std::vector<double2> build_twiddles<double2>(const std::vector<int>&, bool);
template std::vector<float2> build_half_twiddles<float2>(long long, bool);
template std::vector<double2> build_half_twiddles<double2>(long long, bool);

namespace {

// Kernel argument blocks. The fp64 build of a kernel sees the same structs with float -> double (rtc_prelude.cuh), so
// the host fills a struct of that layout.
struct RowsArgs64 { const void* in; double2* out; const double2* tw; long long nrows; double scale; int do_scale; };
struct ColsArgs64 { const void* in; double2* out; const double2* tw; long long inner; int tiles_per_outer; double scale; int do_scale; int reverse; };
struct HalfArgs64 { const void* in; void* out; const double2* tw; const double2* tw2; long long nrows; double scale; };
struct SplitArgs64 {
  const void* in; double2* out; const double2* tw; const double2* twN; const double2* tw2; long long inner; long long nrows;
  int tiles_per_outer; int n1, n2; double scale; int do_scale;
};

template <bool F64> struct Args;
template <> struct Args<false> { using T2 = float2; using Rows = RowsArgs; using Cols = ColsArgs; using Half = HalfArgs; using Split = SplitArgs; };
template <> struct Args<true> { using T2 = double2; using Rows = RowsArgs64; using Cols = ColsArgs64; using Half = HalfArgs64; using Split = SplitArgs64; };

template <bool F64>
typename Args<F64>::Cols cols_args(const TilePass& p, const void* src, void* dst) {
  using T2 = typename Args<F64>::T2;
  typename Args<F64>::Cols a;
  a.in = src;
  a.out = reinterpret_cast<T2*>(dst);
  a.tw = reinterpret_cast<const T2*>(p.tw);
  a.inner = p.view.inner;
  a.tiles_per_outer = (int)((p.view.inner + p.spec.tile - 1) / p.spec.tile);
  a.scale = p.scale;
  a.do_scale = p.do_scale;
  a.reverse = p.reverse_order ? 1 : 0;
  return a;
}

template <bool F64>
int tile_launch(const TilePass& p, const void* src, void* dst, long long outer, cudaStream_t stream) {
  using T2 = typename Args<F64>::T2;
  const TileSpec& s = p.spec;
  const long long row_tiles = (outer + s.tile - 1) / s.tile;
  switch (s.kind) {
    case TILE_ROWS:
    case TILE_ROWS_IP: {
      typename Args<F64>::Rows a;
      a.in = src;
      a.out = reinterpret_cast<T2*>(dst);
      a.tw = reinterpret_cast<const T2*>(p.tw);
      a.nrows = outer;
      a.scale = p.scale;
      a.do_scale = p.do_scale;
      void* params[1] = {&a};
      return launch_tile(p.k, row_tiles, s.threads, p.smem, false, params, stream);
    }
    case TILE_COLS: {
      typename Args<F64>::Cols a = cols_args<F64>(p, src, dst);
      void* params[1] = {&a};
      return launch_tile(p.k, outer * a.tiles_per_outer, s.threads, p.smem, true, params, stream);
    }
    case TILE_COLS_TMA: {
      CUtensorMap mi, mo;
      const int box_rows = tma_box_rows(s.n);
      if (!encode_axis_map(&mi, src, p.view.inner, p.view.n, outer, s.tile, box_rows) ||
          !encode_axis_map(&mo, dst, p.view.inner, p.view.n, outer, s.tile, box_rows))
        return fail(B200FFT_ERR_CUDA, "cuTensorMapEncodeTiled failed for the strided-axis pass");
      ColsTmaArgs a;
      a.tw = reinterpret_cast<const float2*>(p.tw);
      a.tiles_per_outer = (int)((p.view.inner + s.tile - 1) / s.tile);
      a.scale = (float)p.scale;
      a.do_scale = p.do_scale;
      void* params[3] = {&mi, &mo, &a};
      return launch_tile(p.k, outer * a.tiles_per_outer, s.threads, p.smem, false, params, stream);
    }
    case TILE_SCATTER_Z: return fail(B200FFT_ERR_UNSUPPORTED, "%s only runs as a scattering store", p.text.c_str());
    default: {  // the half-spectrum row forms; the C2R pass is the last pass of its plan
      typename Args<F64>::Half a;
      a.in = src;
      a.out = dst;
      a.tw = reinterpret_cast<const T2*>(p.tw);
      a.tw2 = reinterpret_cast<const T2*>(p.tw2);
      a.nrows = outer;
      a.scale = p.scale;
      void* params[1] = {&a};
      const bool dependent = s.kind == TILE_C2R || s.kind == TILE_C2R_ODD;
      return launch_tile(p.k, row_tiles, s.threads, p.smem, dependent, params, stream);
    }
  }
}

template <bool F64>
int split_launch(const SplitPass& p, const void* src, void* dst, long long outer, cudaStream_t stream) {
  using T2 = typename Args<F64>::T2;
  typename Args<F64>::Split a;
  memset(&a, 0, sizeof a);
  a.inner = p.view.inner;
  a.n1 = (int)p.len[0];
  void* params[1] = {&a};
  long long before = 1;  // product of the lengths of the earlier stages
  for (int i = 0; i < p.count; ++i) {
    const SplitPass::Stage& st = p.st[i];
    const bool last = i == p.count - 1;
    a.in = i == 0 ? src : p.tmp;
    a.out = reinterpret_cast<T2*>(last ? dst : p.tmp);
    a.tw = reinterpret_cast<const T2*>(st.tw);
    a.twN = reinterpret_cast<const T2*>(st.twN);
    a.tw2 = reinterpret_cast<const T2*>(st.tw2);
    a.n2 = st.n2;
    if (last) {
      a.scale = p.scale;
      a.do_scale = p.do_scale;
    }
    long long grid;
    if (st.spec.kind == TILE_SPLIT_B_R2C) {  // (n1/2 + 1) row pairs per transform, tile/2 of them per CTA
      a.tiles_per_outer = (int)((p.len[0] / 2 + 1 + st.spec.tile / 2 - 1) / (st.spec.tile / 2));
      grid = outer * a.tiles_per_outer;
    } else if (st.spec.strided()) {  // view (outer * earlier lengths, this length, later lengths * inner)
      long long cols = p.view.inner;
      for (int j = i + 1; j < p.count; ++j) cols *= p.len[j];
      a.tiles_per_outer = (int)((cols + st.spec.tile - 1) / st.spec.tile);
      grid = outer * before * a.tiles_per_outer;
    } else {  // contiguous rows
      a.nrows = outer * before;
      grid = (a.nrows + st.spec.tile - 1) / st.spec.tile;
    }
    const int rc = launch_tile(st.k, grid, st.spec.threads, st.smem, false, params, stream);
    if (rc != B200FFT_OK) return rc;
    before *= p.len[i];
  }
  return B200FFT_OK;
}

// the StrLay forms: the kernel's argument block followed by the pass's geometry (fast.cuh: StrLay::Args)
template <bool F64>
int strided_launch(const StridedPass& p, const void* src, void* dst, cudaStream_t stream) {
  using T2 = typename Args<F64>::T2;
  const TileSpec& s = p.spec;
  const long long row_tiles = (p.count + s.tile - 1) / s.tile;
  switch (s.kind) {
    case TILE_ROWS:
    case TILE_ROWS_IP: {
      typename StrLay::template Args<typename Args<F64>::Rows> a;
      memset(&a, 0, sizeof a);
      a.in = src;
      a.out = reinterpret_cast<T2*>(dst);
      a.tw = reinterpret_cast<const T2*>(p.tw);
      a.nrows = p.count;
      a.scale = p.scale;
      a.do_scale = p.do_scale;
      a.g = p.geo;
      void* params[1] = {&a};
      return launch_tile(p.k, row_tiles, s.threads, p.smem, p.dependent, params, stream);
    }
    case TILE_COLS: {
      typename StrLay::template Args<typename Args<F64>::Cols> a;
      memset(&a, 0, sizeof a);
      a.in = src;
      a.out = reinterpret_cast<T2*>(dst);
      a.tw = reinterpret_cast<const T2*>(p.tw);
      a.inner = p.ncols;
      a.tiles_per_outer = (int)((p.ncols + s.tile - 1) / s.tile);
      a.scale = p.scale;
      a.do_scale = p.do_scale;
      a.g = p.geo;
      void* params[1] = {&a};
      return launch_tile(p.k, p.count * a.tiles_per_outer, s.threads, p.smem, p.dependent, params, stream);
    }
    default: {  // the half-spectrum row forms
      typename StrLay::template Args<typename Args<F64>::Half> a;
      memset(&a, 0, sizeof a);
      a.in = src;
      a.out = dst;
      a.tw = reinterpret_cast<const T2*>(p.tw);
      a.tw2 = reinterpret_cast<const T2*>(p.tw2);
      a.nrows = p.count;
      a.scale = p.scale;
      a.g = p.geo;
      void* params[1] = {&a};
      return launch_tile(p.k, row_tiles, s.threads, p.smem, p.dependent, params, stream);
    }
  }
}

}  // namespace

int StridedPass::launch(const void* src, void* dst, int64_t, cudaStream_t stream) {
  return spec.f64 ? strided_launch<true>(*this, src, dst, stream) : strided_launch<false>(*this, src, dst, stream);
}

int TilePass::launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) {
  const long long outer = nbatch * view.outer_per_batch;
  return spec.f64 ? tile_launch<true>(*this, src, dst, outer, stream) : tile_launch<false>(*this, src, dst, outer, stream);
}

int TilePass::prepare_scatter() {
  if (spec.kind == TILE_SCATTER_Z) return B200FFT_OK;  // the pass's own kernel, built with it (jit.cu: make_jit_scatter_z_pass)
  if (spec.kind != TILE_COLS || spec.real_in || spec.in_dtype != (spec.f64 ? B200FFT_F64 : B200FFT_F32) || (k.sym && !k_scatter.sym))
    return fail(B200FFT_ERR_UNSUPPORTED, "no scattering store for %s", text.c_str());
  if (!k.sym && !k_scatter.fn) {
    TileSpec sp = spec;
    sp.kind = TILE_SCATTER;
    int cur = -1;
    cudaGetDevice(&cur);
    if (cur != device) cudaSetDevice(device);
    k_scatter = jit_tile_kernel(sp, device);
    if (cur != device && cur >= 0) cudaSetDevice(cur);
    if (!k_scatter.fn) return fail(B200FFT_ERR_UNSUPPORTED, "could not specialise the scattering store for %s", text.c_str());
  }
  return B200FFT_OK;
}

namespace {
// the scattering column kernel `k` with the store policy's argument block `sa` (pointers and integers only: the same block
// for both precisions)
template <class SA>
int scatter_launch(const TilePass& p, const TileKernel& k, const void* src, SA sa, long long outer, cudaStream_t stream) {
  if (p.spec.f64) {
    ColsArgs64 ca = cols_args<true>(p, src, nullptr);
    void* params[2] = {&ca, &sa};
    return launch_tile(k, outer * ca.tiles_per_outer, p.spec.threads, p.smem, false, params, stream);
  }
  ColsArgs ca = cols_args<false>(p, src, nullptr);
  void* params[2] = {&ca, &sa};
  return launch_tile(k, outer * ca.tiles_per_outer, p.spec.threads, p.smem, false, params, stream);
}
}  // namespace

int TilePass::launch_scatter(const void* src, const Scatter& sc, int64_t nbatch, cudaStream_t stream) {
  if (int rc = prepare_scatter()) return rc;
  if (sc.npeers < 1 || sc.npeers > 16 || view.n % sc.npeers)
    return fail(B200FFT_ERR_INVALID_ARG, "split axis length %lld is not divisible by %d peers", (long long)view.n, sc.npeers);
  const long long outer = nbatch * view.outer_per_batch;
  if (spec.kind == TILE_SCATTER_Z) {  // this rank's columns are block my_rank of every row of a peer's slab
    ScatterZArgs za;
    for (int i = 0; i < 16; ++i) za.peer[i] = i < sc.npeers ? reinterpret_cast<float2*>(sc.peer_out[i]) : nullptr;
    za.rows = (int)(view.n / sc.npeers);
    za.col0 = (long long)sc.my_rank * view.inner;
    za.stride = (long long)sc.npeers * view.inner;
    return scatter_launch(*this, k, src, za, outer, stream);
  }
  ScatterArgs sa;
  for (int i = 0; i < 16; ++i) sa.peer[i] = i < sc.npeers ? reinterpret_cast<float2*>(sc.peer_out[i]) : nullptr;
  sa.yl = (int)(view.n / sc.npeers);
  sa.zbase = sc.zbase >= 0 ? sc.zbase : (long long)sc.my_rank * outer;
  return scatter_launch(*this, k_scatter, src, sa, outer, stream);
}

int SplitPass::launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) {
  const long long outer = nbatch * view.outer_per_batch;
  if (outer <= 0) return B200FFT_OK;
  return st[0].spec.f64 ? split_launch<true>(*this, src, dst, outer, stream) : split_launch<false>(*this, src, dst, outer, stream);
}

}  // namespace b200fft

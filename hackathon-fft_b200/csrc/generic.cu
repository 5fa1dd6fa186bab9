// Generic runtime-radix axis pass: any length whose tile fits shared memory, any
// radix list (any prime, any composite), any input dtype, rows or strided axes.
//
// It is the universal-coverage kernel (and the B200FFT_FLAG_FORCE_GENERIC path):
// one CTA stages a tile of C sub-transforms in shared memory, runs every Stockham
// stage with the reference's per-output-point formulation
// (fft/fft/_fft.mojo:228-296, SURVEY Appendix A.3)
//     u = i mod Q, n = (i div Q)*P + (u mod P)
//     Y[i] = X[n] + sum_{j=1..r-1} W_N^{((j*u) mod Q)*rho} * X[n + j*N/r]
// ping-ponging between two shared buffers, and writes the tile back once. Global
// memory is read once and written once per axis; strided axes are tiled so that no
// transpose kernel exists (the reference needs 2*(ndims-1) of them,
// _ndim_fft_gpu.mojo:617-642). The hot shapes are served by the compile-time
// kernels in fast_*.cu; this kernel is O(sum r) per point and exists for coverage.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>

#include "device_utils.cuh"
#include "plan.hpp"

namespace b200fft {

constexpr int GEN_MAX_STAGES = 40;
constexpr int GEN_THREADS = 256;
constexpr size_t MAX_SMEM = 227 * 1024;

struct GenParams {
  const void* src;
  void* dst;
  const void* tw;
  long long outer, inner, tiles_per_outer, ntiles;
  int n, nstages, C, row, src_dtype, src_comps;
  int half;  // HalfMode (rows only): R2C stores bins 0..n/2 with row pitch n/2+1; C2R loads the
             // half spectrum with Hermitian extension X[n-k] = conj(X[k]) and stores real parts
  double scale;
  int radix[GEN_MAX_STAGES];
};

template <typename T>
__global__ void __launch_bounds__(GEN_THREADS) gen_fft_kernel(const __grid_constant__ GenParams p) {
  using T2 = typename Vec2<T>::type;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T2* buf0 = reinterpret_cast<T2*>(smem_raw);
  T2* buf1 = buf0 + (size_t)p.n * p.C;
  const T2* __restrict__ tw = reinterpret_cast<const T2*>(p.tw);
  T2* __restrict__ dst = reinterpret_cast<T2*>(p.dst);
  const int n = p.n;
  const int tid = threadIdx.x;

  for (long long tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    long long base, sn, sc;
    int cc;
    const int hb = n / 2 + 1;  // bins of a half spectrum
    if (p.row) {
      const long long o0 = tile * p.C;
      cc = (int)min((long long)p.C, p.outer - o0);
      base = o0 * n;
      sn = 1;
      sc = n;
      if (p.half == HALF_C2R) {
        // Hermitian-extended load of rows that hold n/2+1 bins
        for (int f = tid; f < n * cc; f += GEN_THREADS) {
          const int c = f / n, nn = f - c * n;
          const long long rowb = (o0 + c) * hb;
          T2 v;
          if (nn < hb) v = load_any<T>(p.src, p.src_dtype, 2, rowb + nn);
          else { v = load_any<T>(p.src, p.src_dtype, 2, rowb + (n - nn)); v.y = -v.y; }
          buf0[f] = v;
        }
      }
    } else {
      const long long o = tile / p.tiles_per_outer;
      const long long i0 = (tile - o * p.tiles_per_outer) * p.C;
      cc = (int)min((long long)p.C, p.inner - i0);
      base = o * n * p.inner + i0;
      sn = p.inner;
      sc = 1;
    }
    const int total = n * cc;

    // stage the tile: shared index == flat index f in both layouts
    // (rows: [c][n], n fastest; strided: [n][cc], c fastest)
    if (!(p.row && p.half == HALF_C2R)) {
      for (int f = tid; f < total; f += GEN_THREADS) {
        int nn, c;
        if (p.row) { c = f / n; nn = f - c * n; }
        else { nn = f / cc; c = f - nn * cc; }
        buf0[f] = load_any<T>(p.src, p.src_dtype, p.src_comps, base + nn * sn + c * sc);
      }
    }
    __syncthreads();

    T2* cur = buf0;
    T2* nxt = buf1;
    int P = 1;
    for (int s = 0; s < p.nstages; ++s) {
      const int r = p.radix[s];
      const int Q = P * r, rho = n / Q, step = n / r;
      const bool last = (s == p.nstages - 1);
      const int da = p.row ? step : step * cc;
      for (int f = tid; f < total; f += GEN_THREADS) {
        int i, c;
        if (p.row) { c = f / n; i = f - c * n; }
        else { i = f / cc; c = f - i * cc; }
        const int q = i / Q;
        const int u = i - q * Q;
        const int nn = q * P + (u % P);
        const int a0 = p.row ? c * n + nn : nn * cc + c;
        // r - 1 terms in one running sum lose accuracy like sqrt(r) (fp32 at a radix-14519 stage: 3e-6 relative L2), so
        // the running sum takes at most 32 terms before it is folded into the total. Up to radix 32 the total is
        // still zero at the end, and adding it leaves the single running sum's value.
        T2 part = cur[a0];
        T2 acc;
        acc.x = acc.y = (T)0;
        int k = 0;
        for (int j = 1; j < r; ++j) {
          k += u;
          if (k >= Q) k -= Q;
          part = cfma(__ldg(&tw[(size_t)k * rho]), cur[a0 + j * da], part);
          if ((j & 31) == 0) {
            acc.x += part.x;
            acc.y += part.y;
            part.x = part.y = (T)0;
          }
        }
        acc.x += part.x;
        acc.y += part.y;
        if (last) { acc.x *= (T)p.scale; acc.y *= (T)p.scale; }
        nxt[f] = acc;
      }
      __syncthreads();
      T2* t = cur; cur = nxt; nxt = t;
      P = Q;
    }

    if (p.row && p.half == HALF_R2C) {
      for (int f = tid; f < hb * cc; f += GEN_THREADS) {
        const int c = f / hb, nn = f - c * hb;
        dst[(tile * p.C + c) * hb + nn] = cur[c * n + nn];
      }
    } else if (p.row && p.half == HALF_C2R) {
      T* __restrict__ rdst = reinterpret_cast<T*>(p.dst);
      for (int f = tid; f < total; f += GEN_THREADS) rdst[base + f] = cur[f].x;
    } else {
      for (int f = tid; f < total; f += GEN_THREADS) {
        int nn, c;
        if (p.row) { c = f / n; nn = f - c * n; }
        else { nn = f / cc; c = f - nn * cc; }
        dst[base + nn * sn + c * sc] = cur[f];
      }
    }
    __syncthreads();
  }
}

namespace {

struct GenericPass : Pass {
  GenParams base{};
  int64_t outer_per_batch = 1;
  size_t smem = 0;
  bool f64 = false;
  int sm_count = 148;
  int axis = 0;
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    return launch_outer(src, dst, nbatch * outer_per_batch, stream);
  }
  int launch_outer(const void* src, void* dst, long long outer, cudaStream_t stream) {
    GenParams p = base;
    p.src = src;
    p.dst = dst;
    p.outer = outer;
    if (p.row) {
      p.tiles_per_outer = 1;
      p.ntiles = (p.outer + p.C - 1) / p.C;
    } else {
      p.tiles_per_outer = (p.inner + p.C - 1) / p.C;
      p.ntiles = p.outer * p.tiles_per_outer;
    }
    const int per_sm = std::max<int>(1, std::min<size_t>(8, MAX_SMEM / std::max<size_t>(smem, 1)));
    const long long grid = std::min<long long>(p.ntiles, (long long)sm_count * per_sm);
    if (grid <= 0) return B200FFT_OK;
    if (f64) gen_fft_kernel<double><<<(unsigned)grid, GEN_THREADS, smem, stream>>>(p);
    else gen_fft_kernel<float><<<(unsigned)grid, GEN_THREADS, smem, stream>>>(p);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    B200_CUDA_CHECK(cudaGetLastError());
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
};

}  // namespace

std::unique_ptr<Pass> make_generic_pass(const b200fft_plan& plan, int axis, const AxisView& view,
                                        const IoSpec& src, bool scale_inverse, HalfMode half) {
  const AxisSpec& ax = plan.prob.axes[axis];
  const bool f64 = plan.prob.desc.out_dtype == B200FFT_F64;
  const size_t sz = f64 ? 16 : 8;
  if (ax.ordered.size() > (size_t)GEN_MAX_STAGES) {
    fail(B200FFT_ERR_UNSUPPORTED, "axis %d: more than %d stages", axis, GEN_MAX_STAGES);
    return nullptr;
  }
  const size_t per_transform = 2 * (size_t)view.n * sz;
  if (per_transform > MAX_SMEM) {
    fail(B200FFT_ERR_UNSUPPORTED,
         "axis %d: length %lld does not fit the generic kernel's shared-memory tile (%zu B > %zu B)", axis,
         (long long)view.n, per_transform, MAX_SMEM);
    return nullptr;
  }
  auto pass = std::make_unique<GenericPass>();
  GenParams& p = pass->base;
  p.tw = plan.tw[axis].ptr;
  p.n = (int)view.n;
  p.inner = view.inner;
  p.row = view.inner == 1;
  p.nstages = (int)ax.ordered.size();
  for (int s = 0; s < p.nstages; ++s) p.radix[s] = (int)ax.ordered[s];
  p.src_dtype = src.dtype;
  p.src_comps = src.comps;
  p.half = (int)half;
  p.scale = scale_inverse ? 1.0 / (double)view.n : 1.0;
  int C;
  if (p.row) {
    // enough sub-transforms for the 256 threads, two CTAs per SM when possible
    const size_t budget = 100 * 1024;
    C = (int)std::max<size_t>(1, std::min<size_t>(64, budget / per_transform));
    while (C > 1 && (size_t)C * view.n > 8192) C /= 2;
    C = std::max(C, 1);
  } else {
    C = f64 ? 8 : 16;  // 128 contiguous bytes per tile row
    while (C > 1 && (size_t)C * per_transform > MAX_SMEM) C /= 2;
    while (C > 1 && (size_t)C * per_transform > 100 * 1024 && C * sz > 64) C /= 2;
    C = (int)std::min<int64_t>(C, view.inner);
  }
  p.C = C;
  pass->smem = (size_t)C * per_transform;
  pass->outer_per_batch = view.outer_per_batch;
  pass->f64 = f64;
  pass->sm_count = plan.sm_count;
  pass->axis = axis;
  cudaError_t e = f64 ? cudaFuncSetAttribute(gen_fft_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MAX_SMEM)
                      : cudaFuncSetAttribute(gen_fft_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MAX_SMEM);
  if (e != cudaSuccess) {
    fail(B200FFT_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return nullptr;
  }
  char buf[256];
  std::string radices;
  for (uint32_t r : ax.ordered) radices += (radices.empty() ? "" : ",") + std::to_string(r);
  snprintf(buf, sizeof buf, "axis %d: generic<%s>%s n=%lld inner=%lld tile=%d smem=%zuB stages=[%s]", axis,
           f64 ? "f64" : "f32", half == HALF_R2C ? " r2c" : half == HALF_C2R ? " c2r" : "", (long long)view.n,
           (long long)view.inner, C, pass->smem, radices.c_str());
  pass->text = buf;
  return pass;
}

}  // namespace b200fft

// One description and one launch path for the tile kernels of fast.cuh and plane.cuh, whether an instantiation is
// compiled into the library (fast_reg_*.cu, split_registry.cu) or specialised at plan time through NVRTC (jit.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <string>
#include <vector>

#include "plan.hpp"

namespace b200fft {

// Which kernel template an instantiation comes from (fast.cuh / plane.cuh).
enum TileKind {
  TILE_ROWS = 0,     // rows_kernel<N, RL, C, NT, INV, REAL, VEC>: `tile` contiguous transforms per CTA
  TILE_COLS,         // cols_kernel<N, RL, CW, NT, INV, REAL>: all N points of `tile` adjacent columns of a strided axis
  TILE_SCATTER,      // cols_scatter_kernel<N, RL, CW, NT, INV>: the same with the slab exchange in its stores
  TILE_R2C,          // rows_r2c_kernel<H, RL, C, NT>: n = 2H real points as an H-point complex row + shared-memory unpack
  TILE_R2C_REG,      // rows_r2c_reg_kernel<H, RL, C, NT>: Hermitian unpack in registers (warp shuffles)
  TILE_R2C_ODD,      // rows_r2c_odd_kernel<N, RL, C, NT>: odd n, the n-point row kernel on real rows, bins 0..n/2 stored
  TILE_C2R,          // rows_c2r_kernel<H, RL, C, NT>: Hermitian pack fused into stage 0 of the H-point inverse
  TILE_C2R_ODD,      // rows_c2r_odd_kernel<N, RL, C, NT>: odd n, Hermitian-extended load, real rows stored
  // long axes as two passes, N = N1 * N2 (fast.cuh, "four-step"):
  TILE_SPLIT_A,      // cols_split_a_kernel<N1, RL, CW, NT, INV>: N1-point strided transforms, W_N^{k1 n2} fused into the store
  TILE_SPLIT_B_COLS, // cols_split_b_kernel<N2, RL, CW, NT, INV>: N2-point strided transforms, natural-order store
  TILE_SPLIT_B_ROWS, // rows_split_b_kernel<N2, RL, C, NT, INV>: the same for a contiguous axis
  // the two innermost axes in one in-place tile per (y, x) plane (plane.cuh); n = NY, n2 = NX (R2C: H), radices = y, radices2 = x
  TILE_PLANE_C2C,    // c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, INV, REAL>
  TILE_PLANE_R2C,    // r2c_plane_ip_kernel<NY, H, RLY, RLX, NT>
  TILE_ROWS_IP,      // rows_ip_kernel<N, RL, C, NT, INV, REAL>: `tile` rows per CTA, 3-5 stages in ONE shared buffer
  // long half-spectrum rows as two passes (split length H = n/2 for even n, n for odd n); pass A of a real-input or
  // dtype-casting axis is TILE_SPLIT_A with real_in / in_dtype
  TILE_SPLIT_B_R2C,     // rows_split_b_r2c_kernel<N2, RL, C, NT>: even R2C, (k1, N1 - k1) row pairs, Hermitian unpack in the store
  TILE_SPLIT_A_C2R,     // cols_split_a_c2r_kernel<N1, RL, CW, NT, false>: even C2R, Hermitian pack in the load
  TILE_SPLIT_A_C2R_ODD, // cols_split_a_c2r_kernel<N1, RL, CW, NT, true>: odd C2R, Hermitian-extended load
  TILE_SPLIT_B_HALF,    // rows_split_b_kernel<N2, RL, C, NT, false, 1>: odd R2C, bins 0..n/2 stored
  TILE_SPLIT_B_REAL,    // rows_split_b_kernel<N2, RL, C, NT, true, 2>: odd C2R, real parts stored
  // contiguous axes longer than 2^24 points as three passes, n = N1 * N2 * N3 (fast.cuh):
  TILE_SPLIT3_A,        // cols_split_a_kernel<N, RL, CW, NT, INV, REAL, true>: passes 1 and 2, the twiddle from two tables
  TILE_SPLIT3_C,        // rows_split_c_kernel<N3, RL, C, NT, INV>: pass 3, rows (k1, k2), natural-order store
  TILE_COLS_TMA         // cols_tma_kernel<N, RL, CW, NT, INV>: strided tiles moved by TMA (compiled-in variants only)
};

size_t in_scalar_bytes(int dtype);

// One instantiation of a tile kernel: its template arguments and the tile geometry.
struct TileSpec {
  TileKind kind = TILE_ROWS;
  int n = 0;  // length of the complex transform the kernel runs (H = n_real / 2 for R2C / R2C_REG / C2R)
  std::vector<int> radices;
  int n2 = 0;                  // plane kinds: the x extent (R2C: H)
  std::vector<int> radices2;   // plane kinds: the x stages
  int tile = 0, threads = 0;
  bool inverse = false, real_in = false, packed = false;
  bool vec = false;            // rows: 128-bit global accesses for complex input ("rowsV" variants)
  bool f64 = false;            // working precision (the plan's out_dtype): fp64 = the same kernels with the scalar type swapped
  int in_dtype = B200FFT_F32;  // element type of the array the kernel READS (cast on load)
  int tile_divides = 0;        // geometry only: the tile must divide this (split pass B rows never straddle transforms)
  long long rows_hint = 0;     // geometry only: transforms per call when the planner knows it (few rows: more threads per row)

  size_t esz() const { return f64 ? sizeof(double2) : sizeof(float2); }
  bool plane() const { return kind == TILE_PLANE_C2C || kind == TILE_PLANE_R2C; }
  bool strided() const {
    return kind == TILE_COLS || kind == TILE_SCATTER || kind == TILE_SPLIT_A || kind == TILE_SPLIT_B_COLS || kind == TILE_SPLIT_A_C2R ||
           kind == TILE_SPLIT_A_C2R_ODD || kind == TILE_SPLIT3_A || kind == TILE_COLS_TMA;
  }
  // Host mirror of fast.cuh's shared-memory formulas for the kinds the plan-time tier builds: used to choose the tile
  // before anything is compiled, and checked against the value the compiled module reports.
  // RowLayout pads a Q-block by P elements when P < 16, Q even and Q < N; DenseLayout is N x CW.
  size_t smem() const {
    if (plane()) return esz() * (size_t)n * (size_t)(n2 + n2 / radices2[0]);  // one buffer of NY rows, pitch NX + NX / r0
    long long P = 1, ex = 0;
    if (kind == TILE_ROWS_IP) {  // rows_ip_smem_bytes: the largest exchange layout, once
      for (size_t s = 0; s + 1 < radices.size(); ++s) {
        const long long Q = P * radices[s];
        ex = std::max(ex, (P < 16 && Q % 2 == 0 && Q < n) ? n + n / Q * P : (long long)n);
        P = Q;
      }
      return esz() * (size_t)ex * (size_t)tile;
    }
    for (size_t s = 0; s + 1 < radices.size(); ++s) {
      const long long Q = P * radices[s];
      long long elems;
      if (strided()) {
        elems = (long long)n * tile;
      } else {
        const bool padded = P < 16 && Q % 2 == 0 && Q < n;
        elems = (long long)tile * (padded ? n + n / Q * P : n);
      }
      ex = std::max(ex, elems);
      P = Q;
    }
    const size_t pingpong = radices.size() > 2 ? 2 : 1;
    switch (kind) {
      case TILE_R2C:
      case TILE_SPLIT_B_R2C: return esz() * (size_t)std::max<long long>(ex, (long long)tile * n) * 2;
      default: return esz() * (size_t)ex * pingpong;
    }
  }
};

// Byte alignment the kernels of a pass (its stages in launch order) need of the buffer they read (src) or write (!src),
// beyond one element of it (Pass::min_align).
size_t tile_min_align(const std::vector<const TileSpec*>& stages, bool src);

// A kernel to launch: the host stub of a compiled-in __global__ instantiation, or a function of a module that NVRTC
// built (jit.cu keeps those modules loaded for the life of the process).
struct TileKernel {
  const void* sym = nullptr;
  CUfunction fn = nullptr;
  std::string name;  // for the error text of a failed launch
};

// Launch `k` on a 1-D grid. An empty grid launches nothing; a grid above 2^31 - 1 is refused. A dependent launch may set
// its grid up while the previous kernel of the stream still runs (fast.cuh: pdl_wait) unless B200FFT_PDL=0.
int launch_tile(const TileKernel& k, long long grid, int threads, size_t smem, bool dependent, void** params, cudaStream_t stream);

// Raise the dynamic shared-memory limit of a compiled-in instantiation that needs more than 48 KB.
cudaError_t prepare_tile(const void* sym, size_t smem);

// driver entry points through the runtime (no link against libcuda); jit.cu resolves them
struct Driver {
  CUresult (*ModuleLoadData)(CUmodule*, const void*) = nullptr;
  CUresult (*ModuleUnload)(CUmodule) = nullptr;
  CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*) = nullptr;
  CUresult (*ModuleGetGlobal)(CUdeviceptr*, size_t*, CUmodule, const char*) = nullptr;
  CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int) = nullptr;
  CUresult (*FuncGetAttribute)(int*, CUfunction_attribute, CUfunction) = nullptr;
  CUresult (*LaunchKernelEx)(const CUlaunchConfig*, CUfunction, void**, void**) = nullptr;
  bool ok = false;
};
const Driver& driver();
// the NVRTC build of `spec` for `device` (compiled or taken from the caches); fn == nullptr when it cannot be built
TileKernel jit_tile_kernel(const TileSpec& spec, int device);

// per-stage twiddle table: stage s >= 1 holds tw[(j-1)*P + p] = W_{P*R}^{j*p}
// (float2 evaluated in double, double2 in long double)
template <class T2 = float2>
std::vector<T2> build_twiddles(const std::vector<int>& radices, bool inverse);
// W_n^{+-k}, k = 0..n/2, for the R2C unpack / C2R pack (same precisions)
template <class T2 = float2>
std::vector<T2> build_half_twiddles(long long n, bool inverse);

// A single-tile pass over one axis: rows, rowsIP, cols, colsT, the half-spectrum row forms, and (launch_scatter) the
// scattering column store.
struct TilePass : Pass {
  TileSpec spec;
  TileKernel k;
  TileKernel k_scatter;  // compiled-in: the variant's scatter instantiation (may be absent); NVRTC: built on first use
  size_t smem = 0;
  AxisView view;
  int device = 0;
  bool do_scale = false;
  double scale = 1.0;
  void* tw = nullptr;   // stage twiddles, float2 or double2
  void* tw2 = nullptr;  // W_n^{+-k} of the Hermitian unpack / pack
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override;
  int launch_scatter(const void* src, const Scatter& sc, int64_t nbatch, cudaStream_t stream) override;
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override { return tile_min_align({&spec}, src); }
};

// An axis too long for one tile as two or three passes through one plan-owned temporary (fast.cuh: cols_split_a,
// cols_split_b, rows_split_b, rows_split_c and their half-spectrum forms).
struct SplitPass : Pass {
  struct Stage {
    TileSpec spec;
    TileKernel k;
    size_t smem = 0;
    const void* tw = nullptr;   // stage twiddles of this pass's kernel
    const void* twN = nullptr;  // SplitArgs::twN / tw2 as this stage reads them
    const void* tw2 = nullptr;
    int n2 = 0;                 // SplitArgs::n2 of this stage
  };
  Stage st[3];
  int count = 2;
  long long len[3] = {1, 1, 1};  // transform length of each stage: N1, N2 (, N3)
  AxisView view;
  bool do_scale = false;
  double scale = 1.0;
  void* tmp = nullptr;
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override;
  std::string describe() const override { return text; }
  int launches() const override { return count; }
  size_t min_align(bool src) const override {
    std::vector<const TileSpec*> s;
    for (int i = 0; i < count; ++i) s.push_back(&st[i].spec);
    return tile_min_align(s, src);
  }
};

}  // namespace b200fft

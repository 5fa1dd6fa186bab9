// Plan-time specialisation tier: the compile-time kernels of fast.cuh instantiated at plan creation for axis lengths
// that have no hand-registered variant.
//
// The reference specialises EVERY shape at compile time (Mojo `comptime` parameters: length, bases, layouts are all
// template arguments of `_intra_something_gpu_fft_kernel_radix_n_multi_dim`, _ndim_fft_gpu.mojo:279-450). A C ABI
// takes them at run time, so the equivalent here is run-time compilation: `b200fft_plan_create` hands the very same
// headers the registered variants are built from (rtc_prelude.cuh, dft.cuh, tma.cuh, fast.cuh — embedded in the
// library as text) to NVRTC with the axis length, the grouped super-stage list, the tile shape and the direction as
// template arguments, gets a cubin for sm_100a back, loads it with the driver API and launches it like any other pass.
// One compile per distinct (kind, N, radices, tile, threads, direction, input kind) per device, cached for the life of
// the process. If libnvrtc cannot be loaded or the compile fails, the axis falls to the runtime-length tier (rt.cu).
// Compiled kernels are also kept on disk (see disk_cache_dir below), so only the first process ever to plan a shape pays.
//   B200FFT_JIT=0        disable this tier          B200FFT_JIT_VERBOSE=1   print compile times / logs to stderr
//   B200FFT_JIT_CACHE=0  no on-disk cache           B200FFT_JIT_CACHE_DIR   where it lives (default ~/.cache/b200fft)
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cerrno>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "fast_registry.hpp"
#include "plan.hpp"
#include "plane.cuh"

namespace b200fft {

namespace {

#include "jit_embed.inc"  // k_src_rtc_prelude, k_src_dft, k_src_tma, k_src_fast: the device headers as text

// ---- NVRTC, loaded lazily (no link-time dependency) ----------------------------------------------------------------
struct Nvrtc {
  using Program = void*;
  int (*CreateProgram)(Program*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  int (*DestroyProgram)(Program*) = nullptr;
  int (*CompileProgram)(Program, int, const char* const*) = nullptr;
  int (*GetCUBINSize)(Program, size_t*) = nullptr;
  int (*GetCUBIN)(Program, char*) = nullptr;
  int (*GetProgramLogSize)(Program, size_t*) = nullptr;
  int (*GetProgramLog)(Program, char*) = nullptr;
  int (*AddNameExpression)(Program, const char*) = nullptr;
  int (*GetLoweredName)(Program, const char*, const char**) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  std::string why;
};

const Nvrtc& nvrtc() {
  static const Nvrtc api = [] {
    Nvrtc n;
    void* h = nullptr;
    for (const char* name : {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"}) {
      h = dlopen(name, RTLD_NOW | RTLD_LOCAL);
      if (h) break;
    }
    if (!h) {
      n.why = "libnvrtc.so.12 not found";
      return n;
    }
    auto sym = [&](const char* s) { return dlsym(h, s); };
#define B200_NVRTC_SYM(field, name) \
  n.field = reinterpret_cast<decltype(n.field)>(sym(name)); \
  if (!n.field) { n.why = std::string("missing ") + name; return n; }
    B200_NVRTC_SYM(CreateProgram, "nvrtcCreateProgram")
    B200_NVRTC_SYM(DestroyProgram, "nvrtcDestroyProgram")
    B200_NVRTC_SYM(CompileProgram, "nvrtcCompileProgram")
    B200_NVRTC_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
    B200_NVRTC_SYM(GetCUBIN, "nvrtcGetCUBIN")
    B200_NVRTC_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
    B200_NVRTC_SYM(GetProgramLog, "nvrtcGetProgramLog")
    B200_NVRTC_SYM(AddNameExpression, "nvrtcAddNameExpression")
    B200_NVRTC_SYM(GetLoweredName, "nvrtcGetLoweredName")
    B200_NVRTC_SYM(GetErrorString, "nvrtcGetErrorString")
#undef B200_NVRTC_SYM
    n.ok = true;
    return n;
  }();
  return api;
}

// ---- driver entry points through the runtime (no link against libcuda, like the tensor-map encoder) ----------------
struct Driver {
  CUresult (*ModuleLoadData)(CUmodule*, const void*) = nullptr;
  CUresult (*ModuleUnload)(CUmodule) = nullptr;
  CUresult (*ModuleGetFunction)(CUfunction*, CUmodule, const char*) = nullptr;
  CUresult (*ModuleGetGlobal)(CUdeviceptr*, size_t*, CUmodule, const char*) = nullptr;
  CUresult (*FuncSetAttribute)(CUfunction, CUfunction_attribute, int) = nullptr;
  CUresult (*FuncGetAttribute)(int*, CUfunction_attribute, CUfunction) = nullptr;
  CUresult (*LaunchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void**,
                           void**) = nullptr;
  CUresult (*LaunchKernelEx)(const CUlaunchConfig*, CUfunction, void**, void**) = nullptr;  // optional (dependent launches)
  bool ok = false;
};

const Driver& driver() {
  static const Driver api = [] {
    Driver d;
    auto get = [](const char* name) -> void* {
      void* p = nullptr;
      cudaDriverEntryPointQueryResult q;
      if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return nullptr;
      }
      return p;
    };
    d.ModuleLoadData = reinterpret_cast<decltype(d.ModuleLoadData)>(get("cuModuleLoadData"));
    d.ModuleUnload = reinterpret_cast<decltype(d.ModuleUnload)>(get("cuModuleUnload"));
    d.ModuleGetFunction = reinterpret_cast<decltype(d.ModuleGetFunction)>(get("cuModuleGetFunction"));
    d.ModuleGetGlobal = reinterpret_cast<decltype(d.ModuleGetGlobal)>(get("cuModuleGetGlobal"));
    d.FuncSetAttribute = reinterpret_cast<decltype(d.FuncSetAttribute)>(get("cuFuncSetAttribute"));
    d.FuncGetAttribute = reinterpret_cast<decltype(d.FuncGetAttribute)>(get("cuFuncGetAttribute"));
    d.LaunchKernel = reinterpret_cast<decltype(d.LaunchKernel)>(get("cuLaunchKernel"));
    d.LaunchKernelEx = reinterpret_cast<decltype(d.LaunchKernelEx)>(get("cuLaunchKernelEx"));
    d.ok = d.ModuleLoadData && d.ModuleUnload && d.ModuleGetFunction && d.ModuleGetGlobal && d.FuncSetAttribute && d.FuncGetAttribute && d.LaunchKernel;
    return d;
  }();
  return api;
}

// ---- what to compile ------------------------------------------------------------------------------------------------
enum JitKind {
  JIT_ROWS = 0,     // rows_kernel<N, RL, C, NT, INV, REAL>: `tile` contiguous transforms per CTA
  JIT_COLS,         // cols_kernel<N, RL, CW, NT, INV, REAL>: all N points of `tile` adjacent columns of a strided axis
  JIT_SCATTER,      // cols_scatter_kernel<N, RL, CW, NT, INV>: the same with the slab exchange in its stores
  JIT_R2C,          // rows_r2c_kernel<H, RL, C, NT>: n = 2H real points as an H-point complex row + shared-memory unpack
  JIT_R2C_REG,      // rows_r2c_reg_kernel<H, RL, C, NT>: Hermitian unpack in registers (warp shuffles)
  JIT_R2C_ODD,      // rows_r2c_odd_kernel<N, RL, C, NT>: odd n, the n-point row kernel on real rows, bins 0..n/2 stored
  JIT_C2R,          // rows_c2r_kernel<H, RL, C, NT>: Hermitian pack fused into stage 0 of the H-point inverse
  JIT_C2R_ODD,      // rows_c2r_odd_kernel<N, RL, C, NT>: odd n, Hermitian-extended load, real rows stored
  // long axes as two passes, N = N1 * N2 (fast.cuh, "four-step"):
  JIT_SPLIT_A,      // cols_split_a_kernel<N1, RL, CW, NT, INV>: N1-point strided transforms, W_N^{k1 n2} fused into the store
  JIT_SPLIT_B_COLS, // cols_split_b_kernel<N2, RL, CW, NT, INV>: N2-point strided transforms, natural-order store
  JIT_SPLIT_B_ROWS, // rows_split_b_kernel<N2, RL, C, NT, INV>: the same for a contiguous axis
  // the two innermost axes in one in-place tile per (y, x) plane (plane.cuh); n = NY, n2 = NX (R2C: H), radices = y, radices2 = x
  JIT_PLANE_C2C,    // c2c_plane_ip_kernel<NY, NX, RLY, RLX, NT, INV, REAL>
  JIT_PLANE_R2C,    // r2c_plane_ip_kernel<NY, H, RLY, RLX, NT>
  JIT_ROWS_IP,      // rows_ip_kernel<N, RL, C, NT, INV, REAL>: `tile` rows per CTA, 3-5 stages in ONE shared buffer
  // long half-spectrum rows as two passes (split length H = n/2 for even n, n for odd n); pass A of a real-input or
  // dtype-casting axis is JIT_SPLIT_A with real_in / in_dtype
  JIT_SPLIT_B_R2C,     // rows_split_b_r2c_kernel<N2, RL, C, NT>: even R2C, (k1, N1 - k1) row pairs, Hermitian unpack in the store
  JIT_SPLIT_A_C2R,     // cols_split_a_c2r_kernel<N1, RL, CW, NT, false>: even C2R, Hermitian pack in the load
  JIT_SPLIT_A_C2R_ODD, // cols_split_a_c2r_kernel<N1, RL, CW, NT, true>: odd C2R, Hermitian-extended load
  JIT_SPLIT_B_HALF,    // rows_split_b_kernel<N2, RL, C, NT, false, 1>: odd R2C, bins 0..n/2 stored
  JIT_SPLIT_B_REAL,    // rows_split_b_kernel<N2, RL, C, NT, true, 2>: odd C2R, real parts stored
  // contiguous axes longer than 2^24 points as three passes, n = N1 * N2 * N3 (fast.cuh):
  JIT_SPLIT3_A,        // cols_split_a_kernel<N, RL, CW, NT, INV, REAL, true>: passes 1 and 2, the twiddle from two tables
  JIT_SPLIT3_C         // rows_split_c_kernel<N3, RL, C, NT, INV>: pass 3, rows (k1, k2), natural-order store
};

struct JitSpec {
  JitKind kind = JIT_ROWS;
  int n = 0;  // length of the complex transform the kernel runs (H = n_real / 2 for R2C / R2C_REG / C2R)
  std::vector<int> radices;
  int n2 = 0;                  // plane kinds: the x extent (R2C: H)
  std::vector<int> radices2;   // plane kinds: the x stages
  int tile = 0, threads = 0;
  bool inverse = false, real_in = false, packed = false;
  bool f64 = false;            // working precision (the plan's out_dtype): fp64 = the same kernels with the scalar type swapped
  int in_dtype = B200FFT_F32;  // element type of the array the kernel READS (cast on load)

  size_t esz() const { return f64 ? sizeof(double2) : sizeof(float2); }
  int tile_divides = 0;        // geometry only: the tile must divide this (split pass B rows never straddle transforms)
  long long rows_hint = 0;     // geometry only: transforms per call when the planner knows it (few rows: more threads per row)
  bool plane() const { return kind == JIT_PLANE_C2C || kind == JIT_PLANE_R2C; }
  std::string plane_args() const {  // "<NY, NX, Radices<y...>, Radices<x...>"
    std::string ry, rx;
    for (int r : radices) ry += (ry.empty() ? "" : ", ") + std::to_string(r);
    for (int r : radices2) rx += (rx.empty() ? "" : ", ") + std::to_string(r);
    return std::to_string(n) + ", " + std::to_string(n2) + ", b200fft::Radices<" + ry + ">, b200fft::Radices<" + rx + ">";
  }
  bool strided() const {
    return kind == JIT_COLS || kind == JIT_SCATTER || kind == JIT_SPLIT_A || kind == JIT_SPLIT_B_COLS || kind == JIT_SPLIT_A_C2R ||
           kind == JIT_SPLIT_A_C2R_ODD || kind == JIT_SPLIT3_A;
  }
  std::string radix_list() const {
    std::string s;
    for (int r : radices) s += (s.empty() ? "" : ", ") + std::to_string(r);
    return s;
  }
  std::string shape_args() const {  // "<N, Radices<...>, tile" shared by every kernel and smem-size template
    return std::to_string(n) + ", b200fft::Radices<" + radix_list() + ">, " + std::to_string(tile);
  }
  std::string expression() const {  // the template-id NVRTC instantiates
    const std::string head = shape_args() + ", " + std::to_string(threads);
    const char* inv = inverse ? "true" : "false";
    const char* real = real_in ? "true" : "false";
    switch (kind) {
      case JIT_PLANE_C2C: return "b200fft::c2c_plane_ip_kernel<" + plane_args() + ", " + std::to_string(threads) + ", " + inv + ", " + real + ">";
      case JIT_PLANE_R2C: return "b200fft::r2c_plane_ip_kernel<" + plane_args() + ", " + std::to_string(threads) + ">";
      case JIT_ROWS: return "b200fft::rows_kernel<" + head + ", " + inv + ", " + real + ">";
      case JIT_ROWS_IP:
        return "b200fft::rows_ip_kernel<" + head + ", " + inv + ", " + real + ">";
      case JIT_COLS: return "b200fft::cols_kernel<" + head + ", " + inv + ", " + real + ">";
      case JIT_SCATTER: return "b200fft::cols_scatter_kernel<" + head + ", " + inv + ">";
      case JIT_R2C: return "b200fft::rows_r2c_kernel<" + head + ">";
      case JIT_R2C_REG: return "b200fft::rows_r2c_reg_kernel<" + head + ">";
      case JIT_R2C_ODD: return "b200fft::rows_r2c_odd_kernel<" + head + ">";
      case JIT_C2R_ODD: return "b200fft::rows_c2r_odd_kernel<" + head + ">";
      case JIT_SPLIT_A: return "b200fft::cols_split_a_kernel<" + head + ", " + inv + (real_in ? ", true>" : ">");
      case JIT_SPLIT_A_C2R: return "b200fft::cols_split_a_c2r_kernel<" + head + ", false>";
      case JIT_SPLIT_A_C2R_ODD: return "b200fft::cols_split_a_c2r_kernel<" + head + ", true>";
      case JIT_SPLIT_B_R2C: return "b200fft::rows_split_b_r2c_kernel<" + head + ">";
      case JIT_SPLIT_B_HALF: return "b200fft::rows_split_b_kernel<" + head + ", false, 1>";
      case JIT_SPLIT_B_REAL: return "b200fft::rows_split_b_kernel<" + head + ", true, 2>";
      case JIT_SPLIT_B_COLS: return "b200fft::cols_split_b_kernel<" + head + ", " + inv + ">";
      case JIT_SPLIT_B_ROWS: return "b200fft::rows_split_b_kernel<" + head + ", " + inv + ">";
      case JIT_SPLIT3_A: return "b200fft::cols_split_a_kernel<" + head + ", " + inv + ", " + real + ", true>";
      case JIT_SPLIT3_C: return "b200fft::rows_split_c_kernel<" + head + ", " + inv + ">";
      default: return "b200fft::rows_c2r_kernel<" + head + ">";
    }
  }
  std::string smem_expression() const {  // fast.cuh's own constexpr for the instantiation's dynamic shared memory
    switch (kind) {
      case JIT_PLANE_C2C:
        return "b200fft::c2c_plane_ip_smem_bytes<" + std::to_string(n) + ", " + std::to_string(n2) + ", b200fft::Radices<" +
               std::to_string(radices2[0]) + ", " + std::to_string(radices2[1]) + ">>()";
      case JIT_PLANE_R2C:
        return "b200fft::r2c_plane_ip_smem_bytes<" + std::to_string(n) + ", " + std::to_string(n2) + ", b200fft::Radices<" +
               std::to_string(radices2[0]) + ", " + std::to_string(radices2[1]) + ">>()";
      case JIT_ROWS_IP: return "b200fft::rows_ip_smem_bytes<" + shape_args() + ">()";
      case JIT_ROWS:
      case JIT_SPLIT_B_ROWS:
      case JIT_SPLIT_B_HALF:
      case JIT_SPLIT_B_REAL:
      case JIT_SPLIT3_C:
      case JIT_C2R_ODD:
      case JIT_R2C_ODD: return "b200fft::rows_smem_bytes<" + shape_args() + ">()";
      case JIT_COLS:
      case JIT_SPLIT_A:
      case JIT_SPLIT_B_COLS:
      case JIT_SPLIT_A_C2R:
      case JIT_SPLIT_A_C2R_ODD:
      case JIT_SPLIT3_A:
      case JIT_SCATTER: return "b200fft::cols_smem_bytes<" + shape_args() + ">()";
      case JIT_R2C:
      case JIT_SPLIT_B_R2C: return "b200fft::rows_r2c_smem_bytes<" + shape_args() + ">()";
      case JIT_R2C_REG: return "b200fft::rows_r2c_reg_smem_bytes<" + shape_args() + ">()";
      default: return "b200fft::rows_c2r_smem_bytes<" + shape_args() + ">()";
    }
  }
  std::string name() const {
    static const char* const tag[] = {"jitrows", "jitcols", "jitscatter", "jitr2c", "jitr2creg", "jitr2codd", "jitc2r", "jitc2rodd",
                                      "jitsplitA", "jitsplitBcols", "jitsplitBrows", "jitplane", "jitr2cplane", "jitrowsIP",
                                      "jitsplitBr2c", "jitsplitAc2r", "jitsplitAc2rodd", "jitsplitBhalf", "jitsplitBreal",
                                      "jitsplit3A", "jitsplit3C"};
    if (plane())
      return std::string(tag[kind]) + std::to_string(n) + "x" + std::to_string(kind == JIT_PLANE_R2C ? 2 * n2 : n2) + "(" + radix_name(radices) +
             ";" + radix_name(radices2) + ")_inplace_t" + std::to_string(threads) + (f64 ? "_f64" : "");
    return std::string(tag[kind]) + std::to_string(n) + "_" + radix_name(radices) + (strided() ? "_w" : "_c") + std::to_string(tile) +
           "_t" + std::to_string(threads) + (f64 ? "_f64" : "") + ((kind == JIT_SPLIT_A || kind == JIT_SPLIT3_A) && real_in ? "_realin" : "") + (in_dtype == B200FFT_U8 ? "_inu8" : in_dtype == (f64 ? B200FFT_F32 : B200FFT_F64) ? (f64 ? "_inf32" : "_inf64") : "");
  }
  std::string defines() const {  // rtc_prelude.cuh reads these
    std::string d;
    if (in_dtype == B200FFT_U8) d += "#define B200FFT_JIT_IN_U8 1\n";
    if (in_dtype == B200FFT_F64) d += "#define B200FFT_JIT_IN_F64 1\n";
    if (f64) d += "#define B200FFT_JIT_F64 1\n";
    if (packed && !f64) d += "#define B200FFT_PACKED 1\n";
    return d;
  }
  std::string key() const { return expression() + "|" + defines(); }
  // Host mirror of the smem_expression() formulas (fast.cuh): used to choose the tile before anything is compiled, and
  // checked against the value the compiled module reports (b200fft_jit_smem_bytes) when it is loaded.
  // RowLayout pads a Q-block by P elements when P < 16, Q even and Q < N; DenseLayout is N x CW.
  size_t smem() const {
    if (plane()) return esz() * (size_t)n * (size_t)(n2 + n2 / radices2[0]);  // one buffer of NY rows, pitch NX + NX / r0
    long long P = 1, ex = 0;
    if (kind == JIT_ROWS_IP) {  // rows_ip_smem_bytes: the largest exchange layout, once
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
      case JIT_R2C:
      case JIT_SPLIT_B_R2C: return esz() * (size_t)std::max<long long>(ex, (long long)tile * n) * 2;
      default: return esz() * (size_t)ex * pingpong;
    }
  }
};

struct JitKernel {
  CUmodule module = nullptr;
  CUfunction fn = nullptr;
  int regs = 0, local_bytes = 0;
  size_t cubin_bytes = 0;
  double compile_ms = 0;
};

// compile `spec` to a cubin for sm_100a; `lowered` receives the kernel's mangled name
int compile(const JitSpec& spec, std::vector<char>* cubin, std::string* lowered, std::string* log, double* ms) {
  const Nvrtc& rtc = nvrtc();
  if (!rtc.ok) return fail(B200FFT_ERR_UNSUPPORTED, "run-time compilation unavailable: %s", rtc.why.c_str());
  const auto t0 = std::chrono::steady_clock::now();
  std::string src = spec.defines();
  src += "#include \"fast.cuh\"\n#include \"plane.cuh\"\n";
  src += "extern \"C\" __device__ unsigned long long b200fft_jit_smem_bytes = (unsigned long long)" + spec.smem_expression() + ";\n";
  const char* headers[] = {k_src_rtc_prelude, k_src_dft, k_src_tma, k_src_fast, k_src_plane};
  const char* names[] = {"rtc_prelude.cuh", "dft.cuh", "tma.cuh", "fast.cuh", "plane.cuh"};
  Nvrtc::Program prog = nullptr;
  int rc = rtc.CreateProgram(&prog, src.c_str(), "b200fft_jit.cu", 5, headers, names);
  if (rc) return fail(B200FFT_ERR_CUDA, "nvrtcCreateProgram: %s", rtc.GetErrorString(rc));
  const std::string expr = spec.expression();
  rc = rtc.AddNameExpression(prog, expr.c_str());
  // -default-device: the headers' plain constexpr helpers (index arithmetic, compile-time trigonometry) are device
  // functions here, which is what --expt-relaxed-constexpr gives them under nvcc
  const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "-default-device"};
  if (!rc) rc = rtc.CompileProgram(prog, 4, opts);
  size_t ln = 0;
  if (rtc.GetProgramLogSize(prog, &ln) == 0 && ln > 1) {
    log->resize(ln);
    rtc.GetProgramLog(prog, &(*log)[0]);
  }
  if (rc) {
    rtc.DestroyProgram(&prog);
    return fail(B200FFT_ERR_CUDA, "NVRTC could not compile %s: %s\n%s", expr.c_str(), rtc.GetErrorString(rc), log->c_str());
  }
  const char* low = nullptr;
  size_t nb = 0;
  if ((rc = rtc.GetLoweredName(prog, expr.c_str(), &low)) || (rc = rtc.GetCUBINSize(prog, &nb)) || nb == 0) {
    rtc.DestroyProgram(&prog);
    return fail(B200FFT_ERR_CUDA, "NVRTC produced no cubin for %s", expr.c_str());
  }
  *lowered = low;
  cubin->resize(nb);
  rc = rtc.GetCUBIN(prog, cubin->data());
  rtc.DestroyProgram(&prog);
  if (rc) return fail(B200FFT_ERR_CUDA, "nvrtcGetCUBIN: %s", rtc.GetErrorString(rc));
  *ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  if (const char* dir = getenv("B200FFT_JIT_DUMP_DIR")) {  // keep the cubin (cuobjdump -sass <file>: profiles/sass/)
    const std::string path = std::string(dir) + "/" + spec.name() + ".cubin";
    if (FILE* f = fopen(path.c_str(), "wb")) {
      fwrite(cubin->data(), 1, cubin->size(), f);
      fclose(f);
    }
  }
  return B200FFT_OK;
}

// ---- on-disk cache of compiled kernels: a new process does not pay NVRTC again for a kernel some earlier process built.
// One file per kernel, named by a hash of the specialisation key AND of the embedded header text (a rebuilt library never
// picks up a stale cubin). Directory: $B200FFT_JIT_CACHE_DIR, else $XDG_CACHE_HOME/b200fft, else $HOME/.cache/b200fft;
// B200FFT_JIT_CACHE=0 turns it off; an unwritable directory is silently not used.
uint64_t fnv1a(const char* p, size_t n, uint64_t h = 1469598103934665603ull) {
  for (size_t i = 0; i < n; ++i) h = (h ^ (unsigned char)p[i]) * 1099511628211ull;
  return h;
}
std::string disk_cache_dir() {
  if (const char* e = getenv("B200FFT_JIT_CACHE"))
    if (atoi(e) == 0) return "";
  std::string dir;
  if (const char* e = getenv("B200FFT_JIT_CACHE_DIR")) dir = e;
  else if (const char* x = getenv("XDG_CACHE_HOME")) dir = std::string(x) + "/b200fft";
  else if (const char* h = getenv("HOME")) dir = std::string(h) + "/.cache/b200fft";
  if (dir.empty()) return "";
  std::string partial;
  for (size_t i = 0; i <= dir.size(); ++i)  // mkdir -p
    if (i == dir.size() || (dir[i] == '/' && i > 0)) {
      partial = dir.substr(0, i);
      if (mkdir(partial.c_str(), 0755) != 0 && errno != EEXIST) return "";
    }
  return dir;
}
std::string disk_cache_path(const JitSpec& spec) {
  static const uint64_t src_hash = [] {
    uint64_t h = fnv1a(k_src_rtc_prelude, strlen(k_src_rtc_prelude));
    h = fnv1a(k_src_dft, strlen(k_src_dft), h);
    h = fnv1a(k_src_tma, strlen(k_src_tma), h);
    h = fnv1a(k_src_fast, strlen(k_src_fast), h);
    return fnv1a(k_src_plane, strlen(k_src_plane), h);
  }();
  static const std::string dir = disk_cache_dir();
  if (dir.empty()) return "";
  const std::string key = spec.key() + "|" + spec.smem_expression();
  char name[64];
  snprintf(name, sizeof name, "/%016llx.cubin", (unsigned long long)fnv1a(key.data(), key.size(), src_hash));
  return dir + name;
}
// file = "B2FJ" | u32 name length | lowered name | cubin
bool disk_cache_load(const std::string& path, std::vector<char>* cubin, std::string* lowered) {
  if (path.empty()) return false;
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  char magic[4];
  uint32_t n = 0;
  bool ok = fread(magic, 1, 4, f) == 4 && memcmp(magic, "B2FJ", 4) == 0 && fread(&n, 4, 1, f) == 1 && n > 0 && n < 4096;
  if (ok) {
    lowered->resize(n);
    ok = fread(&(*lowered)[0], 1, n, f) == n;
  }
  if (ok) {
    const long at = ftell(f);
    fseek(f, 0, SEEK_END);
    const long end = ftell(f);
    fseek(f, at, SEEK_SET);
    ok = end > at;
    if (ok) {
      cubin->resize((size_t)(end - at));
      ok = fread(cubin->data(), 1, cubin->size(), f) == cubin->size();
    }
  }
  fclose(f);
  return ok;
}
void disk_cache_store(const std::string& path, const std::vector<char>& cubin, const std::string& lowered) {
  if (path.empty()) return;
  const std::string tmp = path + ".tmp" + std::to_string((long long)getpid());
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return;
  const uint32_t n = (uint32_t)lowered.size();
  const bool ok = fwrite("B2FJ", 1, 4, f) == 4 && fwrite(&n, 4, 1, f) == 1 && fwrite(lowered.data(), 1, n, f) == n &&
                  fwrite(cubin.data(), 1, cubin.size(), f) == cubin.size();
  fclose(f);
  if (!ok || rename(tmp.c_str(), path.c_str()) != 0) remove(tmp.c_str());  // rename: readers never see a partial file
}

std::mutex g_jit_mutex;
std::map<std::string, std::shared_ptr<JitKernel>>& cache() {
  static std::map<std::string, std::shared_ptr<JitKernel>> c;  // key = device ordinal + spec key; modules live until exit
  return c;
}

// compiled + loaded kernel for `spec` on `device` (the current device), from the cache when it was built before
std::shared_ptr<JitKernel> get_kernel(const JitSpec& spec, int device) {
  const Driver& drv = driver();
  if (!drv.ok) {
    fail(B200FFT_ERR_UNSUPPORTED, "driver entry points for module loading are unavailable");
    return nullptr;
  }
  const std::string key = std::to_string(device) + "|" + spec.key();
  std::lock_guard<std::mutex> lock(g_jit_mutex);
  auto it = cache().find(key);
  if (it != cache().end()) return it->second;
  std::vector<char> cubin;
  std::string lowered, log;
  double ms = 0;
  const std::string on_disk = disk_cache_path(spec);
  const bool from_disk = disk_cache_load(on_disk, &cubin, &lowered);
  if (!from_disk) {
    if (compile(spec, &cubin, &lowered, &log, &ms) != B200FFT_OK) {
      if (getenv("B200FFT_JIT_VERBOSE")) fprintf(stderr, "[b200fft jit] %s\n", last_error().c_str());
      cache()[key] = nullptr;  // do not retry a failing compile on every plan
      return nullptr;
    }
    disk_cache_store(on_disk, cubin, lowered);
  }
  auto k = std::make_shared<JitKernel>();
  k->cubin_bytes = cubin.size();
  k->compile_ms = ms;
  cudaFree(0);  // make sure the primary context of the current device exists and is current
  if (drv.ModuleLoadData(&k->module, cubin.data()) != CUDA_SUCCESS || drv.ModuleGetFunction(&k->fn, k->module, lowered.c_str()) != CUDA_SUCCESS) {
    fail(B200FFT_ERR_CUDA, "cannot load the compiled module for %s", spec.expression().c_str());
    if (k->module) drv.ModuleUnload(k->module);
    if (from_disk) remove(on_disk.c_str());  // a damaged cache file: the next plan compiles afresh
    cache()[key] = nullptr;
    return nullptr;
  }
  {  // the instantiation's own idea of its dynamic shared memory must agree with the host mirror the tile was sized with
    CUdeviceptr gp = 0;
    size_t gb = 0;
    unsigned long long reported = ~0ull;
    if (drv.ModuleGetGlobal(&gp, &gb, k->module, "b200fft_jit_smem_bytes") != CUDA_SUCCESS || gb != sizeof reported ||
        cudaMemcpy(&reported, reinterpret_cast<const void*>(gp), sizeof reported, cudaMemcpyDeviceToHost) != cudaSuccess ||
        reported != (unsigned long long)spec.smem()) {
      cudaGetLastError();
      fail(B200FFT_ERR_CUDA, "%s: module reports %llu B of shared memory, the planner computed %zu", spec.name().c_str(), reported,
           spec.smem());
      if (getenv("B200FFT_JIT_VERBOSE")) fprintf(stderr, "[b200fft jit] %s\n", last_error().c_str());
      drv.ModuleUnload(k->module);
      cache()[key] = nullptr;
      return nullptr;
    }
  }
  drv.FuncGetAttribute(&k->regs, CU_FUNC_ATTRIBUTE_NUM_REGS, k->fn);
  drv.FuncGetAttribute(&k->local_bytes, CU_FUNC_ATTRIBUTE_LOCAL_SIZE_BYTES, k->fn);
  const size_t smem = spec.smem();
  if (smem > 48 * 1024 && drv.FuncSetAttribute(k->fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem) != CUDA_SUCCESS) {
    fail(B200FFT_ERR_CUDA, "cannot reserve %zu B of shared memory for %s", smem, spec.name().c_str());
    drv.ModuleUnload(k->module);
    cache()[key] = nullptr;
    return nullptr;
  }
  if (getenv("B200FFT_JIT_VERBOSE"))
    fprintf(stderr, "[b200fft jit] %s: %.0f ms, cubin %zu B, %d registers, %d B local\n", spec.expression().c_str(), ms, cubin.size(),
            k->regs, k->local_bytes);
  cache()[key] = k;
  return k;
}

// Group the user's ordered stage list into super-stages (register codelets): products <= 32, fewest stages, balanced
// (the longest-processing-time rule rt.cu uses); a prime base above 32 (the reference allows any prime, fft.mojo:83-104
// lists up to 97) becomes a stage of its own, up to JIT_MAX_PRIME.
constexpr int JIT_MAX_RADIX = 32;
constexpr int JIT_MAX_PRIME = 127;  // unrolled codelets up to 61, looped ones above (dft.cuh: looped_prime)
constexpr int JIT_MAX_STAGES = 5;

bool jit_group_cap(const std::vector<uint32_t>& ordered, int cap, std::vector<int>* out, int max_stages = JIT_MAX_STAGES) {
  std::vector<uint32_t> small;
  std::vector<int> big;
  auto is_prime = [](uint32_t r) {
    for (uint32_t f = 2; f * f <= r; ++f)
      if (r % f == 0) return false;
    return r > 1;
  };
  for (uint32_t r : ordered) {
    if (r > (uint32_t)JIT_MAX_PRIME) return false;
    // a user base above the cap is a stage of its own: primes up to JIT_MAX_PRIME (looped above 64), composites up to 64 (a
    // fully unrolled Cooley-Tukey codelet; larger ones would take NVRTC tens of seconds and 200+ registers)
    if (r > (uint32_t)cap && !is_prime(r) && r > 64) return false;
    if (r > (uint32_t)cap) big.push_back((int)r);
    else small.push_back(r);
  }
  std::sort(small.begin(), small.end(), [](uint32_t x, uint32_t y) { return x > y; });
  for (int want = small.empty() ? 0 : 1; want + (int)big.size() <= max_stages; ++want) {
    std::vector<long long> g((size_t)want, 1);
    bool ok = true;
    for (uint32_t b : small) {
      int best = -1;
      for (int i = 0; i < want; ++i)
        if (g[i] * b <= cap && (best < 0 || g[i] < g[best])) best = i;
      if (best < 0) { ok = false; break; }
      g[best] *= b;
    }
    if (!ok) continue;
    out->clear();
    for (int b : big) out->push_back(b);
    for (long long v : g)
      if (v > 1) out->push_back((int)v);
    std::sort(out->begin(), out->end(), [](int x, int y) { return x > y; });  // largest radix first
    if (out->empty()) out->push_back(1);
    return true;
  }
  return false;
}

// Codelets of radix <= 32 keep a butterfly in ~64 data registers; when that needs three or more exchanges-worth of
// stages, codelets up to JIT_WIDE_RADIX are tried and kept if they save a stage (1000 = 10 x 10 x 10 -> 40 x 25: one
// shared-memory exchange instead of two).   B200FFT_JIT_MAX_RADIX=<r> overrides the wide cap (A/B knob).
constexpr int JIT_WIDE_RADIX = 50;
constexpr int JIT_MAX_RADIX_F64 = 16;  // a radix-16 fp64 butterfly already holds 64 registers of data
bool jit_group(const std::vector<uint32_t>& ordered, std::vector<int>* out, bool f64 = false) {
  if (f64) return jit_group_cap(ordered, JIT_MAX_RADIX_F64, out);
  if (!jit_group_cap(ordered, JIT_MAX_RADIX, out)) return false;
  int wide = JIT_WIDE_RADIX;
  if (const char* e = getenv("B200FFT_JIT_MAX_RADIX")) wide = std::max(2, std::min(64, atoi(e)));
  if (out->size() >= 3 && wide > JIT_MAX_RADIX) {
    std::vector<int> w;
    if (jit_group_cap(ordered, wide, &w) && w.size() < out->size()) *out = w;
  }
  return true;
}

// Tile shape and CTA size, following the hand-tuned variants (fast_reg_*.cu): about one thread per butterfly of the
// stage with the LARGEST radix (fewest butterflies; up to four rounds when that would be too many threads), tiles of
// 16-48 KB so several CTAs share an SM, strided tiles 16 columns wide (128 contiguous bytes per axis step) unless the
// axis is so long that only 8 fit. Every candidate (tile, rounds) is scored; the cheapest wins.
bool jit_geometry(JitSpec* s, long long inner) {
  const int rmax = *std::max_element(s->radices.begin(), s->radices.end());
  const int rlast = s->radices.back();
  const long long per = (long long)s->n / rmax;  // butterflies of the widest stage per sub-transform
  std::vector<int> tiles;
  if (s->strided()) {
    for (int t : {8, 16, 32, 64})
      if (t <= std::max<long long>(8, (inner + 7) / 8 * 8)) tiles.push_back(t);
    if (inner < 8) tiles.assign(1, (int)inner);
  } else {
    for (int t = 1; t <= 256; ++t) tiles.push_back(t);
  }
  double best = 1e30;
  int best_tile = 0, best_nt = 0;
  for (int tile : tiles) {
    s->tile = tile;
    const size_t smem = s->smem();
    if (smem > 200 * 1024) continue;
    if (s->kind == JIT_R2C_REG && ((long long)tile * (s->n / rlast)) % 32 != 0) continue;  // r2c_reg_ok(): whole warps per row group
    if (s->tile_divides > 0 && s->tile_divides % tile != 0) continue;
    if (s->kind == JIT_SPLIT_B_R2C && tile % 2) continue;  // whole (k1, N1 - k1) row pairs
    const long long work = tile * per;
    const double bytes = (double)tile * s->n * (double)s->esz();
    for (int rounds = 1; rounds <= 4; ++rounds) {
      long long nt = ((work + rounds - 1) / rounds + 31) / 32 * 32;
      if (nt < 64 && rounds > 1) continue;
      if (nt < 32 || nt > 512) continue;
      const double waste = (double)(nt * rounds - work) / (double)(nt * rounds);
      double score = 4.0 * waste + 0.5 * std::fabs(std::log2(bytes / 32768.0)) + 0.3 * std::fabs(std::log2((double)nt / 256.0)) +
                     0.15 * (rounds - 1) + (smem > 64 * 1024 ? 0.5 : 0.0);
      if (s->strided() && tile < 16) score += 0.6;  // 64-byte runs: only when nothing wider fits
      if (score < best) {
        best = score;
        best_tile = tile;
        best_nt = (int)nt;
      }
    }
  }
  if (!best_tile) return false;
  s->tile = best_tile;
  s->threads = best_nt;
  return s->smem() <= 227 * 1024;
}

// rows_ip_kernel (fast.cuh): one row per CTA; the in-place middle stage holds rounds * r1 points per thread in registers
bool jit_rows_ip_geometry(JitSpec* s) {
  if (s->radices.size() < 3 || s->radices.size() > 5) return false;
  const char* env = getenv("B200FFT_ROWS_INPLACE");
  if (env && env[0] == '0') return false;
  double best = 1e30;
  int best_nt = 0, best_tile = 0;
  std::vector<int> order = s->radices, best_order;
  std::sort(order.begin(), order.end());
  const bool few_rows = s->rows_hint > 0 && s->rows_hint <= 2 * 148;
  do {  // the stage ORDER is free (same transform): one whose middle stages fit the register budget
    // one row per CTA: two or three rows per CTA measured no better (11986 x 2187: 0.078 ms at c1 t128, 0.088 at c2 t192;
    // 10485 x 2500: 0.078 vs 0.087), and rows short enough to need it stay on the two-buffer tile (jit_plan_axis)
    for (int tile : {1}) {
      for (int nt = 96; nt <= 512; nt += 32) {
        const long long budget = std::min(64, (std::min(255, 65536 / nt) - 40) / 2);
        long long held = 0;  // complex values a thread keeps across the barrier of an in-place stage
        for (size_t i = 1; i + 1 < order.size(); ++i)
          held = std::max<long long>(held, ((long long)tile * s->n / order[i] + nt - 1) / nt * order[i]);
        if (held > budget) continue;
        double waste = 0;
        for (int r : order) {
          const long long work = (long long)tile * s->n / r, rounds = (work + nt - 1) / nt;
          waste += (double)(rounds * nt - work) / (double)(rounds * nt);
        }
        // under two waves of CTAs the kernel is latency-bound: as many threads per row as the stages feed (10000 points,
        // 100 rows: 0.0125 ms at 256 threads, 0.0105 at 512); 64-thread CTAs run out of CTA slots (14563 x 1800: 0.111 ms)
        const double want_nt = few_rows ? 512.0 : 256.0;
        double score = 4.0 * waste + 0.3 * std::fabs(std::log2((double)nt / want_nt)) + (held > 40 ? 0.5 : 0.0);
        // a permuted order only when the given one does not fit (8738 x 3000: 20x15x10 0.083 ms, 10x20x15 0.128)
        if (order != s->radices) score += 1.0;
        if (score < best) { best = score; best_nt = nt; best_order = order; best_tile = tile; }
      }
    }
  } while (std::next_permutation(order.begin(), order.end()));
  if (!best_nt) return false;
  s->threads = best_nt;
  s->tile = best_tile;
  s->radices = best_order;
  return s->smem() <= 200 * 1024;
}

size_t in_scalar_bytes(int dtype) { return dtype == B200FFT_U8 ? 1 : dtype == B200FFT_F64 ? 8 : 4; }

// rows_r2c_reg_kernel's precondition (fast.cuh: r2c_reg_ok) apart from the tile, which jit_geometry picks
bool r2c_reg_shape_ok(const JitSpec& s) {
  const int P = s.n / s.radices.back();
  return s.radices.size() >= 1 && P >= 8 && P <= 32 && 32 % P == 0;
}

struct JitPass : Pass {
  JitSpec spec;
  std::shared_ptr<JitKernel> k;
  std::shared_ptr<JitKernel> k_scatter;  // compiled on the first launch_scatter
  AxisView view;
  int device = 0;
  bool do_scale = false;
  double scale = 1.0;
  void* d_tw = nullptr;   // stage twiddles, float2 or double2
  void* d_tw2 = nullptr;  // W_n^{+-k} of the Hermitian unpack / pack
  size_t smem = 0;
  std::string text;

  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    return launch_outer(src, dst, nbatch * view.outer_per_batch, stream);
  }
  int run(const JitKernel& kern, const JitSpec& sp, long long grid, void** params, cudaStream_t stream) {
    if (grid <= 0) return B200FFT_OK;
    if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many tiles");
    // a pass that follows another pass of the plan: programmatic dependent launch (fast.cuh: pdl_wait; profiles/r2_pdl.md)
    const bool dependent = (sp.kind == JIT_COLS || sp.kind == JIT_C2R || sp.kind == JIT_C2R_ODD) && driver().LaunchKernelEx && pdl_enabled();
    CUresult r;
    if (dependent) {
      CUlaunchConfig cfg;
      memset(&cfg, 0, sizeof cfg);
      cfg.gridDimX = (unsigned)grid;
      cfg.gridDimY = cfg.gridDimZ = 1;
      cfg.blockDimX = (unsigned)sp.threads;
      cfg.blockDimY = cfg.blockDimZ = 1;
      cfg.sharedMemBytes = (unsigned)sp.smem();
      cfg.hStream = (CUstream)stream;
      CUlaunchAttribute attr;
      memset(&attr, 0, sizeof attr);
      attr.id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
      attr.value.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = &attr;
      cfg.numAttrs = 1;
      r = driver().LaunchKernelEx(&cfg, kern.fn, params, nullptr);
    } else {
      r = driver().LaunchKernel(kern.fn, (unsigned)grid, 1, 1, (unsigned)sp.threads, 1, 1, (unsigned)sp.smem(), (CUstream)stream, params,
                                nullptr);
    }
    if (r != CUDA_SUCCESS) return fail(B200FFT_ERR_CUDA, "launch of %s failed (CUresult %d)", sp.name().c_str(), (int)r);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return B200FFT_OK;
  }
  // Kernel argument blocks. The fp64 build of a kernel sees the same structs with float -> double (rtc_prelude.cuh), so
  // the host fills a struct of that layout.
  struct RowsArgs64 { const void* in; double2* out; const double2* tw; long long nrows; double scale; int do_scale; };
  struct ColsArgs64 { const void* in; double2* out; const double2* tw; long long inner; int tiles_per_outer; double scale; int do_scale; int reverse; };
  struct HalfArgs64 { const void* in; void* out; const double2* tw; const double2* tw2; long long nrows; double scale; };
  template <class A, class T2>
  A cols_args(const void* src, void* dst) const {
    A ca;
    ca.in = src;
    ca.out = reinterpret_cast<T2*>(dst);
    ca.tw = reinterpret_cast<const T2*>(d_tw);
    ca.inner = view.inner;
    ca.tiles_per_outer = (int)((view.inner + spec.tile - 1) / spec.tile);
    ca.scale = scale;
    ca.do_scale = do_scale;
    ca.reverse = reverse_order ? 1 : 0;
    return ca;
  }
  template <class A, class T2>
  int launch_rows(const void* src, void* dst, int64_t outer, cudaStream_t stream) {
    A ra;
    ra.in = src;
    ra.out = reinterpret_cast<T2*>(dst);
    ra.tw = reinterpret_cast<const T2*>(d_tw);
    ra.nrows = outer;
    ra.scale = scale;
    ra.do_scale = do_scale;
    void* params[1] = {&ra};
    return run(*k, spec, (outer + spec.tile - 1) / spec.tile, params, stream);
  }
  template <class A, class T2>
  int launch_half(const void* src, void* dst, int64_t outer, cudaStream_t stream) {
    A ha;
    ha.in = src;
    ha.out = dst;
    ha.tw = reinterpret_cast<const T2*>(d_tw);
    ha.tw2 = reinterpret_cast<const T2*>(d_tw2);
    ha.nrows = outer;
    ha.scale = scale;
    void* params[1] = {&ha};
    return run(*k, spec, (outer + spec.tile - 1) / spec.tile, params, stream);
  }
  int launch_outer(const void* src, void* dst, int64_t outer, cudaStream_t stream) {
    if (spec.kind == JIT_ROWS || spec.kind == JIT_ROWS_IP)
      return spec.f64 ? launch_rows<RowsArgs64, double2>(src, dst, outer, stream) : launch_rows<RowsArgs, float2>(src, dst, outer, stream);
    if (spec.kind == JIT_COLS) {
      void* params[1];
      if (spec.f64) {
        ColsArgs64 ca = cols_args<ColsArgs64, double2>(src, dst);
        params[0] = &ca;
        return run(*k, spec, outer * ca.tiles_per_outer, params, stream);
      }
      ColsArgs ca = cols_args<ColsArgs, float2>(src, dst);
      params[0] = &ca;
      return run(*k, spec, outer * ca.tiles_per_outer, params, stream);
    }
    return spec.f64 ? launch_half<HalfArgs64, double2>(src, dst, outer, stream) : launch_half<HalfArgs, float2>(src, dst, outer, stream);
  }
  int launch_scatter(const void* src, const Scatter& sc, int64_t nbatch, cudaStream_t stream) override {
    if (spec.kind != JIT_COLS || spec.real_in || spec.in_dtype != (spec.f64 ? B200FFT_F64 : B200FFT_F32)) return fail(B200FFT_ERR_UNSUPPORTED, "no scattering store for %s", text.c_str());
    if (sc.npeers < 1 || sc.npeers > 16 || view.n % sc.npeers)
      return fail(B200FFT_ERR_INVALID_ARG, "split axis length %lld is not divisible by %d peers", (long long)view.n, sc.npeers);
    JitSpec sp = spec;
    sp.kind = JIT_SCATTER;
    if (!k_scatter) {
      int cur = -1;
      cudaGetDevice(&cur);
      if (cur != device) cudaSetDevice(device);
      k_scatter = get_kernel(sp, device);
      if (cur != device && cur >= 0) cudaSetDevice(cur);
      if (!k_scatter) return fail(B200FFT_ERR_UNSUPPORTED, "could not specialise the scattering store for %s", text.c_str());
    }
    ScatterArgs sa;  // pointers and integers only: the same block for both precisions
    for (int i = 0; i < 16; ++i) sa.peer[i] = i < sc.npeers ? reinterpret_cast<float2*>(sc.peer_out[i]) : nullptr;
    sa.yl = (int)(view.n / sc.npeers);
    const long long outer = nbatch * view.outer_per_batch;
    sa.zbase = sc.zbase >= 0 ? sc.zbase : (long long)sc.my_rank * outer;
    if (spec.f64) {
      ColsArgs64 ca = cols_args<ColsArgs64, double2>(src, nullptr);
      void* params[2] = {&ca, &sa};
      return run(*k_scatter, sp, outer * ca.tiles_per_outer, params, stream);
    }
    ColsArgs ca = cols_args<ColsArgs, float2>(src, nullptr);
    void* params[2] = {&ca, &sa};
    return run(*k_scatter, sp, outer * ca.tiles_per_outer, params, stream);
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override {
    // even half spectrum: R2C reads the real row as complex pairs, C2R stores it as complex pairs
    if (src) return spec.kind == JIT_R2C || spec.kind == JIT_R2C_REG ? 2 * in_scalar_bytes(spec.in_dtype) : 0;
    return spec.kind == JIT_C2R ? spec.esz() : 0;
  }
};

// fp64 forms of build_twiddles / build_half_twiddles (fast_registry.cu): tw[(j-1)*P + p] = W_{P*R}^{j*p} per stage s >= 1
std::vector<double2> stage_twiddles64(const std::vector<int>& radices, bool inverse) {
  std::vector<double2> t;
  long long P = 1;
  for (size_t s = 0; s < radices.size(); ++s) {
    const int R = radices[s];
    if (s > 0) {
      const long long Q = P * R;
      for (int j = 1; j < R; ++j)
        for (long long p = 0; p < P; ++p) {
          const long double th = 2.0L * 3.14159265358979323846264338327950288L * (long double)((j * p) % Q) / (long double)Q;
          t.push_back(make_double2((double)cosl(th), (double)((inverse ? 1.0L : -1.0L) * sinl(th))));
        }
    }
    P *= R;
  }
  if (t.empty()) t.push_back(make_double2(1.0, 0.0));
  return t;
}
std::vector<double2> half_twiddles64(long long n, bool inverse) {
  std::vector<double2> t;
  for (long long k = 0; k <= n / 2; ++k) {
    const long double th = 2.0L * 3.14159265358979323846264338327950288L * (long double)k / (long double)n;
    t.push_back(make_double2((double)cosl(th), (double)((inverse ? 1.0L : -1.0L) * sinl(th))));
  }
  return t;
}

bool jit_enabled() {
  const char* e = getenv("B200FFT_JIT");
  return !(e && atoi(e) == 0);
}

// kind + transform length + stage list for one axis; false when this tier does not serve it
bool jit_plan_axis(const AxisSpec& ax, const AxisView& view, const IoSpec& src, bool inverse, HalfMode half, bool f64,
                   JitSpec* spec, long long rows_hint = 0) {
  spec->rows_hint = rows_hint;
  spec->inverse = inverse;
  spec->real_in = src.comps == 1;
  spec->f64 = f64;
  spec->in_dtype = src.dtype;
  if (half == HALF_C2R && src.dtype != (f64 ? B200FFT_F64 : B200FFT_F32)) return false;  // the staged half spectrum is read as is
  if (half != HALF_NONE && src.dtype == B200FFT_U8) return false;
  if (half == HALF_NONE) {
    spec->kind = view.inner != 1 ? JIT_COLS : JIT_ROWS;
    spec->n = (int)view.n;
    if (!jit_group(ax.ordered, &spec->radices, f64)) return false;
  } else {
    if (view.inner != 1) return false;  // half-spectrum handling is a row pass
    if (view.n % 2) {
      spec->kind = half == HALF_R2C ? JIT_R2C_ODD : JIT_C2R_ODD;
      spec->n = (int)view.n;
      if (!jit_group(ax.ordered, &spec->radices, f64)) return false;
    } else {
      // n = 2H real points as an H-point complex transform: the user's stage list with one factor 2 removed
      spec->n = (int)(view.n / 2);
      bool ok = false;
      for (const auto& o : drop_factor_two(ax.ordered))
        if (jit_group(o, &spec->radices, f64)) { ok = true; break; }
      if (!ok) return false;
      if (spec->n == 1) return false;
      spec->kind = half == HALF_C2R ? JIT_C2R : JIT_R2C;
      if (half == HALF_R2C && r2c_reg_shape_ok(*spec) && !getenv("B200FFT_R2C_SMEM")) spec->kind = JIT_R2C_REG;
    }
    spec->inverse = half == HALF_C2R;
    spec->real_in = false;
  }
  // packed FADD2 adds: the measured win for mixed-radix and strided kernels, a loss for contiguous power-of-two rows
  // (dft.cuh, profiles/r1_packed_fadd2.md)
  spec->packed = !f64 && (spec->strided() || (spec->n & (spec->n - 1)) != 0);
  // long contiguous rows: two exchange buffers leave one CTA per SM (4096 points, measured 2x slower) or do not fit at
  // all (beyond ~14000); one buffer with the middle stage exchanged in place (profiles/r2_long_rows.md)
  static const long long ip_min_bytes = [] {
    const char* e = getenv("B200FFT_ROWS_INPLACE_MIN");  // row bytes from which the one-buffer kernel is tried
    return e ? atoll(e) : 16384LL;
  }();
  // every 3+-stage row from 2048 points gains at large batch (11986 x 2187: 0.126 -> 0.078 ms, 8738 x 3000: 0.113 -> 0.083;
  // 14563 x 1800 does not: 0.091 -> 0.092); under two waves of CTAs the short ones are a wash or lose a little
  // (100 x 3600: 0.0064 -> 0.0075), so those keep the two-buffer tile
  const long long row_bytes = (long long)spec->n * (long long)spec->esz();
  const bool few_rows = rows_hint > 0 && rows_hint <= 2 * 148;
  // two wide stages containing a radix-40 / 50 codelet lose to three narrow stages in one buffer (26214 x 1000: 40x25
  // 0.097 ms, 10x10x10 in place 0.082; 13107 x 2000: 50x40 0.104, 20x10x10 0.084; 40x40, 36x36 and 48x32 do not)
  if (spec->kind == JIT_ROWS && !f64 && !few_rows && spec->n >= 1000 && spec->radices.size() == 2 && !getenv("B200FFT_JIT_MAX_RADIX")) {
    const int n40 = (int)std::count(spec->radices.begin(), spec->radices.end(), 40);
    const int n50 = (int)std::count(spec->radices.begin(), spec->radices.end(), 50);
    JitSpec narrow = *spec;
    if ((n50 > 0 || n40 == 1) && jit_group_cap(ax.ordered, JIT_MAX_RADIX, &narrow.radices) && narrow.radices.size() == 3) {
      narrow.kind = JIT_ROWS_IP;
      if (jit_rows_ip_geometry(&narrow)) {
        *spec = narrow;
        return true;
      }
    }
  }
  if (spec->kind == JIT_ROWS && row_bytes >= ip_min_bytes && (row_bytes >= 32768 || !few_rows)) {
    spec->kind = JIT_ROWS_IP;
    if (jit_rows_ip_geometry(spec)) return true;
    spec->kind = JIT_ROWS;
  }
  if (!jit_geometry(spec, view.inner)) {
    if (spec->kind != JIT_R2C_REG) return false;
    spec->kind = JIT_R2C;  // no tile keeps whole warps per row group: the shared-memory unpack
    if (!jit_geometry(spec, view.inner)) return false;
  }
  return true;
}

// ---- long axes: N = N1 * N2 as two specialised passes and one plan-owned temporary (split_registry.cu does this for a
// fixed list of (N1, N2); here any factorisation the stage list allows) ---------------------------------------------------
struct JitSplitPass : Pass {
  JitSpec sa, sb;
  std::shared_ptr<JitKernel> ka, kb;
  AxisView view;
  int n1 = 0, n2 = 0;
  bool do_scale = false;
  double scale = 1.0;
  void *twa = nullptr, *twb = nullptr, *tw2 = nullptr, *tmp = nullptr;
  const void* twN = nullptr;
  std::string text;

  struct SplitArgs64 {
    const void* in; double2* out; const double2* tw; const double2* twN; const double2* tw2; long long inner; long long nrows;
    int tiles_per_outer; int n1, n2; double scale; int do_scale;
  };
  template <class A, class T2>
  int go(const void* src, void* dst, long long outer, cudaStream_t stream) {
    A a;
    memset(&a, 0, sizeof a);
    a.inner = view.inner;
    a.n1 = n1;
    a.n2 = n2;
    a.in = src;  // pass A: view (outer, n1, n2 * inner)
    a.out = reinterpret_cast<T2*>(tmp);
    a.tw = reinterpret_cast<const T2*>(twa);
    a.twN = reinterpret_cast<const T2*>(twN);
    a.tw2 = reinterpret_cast<const T2*>(tw2);
    const long long vinner = (long long)n2 * view.inner;
    a.tiles_per_outer = (int)((vinner + sa.tile - 1) / sa.tile);
    void* params[1] = {&a};
    int rc = launch_one(*ka, sa, outer * a.tiles_per_outer, params, stream);
    if (rc != B200FFT_OK) return rc;
    a.in = tmp;  // pass B
    a.out = reinterpret_cast<T2*>(dst);
    a.tw = reinterpret_cast<const T2*>(twb);
    a.scale = scale;
    a.do_scale = do_scale;
    long long grid;
    if (sb.kind == JIT_SPLIT_B_R2C) {  // (n1/2 + 1) row pairs per transform, tile/2 of them per CTA
      a.tiles_per_outer = (int)((n1 / 2 + 1 + sb.tile / 2 - 1) / (sb.tile / 2));
      grid = outer * a.tiles_per_outer;
    } else if (sb.kind != JIT_SPLIT_B_COLS) {
      a.nrows = outer * n1;
      grid = (a.nrows + sb.tile - 1) / sb.tile;
    } else {
      a.tiles_per_outer = (int)((view.inner + sb.tile - 1) / sb.tile);
      grid = outer * n1 * a.tiles_per_outer;
    }
    return launch_one(*kb, sb, grid, params, stream);
  }
  static int launch_one(const JitKernel& kern, const JitSpec& sp, long long grid, void** params, cudaStream_t stream) {
    if (grid <= 0) return B200FFT_OK;
    if (grid > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many tiles");
    const CUresult r = driver().LaunchKernel(kern.fn, (unsigned)grid, 1, 1, (unsigned)sp.threads, 1, 1, (unsigned)sp.smem(),
                                             (CUstream)stream, params, nullptr);
    if (r != CUDA_SUCCESS) return fail(B200FFT_ERR_CUDA, "launch of %s failed (CUresult %d)", sp.name().c_str(), (int)r);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return B200FFT_OK;
  }
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    const long long outer = nbatch * view.outer_per_batch;
    if (outer <= 0) return B200FFT_OK;
    return sa.f64 ? go<SplitArgs64, double2>(src, dst, outer, stream) : go<SplitArgs, float2>(src, dst, outer, stream);
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override {
    // even half spectrum: R2C pass A reads the real row as H complex pairs, C2R pass B stores it as H complex pairs
    if (src) return sb.kind == JIT_SPLIT_B_R2C ? 2 * in_scalar_bytes(sa.in_dtype) : 0;
    return sa.kind == JIT_SPLIT_A_C2R ? sb.esz() : 0;
  }
  int launches() const override { return 2; }
};

// Split the grouped super-stage list into the stages of pass A (product N1) and pass B (product N2): both as close to
// sqrt(N) as the radices allow, each short enough for one tile.
bool jit_split_stages(const std::vector<int>& radices, std::vector<int>* a, std::vector<int>* b) {
  const size_t m = radices.size();
  if (m < 2 || m > 12) return false;
  double best = 1e300;
  for (unsigned mask = 1; mask + 1 < (1u << m); ++mask) {
    long long p1 = 1, p2 = 1;
    int c1 = 0, c2 = 0;
    for (size_t i = 0; i < m; ++i) {
      if (mask >> i & 1) { p1 *= radices[i]; ++c1; }
      else { p2 *= radices[i]; ++c2; }
    }
    if (p1 > 8192 || p2 > 8192 || c1 > 4 || c2 > 4) continue;
    const double score = std::fabs(std::log2((double)p1 / (double)p2)) + 0.25 * (c1 > c2 ? c1 - c2 : c2 - c1);
    if (score < best) {
      best = score;
      a->clear();
      b->clear();
      for (size_t i = 0; i < m; ++i) ((mask >> i & 1) ? a : b)->push_back(radices[i]);
    }
  }
  return best < 1e299;
}

// The two passes of one long axis, decided on the host alone (the plan and b200fft_jit_split_probe share it).
//   complex / real input / cast on load: split n; pass A reads the user's array (real scalars or complex pairs)
//   even-n R2C: split H = n/2 (the real row read as H complex); pass B unpacks mirrored row pairs into n/2+1 bins
//   even-n C2R: split H; pass A packs the half spectrum in its load; pass B writes H complex = the n reals
//   odd-n R2C / C2R: split n; pass B keeps bins 0..n/2 / pass A extends the half spectrum, pass B keeps real parts
struct JitSplitChoice {
  JitSpec sa, sb;
  long long n1 = 0, n2 = 0;
  long long len = 0;  // length of the complex transform the two passes run (H for even half-spectrum rows)
};
bool jit_split_plan(const std::vector<uint32_t>& ordered, const AxisView& view, const IoSpec& src, bool inverse, HalfMode half,
                    bool f64, JitSplitChoice* c) {
  const int work = f64 ? B200FFT_F64 : B200FFT_F32;
  const bool even_half = half != HALF_NONE && view.n % 2 == 0;
  if (half != HALF_NONE) {  // the same input rules as the single-tile half-spectrum kernels (jit_plan_axis)
    if (view.inner != 1 || src.dtype == B200FFT_U8 || (half == HALF_C2R && src.dtype != work)) return false;
  }
  c->len = even_half ? view.n / 2 : view.n;
  if (c->len > SPLIT2_MAX_N) return false;
  const std::vector<std::vector<uint32_t>> options = even_half ? drop_factor_two(ordered) : std::vector<std::vector<uint32_t>>{ordered};
  std::vector<int> all, ra, rb;
  bool ok = false;
  // more stages than one tile takes: the cap on the stage count does not apply to the union of the two passes
  for (const auto& o : options)
    if (jit_group_cap(o, f64 ? JIT_MAX_RADIX_F64 : JIT_MAX_RADIX, &all, 8) && jit_split_stages(all, &ra, &rb)) { ok = true; break; }
  if (!ok) return false;
  c->n1 = c->n2 = 1;
  for (int r : ra) c->n1 *= r;
  for (int r : rb) c->n2 *= r;
  for (JitSpec* s : {&c->sa, &c->sb}) {
    s->inverse = half == HALF_NONE ? inverse : half == HALF_C2R;
    s->f64 = f64;
    s->in_dtype = work;  // pass B reads the temporary
    s->packed = !f64;
  }
  c->sa.in_dtype = src.dtype;
  c->sa.n = (int)c->n1;
  c->sa.radices = ra;
  c->sb.n = (int)c->n2;
  c->sb.radices = rb;
  if (half == HALF_NONE) {
    c->sa.kind = JIT_SPLIT_A;
    c->sa.real_in = src.comps == 1;
    c->sb.kind = view.inner == 1 ? JIT_SPLIT_B_ROWS : JIT_SPLIT_B_COLS;
  } else if (half == HALF_R2C) {
    c->sa.kind = JIT_SPLIT_A;
    c->sa.real_in = !even_half;  // even n: the real row's bytes are H complex pairs
    c->sb.kind = even_half ? JIT_SPLIT_B_R2C : JIT_SPLIT_B_HALF;
  } else {
    c->sa.kind = even_half ? JIT_SPLIT_A_C2R : JIT_SPLIT_A_C2R_ODD;
    c->sb.kind = even_half ? JIT_SPLIT_B_ROWS : JIT_SPLIT_B_REAL;
  }
  if (view.inner == 1 && c->sb.kind != JIT_SPLIT_B_R2C) c->sb.tile_divides = (int)c->n1;  // row tiles never straddle transforms
  return jit_geometry(&c->sa, c->n2 * view.inner) && jit_geometry(&c->sb, view.inner);
}

std::unique_ptr<Pass> make_jit_split_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src, bool scale_inverse,
                                          HalfMode half) {
  const Problem& p = plan.prob;
  const bool f64 = p.desc.out_dtype == B200FFT_F64;
  JitSplitChoice c;
  if (!jit_split_plan(p.axes[axis].ordered, view, src, p.desc.inverse != 0, half, f64, &c)) return nullptr;
  const bool even_half = half != HALF_NONE && c.len != view.n;
  if (!even_half && !plan.tw[axis].ptr) return nullptr;
  auto pass = std::make_unique<JitSplitPass>();
  pass->sa = c.sa;
  pass->sb = c.sb;
  pass->n1 = (int)c.n1;
  pass->n2 = (int)c.n2;
  pass->view = view;
  pass->ka = get_kernel(pass->sa, plan.device);
  pass->kb = pass->ka ? get_kernel(pass->sb, plan.device) : nullptr;
  if (!pass->ka || !pass->kb) return nullptr;
  // the half-spectrum inverse is always normalised (like the single-tile C2R kernels)
  pass->do_scale = scale_inverse || half == HALF_C2R;
  pass->scale = pass->do_scale ? 1.0 / (double)view.n : 1.0;
  auto upload = [&](const void* data, size_t bytes, void** d) {
    if (cudaMalloc(d, bytes) != cudaSuccess) { cudaGetLastError(); return false; }
    plan.owned_device.push_back(*d);
    return cudaMemcpy(*d, data, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  const bool inv = pass->sa.inverse;
  bool ok;
  if (f64) {
    const auto ta = stage_twiddles64(c.sa.radices, inv), tb = stage_twiddles64(c.sb.radices, inv);
    ok = upload(ta.data(), ta.size() * sizeof(double2), &pass->twa) && upload(tb.data(), tb.size() * sizeof(double2), &pass->twb);
  } else {
    const auto ta = build_twiddles(c.sa.radices, inv), tb = build_twiddles(c.sb.radices, inv);
    ok = upload(ta.data(), ta.size() * sizeof(float2), &pass->twa) && upload(tb.data(), tb.size() * sizeof(float2), &pass->twb);
  }
  if (!ok) return nullptr;
  if (!even_half) {
    pass->twN = plan.tw[axis].ptr;  // W_n^m, m in [0, n), in the working precision (api.cu: upload_twiddles)
  } else {
    // the split runs on H = n/2 points: pass A's twiddle is W_H^m, m in [0, H), and the unpack / pack needs W_n^{-+k}, k = 0..H
    void* d = nullptr;
    if (f64) {
      const std::vector<double2> th = half_twiddles64(c.len, inv);  // W_H^m for m = 0..H/2; the rest by symmetry below
      std::vector<double2> full((size_t)c.len);
      for (long long m = 0; m < c.len; ++m) full[(size_t)m] = m <= c.len / 2 ? th[(size_t)m] : make_double2(th[(size_t)(c.len - m)].x, -th[(size_t)(c.len - m)].y);
      const std::vector<double2> t2 = half_twiddles64(view.n, inv);
      ok = upload(full.data(), full.size() * sizeof(double2), &d) && upload(t2.data(), t2.size() * sizeof(double2), &pass->tw2);
    } else {
      std::vector<float2> full((size_t)c.len);
      for (long long m = 0; m < c.len; ++m) {
        const double th = 2.0 * M_PI * (double)m / (double)c.len;
        full[(size_t)m] = make_float2((float)std::cos(th), (float)((inv ? 1.0 : -1.0) * std::sin(th)));
      }
      const std::vector<float2> t2 = build_half_twiddles(view.n, inv);
      ok = upload(full.data(), full.size() * sizeof(float2), &d) && upload(t2.data(), t2.size() * sizeof(float2), &pass->tw2);
    }
    if (!ok) return nullptr;
    pass->twN = d;
  }
  const size_t tmp_bytes = (size_t)p.batch * view.outer_per_batch * c.len * view.inner * pass->sa.esz();
  if (cudaMalloc(&pass->tmp, tmp_bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  plan.owned_device.push_back(pass->tmp);
  plan.workspace_bytes += tmp_bytes;
  std::string stages;
  for (uint32_t r : p.axes[axis].ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  if (stages.size() > 120) stages = stages.substr(0, 117) + "...";
  const char* form = "";
  const char* a_note = "(+W_n twiddle)";
  const char* b_note = "(natural-order store)";
  if (half == HALF_R2C && even_half) {
    form = " r2c";
    a_note = "(+W_H twiddle)";
    b_note = "(mirrored row pairs, unpack in the store)";
  } else if (half == HALF_R2C) {
    form = " r2c";
    a_note = "(real rows, +W_n twiddle)";
    b_note = "(bins 0..n/2 stored)";
  } else if (half == HALF_C2R && even_half) {
    form = " c2r";
    a_note = "(Hermitian pack in the load, +W_H twiddle)";
    b_note = "(natural-order store, 1/n)";
  } else if (half == HALF_C2R) {
    form = " c2r";
    a_note = "(Hermitian-extended load, +W_n twiddle)";
    b_note = "(real parts stored, 1/n)";
  } else if (src.comps == 1) {
    form = " real-in";
  }
  char buf[700];
  snprintf(buf, sizeof buf, "axis %d: split n=%lld%s = %lld x %lld%s inner=%lld: %s %s -> %s %s; temp=%zuB user "
           "stages=[%s] [NVRTC, %.0f + %.0f ms]", axis, (long long)view.n, form, c.n1, c.n2, even_half ? " (H points)" : "",
           (long long)view.inner, pass->sa.name().c_str(), a_note, pass->sb.name().c_str(), b_note, tmp_bytes, stages.c_str(),
           pass->ka->compile_ms, pass->kb->compile_ms);
  pass->text = buf;
  return pass;
}

// ---- contiguous axes longer than 2^24 points: n = N1 * N2 * N3 as three specialised passes and one plan-owned temporary
// (fast.cuh: rows_split_c_kernel). Both twiddles come from two tables of about sqrt(L) entries (SplitTw2Dst), so nothing
// the plan holds grows like n except the temporary.
struct JitSplit3Pass : Pass {
  JitSpec s[3];
  std::shared_ptr<JitKernel> k[3];
  AxisView view;
  int n1 = 0, n2 = 0, n3 = 0;
  bool do_scale = false;
  double scale = 1.0;
  void* tw[3] = {};               // stage twiddles of each pass
  void *hi[2] = {}, *lo[2] = {};  // T_hi / T_lo of W_n (pass 1) and W_M (pass 2)
  void* tmp = nullptr;
  std::string text;

  template <class A, class T2>
  int go(const void* src, void* dst, long long outer, cudaStream_t stream) {
    A a;
    memset(&a, 0, sizeof a);
    void* params[1] = {&a};
    a.inner = 1;
    a.n1 = n1;
    for (int p = 0; p < 2; ++p) {  // 1: view (outer, N1, M), input -> temporary; 2: view (outer N1, N2, N3) in place
      const long long cols = p == 0 ? (long long)n2 * n3 : n3;
      a.in = p == 0 ? src : tmp;
      a.out = reinterpret_cast<T2*>(tmp);
      a.tw = reinterpret_cast<const T2*>(tw[p]);
      a.twN = reinterpret_cast<const T2*>(hi[p]);
      a.tw2 = reinterpret_cast<const T2*>(lo[p]);
      a.n2 = (int)cols;
      a.tiles_per_outer = (int)((cols + s[p].tile - 1) / s[p].tile);
      const int rc = JitSplitPass::launch_one(*k[p], s[p], (p == 0 ? outer : outer * n1) * a.tiles_per_outer, params, stream);
      if (rc != B200FFT_OK) return rc;
    }
    a.in = tmp;  // 3: rows (k1, k2) of the temporary -> natural order
    a.out = reinterpret_cast<T2*>(dst);
    a.tw = reinterpret_cast<const T2*>(tw[2]);
    a.twN = a.tw2 = nullptr;
    a.n2 = n2;
    a.nrows = outer * n1 * n2;
    a.scale = scale;
    a.do_scale = do_scale;
    return JitSplitPass::launch_one(*k[2], s[2], (a.nrows + s[2].tile - 1) / s[2].tile, params, stream);
  }
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    const long long outer = nbatch * view.outer_per_batch;
    if (outer <= 0) return B200FFT_OK;
    return s[0].f64 ? go<JitSplitPass::SplitArgs64, double2>(src, dst, outer, stream) : go<SplitArgs, float2>(src, dst, outer, stream);
  }
  std::string describe() const override { return text; }
  int launches() const override { return 3; }
};

// Every split of the grouped super-stage list into three sets (products N1, N2, N3) of at most 8192 points and 4 stages,
// most balanced first (the measure jit_split_stages applies to two): each assignment of the m <= 12 groups is scored.
// The strided passes 1 and 2 hold fewer points per tile than the row pass 3, so the caller takes the first split whose
// three tiles fit. Each split is returned as its assignment in base 3 (digit i: the set of group i).
std::vector<long long> jit_split3_stages(const std::vector<int>& radices) {
  const size_t m = radices.size();
  std::vector<std::pair<double, long long>> scored;  // (score, assignment)
  if (m < 3 || m > 12) return {};
  long long total = 1;
  for (size_t i = 0; i < m; ++i) total *= 3;
  for (long long code = 0; code < total; ++code) {
    long long p[3] = {1, 1, 1};
    int cnt[3] = {0, 0, 0};
    long long rest = code;
    for (size_t i = 0; i < m; ++i, rest /= 3) {
      p[rest % 3] *= radices[i];
      ++cnt[rest % 3];
    }
    bool ok = true;
    for (int j = 0; j < 3; ++j) ok = ok && cnt[j] > 0 && cnt[j] <= 4 && p[j] <= 8192;
    if (!ok) continue;
    const long long pmax = std::max({p[0], p[1], p[2]}), pmin = std::min({p[0], p[1], p[2]});
    const int cmax = std::max({cnt[0], cnt[1], cnt[2]}), cmin = std::min({cnt[0], cnt[1], cnt[2]});
    scored.emplace_back(std::log2((double)pmax / (double)pmin) + 0.25 * (cmax - cmin), code);
  }
  std::stable_sort(scored.begin(), scored.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
  std::vector<long long> out(scored.size());
  for (size_t k = 0; k < scored.size(); ++k) out[k] = scored[k].second;
  return out;
}

// The three passes of a contiguous axis longer than SPLIT2_MAX_N points, decided on the host alone (the plan and
// b200fft_jit_split3_probe share it). Complex input, or real input with the full spectrum, of any input dtype (cast on
// load in pass 1). False, with the reason in last_error(), for every axis it does not serve.
struct JitSplit3Choice {
  JitSpec s[3];
  long long n[3] = {0, 0, 0};
};
bool jit_split3_plan(const std::vector<uint32_t>& ordered, const AxisView& view, const IoSpec& src, bool inverse, HalfMode half,
                     bool f64, JitSplit3Choice* c) {
  const long long n = view.n;
  const char* why = nullptr;
  char radix_why[64];
  if (n <= SPLIT2_MAX_N) why = "axes up to 2^24 points take the two-pass split";
  else if (half != HALF_NONE)
    why = "half-spectrum rows whose split length is above 2^24 points are not served (B200FFT_REAL_FULL serves real input with "
          "the full spectrum)";
  else if (view.inner != 1) why = "strided axes (inner > 1) longer than 2^24 points are not served; the three-pass split takes contiguous axes";
  for (uint32_t r : ordered)
    if (!why && r > (uint32_t)JIT_MAX_PRIME) {
      snprintf(radix_why, sizeof radix_why, "radix %u is above %d", r, JIT_MAX_PRIME);
      why = radix_why;
    }
  std::vector<int> all;
  std::vector<long long> splits;
  if (!why && jit_group_cap(ordered, f64 ? JIT_MAX_RADIX_F64 : JIT_MAX_RADIX, &all, 12)) splits = jit_split3_stages(all);
  if (!why && splits.empty()) why = "the stage list does not split into three tiles of at most 8192 points and 4 stages each";
  if (why) {
    fail(B200FFT_ERR_UNSUPPORTED, "%lld points: %s", n, why);
    return false;
  }
  const int work = f64 ? B200FFT_F64 : B200FFT_F32;
  for (long long code : splits) {
    std::vector<int> sets[3];
    for (size_t i = 0; i < all.size(); ++i, code /= 3) sets[code % 3].push_back(all[i]);
    for (int j = 0; j < 3; ++j) {
      JitSpec& s = c->s[j];
      s = JitSpec();
      c->n[j] = 1;
      for (int r : sets[j]) c->n[j] *= r;
      s.kind = j < 2 ? JIT_SPLIT3_A : JIT_SPLIT3_C;
      s.n = (int)c->n[j];
      s.radices = sets[j];
      s.inverse = inverse;
      s.f64 = f64;
      s.in_dtype = work;  // passes 2 and 3 read the temporary
      s.packed = !f64;
    }
    c->s[0].in_dtype = src.dtype;
    c->s[0].real_in = src.comps == 1;
    c->s[2].tile_divides = (int)c->n[0];  // a CTA's rows share k2
    if (jit_geometry(&c->s[0], c->n[1] * c->n[2]) && jit_geometry(&c->s[1], c->n[2]) && jit_geometry(&c->s[2], 1)) return true;
  }
  fail(B200FFT_ERR_UNSUPPORTED, "%lld points: no split into three tiles fits shared memory", n);
  return false;
}

// W_L^e = T_hi[e >> s] * T_lo[e & (2^s - 1)] (fast.cuh: SplitTw2Dst): T_hi[h] = W_L^{h 2^s}, h < ceil(L / 2^s), and
// T_lo[j] = W_L^j, j < 2^s; evaluated in double, stored in the working precision T2
template <class T2>
void split_tw2_tables(long long L, bool inverse, std::vector<T2>* thi, std::vector<T2>* tlo) {
  const int s = split_tw_shift(L);
  const long long lo = 1LL << s, hi = (L + lo - 1) / lo;
  auto w = [&](long long e) {
    const double th = 2.0 * M_PI * ((double)e / (double)L);
    T2 v;
    v.x = std::cos(th);
    v.y = (inverse ? 1.0 : -1.0) * std::sin(th);
    return v;
  };
  thi->resize((size_t)hi);
  tlo->resize((size_t)lo);
  for (long long h = 0; h < hi; ++h) (*thi)[(size_t)h] = w(h * lo);
  for (long long j = 0; j < lo; ++j) (*tlo)[(size_t)j] = w(j);
}

// nullptr when the three-pass split does not serve the axis; *status = B200FFT_ERR_ALLOC (not 4) when it would but its
// device memory cannot be allocated
std::unique_ptr<Pass> make_jit_split3_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src, bool scale_inverse,
                                           HalfMode half, int* status) {
  const Problem& p = plan.prob;
  const bool f64 = p.desc.out_dtype == B200FFT_F64;
  JitSplit3Choice c;
  if (!jit_split3_plan(p.axes[axis].ordered, view, src, p.desc.inverse != 0, half, f64, &c)) return nullptr;
  auto pass = std::make_unique<JitSplit3Pass>();
  pass->view = view;
  pass->n1 = (int)c.n[0];
  pass->n2 = (int)c.n[1];
  pass->n3 = (int)c.n[2];
  for (int j = 0; j < 3; ++j) {
    pass->s[j] = c.s[j];
    pass->k[j] = get_kernel(c.s[j], plan.device);
    if (!pass->k[j]) return nullptr;
  }
  pass->do_scale = scale_inverse;
  pass->scale = scale_inverse ? 1.0 / (double)view.n : 1.0;
  auto upload = [&](const void* data, size_t bytes, void** d) {
    if (cudaMalloc(d, bytes) != cudaSuccess) {
      cudaGetLastError();
      *status = fail(B200FFT_ERR_ALLOC, "axis %d: cannot allocate %zu B of three-pass split tables", axis, bytes);
      return false;
    }
    plan.owned_device.push_back(*d);
    return cudaMemcpy(*d, data, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  const bool inv = p.desc.inverse != 0;
  const long long L[2] = {view.n, c.n[1] * c.n[2]};
  bool ok = true;
  if (f64) {
    std::vector<double2> hi, lo;
    for (int j = 0; j < 3 && ok; ++j) {
      const auto t = stage_twiddles64(c.s[j].radices, inv);
      ok = upload(t.data(), t.size() * sizeof(double2), &pass->tw[j]);
    }
    for (int j = 0; j < 2 && ok; ++j) {
      split_tw2_tables(L[j], inv, &hi, &lo);
      ok = upload(hi.data(), hi.size() * sizeof(double2), &pass->hi[j]) && upload(lo.data(), lo.size() * sizeof(double2), &pass->lo[j]);
    }
  } else {
    std::vector<float2> hi, lo;
    for (int j = 0; j < 3 && ok; ++j) {
      const auto t = build_twiddles(c.s[j].radices, inv);
      ok = upload(t.data(), t.size() * sizeof(float2), &pass->tw[j]);
    }
    for (int j = 0; j < 2 && ok; ++j) {
      split_tw2_tables(L[j], inv, &hi, &lo);
      ok = upload(hi.data(), hi.size() * sizeof(float2), &pass->hi[j]) && upload(lo.data(), lo.size() * sizeof(float2), &pass->lo[j]);
    }
  }
  if (!ok) return nullptr;
  const size_t tmp_bytes = (size_t)p.batch * (size_t)view.outer_per_batch * (size_t)view.n * c.s[1].esz();
  if (cudaMalloc(&pass->tmp, tmp_bytes) != cudaSuccess) {
    cudaGetLastError();
    *status = fail(B200FFT_ERR_ALLOC, "axis %d: cannot allocate the %zu B temporary of the three-pass split", axis, tmp_bytes);
    return nullptr;
  }
  plan.owned_device.push_back(pass->tmp);
  plan.workspace_bytes += tmp_bytes;
  std::string stages;
  for (uint32_t r : p.axes[axis].ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  if (stages.size() > 120) stages = stages.substr(0, 117) + "...";
  char buf[800];
  snprintf(buf, sizeof buf, "axis %d: split3 n=%lld%s = %lld x %lld x %lld inner=1: %s (+W_n twiddle, two tables) -> %s (in place, "
           "+W_M twiddle, two tables) -> %s (natural-order store%s); temp=%zuB user stages=[%s] [NVRTC, %.0f + %.0f + %.0f ms]",
           axis, (long long)view.n, src.comps == 1 ? " real-in" : "", c.n[0], c.n[1], c.n[2], c.s[0].name().c_str(),
           c.s[1].name().c_str(), c.s[2].name().c_str(), scale_inverse ? ", 1/n" : "", tmp_bytes, stages.c_str(),
           pass->k[0]->compile_ms, pass->k[1]->compile_ms, pass->k[2]->compile_ms);
  pass->text = buf;
  return pass;
}

}  // namespace

std::unique_ptr<Pass> make_jit_pass(b200fft_plan& plan, int axis, const AxisView& view, const IoSpec& src, bool scale_inverse,
                                    HalfMode half, int* status) {
  const Problem& p = plan.prob;
  if (!jit_enabled() || view.n < 2) {
    if (view.n > SPLIT2_MAX_N)
      fail(B200FFT_ERR_UNSUPPORTED, "%lld points: axes longer than 2^24 points need the plan-time specialisation tier, which "
           "B200FFT_JIT=0 turns off", (long long)view.n);
    return nullptr;
  }
  const bool f64 = p.desc.out_dtype == B200FFT_F64;
  JitSpec spec;
  const long long rows = view.inner == 1 ? (long long)p.batch * view.outer_per_batch : 0;
  if ((view.n > 16384 && view.inner != 1) || view.n > 32768 ||
      !jit_plan_axis(p.axes[axis], view, src, p.desc.inverse != 0, half, f64, &spec, rows)) {
    // too long (or too many stages) for one tile: two passes, or three beyond what two serve
    if (view.n < 1024) return nullptr;
    std::unique_ptr<Pass> pass = make_jit_split_pass(plan, axis, view, src, scale_inverse, half);
    if (!pass && view.n > SPLIT2_MAX_N) pass = make_jit_split3_pass(plan, axis, view, src, scale_inverse, half, status);
    return pass;
  }
  std::shared_ptr<JitKernel> k = get_kernel(spec, plan.device);
  if (!k) return nullptr;
  auto pass = std::make_unique<JitPass>();
  pass->spec = spec;
  pass->k = k;
  pass->view = view;
  pass->device = plan.device;
  pass->do_scale = scale_inverse;
  pass->scale = (scale_inverse || half == HALF_C2R) ? 1.0 / (double)view.n : 1.0;  // the half-spectrum inverse is always normalised
  pass->smem = spec.smem();
  auto upload = [&](const void* data, size_t bytes, void** d) {
    if (cudaMalloc(d, bytes) != cudaSuccess) { cudaGetLastError(); return false; }
    plan.owned_device.push_back(*d);  // owned by the plan before the copy: a failed copy must not leak it
    return cudaMemcpy(*d, data, bytes, cudaMemcpyHostToDevice) == cudaSuccess;
  };
  const bool need_tw2 = half != HALF_NONE && spec.kind != JIT_R2C_ODD && spec.kind != JIT_C2R_ODD;
  if (f64) {
    const std::vector<double2> tw = stage_twiddles64(spec.radices, spec.inverse);
    if (!upload(tw.data(), tw.size() * sizeof(double2), &pass->d_tw)) return nullptr;
    if (need_tw2) {
      const std::vector<double2> t2 = half_twiddles64(view.n, half == HALF_C2R);
      if (!upload(t2.data(), t2.size() * sizeof(double2), &pass->d_tw2)) return nullptr;
    }
  } else {
    const std::vector<float2> tw = build_twiddles(spec.radices, spec.inverse);
    if (!upload(tw.data(), tw.size() * sizeof(float2), &pass->d_tw)) return nullptr;
    if (need_tw2) {
      const std::vector<float2> t2 = build_half_twiddles(view.n, half == HALF_C2R);
      if (!upload(t2.data(), t2.size() * sizeof(float2), &pass->d_tw2)) return nullptr;
    }
  }
  std::string stages;
  for (uint32_t r : p.axes[axis].ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  char buf[400];
  snprintf(buf, sizeof buf, "axis %d: %s n=%lld inner=%lld smem=%zuB regs=%d%s user stages=[%s] fused as %s(%s)%s [NVRTC, %.0f ms]", axis,
           spec.name().c_str(), (long long)view.n, (long long)view.inner, pass->smem, k->regs,
           k->local_bytes ? (" local=" + std::to_string(k->local_bytes) + "B").c_str() : "", stages.c_str(),
           need_tw2 ? "(2)" : "", radix_name(spec.radices).c_str(),
           half == HALF_R2C ? (spec.kind == JIT_R2C_ODD ? " r2c (real rows, bins 0..n/2 stored)" : " r2c")
           : half == HALF_C2R ? (spec.kind == JIT_C2R_ODD ? " c2r (Hermitian-extended load)" : " c2r") : spec.real_in ? " real-in" : "",
           k->compile_ms);
  pass->text = buf;
  return pass;
}

// ---- plane passes for plane sizes without a registered variant: the in-place plane kernels of plane.cuh specialised at
// plan time (any NY x NX whose axes each split into two register stages and whose padded plane fits shared memory) ------
namespace {

struct JitPlanePass : Pass {
  JitSpec spec;
  std::shared_ptr<JitKernel> k;
  long long planes_per_batch = 1;
  float scale = 1.f;
  void *twx = nullptr, *twy = nullptr, *tw2 = nullptr;
  std::string text;
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    PlaneFwdArgs a;
    a.in = src;
    a.out = reinterpret_cast<float2*>(dst);
    a.twx = reinterpret_cast<const float2*>(twx);
    a.twy = reinterpret_cast<const float2*>(twy);
    a.tw2 = reinterpret_cast<const float2*>(tw2);
    a.planes = nbatch * planes_per_batch;
    a.scale = scale;
    a.do_scale = spec.inverse ? 1 : 0;
    if (a.planes <= 0) return B200FFT_OK;
    if (a.planes > 0x7fffffffLL) return fail(B200FFT_ERR_UNSUPPORTED, "too many planes");
    void* params[1] = {&a};
    const CUresult r = driver().LaunchKernel(k->fn, (unsigned)a.planes, 1, 1, (unsigned)spec.threads, 1, 1, (unsigned)spec.smem(),
                                             (CUstream)stream, params, nullptr);
    if (r != CUDA_SUCCESS) return fail(B200FFT_ERR_CUDA, "launch of %s failed (CUresult %d)", spec.name().c_str(), (int)r);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    return B200FFT_OK;
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override {
    // R2C planes read the real rows as complex pairs of the input element type
    return src && spec.kind == JIT_PLANE_R2C ? 2 * in_scalar_bytes(spec.in_dtype) : 0;
  }
};

// exactly two register stages of at most 32 for one axis, or false
bool two_stages(const std::vector<uint32_t>& ordered, std::vector<int>* out) {
  std::vector<uint32_t> bases(ordered);
  std::sort(bases.begin(), bases.end(), [](uint32_t x, uint32_t y) { return x > y; });
  long long g[2] = {1, 1};
  for (uint32_t b : bases) {  // longest-processing-time rule into exactly two groups of product <= 32
    const int i = g[0] <= g[1] ? 0 : 1;
    if (g[i] * b <= JIT_MAX_RADIX) g[i] *= b;
    else if (g[1 - i] * b <= JIT_MAX_RADIX) g[1 - i] *= b;
    else return false;
  }
  if (g[0] < 2 || g[1] < 2) return false;
  out->assign({(int)std::max(g[0], g[1]), (int)std::min(g[0], g[1])});
  return true;
}

}  // namespace

std::unique_ptr<Pass> make_jit_plane_pass(b200fft_plan& plan) {
  const Problem& p = plan.prob;
  if (!jit_enabled() || p.rank < 2 || (p.half && p.desc.inverse)) return nullptr;
  if (const char* e = getenv("B200FFT_JIT_PLANE"))
    if (atoi(e) == 0) return nullptr;
  if (p.desc.out_dtype != B200FFT_F32 || p.desc.in_dtype != B200FFT_F32) return nullptr;
  const int last = p.rank - 1;
  if (!p.axes[last].transformed || !p.axes[last - 1].transformed) return nullptr;
  const bool real_in = !p.half && p.desc.in_components == 1;
  if (real_in && p.desc.inverse) return nullptr;
  if (p.half && p.axes[last].n % 2) return nullptr;
  JitSpec spec;
  spec.kind = p.half ? JIT_PLANE_R2C : JIT_PLANE_C2C;
  spec.n = (int)p.axes[last - 1].n;
  spec.n2 = (int)(p.half ? p.axes[last].n / 2 : p.axes[last].n);
  spec.inverse = p.desc.inverse != 0;
  spec.real_in = real_in;
  if ((long long)spec.n * spec.n2 < 256 || spec.n > 1024 || spec.n2 > 1024) return nullptr;
  if (!two_stages(p.axes[last - 1].ordered, &spec.radices)) return nullptr;
  if (p.half) {
    bool ok = false;
    for (const auto& o : drop_factor_two(p.axes[last].ordered))
      if (two_stages(o, &spec.radices2)) { ok = true; break; }
    if (!ok) return nullptr;
  } else if (!two_stages(p.axes[last].ordered, &spec.radices2)) {
    return nullptr;
  }
  spec.packed = true;
  if (spec.smem() > 150 * 1024) return nullptr;
  // threads: every in-place stage must hold its share of the tile in registers (run_stage_inplace: ROUNDS * R <= 40)
  const long long cols = p.half ? spec.n2 + 1 : spec.n2;
  const long long total_x1 = (long long)spec.n * (spec.n2 / spec.radices2[1]);
  const long long total_y0 = (long long)(spec.n / spec.radices[0]) * cols;
  spec.threads = 0;
  for (int nt : {128, 256, 512, 1024}) {
    const long long rx = (total_x1 + nt - 1) / nt * spec.radices2[1], ry = (total_y0 + nt - 1) / nt * spec.radices[0];
    if (rx <= 40 && ry <= 40 && rx <= 32 + 8 && ry <= 32 + 8) {
      spec.threads = nt;
      if (nt >= 256 || (rx <= 16 && ry <= 16)) break;  // prefer >= 256 threads unless the tile is small
    }
  }
  if (!spec.threads) return nullptr;
  std::shared_ptr<JitKernel> k = get_kernel(spec, plan.device);
  if (!k) return nullptr;
  auto pass = std::make_unique<JitPlanePass>();
  pass->spec = spec;
  pass->k = k;
  pass->planes_per_batch = 1;
  for (int a = 0; a < last - 1; ++a) pass->planes_per_batch *= p.axes[a].n;
  pass->scale = spec.inverse ? (float)(1.0 / ((double)spec.n * spec.n2)) : 1.f;
  auto upload = [&](const std::vector<float2>& t, void** d) {
    if (cudaMalloc(d, t.size() * sizeof(float2)) != cudaSuccess) { cudaGetLastError(); return false; }
    plan.owned_device.push_back(*d);
    return cudaMemcpy(*d, t.data(), t.size() * sizeof(float2), cudaMemcpyHostToDevice) == cudaSuccess;
  };
  if (!upload(build_twiddles(spec.radices, spec.inverse), &pass->twy) || !upload(build_twiddles(spec.radices2, spec.inverse), &pass->twx))
    return nullptr;
  if (p.half && !upload(build_half_twiddles(p.axes[last].n, false), &pass->tw2)) return nullptr;
  char buf[360];
  snprintf(buf, sizeof buf, "axes %d,%d: %s: one in-place tile per (y, x) plane%s, smem=%zuB regs=%d [NVRTC, %.0f ms]", last - 1, last,
           spec.name().c_str(), real_in ? " real-in" : "", spec.smem(), k->regs, k->compile_ms);
  pass->text = buf;
  return pass;
}

namespace {
// compile `spec` (or load it from the on-disk cache) and describe the result; no CUDA device involved
int probe_compile(const JitSpec& spec, std::string* report) {
  std::vector<char> cubin;
  std::string lowered, log;
  double ms = 0;
  const std::string on_disk = disk_cache_path(spec);
  const bool from_disk = disk_cache_load(on_disk, &cubin, &lowered);
  if (!from_disk) {
    const int rc = compile(spec, &cubin, &lowered, &log, &ms);
    if (rc != B200FFT_OK) return rc;
    disk_cache_store(on_disk, cubin, lowered);
  }
  char buf[700];
  snprintf(buf, sizeof buf, "%s: %s, smem=%zuB, cubin=%zuB, %.0f ms%s, symbol %s", spec.name().c_str(), spec.expression().c_str(), spec.smem(),
           cubin.size(), ms, from_disk ? " (disk cache)" : "", lowered.c_str());
  *report = buf;
  return B200FFT_OK;
}
}  // namespace

// Host-only probe (no CUDA device needed): compile the kernel the planner would pick for one axis and report it.
// half: 0 = complex / real-input full spectrum, 1 = R2C rows, 2 = C2R rows
int jit_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
              int in_dtype, int out_dtype, std::string* report) {
  AxisSpec ax;
  ax.n = n;
  ax.ordered = ordered;
  AxisView view;
  view.n = n;
  view.inner = inner;
  IoSpec src;
  src.comps = real_in ? 1 : 2;
  src.dtype = in_dtype;
  JitSpec spec;
  if (!jit_plan_axis(ax, view, src, inverse, (HalfMode)half, out_dtype == B200FFT_F64, &spec))
    return fail(B200FFT_ERR_UNSUPPORTED, "the specialisation tier does not serve this axis (radix above %d, or no tile fits)", JIT_MAX_PRIME);
  return probe_compile(spec, report);
}

// The same for the two passes the planner builds for a long axis (make_jit_split_pass): "<pass A report>; <pass B report>"
int jit_split_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
                    int in_dtype, int out_dtype, std::string* report) {
  AxisView view;
  view.n = n;
  view.inner = inner;
  IoSpec src;
  src.comps = real_in ? 1 : 2;
  src.dtype = in_dtype;
  JitSplitChoice c;
  if (!jit_split_plan(ordered, view, src, inverse, (HalfMode)half, out_dtype == B200FFT_F64, &c))
    return fail(B200FFT_ERR_UNSUPPORTED, "no two-pass split of this axis (a radix above %d, more than 2^24 points, or no tile fits)",
                JIT_MAX_PRIME);
  std::string ra, rb;
  int rc = probe_compile(c.sa, &ra);
  if (rc == B200FFT_OK) rc = probe_compile(c.sb, &rb);
  if (rc != B200FFT_OK) return rc;
  *report = ra + "; " + rb;
  return B200FFT_OK;
}

// The same for the three passes of an axis longer than 2^24 points (make_jit_split3_pass): "<pass 1>; <pass 2>; <pass 3>"
int jit_split3_probe(int64_t n, int64_t inner, const std::vector<uint32_t>& ordered, bool inverse, bool real_in, int half,
                     int in_dtype, int out_dtype, std::string* report) {
  AxisView view;
  view.n = n;
  view.inner = inner;
  IoSpec src;
  src.comps = real_in ? 1 : 2;
  src.dtype = in_dtype;
  JitSplit3Choice c;
  if (!jit_split3_plan(ordered, view, src, inverse, (HalfMode)half, out_dtype == B200FFT_F64, &c)) return B200FFT_ERR_UNSUPPORTED;
  std::string r[3];
  for (int j = 0; j < 3; ++j) {
    const int rc = probe_compile(c.s[j], &r[j]);
    if (rc != B200FFT_OK) return rc;
  }
  *report = r[0] + "; " + r[1] + "; " + r[2];
  return B200FFT_OK;
}

}  // namespace b200fft

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
#include "tile.hpp"

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

}  // namespace

// ---- driver entry points through the runtime (no link against libcuda, like the tensor-map encoder) ----------------
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
    d.LaunchKernelEx = reinterpret_cast<decltype(d.LaunchKernelEx)>(get("cuLaunchKernelEx"));
    d.ok = d.ModuleLoadData && d.ModuleUnload && d.ModuleGetFunction && d.ModuleGetGlobal && d.FuncSetAttribute && d.FuncGetAttribute && d.LaunchKernelEx;
    return d;
  }();
  return api;
}

namespace {

// ---- what to compile: the NVRTC source of a TileSpec (tile.hpp) ----------------------------------------------------
std::string radix_list(const std::vector<int>& radices) {
  std::string s;
  for (int r : radices) s += (s.empty() ? "" : ", ") + std::to_string(r);
  return s;
}
std::string plane_args(const TileSpec& s) {  // "<NY, NX, Radices<y...>, Radices<x...>"
  return std::to_string(s.n) + ", " + std::to_string(s.n2) + ", b200fft::Radices<" + radix_list(s.radices) + ">, b200fft::Radices<" +
         radix_list(s.radices2) + ">";
}
std::string shape_args(const TileSpec& s) {  // "<N, Radices<...>, tile" shared by every kernel and smem-size template
  return std::to_string(s.n) + ", b200fft::Radices<" + radix_list(s.radices) + ">, " + std::to_string(s.tile);
}
std::string expression(const TileSpec& s) {  // the template-id NVRTC instantiates
  const std::string head = shape_args(s) + ", " + std::to_string(s.threads);
  const char* inv = s.inverse ? "true" : "false";
  const char* real = s.real_in ? "true" : "false";
  switch (s.kind) {
    case TILE_PLANE_C2C: return "b200fft::c2c_plane_ip_kernel<" + plane_args(s) + ", " + std::to_string(s.threads) + ", " + inv + ", " + real + ">";
    case TILE_PLANE_R2C: return "b200fft::r2c_plane_ip_kernel<" + plane_args(s) + ", " + std::to_string(s.threads) + ">";
    case TILE_ROWS: return "b200fft::rows_kernel<" + head + ", " + inv + ", " + real + ">";
    case TILE_ROWS_IP:
      return "b200fft::rows_ip_kernel<" + head + ", " + inv + ", " + real + ">";
    case TILE_COLS: return "b200fft::cols_kernel<" + head + ", " + inv + ", " + real + ">";
    case TILE_SCATTER: return "b200fft::cols_scatter_kernel<" + head + ", " + inv + ">";
    case TILE_R2C: return "b200fft::rows_r2c_kernel<" + head + ">";
    case TILE_R2C_REG: return "b200fft::rows_r2c_reg_kernel<" + head + ">";
    case TILE_R2C_ODD: return "b200fft::rows_r2c_odd_kernel<" + head + ">";
    case TILE_C2R_ODD: return "b200fft::rows_c2r_odd_kernel<" + head + ">";
    case TILE_SPLIT_A: return "b200fft::cols_split_a_kernel<" + head + ", " + inv + (s.real_in ? ", true>" : ">");
    case TILE_SPLIT_A_C2R: return "b200fft::cols_split_a_c2r_kernel<" + head + ", false>";
    case TILE_SPLIT_A_C2R_ODD: return "b200fft::cols_split_a_c2r_kernel<" + head + ", true>";
    case TILE_SPLIT_B_R2C: return "b200fft::rows_split_b_r2c_kernel<" + head + ">";
    case TILE_SPLIT_B_HALF: return "b200fft::rows_split_b_kernel<" + head + ", false, 1>";
    case TILE_SPLIT_B_REAL: return "b200fft::rows_split_b_kernel<" + head + ", true, 2>";
    case TILE_SPLIT_B_COLS: return "b200fft::cols_split_b_kernel<" + head + ", " + inv + ">";
    case TILE_SPLIT_B_ROWS: return "b200fft::rows_split_b_kernel<" + head + ", " + inv + ">";
    case TILE_SPLIT3_A: return "b200fft::cols_split_a_kernel<" + head + ", " + inv + ", " + real + ", true>";
    case TILE_SPLIT3_C: return "b200fft::rows_split_c_kernel<" + head + ", " + inv + ">";
    default: return "b200fft::rows_c2r_kernel<" + head + ">";
  }
}
std::string smem_expression(const TileSpec& s) {  // fast.cuh's own constexpr for the instantiation's dynamic shared memory
  switch (s.kind) {
    case TILE_PLANE_C2C:
      return "b200fft::c2c_plane_ip_smem_bytes<" + std::to_string(s.n) + ", " + std::to_string(s.n2) + ", b200fft::Radices<" +
             std::to_string(s.radices2[0]) + ", " + std::to_string(s.radices2[1]) + ">>()";
    case TILE_PLANE_R2C:
      return "b200fft::r2c_plane_ip_smem_bytes<" + std::to_string(s.n) + ", " + std::to_string(s.n2) + ", b200fft::Radices<" +
             std::to_string(s.radices2[0]) + ", " + std::to_string(s.radices2[1]) + ">>()";
    case TILE_ROWS_IP: return "b200fft::rows_ip_smem_bytes<" + shape_args(s) + ">()";
    case TILE_ROWS:
    case TILE_SPLIT_B_ROWS:
    case TILE_SPLIT_B_HALF:
    case TILE_SPLIT_B_REAL:
    case TILE_SPLIT3_C:
    case TILE_C2R_ODD:
    case TILE_R2C_ODD: return "b200fft::rows_smem_bytes<" + shape_args(s) + ">()";
    case TILE_COLS:
    case TILE_SPLIT_A:
    case TILE_SPLIT_B_COLS:
    case TILE_SPLIT_A_C2R:
    case TILE_SPLIT_A_C2R_ODD:
    case TILE_SPLIT3_A:
    case TILE_SCATTER: return "b200fft::cols_smem_bytes<" + shape_args(s) + ">()";
    case TILE_R2C:
    case TILE_SPLIT_B_R2C: return "b200fft::rows_r2c_smem_bytes<" + shape_args(s) + ">()";
    case TILE_R2C_REG: return "b200fft::rows_r2c_reg_smem_bytes<" + shape_args(s) + ">()";
    default: return "b200fft::rows_c2r_smem_bytes<" + shape_args(s) + ">()";
  }
}
std::string jit_name(const TileSpec& s) {
  static const char* const tag[] = {"jitrows", "jitcols", "jitscatter", "jitr2c", "jitr2creg", "jitr2codd", "jitc2r", "jitc2rodd",
                                    "jitsplitA", "jitsplitBcols", "jitsplitBrows", "jitplane", "jitr2cplane", "jitrowsIP",
                                    "jitsplitBr2c", "jitsplitAc2r", "jitsplitAc2rodd", "jitsplitBhalf", "jitsplitBreal",
                                    "jitsplit3A", "jitsplit3C"};
  if (s.plane())
    return std::string(tag[s.kind]) + std::to_string(s.n) + "x" + std::to_string(s.kind == TILE_PLANE_R2C ? 2 * s.n2 : s.n2) + "(" +
           radix_name(s.radices) + ";" + radix_name(s.radices2) + ")_inplace_t" + std::to_string(s.threads) + (s.f64 ? "_f64" : "");
  return std::string(tag[s.kind]) + std::to_string(s.n) + "_" + radix_name(s.radices) + (s.strided() ? "_w" : "_c") + std::to_string(s.tile) +
         "_t" + std::to_string(s.threads) + (s.f64 ? "_f64" : "") + ((s.kind == TILE_SPLIT_A || s.kind == TILE_SPLIT3_A) && s.real_in ? "_realin" : "") +
         (s.in_dtype == B200FFT_U8 ? "_inu8" : s.in_dtype == (s.f64 ? B200FFT_F32 : B200FFT_F64) ? (s.f64 ? "_inf32" : "_inf64") : "");
}
std::string defines(const TileSpec& s) {  // rtc_prelude.cuh reads these
  std::string d;
  if (s.in_dtype == B200FFT_U8) d += "#define B200FFT_JIT_IN_U8 1\n";
  if (s.in_dtype == B200FFT_F64) d += "#define B200FFT_JIT_IN_F64 1\n";
  if (s.f64) d += "#define B200FFT_JIT_F64 1\n";
  if (s.packed && !s.f64) d += "#define B200FFT_PACKED 1\n";
  return d;
}
std::string spec_key(const TileSpec& s) { return expression(s) + "|" + defines(s); }

struct JitKernel {
  CUmodule module = nullptr;
  CUfunction fn = nullptr;
  int regs = 0, local_bytes = 0;
  size_t cubin_bytes = 0;
  double compile_ms = 0;
};

// compile `spec` to a cubin for sm_100a; `lowered` receives the kernel's mangled name
int compile(const TileSpec& spec, std::vector<char>* cubin, std::string* lowered, std::string* log, double* ms) {
  const Nvrtc& rtc = nvrtc();
  if (!rtc.ok) return fail(B200FFT_ERR_UNSUPPORTED, "run-time compilation unavailable: %s", rtc.why.c_str());
  const auto t0 = std::chrono::steady_clock::now();
  std::string src = defines(spec);
  src += "#include \"fast.cuh\"\n#include \"plane.cuh\"\n";
  src += "extern \"C\" __device__ unsigned long long b200fft_jit_smem_bytes = (unsigned long long)" + smem_expression(spec) + ";\n";
  const char* headers[] = {k_src_rtc_prelude, k_src_dft, k_src_tma, k_src_fast, k_src_plane};
  const char* names[] = {"rtc_prelude.cuh", "dft.cuh", "tma.cuh", "fast.cuh", "plane.cuh"};
  Nvrtc::Program prog = nullptr;
  int rc = rtc.CreateProgram(&prog, src.c_str(), "b200fft_jit.cu", 5, headers, names);
  if (rc) return fail(B200FFT_ERR_CUDA, "nvrtcCreateProgram: %s", rtc.GetErrorString(rc));
  const std::string expr = expression(spec);
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
    const std::string path = std::string(dir) + "/" + jit_name(spec) + ".cubin";
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
std::string disk_cache_path(const TileSpec& spec) {
  static const uint64_t src_hash = [] {
    uint64_t h = fnv1a(k_src_rtc_prelude, strlen(k_src_rtc_prelude));
    h = fnv1a(k_src_dft, strlen(k_src_dft), h);
    h = fnv1a(k_src_tma, strlen(k_src_tma), h);
    h = fnv1a(k_src_fast, strlen(k_src_fast), h);
    return fnv1a(k_src_plane, strlen(k_src_plane), h);
  }();
  static const std::string dir = disk_cache_dir();
  if (dir.empty()) return "";
  const std::string key = spec_key(spec) + "|" + smem_expression(spec);
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
std::shared_ptr<JitKernel> get_kernel(const TileSpec& spec, int device) {
  const Driver& drv = driver();
  if (!drv.ok) {
    fail(B200FFT_ERR_UNSUPPORTED, "driver entry points for module loading are unavailable");
    return nullptr;
  }
  const std::string key = std::to_string(device) + "|" + spec_key(spec);
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
    fail(B200FFT_ERR_CUDA, "cannot load the compiled module for %s", expression(spec).c_str());
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
      fail(B200FFT_ERR_CUDA, "%s: module reports %llu B of shared memory, the planner computed %zu", jit_name(spec).c_str(), reported,
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
    fail(B200FFT_ERR_CUDA, "cannot reserve %zu B of shared memory for %s", smem, jit_name(spec).c_str());
    drv.ModuleUnload(k->module);
    cache()[key] = nullptr;
    return nullptr;
  }
  if (getenv("B200FFT_JIT_VERBOSE"))
    fprintf(stderr, "[b200fft jit] %s: %.0f ms, cubin %zu B, %d registers, %d B local\n", expression(spec).c_str(), ms, cubin.size(),
            k->regs, k->local_bytes);
  cache()[key] = k;
  return k;
}

}  // namespace

TileKernel jit_tile_kernel(const TileSpec& spec, int device) {
  const std::shared_ptr<JitKernel> k = get_kernel(spec, device);
  return {nullptr, k ? k->fn : nullptr, jit_name(spec)};
}

namespace {

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
bool jit_geometry(TileSpec* s, long long inner) {
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
    if (s->kind == TILE_R2C_REG && ((long long)tile * (s->n / rlast)) % 32 != 0) continue;  // r2c_reg_ok(): whole warps per row group
    if (s->tile_divides > 0 && s->tile_divides % tile != 0) continue;
    if (s->kind == TILE_SPLIT_B_R2C && tile % 2) continue;  // whole (k1, N1 - k1) row pairs
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
bool jit_rows_ip_geometry(TileSpec* s) {
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

// rows_r2c_reg_kernel's precondition (fast.cuh: r2c_reg_ok) apart from the tile, which jit_geometry picks
bool r2c_reg_shape_ok(const TileSpec& s) {
  const int P = s.n / s.radices.back();
  return s.radices.size() >= 1 && P >= 8 && P <= 32 && 32 % P == 0;
}

bool jit_enabled() {
  const char* e = getenv("B200FFT_JIT");
  return !(e && atoi(e) == 0);
}

// kind + transform length + stage list for one axis; false when this tier does not serve it
bool jit_plan_axis(const AxisSpec& ax, const AxisView& view, const IoSpec& src, bool inverse, HalfMode half, bool f64,
                   TileSpec* spec, long long rows_hint = 0) {
  spec->rows_hint = rows_hint;
  spec->inverse = inverse;
  spec->real_in = src.comps == 1;
  spec->f64 = f64;
  spec->in_dtype = src.dtype;
  if (half == HALF_C2R && src.dtype != (f64 ? B200FFT_F64 : B200FFT_F32)) return false;  // the staged half spectrum is read as is
  if (half != HALF_NONE && src.dtype == B200FFT_U8) return false;
  if (half == HALF_NONE) {
    spec->kind = view.inner != 1 ? TILE_COLS : TILE_ROWS;
    spec->n = (int)view.n;
    if (!jit_group(ax.ordered, &spec->radices, f64)) return false;
  } else {
    if (view.inner != 1) return false;  // half-spectrum handling is a row pass
    if (view.n % 2) {
      spec->kind = half == HALF_R2C ? TILE_R2C_ODD : TILE_C2R_ODD;
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
      spec->kind = half == HALF_C2R ? TILE_C2R : TILE_R2C;
      if (half == HALF_R2C && r2c_reg_shape_ok(*spec) && !getenv("B200FFT_R2C_SMEM")) spec->kind = TILE_R2C_REG;
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
  if (spec->kind == TILE_ROWS && !f64 && !few_rows && spec->n >= 1000 && spec->radices.size() == 2 && !getenv("B200FFT_JIT_MAX_RADIX")) {
    const int n40 = (int)std::count(spec->radices.begin(), spec->radices.end(), 40);
    const int n50 = (int)std::count(spec->radices.begin(), spec->radices.end(), 50);
    TileSpec narrow = *spec;
    if ((n50 > 0 || n40 == 1) && jit_group_cap(ax.ordered, JIT_MAX_RADIX, &narrow.radices) && narrow.radices.size() == 3) {
      narrow.kind = TILE_ROWS_IP;
      if (jit_rows_ip_geometry(&narrow)) {
        *spec = narrow;
        return true;
      }
    }
  }
  if (spec->kind == TILE_ROWS && row_bytes >= ip_min_bytes && (row_bytes >= 32768 || !few_rows)) {
    spec->kind = TILE_ROWS_IP;
    if (jit_rows_ip_geometry(spec)) return true;
    spec->kind = TILE_ROWS;
  }
  if (!jit_geometry(spec, view.inner)) {
    if (spec->kind != TILE_R2C_REG) return false;
    spec->kind = TILE_R2C;  // no tile keeps whole warps per row group: the shared-memory unpack
    if (!jit_geometry(spec, view.inner)) return false;
  }
  return true;
}

// ---- long axes: N = N1 * N2 as two specialised passes and one plan-owned temporary (split_registry.cu does this for a
// fixed list of (N1, N2); here any factorisation the stage list allows) ---------------------------------------------------
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
  TileSpec sa, sb;
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
  for (TileSpec* s : {&c->sa, &c->sb}) {
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
    c->sa.kind = TILE_SPLIT_A;
    c->sa.real_in = src.comps == 1;
    c->sb.kind = view.inner == 1 ? TILE_SPLIT_B_ROWS : TILE_SPLIT_B_COLS;
  } else if (half == HALF_R2C) {
    c->sa.kind = TILE_SPLIT_A;
    c->sa.real_in = !even_half;  // even n: the real row's bytes are H complex pairs
    c->sb.kind = even_half ? TILE_SPLIT_B_R2C : TILE_SPLIT_B_HALF;
  } else {
    c->sa.kind = even_half ? TILE_SPLIT_A_C2R : TILE_SPLIT_A_C2R_ODD;
    c->sb.kind = even_half ? TILE_SPLIT_B_ROWS : TILE_SPLIT_B_REAL;
  }
  if (view.inner == 1 && c->sb.kind != TILE_SPLIT_B_R2C) c->sb.tile_divides = (int)c->n1;  // row tiles never straddle transforms
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
  auto pass = std::make_unique<SplitPass>();
  pass->len[0] = c.n1;
  pass->len[1] = c.n2;
  pass->view = view;
  const TileSpec* spec[2] = {&c.sa, &c.sb};
  std::shared_ptr<JitKernel> k[2];
  for (int i = 0; i < 2; ++i) {
    if (!(k[i] = get_kernel(*spec[i], plan.device))) return nullptr;
    SplitPass::Stage& st = pass->st[i];
    st.spec = *spec[i];
    st.k = {nullptr, k[i]->fn, jit_name(st.spec)};
    st.smem = st.spec.smem();
    st.n2 = (int)c.n2;
  }
  // the half-spectrum inverse is always normalised (like the single-tile C2R kernels)
  pass->do_scale = scale_inverse || half == HALF_C2R;
  pass->scale = pass->do_scale ? 1.0 / (double)view.n : 1.0;
  const bool inv = c.sa.inverse;
  const void *twN = plan.tw[axis].ptr, *tw2 = nullptr;  // W_n^m, m in [0, n), in the working precision (api.cu: upload_twiddles)
  auto tables = [&](auto zero) {
    using T2 = decltype(zero);
    for (int i = 0; i < 2; ++i)
      if (!(pass->st[i].tw = plan_upload(plan, build_twiddles<T2>(spec[i]->radices, inv)))) return false;
    if (!even_half) return true;
    // the split runs on H = n/2 points: pass A's twiddle is W_H^m, m in [0, H), and the unpack / pack needs W_n^{-+k}, k = 0..H
    std::vector<T2> full((size_t)c.len);
    if constexpr (std::is_same<T2, double2>::value) {
      const std::vector<double2> th = build_half_twiddles<double2>(c.len, inv);  // W_H^m for m = 0..H/2; the rest by symmetry
      for (long long m = 0; m < c.len; ++m) full[(size_t)m] = m <= c.len / 2 ? th[(size_t)m] : make_double2(th[(size_t)(c.len - m)].x, -th[(size_t)(c.len - m)].y);
    } else {
      for (long long m = 0; m < c.len; ++m) {
        const double th = 2.0 * M_PI * (double)m / (double)c.len;
        full[(size_t)m] = make_float2((float)std::cos(th), (float)((inv ? 1.0 : -1.0) * std::sin(th)));
      }
    }
    return (twN = plan_upload(plan, full)) && (tw2 = plan_upload(plan, build_half_twiddles<T2>(view.n, inv)));
  };
  if (!(f64 ? tables(double2()) : tables(float2()))) return nullptr;
  for (SplitPass::Stage& st : pass->st) {
    st.twN = twN;
    st.tw2 = tw2;
  }
  const size_t tmp_bytes = (size_t)p.batch * view.outer_per_batch * c.len * view.inner * c.sa.esz();
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
           (long long)view.inner, jit_name(c.sa).c_str(), a_note, jit_name(c.sb).c_str(), b_note, tmp_bytes, stages.c_str(),
           k[0]->compile_ms, k[1]->compile_ms);
  pass->text = buf;
  return pass;
}

// ---- contiguous axes longer than 2^24 points: n = N1 * N2 * N3 as three specialised passes and one plan-owned temporary
// (fast.cuh: rows_split_c_kernel). Both twiddles come from two tables of about sqrt(L) entries (SplitTw2Dst), so nothing
// the plan holds grows like n except the temporary.
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
  TileSpec s[3];
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
      TileSpec& s = c->s[j];
      s = TileSpec();
      c->n[j] = 1;
      for (int r : sets[j]) c->n[j] *= r;
      s.kind = j < 2 ? TILE_SPLIT3_A : TILE_SPLIT3_C;
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
  auto pass = std::make_unique<SplitPass>();
  pass->count = 3;
  pass->view = view;
  std::shared_ptr<JitKernel> k[3];
  for (int j = 0; j < 3; ++j) {
    if (!(k[j] = get_kernel(c.s[j], plan.device))) return nullptr;
    SplitPass::Stage& st = pass->st[j];
    st.spec = c.s[j];
    st.k = {nullptr, k[j]->fn, jit_name(st.spec)};
    st.smem = st.spec.smem();
    pass->len[j] = c.n[j];
  }
  pass->st[0].n2 = (int)(c.n[1] * c.n[2]);  // passes 1 and 2: the columns of their view; pass 3: N2 of the natural-order store
  pass->st[1].n2 = (int)c.n[2];
  pass->st[2].n2 = (int)c.n[1];
  pass->do_scale = scale_inverse;
  pass->scale = scale_inverse ? 1.0 / (double)view.n : 1.0;
  const bool inv = p.desc.inverse != 0;
  const long long L[2] = {view.n, c.n[1] * c.n[2]};
  auto tables = [&](auto zero) {
    using T2 = decltype(zero);
    auto upload = [&](const std::vector<T2>& t, const void** d) {
      if ((*d = plan_upload(plan, t))) return true;
      *status = fail(B200FFT_ERR_ALLOC, "axis %d: cannot allocate %zu B of three-pass split tables", axis, t.size() * sizeof(T2));
      return false;
    };
    std::vector<T2> hi, lo;
    for (int j = 0; j < 3; ++j)
      if (!upload(build_twiddles<T2>(c.s[j].radices, inv), &pass->st[j].tw)) return false;
    for (int j = 0; j < 2; ++j) {  // T_hi / T_lo of W_n (pass 1) and W_M (pass 2)
      split_tw2_tables(L[j], inv, &hi, &lo);
      if (!upload(hi, &pass->st[j].twN) || !upload(lo, &pass->st[j].tw2)) return false;
    }
    return true;
  };
  if (!(f64 ? tables(double2()) : tables(float2()))) return nullptr;
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
           axis, (long long)view.n, src.comps == 1 ? " real-in" : "", c.n[0], c.n[1], c.n[2], jit_name(c.s[0]).c_str(),
           jit_name(c.s[1]).c_str(), jit_name(c.s[2]).c_str(), scale_inverse ? ", 1/n" : "", tmp_bytes, stages.c_str(),
           k[0]->compile_ms, k[1]->compile_ms, k[2]->compile_ms);
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
  TileSpec spec;
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
  auto pass = std::make_unique<TilePass>();
  pass->spec = spec;
  pass->k = {nullptr, k->fn, jit_name(spec)};
  pass->view = view;
  pass->device = plan.device;
  pass->do_scale = scale_inverse;
  pass->scale = (scale_inverse || half == HALF_C2R) ? 1.0 / (double)view.n : 1.0;  // the half-spectrum inverse is always normalised
  pass->smem = spec.smem();
  const bool need_tw2 = half != HALF_NONE && spec.kind != TILE_R2C_ODD && spec.kind != TILE_C2R_ODD;
  auto tables = [&](auto zero) {
    using T2 = decltype(zero);
    return (pass->tw = plan_upload(plan, build_twiddles<T2>(spec.radices, spec.inverse))) &&
           (!need_tw2 || (pass->tw2 = plan_upload(plan, build_half_twiddles<T2>(view.n, half == HALF_C2R))));
  };
  if (!(f64 ? tables(double2()) : tables(float2()))) return nullptr;
  std::string stages;
  for (uint32_t r : p.axes[axis].ordered) stages += (stages.empty() ? "" : ",") + std::to_string(r);
  char buf[400];
  snprintf(buf, sizeof buf, "axis %d: %s n=%lld inner=%lld smem=%zuB regs=%d%s user stages=[%s] fused as %s(%s)%s [NVRTC, %.0f ms]", axis,
           jit_name(spec).c_str(), (long long)view.n, (long long)view.inner, pass->smem, k->regs,
           k->local_bytes ? (" local=" + std::to_string(k->local_bytes) + "B").c_str() : "", stages.c_str(),
           need_tw2 ? "(2)" : "", radix_name(spec.radices).c_str(),
           half == HALF_R2C ? (spec.kind == TILE_R2C_ODD ? " r2c (real rows, bins 0..n/2 stored)" : " r2c")
           : half == HALF_C2R ? (spec.kind == TILE_C2R_ODD ? " c2r (Hermitian-extended load)" : " c2r") : spec.real_in ? " real-in" : "",
           k->compile_ms);
  pass->text = buf;
  return pass;
}

// ---- plane passes for plane sizes without a registered variant: the in-place plane kernels of plane.cuh specialised at
// plan time (any NY x NX whose axes each split into two register stages and whose padded plane fits shared memory) ------
namespace {

struct JitPlanePass : Pass {
  TileSpec spec;
  TileKernel k;
  long long planes_per_batch = 1;
  float scale = 1.f;
  const float2 *twx = nullptr, *twy = nullptr, *tw2 = nullptr;
  std::string text;
  int launch(const void* src, void* dst, int64_t nbatch, cudaStream_t stream) override {
    PlaneFwdArgs a;
    a.in = src;
    a.out = reinterpret_cast<float2*>(dst);
    a.twx = twx;
    a.twy = twy;
    a.tw2 = tw2;
    a.planes = nbatch * planes_per_batch;
    a.scale = scale;
    a.do_scale = spec.inverse ? 1 : 0;
    void* params[1] = {&a};
    return launch_tile(k, a.planes, spec.threads, spec.smem(), false, params, stream);
  }
  std::string describe() const override { return text; }
  size_t min_align(bool src) const override { return tile_min_align({&spec}, src); }
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
  TileSpec spec;
  spec.kind = p.half ? TILE_PLANE_R2C : TILE_PLANE_C2C;
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
  pass->k = {nullptr, k->fn, jit_name(spec)};
  pass->planes_per_batch = 1;
  for (int a = 0; a < last - 1; ++a) pass->planes_per_batch *= p.axes[a].n;
  pass->scale = spec.inverse ? (float)(1.0 / ((double)spec.n * spec.n2)) : 1.f;
  if (!(pass->twy = plan_upload(plan, build_twiddles(spec.radices, spec.inverse))) ||
      !(pass->twx = plan_upload(plan, build_twiddles(spec.radices2, spec.inverse))))
    return nullptr;
  if (p.half && !(pass->tw2 = plan_upload(plan, build_half_twiddles(p.axes[last].n, false)))) return nullptr;
  char buf[360];
  snprintf(buf, sizeof buf, "axes %d,%d: %s: one in-place tile per (y, x) plane%s, smem=%zuB regs=%d [NVRTC, %.0f ms]", last - 1, last,
           jit_name(spec).c_str(), real_in ? " real-in" : "", spec.smem(), k->regs, k->compile_ms);
  pass->text = buf;
  return pass;
}

namespace {
// compile `spec` (or load it from the on-disk cache) and describe the result; no CUDA device involved
int probe_compile(const TileSpec& spec, std::string* report) {
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
  snprintf(buf, sizeof buf, "%s: %s, smem=%zuB, cubin=%zuB, %.0f ms%s, symbol %s", jit_name(spec).c_str(), expression(spec).c_str(), spec.smem(),
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
  TileSpec spec;
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

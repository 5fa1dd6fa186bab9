// Variant table shared by the registration units (fast_reg_*.cu) and the pass factory.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "fast.cuh"
#include "tile.hpp"

namespace b200fft {

// Instantiations a variant may have, one kernel each (null where the variant has none)
enum Form {
  FORM_FWD = 0, FORM_INV, FORM_FWD_REAL, FORM_INV_REAL,  // rows / rowsIP / cols; colsT: FWD and INV only
  FORM_R2C, FORM_C2R, FORM_R2C_REG, FORM_R2C_ODD, FORM_C2R_ODD,  // half-spectrum forms of a row variant
  FORM_SCATTER_FWD, FORM_SCATTER_INV,  // cols: the slab exchange fused into the store
  FORM_COUNT
};

struct Variant {
  std::string name;
  TileKind kind;  // TILE_ROWS, TILE_ROWS_IP, TILE_COLS or TILE_COLS_TMA
  int n;
  std::vector<int> radices;
  int tile, threads;
  size_t smem;
  bool full;   // has inverse and real-input instantiations
  bool vec = false;  // complex-input rows move data with 128-bit accesses ("rowsV")
  // half-spectrum real transforms of length 2*n on top of this n-point row variant (FULL only)
  size_t smem_r2c = 0, smem_c2r = 0;
  size_t smem_r2c_reg = 0;  // R2C with the Hermitian unpack in registers (fast.cuh, R2CRegDst)
  const void* sym[FORM_COUNT] = {};
};

std::vector<Variant>& registry();

// shared with the fused N-d registry (fused_registry.cu)
bool can_group(std::vector<uint32_t> ordered, std::vector<int> target);
std::vector<std::vector<uint32_t>> drop_factor_two(const std::vector<uint32_t>& ordered);
// tensor map over the (inner, n, outer) view of a dense complex64 array, box = (cw, box_rows, 1); false
// when the driver entry point is unavailable or the encode fails
bool encode_axis_map(CUtensorMap* map, const void* base, long long inner, long long n, long long outer, int cw,
                     int box_rows);
bool tensor_maps_available();

template <class RL>
std::vector<int> radix_vec() {
  return std::vector<int>(RL::r, RL::r + RL::count);
}
inline std::string radix_name(const std::vector<int>& r) {
  std::string s;
  for (int v : r) s += (s.empty() ? "" : "x") + std::to_string(v);
  return s;
}

template <int N, int C, int NT, bool FULL, bool VEC, int... Rs>
void reg_rows_impl() {
  using RL = Radices<Rs...>;
  static_assert(RL::product() == N, "radices must multiply to N");
  Variant v;
  v.kind = TILE_ROWS; v.n = N; v.radices = radix_vec<RL>(); v.tile = C; v.threads = NT;
  v.smem = rows_smem_bytes<N, RL, C>();
  v.name = std::string(VEC ? "rowsV" : "rows") + std::to_string(N) + "_" + radix_name(v.radices) + "_c" + std::to_string(C) +
           "_t" + std::to_string(NT);
  v.vec = VEC;
  // FULL variants instantiate forward/inverse x complex/real-input; tuning candidates only forward complex (they are
  // skipped for other requests). Real input keeps the 32-bit loads.
  v.sym[FORM_FWD] = (const void*)rows_kernel<N, RL, C, NT, false, false, VEC>;
  if constexpr (FULL) {
    v.sym[FORM_INV] = (const void*)rows_kernel<N, RL, C, NT, true, false, VEC>;
    v.sym[FORM_FWD_REAL] = (const void*)rows_kernel<N, RL, C, NT, false, true>;
    v.sym[FORM_INV_REAL] = (const void*)rows_kernel<N, RL, C, NT, true, true>;
    v.smem_r2c = rows_r2c_smem_bytes<N, RL, C>();
    v.smem_c2r = rows_c2r_smem_bytes<N, RL, C>();
    if (v.smem_r2c <= 227 * 1024 && v.smem_c2r <= 227 * 1024) {
      v.sym[FORM_R2C] = (const void*)rows_r2c_kernel<N, RL, C, NT>;
      v.sym[FORM_C2R] = (const void*)rows_c2r_kernel<N, RL, C, NT>;
      if constexpr (r2c_reg_ok<N, RL, C, NT>()) {
        v.sym[FORM_R2C_REG] = (const void*)rows_r2c_reg_kernel<N, RL, C, NT>;
        v.smem_r2c_reg = rows_r2c_reg_smem_bytes<N, RL, C>();
      }
    }
    if constexpr (N % 2 == 1) {  // odd n: half-spectrum R2C of length n itself and its inverse on this n-point variant
      v.sym[FORM_R2C_ODD] = (const void*)rows_r2c_odd_kernel<N, RL, C, NT>;
      v.sym[FORM_C2R_ODD] = (const void*)rows_c2r_odd_kernel<N, RL, C, NT>;
    }
  }
  v.full = FULL;
  registry().push_back(v);
}
template <int N, int C, int NT, bool FULL, int... Rs>
void reg_rows() {
  reg_rows_impl<N, C, NT, FULL, false, Rs...>();
}
// 128-bit loads/stores + shuffle exchange for the complex-input instantiations ("rowsV..." variants)
template <int N, int C, int NT, bool FULL, int... Rs>
void reg_rows_v4() {
  reg_rows_impl<N, C, NT, FULL, true, Rs...>();
}
// one long row per CTA, three stages in one shared buffer (rows_ip_kernel): complex or real input, forward and inverse
template <int N, int NT, int... Rs>
void reg_rows_inplace() {
  using RL = Radices<Rs...>;
  static_assert(RL::product() == N, "radices must multiply to N");
  Variant v;
  v.kind = TILE_ROWS_IP; v.n = N; v.radices = radix_vec<RL>(); v.tile = 1; v.threads = NT;
  v.smem = rows_ip_smem_bytes<N, RL>();
  v.name = "rowsIP" + std::to_string(N) + "_" + radix_name(v.radices) + "_c1_t" + std::to_string(NT);
  v.sym[FORM_FWD] = (const void*)rows_ip_kernel<N, RL, 1, NT, false, false>;
  v.sym[FORM_INV] = (const void*)rows_ip_kernel<N, RL, 1, NT, true, false>;
  v.sym[FORM_FWD_REAL] = (const void*)rows_ip_kernel<N, RL, 1, NT, false, true>;
  v.sym[FORM_INV_REAL] = (const void*)rows_ip_kernel<N, RL, 1, NT, true, true>;
  v.full = false;
  registry().push_back(v);
}
template <int N, int CW, int NT, bool FULL, int... Rs>
void reg_cols() {
  using RL = Radices<Rs...>;
  static_assert(RL::product() == N, "radices must multiply to N");
  Variant v;
  v.kind = TILE_COLS; v.n = N; v.radices = radix_vec<RL>(); v.tile = CW; v.threads = NT;
  v.smem = cols_smem_bytes<N, RL, CW>();
  v.name = "cols" + std::to_string(N) + "_" + radix_name(v.radices) + "_w" + std::to_string(CW) + "_t" + std::to_string(NT);
  v.sym[FORM_FWD] = (const void*)cols_kernel<N, RL, CW, NT, false, false>;
  if constexpr (FULL) {
    v.sym[FORM_INV] = (const void*)cols_kernel<N, RL, CW, NT, true, false>;
    v.sym[FORM_FWD_REAL] = (const void*)cols_kernel<N, RL, CW, NT, false, true>;
    v.sym[FORM_INV_REAL] = (const void*)cols_kernel<N, RL, CW, NT, true, true>;
    v.sym[FORM_SCATTER_FWD] = (const void*)cols_scatter_kernel<N, RL, CW, NT, false>;
    v.sym[FORM_SCATTER_INV] = (const void*)cols_scatter_kernel<N, RL, CW, NT, true>;
  }
  v.full = FULL;
  registry().push_back(v);
}

// complex input only: the tensor maps describe complex64 elements
template <int N, int CW, int NT, int... Rs>
void reg_cols_tma() {
  using RL = Radices<Rs...>;
  static_assert(RL::product() == N, "radices must multiply to N");
  Variant v;
  v.kind = TILE_COLS_TMA; v.n = N; v.radices = radix_vec<RL>(); v.tile = CW; v.threads = NT;
  v.smem = cols_tma_smem_bytes<N, CW>();
  v.name = "colsT" + std::to_string(N) + "_" + radix_name(v.radices) + "_w" + std::to_string(CW) + "_t" + std::to_string(NT);
  v.sym[FORM_FWD] = (const void*)cols_tma_kernel<N, RL, CW, NT, false>;
  v.sym[FORM_INV] = (const void*)cols_tma_kernel<N, RL, CW, NT, true>;
  v.full = true;
  registry().push_back(v);
}

}  // namespace b200fft

// Kernels of the two-pass ("four-step") treatment of long axes (fast.cuh: cols_split_a/b, rows_split_b).
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "fast_registry.hpp"

namespace b200fft {

struct SplitKernel {
  std::string name;
  TileKind kind;  // TILE_SPLIT_A, TILE_SPLIT_B_COLS or TILE_SPLIT_B_ROWS
  int n;
  std::vector<int> radices;
  int tile, threads;
  size_t smem;
  const void* sym[2] = {};  // forward, inverse
};

std::vector<SplitKernel>& split_registry();

template <TileKind KIND, int N, int T, int NT, int... Rs>
void reg_split() {
  using RL = Radices<Rs...>;
  static_assert(RL::product() == N, "radices must multiply to N");
  SplitKernel k;
  k.kind = KIND;
  k.n = N;
  k.radices = radix_vec<RL>();
  k.tile = T;
  k.threads = NT;
  const char* tag = KIND == TILE_SPLIT_A ? "splitA_cols" : KIND == TILE_SPLIT_B_COLS ? "splitB_cols" : "splitB_rows";
  k.name = std::string(tag) + std::to_string(N) + "_" + radix_name(k.radices) + (KIND == TILE_SPLIT_B_ROWS ? "_c" : "_w") +
           std::to_string(T) + "_t" + std::to_string(NT);
  if constexpr (KIND == TILE_SPLIT_A) {
    k.smem = cols_smem_bytes<N, RL, T>();
    k.sym[0] = (const void*)cols_split_a_kernel<N, RL, T, NT, false>;
    k.sym[1] = (const void*)cols_split_a_kernel<N, RL, T, NT, true>;
  } else if constexpr (KIND == TILE_SPLIT_B_COLS) {
    k.smem = cols_smem_bytes<N, RL, T>();
    k.sym[0] = (const void*)cols_split_b_kernel<N, RL, T, NT, false>;
    k.sym[1] = (const void*)cols_split_b_kernel<N, RL, T, NT, true>;
  } else {
    k.smem = rows_smem_bytes<N, RL, T>();
    k.sym[0] = (const void*)rows_split_b_kernel<N, RL, T, NT, false>;
    k.sym[1] = (const void*)rows_split_b_kernel<N, RL, T, NT, true>;
  }
  split_registry().push_back(k);
}

}  // namespace b200fft

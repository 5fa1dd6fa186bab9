// Compile-time Stockham kernels: every radix, stride and index is a template constant.
//
// A transform of length N is a fixed list of super-stages R_0..R_{S-1} (prod = N). Stage s
// has P_s = prod_{t<s} R_t, Q_s = P_s*R_s and N/R_s butterflies; butterfly n reads
//     x_j = X[n + j*N/R_s] * W_{Q_s}^{j*(n mod P_s)}          (reference: _fft.mojo:233-267)
// runs the register codelet Dft<R_s> (dft.cuh) and writes Y[(n div P_s)*Q_s + (n mod P_s) + k*P_s].
// Stage 0 reads global memory directly, the last stage writes global memory directly, and
// the S-1 exchanges in between go through shared memory (ping-pong buffers, padded so the
// scatter writes of small-P stages do not bank-conflict). Global memory is touched exactly
// once per element per pass.
//
// One stage template serves three tile shapes through an (outer o, axis index i, inner c)
// index space, c fastest in the butterfly enumeration so a warp's accesses are contiguous:
//   rows   : O = rows per tile, CN = 1     (contiguous 1-D transforms)
//   cols   : O = 1, CN = columns per tile  (strided axis; no transpose kernel)
//   planes : both, back to back, for 2-D tiles that fit shared memory
#pragma once
#include "rtc_prelude.cuh"

#include "dft.cuh"
#include "tma.cuh"

namespace b200fft {

template <int... Rs>
struct Radices {
  static constexpr int count = sizeof...(Rs);
  static constexpr int r[sizeof...(Rs)] = {Rs...};
  static constexpr int product() {
    int p = 1;
    for (int i = 0; i < count; ++i) p *= r[i];
    return p;
  }
  static constexpr int processed(int s) {  // P_s
    int p = 1;
    for (int i = 0; i < s; ++i) p *= r[i];
    return p;
  }
  // offset of stage s in the per-plan twiddle table: stages >= 1 store (R_s - 1) * P_s entries
  static constexpr int tw_offset(int s) {
    int off = 0;
    for (int i = 1; i < s; ++i) off += (r[i] - 1) * processed(i);
    return off;
  }
  static constexpr int tw_total() { return tw_offset(count); }
  static constexpr int max_radix() {
    int m = 0;
    for (int i = 0; i < count; ++i) m = r[i] > m ? r[i] : m;
    return m;
  }
};

// ---- shared-memory exchange layouts --------------------------------------------------------
// rows: element i of row o. After a stage with P < 16 the scatter stride between consecutive
// butterflies is Q (a power of two for the hot sizes): one pad of P elements per Q-block makes
// it odd in units of P, which removes the bank conflicts (see DESIGN.md, exchange padding).
template <int N, int Q, int P>
struct RowLayout {
  static constexpr bool padded = (P < 16) && (Q % 2 == 0) && (Q < N);
  static constexpr int stride = padded ? N + (N / Q) * P : N;
  static constexpr int size(int rows) { return rows * stride; }
  static __device__ __forceinline__ int off(int o, int i, int) {
    if constexpr (padded) return o * stride + i + (i / Q) * P;
    else return o * stride + i;
  }
};
// cols / planes: dense [i][c], c contiguous: conflict-free without padding when CN >= 16
template <int N, int CN>
struct DenseLayout {
  static constexpr int size(int) { return N * CN; }
  static __device__ __forceinline__ int off(int, int i, int c) { return i * CN + c; }
};

// ---- global accessors ------------------------------------------------------------------------
// element (o, i, c) of the tile lives at base[o*so + i*si + c]; rows/columns beyond the valid
// extent (ragged last tile) read as zero and are not written.
// COHERENT: the data may have been written earlier in the SAME kernel by another CTA (fused N-d
// kernel, fused.cuh): read through L2 (ld.global.cg), never through the non-coherent / L1 path.
template <bool REAL, bool COHERENT = false>
struct GlobalSrc {
  const void* __restrict__ base;
  long long so, si;
  int valid_o, valid_c;
  __device__ __forceinline__ float2 load(int o, int i, int c) const {
    if (o >= valid_o || c >= valid_c) return make_float2(0.f, 0.f);
    const long long idx = o * so + i * si + c;
    // in_scalar / in_vec2: the input array's own element type (fp32 except in run-time specialised kernels that read
    // a uint8 / fp64 array, rtc_prelude.cuh), cast to the working precision on load
    if constexpr (REAL) {
      const in_scalar* p = reinterpret_cast<const in_scalar*>(base) + idx;
      return make_float2((float)(COHERENT ? __ldcg(p) : __ldg(p)), 0.f);
    } else {
      const in_vec2* p = reinterpret_cast<const in_vec2*>(base) + idx;
      const in_vec2 v = COHERENT ? __ldcg(p) : __ldg(p);
      return make_float2((float)v.x, (float)v.y);
    }
  }
};
struct GlobalDst {
  float2* __restrict__ base;
  long long so, si;
  int valid_o, valid_c;
  __device__ __forceinline__ void store(int o, int i, int c, float2 v) const {
    if (o >= valid_o || c >= valid_c) return;
    base[o * so + i * si + c] = v;
  }
};
// 128-bit variants for contiguous rows: lanes (2m, 2m+1) own butterflies n = 2m, 2m+1 whose inputs
// x[n + j*NB] and outputs Y[.. + p + k*P] are ADJACENT in memory for every j / k. Each lane moves one
// float4 (both butterflies' element) for half of the j's and the two lanes swap halves with one
// __shfl_xor per element pair: every global access is a 16-byte LDG.128 / STG.128, a warp covers 512
// contiguous bytes, and the exchange between the two butterflies stays inside the warp.
struct GlobalSrcV4 {
  static constexpr bool pairwise = true;
  const float2* __restrict__ base;
  long long so;
  int valid_o;
  __device__ __forceinline__ float4 load2(int o, int i_even) const {
    if (o >= valid_o) return make_float4(0.f, 0.f, 0.f, 0.f);
#ifdef B200FFT_JIT_F64  // never instantiated in fp64 builds (VEC is an fp32 option); there is no 32-byte __ldg
    return *reinterpret_cast<const float4*>(base + o * so + i_even);
#else
    return __ldg(reinterpret_cast<const float4*>(base + o * so + i_even));
#endif
  }
};
struct GlobalDstV4 {
  static constexpr bool pairwise = true;
  float2* __restrict__ base;
  long long so;
  int valid_o;
  __device__ __forceinline__ void store2(int o, int i_even, float4 v) const {
    if (o >= valid_o) return;
    *reinterpret_cast<float4*>(base + o * so + i_even) = v;
  }
};
template <class T, class = void>
struct is_pairwise : std::false_type {};
template <class T>
struct is_pairwise<T, std::enable_if_t<T::pairwise>> : std::true_type {};

// destinations that take a butterfly's R outputs at once (register-level epilogues, e.g. R2CRegDst)
template <class T, class = void>
struct is_whole : std::false_type {};
template <class T>
struct is_whole<T, std::enable_if_t<T::whole>> : std::true_type {};

// sources whose imaginary parts are all zero (real input arrays): stage 0 may use a codelet's real-input form
template <class T>
struct is_real_src : std::false_type {};
template <bool COHERENT>
struct is_real_src<GlobalSrc<true, COHERENT>> : std::true_type {};

template <class Layout>
struct SmemSrc {
  const float2* buf;
  __device__ __forceinline__ float2 load(int o, int i, int c) const { return buf[Layout::off(o, i, c)]; }
};
template <class Layout>
struct SmemDst {
  float2* buf;
  __device__ __forceinline__ void store(int o, int i, int c, float2 v) const { buf[Layout::off(o, i, c)] = v; }
};

// barrier between the stages of a tile: the whole CTA, or (NB) only the NT consumer threads of a
// warp-specialised kernel (named barrier 1; the producer warp never joins it)
template <int NT, bool NB>
__device__ __forceinline__ void tile_sync() {
  if constexpr (NB) asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
  else __syncthreads();
}

// ---- one Stockham stage over a tile -------------------------------------------------------------
// tw points at this stage's table: tw[(j-1)*P + p] = W_{P*R}^{j*p} (conjugated for inverse).
// TWS: `tw` points into shared memory (persistent kernels stage their tables once per CTA)
template <bool TWS>
__device__ __forceinline__ float2 tw_load(const float2* tw, int idx) {
#ifndef B200FFT_JIT_F64  // (the persistent kernels that keep their tables in shared memory are fp32 only)
  if constexpr (TWS) {
    float2 v;
    // volatile + memory clobber: the table is written by other threads of the CTA before a barrier; the
    // compiler must not hoist this load across that barrier (or out of a persistent kernel's tile loop)
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];"
                 : "=f"(v.x), "=f"(v.y)
                 : "r"((unsigned)__cvta_generic_to_shared(tw + idx))
                 : "memory");
    return v;
  }
#endif
  return __ldg(tw + idx);
}

template <int R, int P, int N, int O, int CN, int NT, bool INV, bool TWS = false, class Src, class Dst>
__device__ __forceinline__ void run_stage(const Src& src, const Dst& dst, const float2* __restrict__ tw, float scale,
                                          bool do_scale) {
  constexpr int NB = N / R;  // butterflies per transform
  constexpr int TOTAL = O * NB * CN;
  constexpr int ROUNDS = (TOTAL + NT - 1) / NT;
#pragma unroll(ROUNDS <= 4 ? ROUNDS : 2)
  for (int it = 0; it < ROUNDS; ++it) {
    const int q = (int)threadIdx.x + it * NT;
    if (TOTAL % NT == 0 || q < TOTAL) {
      const int c = (CN == 1) ? 0 : q % CN;
      const int qn = (CN == 1) ? q : q / CN;
      const int n = (O == 1) ? qn : qn % NB;
      const int o = (O == 1) ? 0 : qn / NB;
      const int p = (P == 1) ? 0 : n % P;
      const int g = (P == 1) ? n : n / P;
      float2 x[R];
      if constexpr (is_pairwise<Src>::value) {
        static_assert(CN == 1 && NB % 2 == 0 && R % 2 == 0 && NT % 2 == 0, "pairwise loads: even NB, R, NT");
        const bool odd = (threadIdx.x & 1) != 0;
        const unsigned mask = __activemask();
#pragma unroll
        for (int jj = 0; jj < R / 2; ++jj) {
          // this lane fetches row j = 2jj + odd of the pair (n & ~1, n | 1); the partner fetches the other
          const float4 v = src.load2(o, (n & ~1) + (2 * jj + (odd ? 1 : 0)) * NB);
          const float2 keep = odd ? make_float2(v.z, v.w) : make_float2(v.x, v.y);
          float2 give = odd ? make_float2(v.x, v.y) : make_float2(v.z, v.w);
          give.x = __shfl_xor_sync(mask, give.x, 1);
          give.y = __shfl_xor_sync(mask, give.y, 1);
          x[2 * jj] = odd ? give : keep;
          x[2 * jj + 1] = odd ? keep : give;
        }
      } else {
#pragma unroll
        for (int j = 0; j < R; ++j) x[j] = src.load(o, n + j * NB, c);
      }
      if constexpr (P > 1) {
#pragma unroll
        for (int j = 1; j < R; ++j) x[j] = cmulf(x[j], tw_load<TWS>(tw, (j - 1) * P + p));
      }
      if constexpr (P == 1 && is_real_src<Src>::value && has_run_real<Dft<R, INV>>::value) Dft<R, INV>::run_real(x);
      else Dft<R, INV>::run(x);
      if (do_scale) {
#pragma unroll
        for (int k = 0; k < R; ++k) { x[k].x *= scale; x[k].y *= scale; }
      }
      if constexpr (is_whole<Dst>::value) {
        static_assert(CN == 1 && TOTAL % 32 == 0 && NT % 32 == 0, "whole-butterfly stores: rows, warp-uniform activity");
        dst.template store_all<R, P>(o, g, p, x);
      } else if constexpr (is_pairwise<Dst>::value) {
        static_assert(CN == 1 && P % 2 == 0 && R % 2 == 0 && NT % 2 == 0, "pairwise stores: even P, R, NT");
        const bool odd = (threadIdx.x & 1) != 0;
        const unsigned mask = __activemask();
#pragma unroll
        for (int kk = 0; kk < R / 2; ++kk) {
          // outputs k of butterflies (p & ~1, p | 1) are adjacent: the even lane stores k = 2kk, the odd lane k = 2kk + 1
          float2 give = odd ? x[2 * kk] : x[2 * kk + 1];
          const float2 keep = odd ? x[2 * kk + 1] : x[2 * kk];
          give.x = __shfl_xor_sync(mask, give.x, 1);
          give.y = __shfl_xor_sync(mask, give.y, 1);
          const float4 v = odd ? make_float4(give.x, give.y, keep.x, keep.y) : make_float4(keep.x, keep.y, give.x, give.y);
          dst.store2(o, g * (P * R) + (p & ~1) + (2 * kk + (odd ? 1 : 0)) * P, v);
        }
      } else {
#pragma unroll
        for (int k = 0; k < R; ++k) dst.store(o, g * (P * R) + p + k * P, c, x[k]);
      }
    }
  }
}

// One Stockham stage whose source and destination are the SAME shared-memory buffer: every butterfly of the tile is read
// (and transformed) into registers first, the CTA synchronises, then everything is written back. Needs the whole stage in
// registers — ROUNDS x R complex values per thread — which radix-8 stages of a 64 x 64 plane afford (2 x 8), and halves
// the shared memory of a plane tile: 37 KB instead of 69 KB, six CTAs per SM instead of three.
template <int R, int P, int N, int O, int CN, int NT, bool INV, class Src, class Dst>
__device__ __forceinline__ void run_stage_inplace(const Src& src, const Dst& dst, const float2* __restrict__ tw) {
  constexpr int NB = N / R;
  constexpr int TOTAL = O * NB * CN;
  constexpr int ROUNDS = (TOTAL + NT - 1) / NT;
  static_assert(ROUNDS * R <= 64, "in-place stage: the tile does not fit the register file");
  float2 x[ROUNDS][R];
#pragma unroll
  for (int it = 0; it < ROUNDS; ++it) {
    const int q = (int)threadIdx.x + it * NT;
    if (TOTAL % NT == 0 || q < TOTAL) {
      const int c = (CN == 1) ? 0 : q % CN;
      const int qn = (CN == 1) ? q : q / CN;
      const int n = (O == 1) ? qn : qn % NB;
      const int o = (O == 1) ? 0 : qn / NB;
      const int p = (P == 1) ? 0 : n % P;
#pragma unroll
      for (int j = 0; j < R; ++j) x[it][j] = src.load(o, n + j * NB, c);
      if constexpr (P > 1) {
#pragma unroll
        for (int j = 1; j < R; ++j) x[it][j] = cmulf(x[it][j], __ldg(tw + (j - 1) * P + p));
      }
      Dft<R, INV>::run(x[it]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < ROUNDS; ++it) {
    const int q = (int)threadIdx.x + it * NT;
    if (TOTAL % NT == 0 || q < TOTAL) {
      const int c = (CN == 1) ? 0 : q % CN;
      const int qn = (CN == 1) ? q : q / CN;
      const int n = (O == 1) ? qn : qn % NB;
      const int o = (O == 1) ? 0 : qn / NB;
      const int p = (P == 1) ? 0 : n % P;
      const int g = (P == 1) ? n : n / P;
#pragma unroll
      for (int k = 0; k < R; ++k) dst.store(o, g * (P * R) + p + k * P, c, x[it][k]);
    }
  }
}

// adapters: LayoutFor<Q, P> for a fixed tile shape
template <int N>
struct RowLayoutN {
  template <int Q, int P>
  using type = RowLayout<N, Q, P>;
};
template <int N, int CN>
struct DenseLayoutN {
  template <int Q, int P>
  using type = DenseLayout<N, CN>;
};
// a full 2-D tile [o][i] without padding (hand-over between the two axes of a plane kernel)
template <int NI>
struct PlaneLayout {
  static __device__ __forceinline__ int off(int o, int i, int) { return o * NI + i; }
};

// All stages of one axis over a tile: stage 0 from `src`, last stage to `gdst`; exchange e
// (after stage e) goes through buffer (E0 + e) % 2. LayoutFor<Q, P> gives the exchange layout
// after a stage with those parameters.
template <class RL, int N, int O, int CN, int NT, bool INV, template <int, int> class LayoutFor, int E0 = 0, int S = 0,
          bool NB = false, bool TWS = false, class Src, class GDst>
__device__ __forceinline__ void run_axis(const Src& src, const GDst& gdst, float2* buf0, float2* buf1,
                                         const float2* __restrict__ tw, float scale, bool do_scale) {
  constexpr int R = RL::r[S];
  constexpr int P = RL::processed(S);
  constexpr bool last = (S == RL::count - 1);
  const float2* tws = tw + RL::tw_offset(S);
  if constexpr (last) {
    run_stage<R, P, N, O, CN, NT, INV, TWS>(src, gdst, tws, scale, do_scale);
  } else {
    using L = LayoutFor<P * R, P>;
    float2* buf = ((E0 + S) % 2 == 0) ? buf0 : buf1;
    run_stage<R, P, N, O, CN, NT, INV, TWS>(src, SmemDst<L>{buf}, tws, 1.f, false);
    tile_sync<NT, NB>();
    run_axis<RL, N, O, CN, NT, INV, LayoutFor, E0, S + 1, NB, TWS>(SmemSrc<L>{buf}, gdst, buf0, buf1, tw, scale, do_scale);
  }
}

// largest exchange buffer (in float2) a plan needs
template <class RL, int O, template <int, int> class LayoutFor, int S = 0>
constexpr int max_exchange_elems() {
  if constexpr (S >= RL::count - 1) {
    return 0;
  } else {
    constexpr int P = RL::processed(S);
    constexpr int mine = LayoutFor<P * RL::r[S], P>::size(O);
    constexpr int rest = max_exchange_elems<RL, O, LayoutFor, S + 1>();
    return mine > rest ? mine : rest;
  }
}

// ---- programmatic dependent launch -----------------------------------------------------------------
// A pass that FOLLOWS another pass of a plan is launched with cudaLaunchAttributeProgrammaticStreamSerialization
// (tile.cu: launch_tile): the driver may set its grid up while the previous pass is still running, and its
// CTAs block in pdl_wait until that grid has completed and its writes are visible. For a kernel launched the ordinary way
// pdl_wait is a no-op, so every tile kernel calls it first thing. The previous pass does NOT signal early
// (griddepcontrol.launch_dependents at CTA start was measured: the same gain on most shapes, but the waiting CTAs it lets
// in cost the real-input 2-D shape 3 % and, with plane kernels signalling too, 100 x 64^3 9 %; profiles/r2_pdl.md): what is
// hidden is the launch latency of pass k+1, 2-5 us per boundary.   B200FFT_PDL=0: ordinary launches everywhere.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- kernels ------------------------------------------------------------------------------------
struct RowsArgs {
  const void* in;
  float2* out;
  const float2* tw;
  long long nrows;
  float scale;
  int do_scale;
};

// contiguous rows: tile = C consecutive transforms of length N, one tile per CTA
// VEC: 128-bit global accesses with an intra-warp shuffle exchange (GlobalSrcV4 / GlobalDstV4); needs complex
// input, at least two stages and even N / R_0, R_last, P_last
template <int N, class RL, int C, int NT, bool INV, bool REAL, bool VEC = false>
__global__ void __launch_bounds__(NT) rows_kernel(const __grid_constant__ RowsArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + BUF;
  pdl_wait();
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  const void* in = REAL ? (const void*)(reinterpret_cast<const in_scalar*>(a.in) + row0 * N)
                        : (const void*)(reinterpret_cast<const in_vec2*>(a.in) + row0 * N);
  if constexpr (VEC && !REAL) {
    GlobalSrcV4 src{reinterpret_cast<const float2*>(a.in) + row0 * N, N, valid};
    GlobalDstV4 dst{a.out + row0 * N, N, valid};
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, buf0, buf1, a.tw, a.scale, a.do_scale != 0);
  } else {
    GlobalSrc<REAL> src{in, N, 1, valid, 1};
    GlobalDst dst{a.out + row0 * N, N, 1, valid, 1};
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, buf0, buf1, a.tw, a.scale, a.do_scale != 0);
  }
}
template <int N, class RL, int C>
constexpr size_t rows_smem_bytes() {
  return sizeof(float2) * (size_t)max_exchange_elems<RL, C, RowLayoutN<N>::template type>() * (RL::count > 2 ? 2 : 1);
}

// One LONG contiguous transform per CTA (8192 < N <= ~24000: two exchange buffers no longer fit shared memory): three stages
// in ONE buffer, the middle stage exchanged in place through registers. (100, 16384) — the one published shape that
// ran behind cuFFT as two split passes of ~11 us each — is a single launch of 100 CTAs this way.
template <int N, class RL, int C = 1>
constexpr size_t rows_ip_smem_bytes() {
  int ex = 0;
  for (int s = 0; s + 1 < RL::count; ++s) {  // RowLayout<N, Q, P>::size(C) of every exchange, the largest
    const int P = RL::processed(s), Q = P * RL::r[s];
    const int e = (P < 16 && Q % 2 == 0 && Q < N) ? N + (N / Q) * P : N;
    ex = e > ex ? e : ex;
  }
  return sizeof(float2) * (size_t)ex * C;
}
// stages 1 .. count-2: shared -> registers -> barrier -> the same shared buffer in the next layout
template <int N, class RL, int C, int NT, bool INV, int S>
__device__ __forceinline__ void rows_ip_middle(float2* buf, const float2* __restrict__ tw) {
  if constexpr (S + 1 < RL::count) {
    constexpr int P = RL::processed(S);
    using Lin = RowLayout<N, P, P / RL::r[S - 1]>;
    using Lout = RowLayout<N, P * RL::r[S], P>;
    run_stage_inplace<RL::r[S], P, N, C, 1, NT, INV>(SmemSrc<Lin>{buf}, SmemDst<Lout>{buf}, tw + RL::tw_offset(S));
    __syncthreads();
    rows_ip_middle<N, RL, C, NT, INV, S + 1>(buf, tw);
  }
}
template <int N, class RL, int C, int NT, bool INV, bool REAL = false>
__global__ void __launch_bounds__(NT) rows_ip_kernel(const __grid_constant__ RowsArgs a) {
  static_assert(RL::count >= 3 && RL::product() == N, "three or more stages that multiply to N");
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  const long long row0 = (long long)blockIdx.x * C;
  // one row per CTA: the grid is the row count, no ragged tile, and the accessors' bounds checks fold away
  const int valid = C == 1 ? 1 : (int)min((long long)C, a.nrows - row0);
  constexpr int L = RL::count - 1;
  using L0 = RowLayout<N, RL::r[0], 1>;
  using LL = RowLayout<N, RL::processed(L), RL::processed(L - 1)>;
  const void* in = REAL ? (const void*)(reinterpret_cast<const in_scalar*>(a.in) + row0 * N)
                        : (const void*)(reinterpret_cast<const in_vec2*>(a.in) + row0 * N);
  GlobalSrc<REAL> src{in, N, 1, valid, 1};
  run_stage<RL::r[0], 1, N, C, 1, NT, INV>(src, SmemDst<L0>{smem_f2}, a.tw, 1.f, false);
  __syncthreads();
  rows_ip_middle<N, RL, C, NT, INV, 1>(smem_f2, a.tw);
  GlobalDst dst{a.out + row0 * N, N, 1, valid, 1};
  run_stage<RL::r[L], RL::processed(L), N, C, 1, NT, INV>(SmemSrc<LL>{smem_f2}, dst, a.tw + RL::tw_offset(L), a.scale, a.do_scale != 0);
}

// strided axis, TMA-tiled: the tile [N][CW] is fetched by cp.async.bulk.tensor.3d box loads (tensor
// map over the (inner, N, outer) view of the array) into shared memory, completion on an mbarrier;
// every stage runs shared -> registers -> shared, and the finished tile leaves through a TMA store.
// No thread issues a global load or store: the strided-axis "transpose" is done by the TMA unit.
struct ColsTmaArgs {
  const float2* tw;
  int tiles_per_outer;
  float scale;
  int do_scale;
};

constexpr int tma_box_rows(int n) {
  int r = n < 256 ? n : 256;
  while (n % r) --r;
  return r;
}

template <int N, class RL, int CW, int NT, bool INV>
__global__ void __launch_bounds__(NT) cols_tma_kernel(const __grid_constant__ CUtensorMap map_in,
                                                      const __grid_constant__ CUtensorMap map_out,
                                                      const __grid_constant__ ColsTmaArgs a) {
  extern __shared__ __align__(128) float2 smem_f2[];
  __shared__ __align__(8) uint64_t bar;
  constexpr int BR = tma_box_rows(N);
  constexpr int TILE = N * CW;
  float2* b0 = smem_f2;
  float2* b1 = smem_f2 + TILE;
  const int o = blockIdx.x / a.tiles_per_outer;
  const int c0 = (blockIdx.x - o * a.tiles_per_outer) * CW;
  if (threadIdx.x == 0) {
    tma::prefetch_map(&map_in);
    tma::prefetch_map(&map_out);
    tma::mbar_init(&bar, 1);
    tma::fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    tma::mbar_arrive_expect_tx(&bar, TILE * (uint32_t)sizeof(float2));
#pragma unroll
    for (int b = 0; b < N / BR; ++b) tma::load_3d(b0 + b * BR * CW, &map_in, c0, b * BR, o, &bar);
  }
  tma::mbar_wait(&bar, 0);
  // stage s reads buffer s % 2 and writes buffer (s + 1) % 2; the result ends in buffer S % 2
  float2* res = (RL::count % 2 == 0) ? b0 : b1;
  using L = DenseLayout<N, CW>;
  run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type, /*E0=*/1>(SmemSrc<L>{b0}, SmemDst<L>{res}, b0, b1,
                                                                                 a.tw, a.scale, a.do_scale != 0);
  tma::fence_proxy_async();
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int b = 0; b < N / BR; ++b) tma::store_3d(&map_out, res + b * BR * CW, c0, b * BR, o);
    tma::store_commit();
    tma::store_wait_read();
  }
}
template <int N, int CW>
constexpr size_t cols_tma_smem_bytes() {
  return sizeof(float2) * (size_t)N * CW * 2;
}

// ---- half-spectrum real transforms (last axis, even length n = 2H) -------------------------------
// R2C: the real row x[0..n) is read as H complex z[m] = x[2m] + i x[2m+1] (the same bytes), the
// H-point transform Z runs with its last stage landing in shared memory, and the unpack
//     X[k] = (Z[k] + conj(Z[H-k]))/2 - (i/2) W_n^k (Z[k] - conj(Z[H-k])),  k = 0..H
// writes the n/2+1 bins straight to global memory (one read + one write of HBM per element).
// C2R is the mirror image: rows of n/2+1 bins are staged in shared memory, stage 0 reads
//     Z[k] = (X[k] + conj(X[H-k])) + i W_n^{-k} (X[k] - conj(X[H-k]))
// on the fly, and the H-point inverse writes x as interleaved pairs, scaled by 1/n.
// `tw2` holds W_n^k (R2C) or W_n^{-k} (C2R) for k = 0..H.
struct HalfArgs {
  const void* in;
  void* out;
  const float2* tw;
  const float2* tw2;
  long long nrows;
  float scale;
};

// one tile of C rows: `src` yields the real rows viewed as H complex each, `out` = first output row.
// `after_stage0` runs once the input has been consumed (async kernels release their input buffer there).
template <int H, class RL, int C, int NT, bool NB = false, bool TWS = false, class Src, class Hook>
__device__ __forceinline__ void r2c_tile_from(const Src& src, float2* __restrict__ out, const float2* __restrict__ tw,
                                              const float2* __restrict__ tw2, int valid, float2* smem_f2, Hook after_stage0) {
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<H>::template type>();
  constexpr int BUF = EX > C * H ? EX : C * H;
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + BUF;
  // the last stage writes Z[o][k] densely into the buffer the last exchange did not use
  float2* zbuf = ((RL::count - 1) % 2 == 0) ? buf0 : buf1;
  if constexpr (RL::count == 1) {
    run_stage<RL::r[0], 1, H, C, 1, NT, false>(src, SmemDst<PlaneLayout<H>>{zbuf}, tw, 1.f, false);
    tile_sync<NT, NB>();
    after_stage0();
  } else {
    using L0 = typename RowLayoutN<H>::template type<RL::r[0], 1>;
    run_stage<RL::r[0], 1, H, C, 1, NT, false>(src, SmemDst<L0>{buf0}, tw, 1.f, false);
    tile_sync<NT, NB>();
    after_stage0();
    run_axis<RL, H, C, 1, NT, false, RowLayoutN<H>::template type, 0, 1, NB, TWS>(SmemSrc<L0>{buf0}, SmemDst<PlaneLayout<H>>{zbuf},
                                                                            buf0, buf1, tw, 1.f, false);
    tile_sync<NT, NB>();
  }
  const int total = valid * (H + 1);
  for (int idx = threadIdx.x; idx < total; idx += NT) {
    const int o = idx / (H + 1), k = idx - o * (H + 1);
    const float2 zk = zbuf[o * H + (k == H ? 0 : k)];
    float2 zm = zbuf[o * H + (k == 0 ? 0 : H - k)];
    zm.y = -zm.y;
    const float2 s = make_float2(zk.x + zm.x, zk.y + zm.y), d = make_float2(zk.x - zm.x, zk.y - zm.y);
    const float2 w = __ldg(&tw2[k]);
    const float2 t = cmulf(d, w);  // W * (Z[k] - conj(Z[H-k]))
    // X = (s - i t) / 2
    out[idx] = make_float2(0.5f * (s.x + t.y), 0.5f * (s.y - t.x));
  }
}
template <int H, class RL, int C, int NT, bool COHERENT = false>
__device__ __forceinline__ void r2c_tile(const in_vec2* in, float2* __restrict__ out, const float2* __restrict__ tw,
                                         const float2* __restrict__ tw2, int valid, float2* smem_f2) {
  GlobalSrc<false, COHERENT> src{in, H, 1, valid, 1};
  r2c_tile_from<H, RL, C, NT, false>(src, out, tw, tw2, valid, smem_f2, [] {});
}

template <int H, class RL, int C, int NT>
__global__ void __launch_bounds__(NT) rows_r2c_kernel(const __grid_constant__ HalfArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  r2c_tile<H, RL, C, NT>(reinterpret_cast<const in_vec2*>(a.in) + row0 * H,
                         reinterpret_cast<float2*>(a.out) + row0 * (H + 1), a.tw, a.tw2, valid, smem_f2);
}

// ---- R2C with the Hermitian unpack in registers (warp shuffles instead of a shared-memory pass) ----------
// In the LAST stage (radix R, P = H / R butterflies per row) the thread of butterfly p holds
// Z[p + k*P], k = 0..R-1. The mirrored bins it needs are H - (p + k*P) = (P - p) + (R-1-k)*P: exactly the
// outputs of butterfly P - p of the same row, in reverse order (butterfly 0 mirrors onto itself,
// Z[H - k*P] = its own output R - k, and Z[H] = Z[0]). When P divides 32 the butterflies of a row sit in
// consecutive lanes of one warp, so the partner's value arrives with one __shfl_sync per component and the
// unpacked bins go straight from registers to global memory: no Z buffer, no extra barrier, and the kernel
// needs only the exchange buffer(s) of the H-point transform (none at all for a single-stage H).
template <int H>
struct R2CRegDst {
  static constexpr bool whole = true;
  float2* __restrict__ out;          // first output row of the tile; rows of H + 1 bins
  const float2* __restrict__ tw2;    // W_n^k, k = 0..H
  int valid_o;
  template <int R, int P>
  __device__ __forceinline__ void store_all(int o, int g, int p, const float2 (&x)[R]) const {
    static_assert(P * R == H && P <= 32 && 32 % P == 0, "last stage of an H-point transform, rows inside a warp");
    (void)g;  // always 0 in the last stage
    const int lane = (int)threadIdx.x & 31;
    const int partner = (lane & ~(P - 1)) | ((P - p) & (P - 1));
    float2* __restrict__ row = out + (long long)o * (H + 1);
    const bool live = o < valid_o;
#pragma unroll
    for (int k = 0; k < R; ++k) {
      float2 zm = x[(R - k) % R];  // butterfly 0: its own mirrored output
      if constexpr (P > 1) {
        const float mx = __shfl_sync(0xffffffffu, x[R - 1 - k].x, partner);
        const float my = __shfl_sync(0xffffffffu, x[R - 1 - k].y, partner);
        if (p != 0) zm = make_float2(mx, my);
      }
      const float2 zk = x[k];
      // s = Z[k] + conj(Z[H-k]), d = Z[k] - conj(Z[H-k])
      const float2 s = make_float2(zk.x + zm.x, zk.y - zm.y), d = make_float2(zk.x - zm.x, zk.y + zm.y);
      const float2 t = cmulf(d, __ldg(&tw2[p + k * P]));
      if (live) row[p + k * P] = make_float2(0.5f * (s.x + t.y), 0.5f * (s.y - t.x));  // (s - i t) / 2
    }
    if (p == 0 && live) row[H] = make_float2(x[0].x - x[0].y, 0.f);  // X[H] = Re Z[0] - Im Z[0]
  }
};
template <int H, class RL, int C, int NT>
constexpr bool r2c_reg_ok() {
  constexpr int P = H / RL::r[RL::count - 1];
  // P >= 8: a warp's store covers segments of P consecutive bins; with fewer (single-stage H: P = 1, every lane a
  // different row) the stores are uncoalesced and the shared-memory unpack wins (measured: 100 x 64^3 R2C 0.172 vs 0.208 ms)
  return P >= 8 && P <= 32 && 32 % P == 0 && (C * P) % 32 == 0 && NT % 32 == 0;
}
template <int H, class RL, int C>
constexpr size_t rows_r2c_reg_smem_bytes() {
  return sizeof(float2) * (size_t)max_exchange_elems<RL, C, RowLayoutN<H>::template type>() * (RL::count > 2 ? 2 : 1);
}
template <int H, class RL, int C, int NT>
__global__ void __launch_bounds__(NT) rows_r2c_reg_kernel(const __grid_constant__ HalfArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<H>::template type>();
  pdl_wait();
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  GlobalSrc<false> src{reinterpret_cast<const in_vec2*>(a.in) + row0 * H, H, 1, valid, 1};
  R2CRegDst<H> dst{reinterpret_cast<float2*>(a.out) + row0 * (H + 1), a.tw2, valid};
  run_axis<RL, H, C, 1, NT, false, RowLayoutN<H>::template type>(src, dst, smem_f2, smem_f2 + EX, a.tw, 1.f, false);
}

// ---- R2C of an ODD length n: the n-point transform of the real row on the row kernel's stages, storing only
// bins 0..n/2 (rows of n/2 + 1 bins). One read of 4 B and one write of ~4 B per input point.
struct GlobalHalfDst {
  float2* __restrict__ base;
  int bins;  // n/2 + 1 = output row stride
  int valid_o;
  __device__ __forceinline__ void store(int o, int i, int, float2 v) const {
    if (o >= valid_o || i >= bins) return;
    base[(long long)o * bins + i] = v;
  }
};
template <int N, class RL, int C, int NT>
__global__ void __launch_bounds__(NT) rows_r2c_odd_kernel(const __grid_constant__ HalfArgs a) {
  static_assert(N % 2 == 1, "odd lengths only (even lengths run as an n/2-point complex transform)");
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  GlobalSrc<true> src{reinterpret_cast<const in_scalar*>(a.in) + row0 * N, N, 1, valid, 1};
  GlobalHalfDst dst{reinterpret_cast<float2*>(a.out) + row0 * (N / 2 + 1), N / 2 + 1, valid};
  run_axis<RL, N, C, 1, NT, false, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, 1.f, false);
}

// the same source reading the half spectrum straight from global memory: X[i] and X[H - i] are both in the tile's own
// rows, so the second read of every element is an L1 / L2 hit, and the kernel needs no staging buffer, no staging
// barrier and only the exchange buffer(s) of the H-point transform (rows_c2r_kernel used to stage the C x (H + 1) bins
// in shared memory first: 100 KB per CTA for H = 512, two CTAs per SM, 100000 x 1024 C2R at 0.31 ms; now 3-6 CTAs).
template <int H>
struct HermGlobalSrc {
  const in_vec2* __restrict__ xb;  // [rows][H+1] in global memory
  const float2* __restrict__ tw2;
  int valid_o;
  __device__ __forceinline__ float2 load(int o, int i, int) const {
    if (o >= valid_o) return make_float2(0.f, 0.f);
    const in_vec2 a = __ldg(&xb[(long long)o * (H + 1) + i]);
    const in_vec2 b = __ldg(&xb[(long long)o * (H + 1) + H - i]);
    const float2 xk = make_float2((float)a.x, (float)a.y), xm = make_float2((float)b.x, -(float)b.y);
    const float2 s = make_float2(xk.x + xm.x, xk.y + xm.y), d = make_float2(xk.x - xm.x, xk.y - xm.y);
    const float2 t = cmulf(d, __ldg(&tw2[i]));  // W_n^{-i} * (X[i] - conj(X[H-i]))
    return make_float2(s.x - t.y, s.y + t.x);   // s + i t
  }
};

// (min 3 CTAs per SM for CTAs of up to 256 threads: <512, 32x16, 8, 256> sat at 83 registers = two CTAs)
template <int H, class RL, int C, int NT>
__global__ void __launch_bounds__(NT, NT <= 256 ? 3 : 1) rows_c2r_kernel(const __grid_constant__ HalfArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<H>::template type>();
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + EX;
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  HermGlobalSrc<H> src{reinterpret_cast<const in_vec2*>(a.in) + row0 * (H + 1), a.tw2, valid};
  GlobalDst dst{reinterpret_cast<float2*>(a.out) + row0 * H, H, 1, valid, 1};
  run_axis<RL, H, C, 1, NT, true, RowLayoutN<H>::template type>(src, dst, buf0, buf1, a.tw, a.scale, true);
}

// C2R of an ODD length n: the n-point inverse on the Hermitian-extended row (X[n - k] = conj X[k], read on the fly from
// the n/2 + 1 stored bins), real parts stored. Mirror image of rows_r2c_odd_kernel.
template <int N>
struct HermExtSrc {
  const in_vec2* __restrict__ xb;  // [rows][N/2+1]
  int valid_o;
  __device__ __forceinline__ float2 load(int o, int i, int) const {
    if (o >= valid_o) return make_float2(0.f, 0.f);
    constexpr int BINS = N / 2 + 1;
    const in_vec2 v = __ldg(&xb[(long long)o * BINS + (i < BINS ? i : N - i)]);
    return make_float2((float)v.x, i < BINS ? (float)v.y : -(float)v.y);
  }
};
struct RealDst {
  float* __restrict__ base;
  int n;
  int valid_o;
  __device__ __forceinline__ void store(int o, int i, int, float2 v) const {
    if (o < valid_o) base[(long long)o * n + i] = v.x;
  }
};
template <int N, class RL, int C, int NT>
__global__ void __launch_bounds__(NT) rows_c2r_odd_kernel(const __grid_constant__ HalfArgs a) {
  static_assert(N % 2 == 1, "odd lengths only");
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  const long long row0 = (long long)blockIdx.x * C;
  const int valid = (int)min((long long)C, a.nrows - row0);
  HermExtSrc<N> src{reinterpret_cast<const in_vec2*>(a.in) + row0 * (N / 2 + 1), valid};
  RealDst dst{reinterpret_cast<float*>(a.out) + row0 * N, N, valid};
  run_axis<RL, N, C, 1, NT, true, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale, true);
}
template <int H, class RL, int C>
constexpr size_t rows_r2c_smem_bytes() {
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<H>::template type>();
  return sizeof(float2) * (size_t)(EX > C * H ? EX : C * H) * 2;
}
template <int H, class RL, int C>
constexpr size_t rows_c2r_smem_bytes() {
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<H>::template type>();
  return sizeof(float2) * (size_t)EX * (RL::count > 2 ? 2 : 1);
}

struct ColsArgs {
  const void* in;
  float2* out;
  const float2* tw;
  long long inner;        // element stride along the axis = number of interleaved columns
  int tiles_per_outer;    // ceil(inner / CW)
  float scale;
  int do_scale;
  int reverse;            // walk the tiles from the last to the first: the pass before this one wrote the array front to
                          // back, so its END is what the L2 still holds ("serpentine" pass order, api.cu: build_passes)
};

// strided axis: tile = all N points of CW adjacent columns (CW*8 contiguous bytes per axis step);
// the "transpose" the reference does with separate kernels happens in the tile addressing.
template <int N, class RL, int CW, int NT, bool INV, bool REAL>
__global__ void __launch_bounds__(NT) cols_kernel(const __grid_constant__ ColsArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + BUF;
  pdl_wait();
  const unsigned bid = a.reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
  const long long o = bid / a.tiles_per_outer;
  const long long c0 = (long long)(bid - o * a.tiles_per_outer) * CW;
  const long long base = o * N * a.inner + c0;
  const int valid_c = (int)min((long long)CW, a.inner - c0);
  const void* in = REAL ? (const void*)(reinterpret_cast<const in_scalar*>(a.in) + base)
                        : (const void*)(reinterpret_cast<const in_vec2*>(a.in) + base);
  GlobalSrc<REAL> src{in, 0, a.inner, 1, valid_c};
  GlobalDst dst{a.out + base, 0, a.inner, 1, valid_c};
  run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(src, dst, buf0, buf1, a.tw, a.scale,
                                                                      a.do_scale != 0);
}
// strided axis with a scattering store: the slab decomposition's exchange fused into the pass.
// The tile's output row i (index along the transformed axis, which is the axis being split across
// GPUs) belongs to peer h = i / yl; it is written straight into that peer's buffer at the place it
// has in the peer's [z][yl][x] slab. With peer pointers mapped over NVLink (CUDA IPC) the
// all-to-all happens inside this kernel's stores; with all pointers local it is the pack step of
// an NCCL all-to-all.
struct ScatterArgs {
  float2* peer[16];
  int yl;            // rows of the split axis per peer
  long long zbase;   // first outer index (z plane) of this rank in the peers' slabs
};
struct ScatterDst {
  const ScatterArgs* sa;
  long long tile_off;  // ((zbase + o) * yl) * inner + c0
  long long inner;
  int valid_c;
  __device__ __forceinline__ void store(int, int i, int c, float2 v) const {
    if (c >= valid_c) return;
    const int h = i / sa->yl;
    const int r = i - h * sa->yl;
    sa->peer[h][tile_off + r * inner + c] = v;
  }
};

template <int N, class RL, int CW, int NT, bool INV>
__global__ void __launch_bounds__(NT) cols_scatter_kernel(const __grid_constant__ ColsArgs a,
                                                          const __grid_constant__ ScatterArgs sa) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + BUF;
  const unsigned bid = a.reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
  const long long o = bid / a.tiles_per_outer;
  const long long c0 = (long long)(bid - o * a.tiles_per_outer) * CW;
  const long long base = o * N * a.inner + c0;
  const int valid_c = (int)min((long long)CW, a.inner - c0);
  GlobalSrc<false> src{reinterpret_cast<const float2*>(a.in) + base, 0, a.inner, 1, valid_c};
  ScatterDst dst{&sa, ((sa.zbase + o) * sa.yl) * a.inner + c0, a.inner, valid_c};
  run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(src, dst, buf0, buf1, a.tw, a.scale,
                                                                      a.do_scale != 0);
}

template <int N, class RL, int CW>
constexpr size_t cols_smem_bytes() {
  return sizeof(float2) * (size_t)max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>() *
         (RL::count > 2 ? 2 : 1);
}

// ---- long axes as two passes ("four-step") ---------------------------------------------------------
// An axis of length N = N1*N2 that is too long for one tile is transformed as
//   A: N1-point transforms over n1 (element stride N2*inner), output (k1, n2) multiplied by W_N^{k1*n2}
//   B: N2-point transforms over n2 (element stride inner) for every k1, output k2 stored at index
//      k1 + N1*k2 of the axis (natural order, so no transpose pass)
// Both are ordinary tile passes: A is a strided-axis pass with a twiddling store, B is a strided-axis
// pass (or, for a contiguous axis, a row pass) whose destination uses a different base and stride.
struct SplitArgs {
  const void* in;      // pass A: the user's array (in_scalar / in_vec2 elements); pass B: the temporary (float2)
  float2* out;
  const float2* tw;    // stage twiddles of this pass's variant
  const float2* twN;   // W_N^n, n in [0, N): pass A only (three-pass split: T_hi of SplitTw2Dst)
  const float2* tw2;   // half-spectrum forms: W_n^{-+k}, k = 0..n/2, of the Hermitian unpack (R2C) / pack (C2R)
                       // (three-pass split: T_lo of SplitTw2Dst)
  long long inner;     // element stride of the ORIGINAL axis (1 = contiguous)
  long long nrows;     // rows pass B: outer * N1 rows of N2 points
  int tiles_per_outer; // cols passes: tiles per outer slab of THIS pass's view
  int n1, n2;
  float scale;
  int do_scale;
};

struct SplitTwDst {
  float2* __restrict__ base;
  long long si;
  int valid_c;
  const float2* __restrict__ twN;
  long long c0, inner;
  __device__ __forceinline__ void store(int, int i, int c, float2 v) const {
    if (c >= valid_c) return;
    const int n2 = (int)((c0 + c) / inner);  // k1 * n2 < N1 * N2 = N: no reduction needed
    base[i * si + c] = cmulf(v, __ldg(&twN[i * n2]));
  }
};

// The twiddle of SplitTwDst for a contiguous axis (inner == 1) too long for a table of L entries: W_L^e, e = k * r,
// as T_hi[e >> s] * T_lo[e & (2^s - 1)], two tables of about sqrt(L) entries (split_tw_shift). k < N and r < L / N,
// so e < L needs no reduction; it reaches 2^31 and is formed in 64 bits.
struct SplitTw2Dst {
  float2* __restrict__ base;
  long long si;
  int valid_c;
  const float2* __restrict__ thi;
  const float2* __restrict__ tlo;
  long long c0;
  int s;
  __device__ __forceinline__ void store(int, int i, int c, float2 v) const {
    if (c >= valid_c) return;
    const long long e = (long long)i * (c0 + c);
    const float2 w = cmulf(__ldg(&thi[e >> s]), __ldg(&tlo[e & ((1LL << s) - 1)]));
    base[i * si + c] = cmulf(v, w);
  }
};
// s = ceil(bits(L - 1) / 2): T_lo holds 2^s entries, T_hi ceil(L / 2^s) (the host builds them with the same rule)
__host__ __device__ __forceinline__ int split_tw_shift(long long L) {
  int bits = 0;
  while (bits < 62 && (1LL << bits) < L) ++bits;
  return (bits + 1) / 2;
}

// pass A: view (outer, N1 = N, inner' = n2 * inner). REAL: the input array holds real scalars (in_scalar), read as
// x + 0i; otherwise complex pairs (in_vec2). Both are cast to the working precision on load.
// TW2: the contiguous axis of a three-pass split (inner == 1, L = N * n2): the twiddle from the two tables twN = T_hi
// and tw2 = T_lo (SplitTw2Dst) instead of the L-entry table twN.
template <int N, class RL, int CW, int NT, bool INV, bool REAL = false, bool TW2 = false>
__global__ void __launch_bounds__(NT) cols_split_a_kernel(const __grid_constant__ SplitArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
  const long long vinner = (long long)a.n2 * a.inner;
  const long long o = blockIdx.x / a.tiles_per_outer;
  const long long c0 = (long long)(blockIdx.x - o * a.tiles_per_outer) * CW;
  const long long base = o * N * vinner + c0;
  const int valid_c = (int)min((long long)CW, vinner - c0);
  const void* in = REAL ? (const void*)(reinterpret_cast<const in_scalar*>(a.in) + base)
                        : (const void*)(reinterpret_cast<const in_vec2*>(a.in) + base);
  GlobalSrc<REAL> src{in, 0, vinner, 1, valid_c};
  if constexpr (TW2) {
    SplitTw2Dst dst{a.out + base, vinner, valid_c, a.twN, a.tw2, c0, split_tw_shift(N * vinner)};
    run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, 1.f, false);
  } else {
    SplitTwDst dst{a.out + base, vinner, valid_c, a.twN, c0, a.inner};
    run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, 1.f, false);
  }
}

// ---- long half-spectrum axes (last axis, inner == 1) as two passes ----------------------------------------------------
// Pass A of a long C2R: the Hermitian pack (even n = 2H) or the Hermitian extension (odd n) of the single-tile C2R
// kernels, read straight from the rows of n/2 + 1 bins in global memory, at axis index m = n1 * N2 + n2 of the split
// transform. The mirrored bin of an element lies in another column tile of the same transform's row (an L2 hit when
// the tiles of one transform run close together, which the grid order gives).
//   even: Z[m] = s + i t, s = X[m] + conj X[H-m], t = W_n^{-m} (X[m] - conj X[H-m]); H = N1 * N2, bins = H + 1
//   odd:  Z[m] = X[m] for m <= n/2, conj X[n-m] above;                             n = N1 * N2, bins = n/2 + 1
template <bool ODD>
struct HermSplitSrc {
  const in_vec2* __restrict__ xb;  // first bin of this transform's row
  const float2* __restrict__ tw2;
  int len;                          // H (even) or n (odd)
  int n2;
  long long c0;
  int valid_c;
  __device__ __forceinline__ float2 load(int, int i, int c) const {
    if (c >= valid_c) return make_float2(0.f, 0.f);
    const int m = i * n2 + (int)c0 + c;
    if constexpr (ODD) {
      const int bins = len / 2 + 1;
      const in_vec2 v = __ldg(&xb[m < bins ? m : len - m]);
      return make_float2((float)v.x, m < bins ? (float)v.y : -(float)v.y);
    } else {
      const in_vec2 p = __ldg(&xb[m]);
      const in_vec2 q = __ldg(&xb[len - m]);
      const float2 xk = make_float2((float)p.x, (float)p.y), xm = make_float2((float)q.x, -(float)q.y);
      const float2 s = make_float2(xk.x + xm.x, xk.y + xm.y), d = make_float2(xk.x - xm.x, xk.y - xm.y);
      const float2 t = cmulf(d, __ldg(&tw2[m]));  // W_n^{-m} * (X[m] - conj(X[H-m]))
      return make_float2(s.x - t.y, s.y + t.x);   // s + i t
    }
  }
};
template <int N, class RL, int CW, int NT, bool ODD>
__global__ void __launch_bounds__(NT) cols_split_a_c2r_kernel(const __grid_constant__ SplitArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
  const int len = N * a.n2;
  const long long bins = ODD ? len / 2 + 1 : len + 1;
  const long long o = blockIdx.x / a.tiles_per_outer;
  const long long c0 = (long long)(blockIdx.x - o * a.tiles_per_outer) * CW;
  const int valid_c = (int)min((long long)CW, (long long)a.n2 - c0);
  HermSplitSrc<ODD> src{reinterpret_cast<const in_vec2*>(a.in) + o * bins, a.tw2, len, a.n2, c0, valid_c};
  SplitTwDst dst{a.out + o * len + c0, a.n2, valid_c, a.twN, c0, 1};
  run_axis<RL, N, 1, CW, NT, true, DenseLayoutN<N, CW>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, 1.f, false);
}

// pass B on a strided axis: view (outer * n1, N2 = N, inner); row k2 of slab (o, k1) goes to axis index k1 + n1*k2
template <int N, class RL, int CW, int NT, bool INV>
__global__ void __launch_bounds__(NT) cols_split_b_kernel(const __grid_constant__ SplitArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
  const long long ov = blockIdx.x / a.tiles_per_outer;  // o * n1 + k1
  const long long c0 = (long long)(blockIdx.x - ov * a.tiles_per_outer) * CW;
  const long long o = ov / a.n1, k1 = ov - o * a.n1;
  const int valid_c = (int)min((long long)CW, a.inner - c0);
  GlobalSrc<false> src{reinterpret_cast<const float2*>(a.in) + ov * N * a.inner + c0, 0, a.inner, 1, valid_c};
  GlobalDst dst{a.out + (o * N * a.n1 + k1) * a.inner + c0, 0, (long long)a.n1 * a.inner, 1, valid_c};
  run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale,
                                                                      a.do_scale != 0);
}

// pass B of an odd-length R2C: only bins k = k1 + N1*k2 <= n/2 are stored, into rows of n/2 + 1 (GlobalHalfDst's rule)
struct SplitHalfDst {
  float2* __restrict__ base;  // bin k1 of this tile's transform
  int n1, bins_left;          // bins_left = n/2 + 1 - k1
  int valid_o;
  __device__ __forceinline__ void store(int o, int i, int, float2 v) const {
    const int k = o + n1 * i;
    if (o < valid_o && k < bins_left) base[k] = v;
  }
};
// pass B of an odd-length C2R: the real parts of the n-point inverse (RealDst's rule)
struct SplitRealDst {
  float* __restrict__ base;  // sample k1 of this tile's transform
  int n1;
  int valid_o;
  __device__ __forceinline__ void store(int o, int i, int, float2 v) const {
    if (o < valid_o) base[o + (long long)n1 * i] = v.x;
  }
};

// pass B on a contiguous axis (inner == 1): C consecutive rows k1 of one transform, N2 = N points each.
// STORE 0: complex natural order; 1: bins 0..n/2 of rows of n/2 + 1 (odd R2C); 2: real parts (odd C2R)
template <int N, class RL, int C, int NT, bool INV, int STORE = 0>
__global__ void __launch_bounds__(NT) rows_split_b_kernel(const __grid_constant__ SplitArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  const long long row0 = (long long)blockIdx.x * C;  // rows never straddle transforms: C divides n1
  const int valid = (int)min((long long)C, a.nrows - row0);
  const long long t = row0 / a.n1, k1 = row0 - t * a.n1;
  GlobalSrc<false> src{reinterpret_cast<const float2*>(a.in) + row0 * N, N, 1, valid, 1};
  const long long len = (long long)N * a.n1;
  if constexpr (STORE == 1) {
    const long long bins = len / 2 + 1;
    SplitHalfDst dst{a.out + t * bins + k1, a.n1, (int)(bins - k1), valid};
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale,
                                                                 a.do_scale != 0);
  } else if constexpr (STORE == 2) {
    SplitRealDst dst{reinterpret_cast<float*>(a.out) + t * len + k1, a.n1, valid};
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale,
                                                                 a.do_scale != 0);
  } else {
    GlobalDst dst{a.out + t * len + k1, 1, a.n1, valid, 1};  // element (row o, k2) -> k1 + o + n1 * k2
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale,
                                                                 a.do_scale != 0);
  }
}

// ---- contiguous axes longer than 2^24 points as three passes, n = N1 * N2 * N3, M = N2 * N3 -----------------------
//   1: cols_split_a_kernel<TW2> on the view (outer, N1, M): user array -> temporary, W_n^{k1 (n2 N3 + n3)} in the store
//   2: the same on the view (outer N1, N2, N3), in place on the temporary, W_M^{k2 n3} in the store
//   3: this kernel: the contiguous N3-point rows (k1, k2) of the temporary (row k1 * M + k2 * N3 of transform t),
//      output k3 stored at k1 + N1 * k2 + N1 * N2 * k3, which is natural order
// A CTA takes C rows of consecutive k1 and one k2 (C divides N1), so every store is a run of C elements.
// Args: n1 = N1, n2 = N2, nrows = outer * N1 * N2.
template <int N, class RL, int C, int NT, bool INV>
__global__ void __launch_bounds__(NT) rows_split_c_kernel(const __grid_constant__ SplitArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  const long long row0 = (long long)blockIdx.x * C;  // row = (t * N2 + k2) * N1 + k1
  const int valid = (int)min((long long)C, a.nrows - row0);
  const long long tk2 = row0 / a.n1, k1 = row0 - tk2 * a.n1;
  const long long t = tk2 / a.n2, k2 = tk2 - t * a.n2;
  const long long m = (long long)a.n2 * N;
  const long long len = (long long)a.n1 * m;
  GlobalSrc<false> src{reinterpret_cast<const float2*>(a.in) + t * len + k1 * m + k2 * N, m, 1, valid, 1};
  GlobalDst dst{a.out + t * len + k1 + (long long)a.n1 * k2, 1, (long long)a.n1 * a.n2, valid, 1};
  run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(src, dst, smem_f2, smem_f2 + BUF, a.tw, a.scale,
                                                               a.do_scale != 0);
}

// Pass B of a long even-length R2C (n = 2H, H = N1 * N2) with the Hermitian unpack fused into the store. Pass A has
// transformed the real row read as H complex points; row k1 of the temporary holds Z[k1 + N1*k2] after this pass's
// N2-point transform. The unpack of bin k needs Z[H - k]:
//   k1 > 0: row N1 - k1, column N2 - 1 - k2          k1 = 0: row 0, column (N2 - k2) mod N2
// so a CTA transforms C/2 consecutive rows k1 = p0 .. and their mirror rows N1 - k1 (row 0 and, for even N1, row N1/2
// pair with themselves and are transformed twice), keeps Z of all C rows in shared memory and writes
//   X[k] = ((Z[k] + conj Z[H-k]) - i W_n^k (Z[k] - conj Z[H-k])) / 2
// for both rows of every pair into rows of H + 1 bins (R2CRegDst's arithmetic); row 0 also writes X[H] = Re Z[0] - Im Z[0].
// Grid: outer * tiles_per_outer, tiles_per_outer = ceil((N1/2 + 1) / (C/2)).
// tile slot o: slots 0 .. C/2-1 hold rows p = p0 + o, slots C/2 .. C-1 their mirror rows N1 - p (row 0 for p = 0)
template <int N, int C>
struct PairSrc {
  const float2* __restrict__ z;  // row 0 of this transform in the temporary
  int n1, p0, npairs;
  __device__ __forceinline__ float2 load(int o, int i, int) const {
    const int p = p0 + (o < C / 2 ? o : o - C / 2);
    if (p >= npairs) return make_float2(0.f, 0.f);
    const int row = o < C / 2 || p == 0 ? p : n1 - p;
    return __ldg(&z[(long long)row * N + i]);
  }
};
template <int N, class RL, int C, int NT>
__global__ void __launch_bounds__(NT) rows_split_b_r2c_kernel(const __grid_constant__ SplitArgs a) {
  static_assert(C % 2 == 0, "rows come in (k1, N1 - k1) pairs");
  extern __shared__ __align__(16) float2 smem_f2[];
  pdl_wait();
  constexpr int PC = C / 2;
  constexpr int EX = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
  constexpr int BUF = EX > C * N ? EX : C * N;
  float2* buf0 = smem_f2;
  float2* buf1 = smem_f2 + BUF;
  float2* zbuf = ((RL::count - 1) % 2 == 0) ? buf0 : buf1;  // the buffer the last exchange does not use
  const int n1 = a.n1;
  const int npairs = n1 / 2 + 1;
  const long long t = blockIdx.x / a.tiles_per_outer;
  const int p0 = (int)(blockIdx.x - t * a.tiles_per_outer) * PC;
  const long long H = (long long)n1 * N;
  PairSrc<N, C> src{reinterpret_cast<const float2*>(a.in) + t * H, n1, p0, npairs};
  if constexpr (RL::count == 1) {
    run_stage<RL::r[0], 1, N, C, 1, NT, false>(src, SmemDst<PlaneLayout<N>>{zbuf}, a.tw, 1.f, false);
  } else {
    run_axis<RL, N, C, 1, NT, false, RowLayoutN<N>::template type>(src, SmemDst<PlaneLayout<N>>{zbuf}, buf0, buf1, a.tw, 1.f,
                                                                   false);
  }
  __syncthreads();
  float2* __restrict__ out = a.out + t * (H + 1);
  // pair fastest: consecutive threads store consecutive bins k1 (first rows) or k1 descending (mirror rows)
  for (int idx = threadIdx.x; idx < C * N; idx += NT) {
    const int j = idx % PC, rest = idx / PC;
    const int k2 = rest % N, side = rest / N;
    const int p = p0 + j;
    if (p >= npairs || (side == 1 && (p == 0 || 2 * p == n1))) continue;  // a self-paired row is stored once
    const int slot = side * PC + j, mslot = (1 - side) * PC + j;
    const int mc = p == 0 ? (N - k2) % N : N - 1 - k2;
    const float2 zk = zbuf[slot * N + k2];
    const float2 zm = zbuf[mslot * N + mc];
    const long long k = (side == 0 ? p : n1 - p) + (long long)n1 * k2;
    // s = Z[k] + conj(Z[H-k]), d = Z[k] - conj(Z[H-k])
    const float2 s = make_float2(zk.x + zm.x, zk.y - zm.y), d = make_float2(zk.x - zm.x, zk.y + zm.y);
    const float2 tt = cmulf(d, __ldg(&a.tw2[k]));
    out[k] = make_float2(0.5f * (s.x + tt.y), 0.5f * (s.y - tt.x));  // (s - i t) / 2
    if (k == 0) out[H] = make_float2(zk.x - zk.y, 0.f);              // X[H] = Re Z[0] - Im Z[0]
  }
}

}  // namespace b200fft

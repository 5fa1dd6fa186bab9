// Fused N-d transform: ONE persistent kernel runs every axis pass of a batched N-d FFT, with the
// intermediate kept in L2 instead of making one HBM round trip per axis.
//
// Separate per-axis kernels (fast.cuh) each stream the whole array through HBM: k axes = k reads +
// k writes. Here the passes become PHASES of one kernel. The work of all phases is cut into tiles
// (the same tiles the per-axis kernels use) and laid out in one global order; CTAs take tiles from
// that order with an atomic counter. A tile of phase p > 0 may only start when the phase p-1 tiles it
// reads are finished: those are counted per dependency GROUP (a z plane for the x -> y hand-over, a
// whole transform for -> z), the producer bumps the group's counter after its stores
// (__syncthreads; __threadfence; atomicAdd), the consumer's thread 0 spins on it with ld.acquire.gpu.
// Because every tile only waits for tiles EARLIER in the order, and tiles are taken in order, the
// scheme cannot deadlock whatever the number of resident CTAs.
//
// The host (fused_registry.cu: build_schedule) orders the tiles as a software pipeline over chunks of
// ~16 MB: [phase0(chunk c), phase1(chunk c-1), phase2(chunk c-2)], so a dependent tile is reached one
// full chunk after its producers were handed out (no spinning in steady state) while the data it
// reads was written a few microseconds earlier and is still in the 126 MB L2. HBM then sees one read
// of the input and one write of the output; the in-between traffic stays in L2 (measured on B200:
// ~10 TB/s L2-resident vs ~6.5 TB/s HBM, profiles/r1_l2bw_microbench.jsonl).
//
// Intermediate data is read with ld.global.cg (GlobalSrc<.., COHERENT>): L1 is not coherent across
// SMs and a line may linger from an earlier phase on the same SM.
#pragma once
#include "fast.cuh"
#include "planner.hpp"  // NdSegment, build_schedule

namespace b200fft {

constexpr int ND_MAX_PHASES = 3;

struct NdPhase {
  const float2* tw;              // stage twiddles of the (first) axis of this phase
  const float2* tw2;             // second table: y axis of a plane phase / W_n^k of the R2C unpack
  long long inner;               // cols: element stride along the axis
  long long units_per_transform; // rows / r2c: rows per transform
  int tiles_per_outer;           // cols: tiles per outer slab
  int tiles_per_transform;
  int tiles_per_group;           // tiles of THIS phase per dependency group it signals
  int groups_per_transform;      // counters per transform this phase signals
  int dep_div;                   // this phase's tile j waits for group j / dep_div of the previous phase
  float scale;
  int do_scale;
};

struct NdArgs {
  const void* in;
  float2* out;
  long long in_stride_bytes;  // per transform
  long long out_stride;       // float2 per transform
  NdPhase ph[ND_MAX_PHASES];
  int nphases;
  int nsegs;
  const NdSegment* segs;
  unsigned total_items;
  unsigned* ctrl;                 // [0] next item, [1] CTAs finished, then the group counters
  unsigned* err;                  // mapped HOST word: set to 1 when a dependency wait gave up (checked by the next exec)
  int cnt_off[ND_MAX_PHASES];     // offset of each phase's counters inside ctrl
  int nwords;                     // words to clear at the end (header + counters)
};

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Spin until *cnt >= want. Every tile only waits for tiles that were handed out earlier (v1: in-order atomic fetch;
// v2: static assignment with the whole grid co-resident, guaranteed by the cooperative launch), so the wait always
// ends. Should that ever be violated, the wait gives up after ~2 s, raises the plan's sticky error word (a mapped
// host word the next b200fft_exec reads and reports) and the kernel runs to its end with invalid results: no trap,
// so the CUDA context survives.
__device__ __forceinline__ void wait_counter_gpu(const unsigned* cnt, unsigned want, unsigned sleep_ns, unsigned* err) {
  unsigned spins = 0;
  while (ld_acquire_gpu(cnt) < want) {
    __nanosleep(sleep_ns);
    if (++spins > 30000000u) {
      if (err) atomicExch_system(err, 1u);
      return;
    }
  }
}

// ---- phases: the tile bodies of fast.cuh as device functions --------------------------------------
enum NdKind { ND_NONE = 0, ND_ROWS = 1, ND_COLS = 2, ND_R2C = 3, ND_PLANE = 4, ND_R2C_PLANE = 5 };

struct NdNone {
  using RL = Radices<1>;
  static constexpr bool none = true;
  static constexpr int kind = ND_NONE, n = 1, tile = 1;
  static constexpr bool inverse = false, real = false;
  static constexpr size_t smem = 0;
  template <int NT>
  static __device__ __forceinline__ void run(const NdPhase&, const void*, float2*, int, float2*) {}
};

// contiguous rows: tile = C consecutive rows of the transform
template <int N, class RL_, int C, bool INV, bool REAL>
struct NdRows {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_ROWS, n = N, tile = C;
  static constexpr bool inverse = INV, real = REAL;
  static constexpr size_t smem = rows_smem_bytes<N, RL, C>();
  template <int NT>
  static __device__ __forceinline__ void run(const NdPhase& p, const void* src, float2* dst, int tile, float2* sm) {
    constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    const void* in = REAL ? (const void*)(reinterpret_cast<const float*>(src) + row0 * N)
                          : (const void*)(reinterpret_cast<const float2*>(src) + row0 * N);
    GlobalSrc<REAL, true> s{in, N, 1, valid, 1};
    GlobalDst d{dst + row0 * N, N, 1, valid, 1};
    run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type>(s, d, sm, sm + BUF, p.tw, p.scale, p.do_scale != 0);
  }
};

// strided axis: tile = all N points of CW adjacent columns of one outer slab
template <int N, class RL_, int CW, bool INV>
struct NdCols {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_COLS, n = N, tile = CW;
  static constexpr bool inverse = INV, real = false;
  static constexpr size_t smem = cols_smem_bytes<N, RL, CW>();
  template <int NT>
  static __device__ __forceinline__ void run(const NdPhase& p, const void* src, float2* dst, int tile, float2* sm) {
    constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
    const int o = tile / p.tiles_per_outer;
    const long long c0 = (long long)(tile - o * p.tiles_per_outer) * CW;
    const long long base = (long long)o * N * p.inner + c0;
    const int valid_c = (int)min((long long)CW, p.inner - c0);
    GlobalSrc<false, true> s{reinterpret_cast<const float2*>(src) + base, 0, p.inner, 1, valid_c};
    GlobalDst d{dst + base, 0, p.inner, 1, valid_c};
    run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type>(s, d, sm, sm + BUF, p.tw, p.scale,
                                                                        p.do_scale != 0);
  }
};

// half-spectrum R2C rows (last axis n = 2H): C real rows -> C rows of H+1 bins
template <int H, class RL_, int C>
struct NdR2C {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_R2C, n = 2 * H, tile = C;
  static constexpr bool inverse = false, real = true;
  static constexpr size_t smem = rows_r2c_smem_bytes<H, RL, C>();
  template <int NT>
  static __device__ __forceinline__ void run(const NdPhase& p, const void* src, float2* dst, int tile, float2* sm) {
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    r2c_tile<H, RL, C, NT, true>(reinterpret_cast<const float2*>(src) + row0 * H, dst + row0 * (H + 1), p.tw, p.tw2, valid,
                                 sm);
  }
};

// element (i = y, c = x - c0) of the plane staged in shared memory
template <int NX>
struct PlaneColLayout {
  static __device__ __forceinline__ int off(int, int i, int c) { return i * NX + c; }
};

// two axes in one tile: a whole (NY x NX) plane is transformed along x into shared memory (RG rows at
// a time), then along y out of shared memory (CW columns at a time). One global read + one global
// write for two axes.
template <int NY, int NX, class RLY_, class RLX_, int RG, int CW, bool INV, bool REAL>
struct NdPlane {
  using RL = RLX_;
  static constexpr bool none = false;
  static constexpr int kind = ND_PLANE, n = NX, n2 = NY, tile = 1;
  static constexpr bool inverse = INV, real = REAL;
  using RLY = RLY_;
  static constexpr int EXR = max_exchange_elems<RLX_, RG, RowLayoutN<NX>::template type>();
  static constexpr int EXC = max_exchange_elems<RLY_, 1, DenseLayoutN<NY, CW>::template type>();
  static constexpr int EX = EXR > EXC ? EXR : EXC;
  static constexpr bool two = (RLX_::count > 2) || (RLY_::count > 2);
  static constexpr size_t smem = sizeof(float2) * ((size_t)NY * NX + (size_t)EX * (two ? 2 : 1));
  static_assert(NY % RG == 0 && NX % CW == 0, "plane tile: RG must divide NY and CW must divide NX");
  template <int NT>
  static __device__ __forceinline__ void run(const NdPhase& p, const void* src, float2* dst, int tile, float2* sm) {
    float2* plane = sm;
    float2* ex0 = sm + NY * NX;
    float2* ex1 = ex0 + EX;
    const long long pbase = (long long)tile * NY * NX;
    for (int r0 = 0; r0 < NY; r0 += RG) {
      const void* in = REAL ? (const void*)(reinterpret_cast<const float*>(src) + pbase + (long long)r0 * NX)
                            : (const void*)(reinterpret_cast<const float2*>(src) + pbase + (long long)r0 * NX);
      GlobalSrc<REAL, true> s{in, NX, 1, RG, 1};
      run_axis<RLX_, NX, RG, 1, NT, INV, RowLayoutN<NX>::template type>(s, SmemDst<PlaneLayout<NX>>{plane + r0 * NX}, ex0, ex1,
                                                                       p.tw, 1.f, false);
      __syncthreads();
    }
    for (int c0 = 0; c0 < NX; c0 += CW) {
      GlobalDst d{dst + pbase + c0, 0, NX, 1, CW};
      run_axis<RLY_, NY, 1, CW, NT, INV, DenseLayoutN<NY, CW>::template type>(SmemSrc<PlaneColLayout<NX>>{plane + c0}, d, ex0,
                                                                             ex1, p.tw2, p.scale, p.do_scale != 0);
      __syncthreads();
    }
  }
};

// ---- the persistent kernel ---------------------------------------------------------------------------
template <int PH, int NT, class Phase>
__device__ __forceinline__ void nd_do_phase(const NdArgs& a, long long gtile, float2* sm) {
  const NdPhase& P = a.ph[PH];
  const long long t = gtile / P.tiles_per_transform;
  const int tile = (int)(gtile - t * P.tiles_per_transform);
  if constexpr (PH > 0) {
    if (threadIdx.x == 0) {
      const NdPhase& Q = a.ph[PH - 1];
      const unsigned* cnt = a.ctrl + a.cnt_off[PH - 1] + t * Q.groups_per_transform + tile / P.dep_div;
      const unsigned want = (unsigned)Q.tiles_per_group;
      wait_counter_gpu(cnt, want, 64, a.err);
    }
    __syncthreads();
  }
  const void* src = PH == 0 ? (const void*)(reinterpret_cast<const char*>(a.in) + t * a.in_stride_bytes)
                            : (const void*)(a.out + t * a.out_stride);
  Phase::template run<NT>(P, src, a.out + t * a.out_stride, tile, sm);
  if (PH + 1 < a.nphases) {
    __syncthreads();  // every thread's stores are issued and visible to thread 0 (CTA scope) ...
    if (threadIdx.x == 0) {
      __threadfence();  // ... and ordered before the counter update at GPU scope
      atomicAdd(a.ctrl + a.cnt_off[PH] + t * P.groups_per_transform + tile / P.tiles_per_group, 1u);
    }
  }
}

template <int NT, int MINB, class P0, class P1, class P2>
__global__ void __launch_bounds__(NT, MINB) nd_fused_kernel(const __grid_constant__ NdArgs a) {
  extern __shared__ __align__(16) float2 smem_f2[];
  __shared__ unsigned s_item;
  __shared__ int s_last;
  int seg = 0;
  unsigned next = 0;
  if (threadIdx.x == 0) next = atomicAdd(a.ctrl, 1u);
  while (true) {
    if (threadIdx.x == 0) s_item = next;
    __syncthreads();
    const unsigned item = s_item;
    if (item >= a.total_items) break;
    if (threadIdx.x == 0) next = atomicAdd(a.ctrl, 1u);  // fetched while this tile is processed
    while ((long long)item >= a.segs[seg].first_item + a.segs[seg].count) ++seg;
    const int phase = a.segs[seg].phase;
    const long long gtile = a.segs[seg].first_tile + ((long long)item - a.segs[seg].first_item);
    if (phase == 0) nd_do_phase<0, NT, P0>(a, gtile, smem_f2);
    else if (phase == 1) nd_do_phase<1, NT, P1>(a, gtile, smem_f2);
    else if constexpr (!P2::none) nd_do_phase<2, NT, P2>(a, gtile, smem_f2);
    __syncthreads();  // shared memory and s_item are reused by the next tile
  }
  // the last CTA to leave clears the counters for the next launch (stream-ordered after this one)
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(a.ctrl + 1, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {
    for (int i = threadIdx.x; i < a.nwords; i += NT) a.ctrl[i] = 0u;
  }
}

template <class P0, class P1, class P2>
constexpr size_t nd_fused_smem() {
  size_t m = P0::smem;
  m = P1::smem > m ? P1::smem : m;
  m = P2::smem > m ? P2::smem : m;
  return m;
}

}  // namespace b200fft

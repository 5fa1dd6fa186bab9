// Fused N-d transform, version 2: the persistent kernel of fused.cuh with the global -> shared
// traffic taken off the compute warps.
//
// fused.cuh (v1) keeps HBM traffic at one read + one write but every tile serialises
// "global-load latency -> stage -> barrier -> stage -> stores" inside its CTA (ncu: warps wait on
// barrier / long_scoreboard, every pipe < 25 % busy, profiles/r1_fused_v1.md). Here each CTA is
//   * NT consumer threads that only ever read shared memory and write global memory, and
//   * one producer warp that fetches the next work item (atomic), waits for its dependency group
//     (ld.acquire.gpu), and brings the tile into a shared-memory ring with bulk-async copies:
//     `cp.async.bulk` (1-D, contiguous row / plane tiles) or `cp.async.bulk.tensor.3d` (TMA box of a
//     strided-axis tile), completion on an mbarrier (complete_tx::bytes).
// full[slot] / empty[slot] mbarriers hand the ring slots back and forth; consumers release a slot as
// soon as stage 0 has read it, so the loads of the next one or two tiles are always in flight while
// the current tile is computed, and the dependency wait is off the consumers' critical path.
// Scheduling, counters and the L2-resident software pipeline are those of fused.cuh.
#pragma once
#include "fused.cuh"

namespace b200fft {

constexpr int ND_RING = 2;  // default input ring depth (a kernel template parameter: 1 trades look-ahead for CTAs per SM)

struct NdItem {  // ring slot descriptor, written by the producer before it arrives on full[slot]
  int phase;     // -1 = no more work
  int tile;
  long long t;
};

namespace tma {
// 1-D bulk copy global -> shared, completion on an mbarrier
__device__ __forceinline__ void load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// order earlier generic-proxy accesses (the acquire that observed other SMs' st.global) before later
// async-proxy reads of global memory (the bulk copies)
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
}  // namespace tma

// dense tiles staged in shared memory by the producer
template <int N, bool REAL>
struct StagedRows {  // [o][i]
  const void* buf;
  __device__ __forceinline__ float2 load(int o, int i, int) const {
    if constexpr (REAL) return make_float2(reinterpret_cast<const float*>(buf)[o * N + i], 0.f);
    else return reinterpret_cast<const float2*>(buf)[o * N + i];
  }
};

// ---- phases ---------------------------------------------------------------------------------------------
// load(): executed by the producer warp (lane 0 issues); run(): by the NT consumer threads.
struct ANone {
  using RL = Radices<1>;
  static constexpr bool none = true;
  static constexpr int kind = ND_NONE, n = 1, tile = 1;
  static constexpr bool inverse = false, real = false;
  static constexpr size_t in_bytes = 0, ex_bytes = 0;
  static constexpr int tw_elems = 0, tw2_elems = 0;
  static __device__ __forceinline__ void load(const NdPhase&, const CUtensorMap*, const void*, long long, int, void*,
                                              uint64_t*) {}
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase&, const float2*, const float2*, const void*, float2*, int,
                                             float2*, Rel) {}
};

template <int N, class RL_, int C, bool INV, bool REAL>
struct ARows {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_ROWS, n = N, tile = C;
  static constexpr bool inverse = INV, real = REAL;
  static constexpr int ELEM = REAL ? 4 : 8;
  static constexpr size_t in_bytes = (size_t)C * N * ELEM;
  static constexpr size_t ex_bytes = rows_smem_bytes<N, RL, C>();
  static constexpr int tw_elems = RL::tw_total() > 0 ? RL::tw_total() : 1, tw2_elems = 0;
  static __device__ __forceinline__ void load(const NdPhase& p, const CUtensorMap*, const void* src_t, long long, int tile,
                                              void* in_buf, uint64_t* full) {
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    const uint32_t bytes = (uint32_t)valid * N * ELEM;
    tma::mbar_arrive_expect_tx(full, bytes);
    tma::load_1d(in_buf, reinterpret_cast<const char*>(src_t) + row0 * N * ELEM, bytes, full);
  }
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase& p, const float2* tw, const float2*, const void* in_buf,
                                             float2* dst_t, int tile, float2* ex, Rel release) {
    constexpr int BUF = max_exchange_elems<RL, C, RowLayoutN<N>::template type>();
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    StagedRows<N, REAL> s{in_buf};
    GlobalDst d{dst_t + row0 * N, N, 1, valid, 1};
    if constexpr (RL::count == 1) {
      run_stage<RL::r[0], 1, N, C, 1, NT, INV, true>(s, d, tw, p.scale, p.do_scale != 0);
      tile_sync<NT, true>();
      release();
    } else {
      using L0 = typename RowLayoutN<N>::template type<RL::r[0], 1>;
      run_stage<RL::r[0], 1, N, C, 1, NT, INV, true>(s, SmemDst<L0>{ex}, tw, 1.f, false);
      tile_sync<NT, true>();
      release();
      run_axis<RL, N, C, 1, NT, INV, RowLayoutN<N>::template type, 0, 1, true, true>(SmemSrc<L0>{ex}, d, ex, ex + BUF, tw,
                                                                                    p.scale, p.do_scale != 0);
    }
  }
};

// strided axis: the [N][CW] tile arrives as N / BR boxes of a 3-D tensor map over (inner, N, outer)
template <int N, class RL_, int CW, bool INV>
struct ACols {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_COLS, n = N, tile = CW;
  static constexpr bool inverse = INV, real = false;
  static constexpr int BR = tma_box_rows(N);
  static constexpr size_t in_bytes = (size_t)N * CW * 8;
  static constexpr size_t ex_bytes = cols_smem_bytes<N, RL, CW>();
  static constexpr int tw_elems = RL::tw_total() > 0 ? RL::tw_total() : 1, tw2_elems = 0;
  static __device__ __forceinline__ void load(const NdPhase& p, const CUtensorMap* map, const void*, long long t, int tile,
                                              void* in_buf, uint64_t* full) {
    const int o = tile / p.tiles_per_outer;
    const int c0 = (tile - o * p.tiles_per_outer) * CW;
    const int outer = (int)(t * (p.tiles_per_transform / p.tiles_per_outer) + o);
    tma::mbar_arrive_expect_tx(full, (uint32_t)in_bytes);
#pragma unroll
    for (int b = 0; b < N / BR; ++b)
      tma::load_3d(reinterpret_cast<float2*>(in_buf) + b * BR * CW, map, c0, b * BR, outer, full);
  }
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase& p, const float2* tw, const float2*, const void* in_buf,
                                             float2* dst_t, int tile, float2* ex, Rel release) {
    constexpr int BUF = max_exchange_elems<RL, 1, DenseLayoutN<N, CW>::template type>();
    const int o = tile / p.tiles_per_outer;
    const long long c0 = (long long)(tile - o * p.tiles_per_outer) * CW;
    const long long base = (long long)o * N * p.inner + c0;
    using LI = DenseLayout<N, CW>;
    SmemSrc<LI> s{reinterpret_cast<const float2*>(in_buf)};
    GlobalDst d{dst_t + base, 0, p.inner, 1, CW};
    if constexpr (RL::count == 1) {
      run_stage<RL::r[0], 1, N, 1, CW, NT, INV, true>(s, d, tw, p.scale, p.do_scale != 0);
      tile_sync<NT, true>();
      release();
    } else {
      run_stage<RL::r[0], 1, N, 1, CW, NT, INV, true>(s, SmemDst<LI>{ex}, tw, 1.f, false);
      tile_sync<NT, true>();
      release();
      run_axis<RL, N, 1, CW, NT, INV, DenseLayoutN<N, CW>::template type, 0, 1, true, true>(SmemSrc<LI>{ex}, d, ex, ex + BUF,
                                                                                           tw, p.scale, p.do_scale != 0);
    }
  }
};

// half-spectrum R2C rows: C real rows (= C x H complex, contiguous) -> C rows of H + 1 bins
template <int H, class RL_, int C>
struct AR2C {
  using RL = RL_;
  static constexpr bool none = false;
  static constexpr int kind = ND_R2C, n = 2 * H, tile = C;
  static constexpr bool inverse = false, real = true;
  static constexpr size_t in_bytes = (size_t)C * H * 8;
  static constexpr size_t ex_bytes = rows_r2c_smem_bytes<H, RL, C>();
  static constexpr int tw_elems = RL::tw_total() > 0 ? RL::tw_total() : 1, tw2_elems = 0;  // W_n^k stays in global
  static __device__ __forceinline__ void load(const NdPhase& p, const CUtensorMap*, const void* src_t, long long, int tile,
                                              void* in_buf, uint64_t* full) {
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    const uint32_t bytes = (uint32_t)valid * H * 8;
    tma::mbar_arrive_expect_tx(full, bytes);
    tma::load_1d(in_buf, reinterpret_cast<const char*>(src_t) + row0 * H * 8, bytes, full);
  }
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase& p, const float2* tw, const float2*, const void* in_buf,
                                             float2* dst_t, int tile, float2* ex, Rel release) {
    const long long row0 = (long long)tile * C;
    const int valid = (int)min((long long)C, p.units_per_transform - row0);
    StagedRows<H, false> s{in_buf};
    r2c_tile_from<H, RL, C, NT, true, true>(s, dst_t + row0 * (H + 1), tw, p.tw2, valid, ex, release);
  }
};

// (y, x) plane: x pass from the staged plane into the exchange buffer and back into the SAME staging
// buffer (now the x-transformed plane), y pass out of it; the slot is released after the y pass's stage 0.
template <int NY, int NX, class RLY_, class RLX_, bool INV>
struct APlane {
  using RL = RLX_;
  using RLY = RLY_;
  static constexpr bool none = false;
  static constexpr int kind = ND_PLANE, n = NX, n2 = NY, tile = 1;
  static constexpr bool inverse = INV, real = false;
  static_assert(RLX_::count == 2 && RLY_::count == 2, "plane tiles: two super-stages per axis");
  static constexpr int EXR = max_exchange_elems<RLX_, NY, RowLayoutN<NX>::template type>();
  static constexpr int EXC = NY * NX;
  static constexpr size_t in_bytes = (size_t)NY * NX * 8;
  static constexpr size_t ex_bytes = sizeof(float2) * (size_t)(EXR > EXC ? EXR : EXC);
  static constexpr int tw_elems = RLX_::tw_total(), tw2_elems = RLY_::tw_total();
  static __device__ __forceinline__ void load(const NdPhase&, const CUtensorMap*, const void* src_t, long long, int tile,
                                              void* in_buf, uint64_t* full) {
    tma::mbar_arrive_expect_tx(full, (uint32_t)in_bytes);
    tma::load_1d(in_buf, reinterpret_cast<const float2*>(src_t) + (long long)tile * NY * NX, (uint32_t)in_bytes, full);
  }
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase& p, const float2* tw, const float2* tw2, const void* in_buf,
                                             float2* dst_t, int tile, float2* ex, Rel release) {
    float2* plane = reinterpret_cast<float2*>(const_cast<void*>(in_buf));
    // x: staged plane -> ex (padded rows) -> plane
    using LX = typename RowLayoutN<NX>::template type<RLX_::r[0], 1>;
    run_stage<RLX_::r[0], 1, NX, NY, 1, NT, INV, true>(StagedRows<NX, false>{in_buf}, SmemDst<LX>{ex}, tw, 1.f, false);
    tile_sync<NT, true>();
    run_stage<RLX_::r[1], RLX_::r[0], NX, NY, 1, NT, INV, true>(SmemSrc<LX>{ex}, SmemDst<PlaneLayout<NX>>{plane},
                                                                tw + RLX_::tw_offset(1), 1.f, false);
    tile_sync<NT, true>();
    // y: plane -> ex (dense [y][x]) -> global
    using LY = DenseLayout<NY, NX>;
    run_stage<RLY_::r[0], 1, NY, 1, NX, NT, INV, true>(SmemSrc<LY>{plane}, SmemDst<LY>{ex}, tw2, 1.f, false);
    tile_sync<NT, true>();
    release();
    GlobalDst d{dst_t + (long long)tile * NY * NX, 0, NX, 1, NX};
    run_stage<RLY_::r[1], RLY_::r[0], NY, 1, NX, NT, INV, true>(SmemSrc<LY>{ex}, d, tw2 + RLY_::tw_offset(1), p.scale,
                                                                p.do_scale != 0);
  }
};

// Half-spectrum (y, x) plane: NY real rows of n = 2H points -> the plane's NY x (H + 1) block of the half spectrum,
// x AND y transformed, in one tile. The real plane (NY * n floats, contiguous) arrives by one bulk copy; the rows run as
// H-point complex transforms (the same bytes viewed as z[m] = x[2m] + i x[2m+1]) whose result Z stays in shared memory;
// the y pass then runs over the H + 1 (odd!) bins of every row, its stage 0 forming each bin on the fly with the
// Hermitian unpack X[k] = (Z[k] + conj(Z[H-k]))/2 - (i/2) W_n^k (Z[k] - conj(Z[H-k])), and its last stage stores the
// finished block, which is contiguous in the output. The ragged H + 1 extent that no TMA box or 16-column tile fits
// (33 bins for n = 64) never reaches global memory half-done: the middle pass of the per-axis plan (2 full tiles + 1
// column, profiles/r1_r2c.md) disappears, and HBM sees one read + one write for two axes. The strided z phase that
// follows has inner = NY * (H + 1), a multiple of NY: whole TMA tiles again.
// Shared memory: region R1 = x exchange, later the y exchange; region R2 = Z. The phase's twiddle table is
// [x stage twiddles | W_n^k, k = 0..H] (one table, staged once per CTA), tw2 = the y stage twiddles.
template <int H>
struct UnpackSrc {  // bin c of row i from Z[i][0..H)
  const float2* z;
  const float2* w;  // W_n^k in shared memory
  __device__ __forceinline__ float2 load(int, int i, int c) const {
    const float2 zk = z[i * H + (c == H ? 0 : c)];
    float2 zm = z[i * H + (c == 0 ? 0 : H - c)];
    zm.y = -zm.y;
    const float2 s = make_float2(zk.x + zm.x, zk.y + zm.y), d = make_float2(zk.x - zm.x, zk.y - zm.y);
    const float2 t = cmulf(d, tw_load<true>(w, c));
    return make_float2(0.5f * (s.x + t.y), 0.5f * (s.y - t.x));
  }
};

// ZSLOT: the x result Z is written back into the staging slot (the real plane it replaces has the same size), so the
// exchange area is R1 only and more CTAs fit an SM; the slot is then released after the y pass's stage 0.
template <int NY, int H, class RLY_, class RLX_, bool ZSLOT = false>
struct AR2CPlane {
  using RL = RLX_;
  using RLY = RLY_;
  static constexpr bool none = false;
  static constexpr int kind = ND_R2C_PLANE, n = 2 * H, n2 = NY, tile = 1;
  static constexpr bool inverse = false, real = true;
  static constexpr int HB = H + 1;
  static_assert(RLX_::count == 2 && RLY_::count == 2, "r2c plane tiles: two super-stages per axis");
  static constexpr int EXR = max_exchange_elems<RLX_, NY, RowLayoutN<H>::template type>();
  static constexpr int R1 = EXR > NY * HB ? EXR : NY * HB;
  static constexpr int R2 = ZSLOT ? 0 : NY * H;
  static constexpr size_t in_bytes = (size_t)NY * H * 8;
  static constexpr size_t ex_bytes = sizeof(float2) * (size_t)(R1 + R2);
  static constexpr int tw_elems = RLX_::tw_total() + HB, tw2_elems = RLY_::tw_total();
  static __device__ __forceinline__ void load(const NdPhase&, const CUtensorMap*, const void* src_t, long long, int tile,
                                              void* in_buf, uint64_t* full) {
    tma::mbar_arrive_expect_tx(full, (uint32_t)in_bytes);
    tma::load_1d(in_buf, reinterpret_cast<const float2*>(src_t) + (long long)tile * NY * H, (uint32_t)in_bytes, full);
  }
  template <int NT, class Rel>
  static __device__ __forceinline__ void run(const NdPhase& p, const float2* tw, const float2* tw2, const void* in_buf,
                                             float2* dst_t, int tile, float2* ex, Rel release) {
    float2* r1 = ex;
    float2* r2 = ZSLOT ? reinterpret_cast<float2*>(const_cast<void*>(in_buf)) : ex + R1;
    // x, stage 0: staged real rows (as H complex) -> r1 (padded rows)
    using LX = typename RowLayoutN<H>::template type<RLX_::r[0], 1>;
    run_stage<RLX_::r[0], 1, H, NY, 1, NT, false, true>(StagedRows<H, false>{in_buf}, SmemDst<LX>{r1}, tw, 1.f, false);
    tile_sync<NT, true>();
    if constexpr (!ZSLOT) release();  // the staging slot is free for the next tile's copy
    // x, stage 1: r1 -> Z = r2, dense [row][k]
    run_stage<RLX_::r[1], RLX_::r[0], H, NY, 1, NT, false, true>(SmemSrc<LX>{r1}, SmemDst<PlaneLayout<H>>{r2},
                                                                 tw + RLX_::tw_offset(1), 1.f, false);
    tile_sync<NT, true>();
    // y over the HB bins of every row, unpacked on the fly: Z -> r1 -> global (the plane's block is contiguous)
    using LY = DenseLayout<NY, HB>;
    run_stage<RLY_::r[0], 1, NY, 1, HB, NT, false, true>(UnpackSrc<H>{r2, tw + RLX_::tw_total()}, SmemDst<LY>{r1}, tw2, 1.f,
                                                         false);
    tile_sync<NT, true>();
    if constexpr (ZSLOT) release();
    GlobalDst d{dst_t + (long long)tile * NY * HB, 0, HB, 1, HB};
    run_stage<RLY_::r[1], RLY_::r[0], NY, 1, HB, NT, false, true>(SmemSrc<LY>{r1}, d, tw2 + RLY_::tw_offset(1), 1.f, false);
    (void)p;
  }
};

// ---- kernel ------------------------------------------------------------------------------------------------
struct NdLocate {
  int seg;
  __device__ __forceinline__ void find(const NdArgs& a, unsigned item, int* phase, long long* gtile) {
    while ((long long)item >= a.segs[seg].first_item + a.segs[seg].count) ++seg;
    *phase = a.segs[seg].phase;
    *gtile = a.segs[seg].first_tile + ((long long)item - a.segs[seg].first_item);
  }
};

// Everything the producer needs to stage one tile, resolved ahead of time by one lane of the producer warp.
struct NdTileReq {
  int phase;            // -1: past the end of the schedule
  int tile;
  long long t;
  const unsigned* cnt;  // dependency counter (phase > 0) and the value it must reach
  unsigned want;
  bool ready;
};

template <int PH>
__device__ __forceinline__ void nd_resolve(const NdArgs& a, long long gtile, NdTileReq* r) {
  const NdPhase& P = a.ph[PH];
  r->phase = PH;
  r->t = gtile / P.tiles_per_transform;
  r->tile = (int)(gtile - r->t * P.tiles_per_transform);
  r->cnt = nullptr;
  r->want = 0;
  r->ready = true;
  if constexpr (PH > 0) {
    const NdPhase& Q = a.ph[PH - 1];
    r->cnt = a.ctrl + a.cnt_off[PH - 1] + r->t * Q.groups_per_transform + r->tile / P.dep_div;
    r->want = (unsigned)Q.tiles_per_group;
    r->ready = ld_acquire_gpu(r->cnt) >= r->want;  // usually true: the schedule keeps consumers a chunk behind
  }
}

template <int PH, class Phase>
__device__ __forceinline__ void nd_issue(const NdArgs& a, const CUtensorMap* map, const NdTileReq& r, void* in_buf,
                                         uint64_t* full, NdItem* ring) {
  const NdPhase& P = a.ph[PH];
  ring->phase = PH;
  ring->tile = r.tile;
  ring->t = r.t;
  const void* src_t = PH == 0 ? (const void*)(reinterpret_cast<const char*>(a.in) + r.t * a.in_stride_bytes)
                              : (const void*)(a.out + r.t * a.out_stride);
  Phase::load(P, map, src_t, r.t, r.tile, in_buf, full);
}

template <int PH, int NT, class Phase, class Rel>
__device__ __forceinline__ void nd_consume(const NdArgs& a, const NdItem& it, const float2* tw, const float2* tw2,
                                           const void* in_buf, float2* ex, Rel release) {
  const NdPhase& P = a.ph[PH];
  Phase::template run<NT>(P, tw, tw2, in_buf, a.out + it.t * a.out_stride, it.tile, ex, release);
  if (PH + 1 < a.nphases) {
    tile_sync<NT, true>();  // every consumer's stores are issued (CTA scope) ...
    if (threadIdx.x == 0) {
      __threadfence();      // ... and ordered before the counter update at GPU scope
      atomicAdd(a.ctrl + a.cnt_off[PH] + it.t * P.groups_per_transform + it.tile / P.tiles_per_group, 1u);
    }
  } else {
    tile_sync<NT, true>();  // the exchange buffer is reused by the next tile
  }
}

template <class P0, class P1, class P2>
constexpr size_t nd_async_in_bytes() {
  size_t m = P0::in_bytes;
  m = P1::in_bytes > m ? P1::in_bytes : m;
  m = P2::in_bytes > m ? P2::in_bytes : m;
  return (m + 127) / 128 * 128;
}
template <class P0, class P1, class P2, int RING = ND_RING>
constexpr size_t nd_async_smem() {
  size_t e = P0::ex_bytes;
  e = P1::ex_bytes > e ? P1::ex_bytes : e;
  e = P2::ex_bytes > e ? P2::ex_bytes : e;
  const size_t tw = sizeof(float2) * (size_t)(P0::tw_elems + P0::tw2_elems + P1::tw_elems + P2::tw_elems);
  return RING * nd_async_in_bytes<P0, P1, P2>() + (e + 15) / 16 * 16 + tw + 128;  // +128: manual ring alignment
}
template <class P0, class P1, class P2>
constexpr size_t nd_async_ex_bytes() {
  size_t e = P0::ex_bytes;
  e = P1::ex_bytes > e ? P1::ex_bytes : e;
  e = P2::ex_bytes > e ? P2::ex_bytes : e;
  return (e + 15) / 16 * 16;
}

// block = NT consumer threads + one producer warp
template <int NT, int MINB, class P0, class P1, class P2, int RING = ND_RING>
__global__ void __launch_bounds__(NT + 32, MINB)
    nd_async_kernel(const __grid_constant__ NdArgs a, const __grid_constant__ CUtensorMap map1,
                    const __grid_constant__ CUtensorMap map2) {
  // 128-byte aligned by declaration (TMA destinations); all pointers below are derived from this array by
  // plain pointer arithmetic so the compiler keeps them in the shared address space (LDS/STS, not generic LD/ST:
  // the first version aligned through uintptr_t and paid 16 % of its stall samples on generic loads)
  extern __shared__ __align__(128) unsigned char smem_async[];
  __shared__ __align__(8) uint64_t full[RING];
  __shared__ __align__(8) uint64_t empty[RING];
  __shared__ NdItem ring[RING];
  __shared__ int s_last;
  constexpr size_t IN = nd_async_in_bytes<P0, P1, P2>();
  unsigned char* base = smem_async;
  float2* ex = reinterpret_cast<float2*>(base + RING * IN);
  // stage twiddle tables, copied once per CTA: every later twiddle read is an LDS
  float2* tw0 = reinterpret_cast<float2*>(base + RING * IN + nd_async_ex_bytes<P0, P1, P2>());
  float2* tw0b = tw0 + P0::tw_elems;
  float2* tw1 = tw0b + P0::tw2_elems;
  float2* tw2s = tw1 + P1::tw_elems;
  for (int i = threadIdx.x; i < P0::tw_elems; i += NT + 32) tw0[i] = a.ph[0].tw[i];
  for (int i = threadIdx.x; i < P0::tw2_elems; i += NT + 32) tw0b[i] = a.ph[0].tw2[i];
  for (int i = threadIdx.x; i < P1::tw_elems; i += NT + 32) tw1[i] = a.ph[1].tw[i];
  if constexpr (!P2::none)
    for (int i = threadIdx.x; i < P2::tw_elems; i += NT + 32) tw2s[i] = a.ph[2].tw[i];

  if (threadIdx.x == 0) {
    for (int i = 0; i < RING; ++i) {
      tma::mbar_init(&full[i], 1);   // the producer's arrive.expect_tx (+ the copies' bytes)
      tma::mbar_init(&empty[i], 1);  // consumer thread 0 after the stage-0 barrier
    }
    tma::fence_barrier_init();
  }
  __syncthreads();

  if (threadIdx.x >= NT) {
    // ---------------- producer warp (lane 0). Work is assigned statically, CTA c takes items c, c + G, c + 2G, ...
    // of the global order (the launch is COOPERATIVE, so the whole grid is co-resident and every item's producers are
    // running or done; fused_registry.cu falls back to the per-axis kernels when such a launch is refused):
    // no atomic work fetch, and item k+1 is resolved — segment lookup, dependency counter read with ld.acquire —
    // while the consumers still work on item k, so neither global round trip sits between two copies. Claiming
    // several items per atomic instead was measured slower: it reserves work far ahead of execution and breaks
    // the one-chunk distance between a phase and its consumers (64^3: 0.201 vs 0.173 ms).
    if (threadIdx.x == NT) {
      if constexpr (P1::kind == ND_COLS) tma::prefetch_map(&map1);
      if constexpr (P2::kind == ND_COLS) tma::prefetch_map(&map2);
      NdLocate loc{0};
      auto resolve = [&](unsigned item, NdTileReq* r) {
        r->phase = -1;
        r->ready = true;
        if (item >= a.total_items) return;
        int phase;
        long long gtile;
        loc.find(a, item, &phase, &gtile);
        if (phase == 0) nd_resolve<0>(a, gtile, r);
        else if (phase == 1) nd_resolve<1>(a, gtile, r);
        else nd_resolve<2>(a, gtile, r);
      };
      unsigned item = blockIdx.x;
      NdTileReq r, rn;
      resolve(item, &rn);
      for (unsigned k = 0;; ++k) {
        r = rn;
        const int slot = k % RING;
        if (k >= RING) tma::mbar_wait(&empty[slot], ((k / RING) - 1) & 1);
        if (r.phase < 0) {
          ring[slot].phase = -1;
          tma::mbar_arrive(&full[slot]);
          break;
        }
        if (!r.ready) wait_counter_gpu(r.cnt, r.want, 32, a.err);
        if (r.phase > 0) tma::fence_proxy_async_all();
        void* in_buf = base + slot * IN;
        if (r.phase == 0) nd_issue<0, P0>(a, nullptr, r, in_buf, &full[slot], &ring[slot]);
        else if (r.phase == 1) nd_issue<1, P1>(a, &map1, r, in_buf, &full[slot], &ring[slot]);
        else if constexpr (!P2::none) nd_issue<2, P2>(a, &map2, r, in_buf, &full[slot], &ring[slot]);
        item += gridDim.x;
        resolve(item, &rn);  // look one tile ahead
      }
    }
    return;
  }

  // ---------------- consumers
  for (unsigned k = 0;; ++k) {
    const int slot = k % RING;
    tma::mbar_wait(&full[slot], (k / RING) & 1);
    const NdItem it = ring[slot];
    if (it.phase < 0) break;
    const void* in_buf = base + slot * IN;
    auto release = [&] {
      if (threadIdx.x == 0) tma::mbar_arrive(&empty[slot]);
    };
    if (it.phase == 0) nd_consume<0, NT, P0>(a, it, tw0, tw0b, in_buf, ex, release);
    else if (it.phase == 1) nd_consume<1, NT, P1>(a, it, tw1, nullptr, in_buf, ex, release);
    else if constexpr (!P2::none) nd_consume<2, NT, P2>(a, it, tw2s, nullptr, in_buf, ex, release);
  }
  // the last CTA to leave clears the counters for the next launch (stream-ordered after this one)
  tile_sync<NT, true>();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(a.ctrl + 1, 1u) == gridDim.x - 1;
  }
  tile_sync<NT, true>();
  if (s_last) {
    for (int i = threadIdx.x; i < a.nwords; i += NT) a.ctrl[i] = 0u;
  }
}

}  // namespace b200fft

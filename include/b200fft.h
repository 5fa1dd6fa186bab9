/*
 * b200fft — C ABI of the B200-native batched N-d radix-n FFT.
 *
 * This is the drop-in boundary for martinvuyk/hackathon-fft's `fft` package. The
 * reference has no FFI of its own: its public surface is four Mojo generics in
 * fft/fft/fft.mojo (plan_fft x2, fft x2) whose GPU overloads end in
 * `_run_gpu_nd_fft` (fft/fft/_ndim_fft_gpu.mojo:462-642). Everything those
 * overloads take as compile-time parameters (dtypes, layouts incl. batch,
 * inverse, bases) becomes a runtime descriptor here; the Mojo wrappers in
 * hackathon-fft_b200/mojo/fft/ read the parameters off and call these entry
 * points with `external_call` (see INTEGRATION.md).
 *
 * All functions are `extern "C"`, take plain pointers and sizes, never throw or
 * abort across the ABI, and return an int status (0 = B200FFT_OK). Distinct
 * plans may be used from distinct threads; one plan must not be executed
 * concurrently with itself (same rule as the reference, whose plan owns mutable
 * scratch: fft/fft/_ndim_fft_cpu.mojo:39-45, _ndim_fft_gpu.mojo:176-185).
 *
 * There is no CPU fallback: every entry point that computes fails with
 * B200FFT_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef B200FFT_H
#define B200FFT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200FFT_API __attribute__((visibility("default")))
#else
#define B200FFT_API
#endif

#define B200FFT_MAX_RANK 8

/* status codes */
enum {
  B200FFT_OK = 0,
  B200FFT_ERR_INVALID_ARG = 1, /* NULL pointer, rank/batch out of range                      */
  B200FFT_ERR_LAYOUT = 2,      /* violates _check_layout_conditions_nd (fft.mojo:20-46)      */
  B200FFT_ERR_BASES = 3,       /* bases do not multiply to the axis length / contain 1
                                  (_utils.mojo:205-220 compile-time asserts)                 */
  B200FFT_ERR_UNSUPPORTED = 4, /* valid for the reference, not built yet here (see message)  */
  B200FFT_ERR_CUDA = 5,        /* CUDA runtime / driver error, or no sm_100 device           */
  B200FFT_ERR_ALLOC = 6
};

/* scalar types of the interleaved buffers (the reference's in_dtype / out_dtype parameters) */
enum { B200FFT_U8 = 0, B200FFT_F32 = 1, B200FFT_F64 = 2 };

/* real-input / real-output packing */
enum {
  /* Reference semantics (_fft.mojo:254-255): in_components == 1 feeds reals into
     stage 0 of the last axis and the output is the FULL N-bin complex spectrum. */
  B200FFT_REAL_FULL = 0,
  /* cuFFT-style half spectrum (new functionality, north-star piece 3):
     forward: real (.., n_last) -> complex (.., n_last/2+1)   (n_last even or odd);
     inverse: complex (.., n_last/2+1) -> real (.., n_last), scaled 1/prod(dims). */
  B200FFT_REAL_HALF = 1
};

/* plan flags */
enum {
  /* Force the generic runtime-radix kernel for every axis (debug knob; plays the
     role of the reference's `_test: _GPUTest` path forcer, _ndim_fft_gpu.mojo:453-459). */
  B200FFT_FLAG_FORCE_GENERIC = 1u << 0,
  /* (bit 1 reserved: it named a chunking switch that round 1 never implemented) */
  /* Never use the fused N-d kernel (one persistent kernel for all axes, intermediate kept in L2):
     run one kernel per axis instead. b200fft_exec_scatter needs per-axis passes. */
  B200FFT_FLAG_NO_FUSED = 1u << 2,
  /* Use the fused N-d kernel whenever a variant matches the problem, not only where it was measured to win
     (what the environment variable B200FFT_FUSED=1 does process-wide). */
  B200FFT_FLAG_PREFER_FUSED = 1u << 3,
  /* Skip the compile-time kernels: run every axis on the runtime-length tier (rt.cu), falling back to the generic
     kernel where that tier does not apply. With FORCE_GENERIC / NO_FUSED / PREFER_FUSED this lets one small
     problem exercise every kernel tier, the job `_GPUTest.{BLOCK,WARP,DEVICE_WIDE,CLUSTER}` does in the
     reference (_ndim_fft_gpu.mojo:453-459, fft/tests.mojo:398-417). */
  B200FFT_FLAG_FORCE_RT = 1u << 4
};

/*
 * Runtime form of plan_fft's compile-time parameters (fft.mojo:122-132,160-176).
 * Buffers are dense row-major `(batch, dims[0..rank-1], components)`, interleaved
 * re/im, exactly the LayoutTensor layouts the reference requires.
 */
typedef struct b200fft_desc {
  int32_t rank;                   /* number of non-batch axes, 1..B200FFT_MAX_RANK             */
  int64_t dims[B200FFT_MAX_RANK]; /* out_layout.shape[1:rank+1]; each >= 2                     */
  int64_t batch;                  /* out_layout.shape[0] >= 1                                  */
  int32_t in_components;          /* in_layout last dim: 1 (real) or 2 (complex)               */
  int32_t in_dtype;               /* B200FFT_U8 | F32 | F64 (cast on load, _fft.mojo:257)      */
  int32_t out_dtype;              /* B200FFT_F32 | F64                                         */
  int32_t inverse;                /* 0 forward (unnormalised), 1 inverse (x 1/prod(dims))      */
  int32_t real_mode;              /* B200FFT_REAL_FULL | B200FFT_REAL_HALF                     */
  uint32_t axis_mask;             /* bit a set = transform axis a; 0 = all axes (reference).
                                     Used by the slab decomposition (local 2-D, then z pass).  */
  const uint32_t* bases;          /* user radix bases of all axes, concatenated; NULL = the
                                     reference's GPU default rule (fft.mojo:49-104)            */
  const int32_t* bases_count;     /* [rank] number of bases per axis (0 = default for that axis) */
  int32_t device;                 /* CUDA ordinal, or -1 for the current device                */
  uint32_t flags;                 /* B200FFT_FLAG_*                                            */
} b200fft_desc;

typedef struct b200fft_plan b200fft_plan;

/* ---- plan_fft[...](ctx=ctx)  (fft.mojo:160-210 -> _GPUPlan.__init__, _ndim_fft_gpu.mojo:179-207)
 * Validates the layout and bases, chooses kernels, uploads the twiddle tables. */
B200FFT_API int b200fft_plan_create(b200fft_plan** plan, const b200fft_desc* desc);

/* The same transform over STRIDED buffers (the layouts of cuFFT's advanced plans, or of a torch view). Each array has
 * rank + 1 strides, in ELEMENTS of that buffer, for the dimensions (batch, d0, ..., d_{rank-1}) of its own layout; one
 * element is one complex pair (its two components stay adjacent) or one real scalar, and the complex side of a
 * half-spectrum plan has n/2+1 elements along the last axis. NULL = the dense row-major strides; dense strides, given
 * either way, make exactly b200fft_plan_create's plan. The stride of a dimension of extent 1 is never read: any value
 * stands for the dense one, and no rule below applies to it. Checked before any CUDA call:
 *   - input strides >= 0, output strides >= 1 and no two output elements at one offset: B200FFT_ERR_LAYOUT;
 *   - an offset beyond int64: B200FFT_ERR_INVALID_ARG;
 *   - REAL_HALF: stride 1 along the last axis on both sides (pitched rows), and for an even length every real-side stride
 *     even (the kernels move real rows as pairs): B200FFT_ERR_UNSUPPORTED.
 * Every transformed axis is one pass of the plan-time specialisation tier reading and writing the arrays through their
 * strides (no copy pass): rows when the axis has the smallest stride of the buffer a pass reads, column tiles along the
 * dimension that has it otherwise. One tile holds the whole axis in at most 200 KB of shared memory: rows up to 16384
 * points in fp32 and 8192 in fp64 (some longer lengths fit, such as 20000 and 12500), column tiles over 8 or more
 * columns up to 1024 points in fp32 and 512 in fp64 (two-stage fp32 lengths such as 2304 = 48 x 48 fit; tiles over
 * fewer columns take longer axes). A longer axis, FORCE_GENERIC, FORCE_RT and B200FFT_JIT=0 return
 * B200FFT_ERR_UNSUPPORTED, naming the case. b200fft_exec runs such a plan in place
 * (d_out == d_in) only when that maps every element onto itself: equal strides and element types, or for REAL_HALF real
 * strides twice the complex ones on every dimension but the last (the padded in-place R2C / C2R layout) with equal input
 * and output precision; any other in-place call returns B200FFT_ERR_INVALID_ARG. b200fft_plan_in_bytes / out_bytes report
 * the bytes each buffer spans; exec_host and exec_scatter(_at) take dense plans only (B200FFT_ERR_UNSUPPORTED). */
B200FFT_API int b200fft_plan_create_strided(b200fft_plan** plan, const b200fft_desc* desc, const int64_t* in_strides,
                                            const int64_t* out_strides);

/* ---- fft(output, x, ctx, plan=plan)  (fft.mojo:262-323 -> _run_gpu_nd_fft, _ndim_fft_gpu.mojo:462-642)
 * Asynchronous on `cu_stream` (a CUstream / cudaStream_t; NULL = default stream);
 * the caller synchronises, as bench.mojo:51-52 does. `d_out` and `d_in` are device
 * pointers; out-of-place, or in-place (d_out == d_in) when input and output have the
 * same element type and component count.
 * Alignment: each pointer must be aligned to one element of its buffer (1 B uint8, 4 B fp32 real, 8 B fp32 complex
 * or fp64 real, 16 B fp64 complex) and to what the plan's kernels need beyond that: 16 B where they use 128-bit,
 * TMA or bulk-async global accesses (the default plans of 64-, 128- and 256-point complex rows among them), two
 * scalars where they read or write real rows as pairs (half-spectrum transforms of even length). Any pointer that
 * cudaMalloc or a torch allocation returns satisfies all of these; a view at an element offset may not. A less
 * aligned pointer returns B200FFT_ERR_INVALID_ARG before anything is launched, and b200fft_last_error() names the
 * pointer and the alignment. b200fft_exec_scatter(_at) check d_in, d_work and the peers the same way;
 * b200fft_exec_host stages through its own buffers and has no requirement. */
B200FFT_API int b200fft_exec(b200fft_plan* plan, void* d_out, const void* d_in, void* cu_stream);

/* Blocks until everything enqueued on `cu_stream` has finished (NULL = the legacy default stream, which is
 * where b200fft_exec launches when it is given NULL). A host language whose device context does not expose its
 * CUstream calls exec with NULL and then this, so that correctness never depends on whether the context's own
 * stream is a blocking one (the Mojo wrapper does: hackathon-fft_b200/mojo/fft/fft/_ndim_fft_gpu.mojo). */
B200FFT_API int b200fft_stream_synchronize(void* cu_stream);

/* Same transform with HOST buffers, cut into chunks that flow H2D -> kernels -> D2H on three internal streams
 * with two device buffers per direction; returns after the result is in h_out. The copies are issued straight
 * from / into the caller's memory: pass page-locked buffers (b200fft_host_register, cudaHostAlloc, torch
 * pin_memory) for the copies to run asynchronously and overlap the kernels — with pageable memory the call is
 * still correct but each copy is staged by the driver and serialises. This is the end-to-end call bench.py
 * times as `e2e`, and what the Mojo package's host-tensor overloads of `fft` call. */
B200FFT_API int b200fft_exec_host(b200fft_plan* plan, void* h_out, const void* h_in);
/* Page-lock / unlock a caller-owned host range (cudaHostRegister) so exec_host's copies overlap. */
B200FFT_API int b200fft_host_register(void* h_ptr, size_t bytes);
B200FFT_API int b200fft_host_unregister(void* h_ptr);

/* Slab-decomposition step 1 with the exchange fused into the last pass (multi-GPU, one process
 * per GPU). The plan is the LOCAL transform of this rank's slab, e.g. batch = local z planes,
 * dims = (Y, X). All passes but the last run normally (d_in -> d_work, in place on d_work; d_work
 * may equal d_in, which then gets overwritten). The last pass transforms axis 0 (Y), the axis being
 * re-split across ranks, and stores output row y of local plane z straight into
 *     peer_out[y / (Y/npeers)] [ ((my_rank * batch + z) * (Y/npeers) + y % (Y/npeers)) * X + x ]
 * i.e. into the [Z][Y/npeers][X] slab of the rank that owns row y. With peer_out[] mapped over
 * NVLink (b200fft_ipc_open) the all-to-all happens inside the kernel's stores; with local
 * pointers it is the pack step of an NCCL all-to-all. The caller synchronises the ranks (barrier)
 * before reading its slab and then runs the Z pass with a plan over (Z, Y/npeers, X), axis_mask=1.
 * A forward half-spectrum (B200FFT_REAL_HALF, R2C) plan is served the same way: its last pass is the complex Y pass over
 * the X/2+1 bins, so X above reads X/2+1, and d_work (which receives the half spectrum) must not be d_in (status 1).
 * Inverse (C2R) plans are refused (status 4). */
B200FFT_API int b200fft_exec_scatter(b200fft_plan* plan, void* const* peer_out, int npeers, int my_rank,
                                     const void* d_in, void* d_work, void* cu_stream);

/* The same for a SUB-RANGE of a rank's planes: the plan's `batch` planes are planes [z_first, z_first + batch) of the
 * global volume (exec_scatter is the case z_first = my_rank * batch). Lets a caller cut its slab into chunks and overlap
 * the X pass of one chunk with the NVLink-bound scattering Y pass of the previous one. */
B200FFT_API int b200fft_exec_scatter_at(b200fft_plan* plan, void* const* peer_out, int npeers, int64_t z_first,
                                        const void* d_in, void* d_work, void* cu_stream);

/* Device buffers that can be shared with the other ranks of the node (cudaMalloc + CUDA IPC). */
#define B200FFT_IPC_HANDLE_BYTES 64
B200FFT_API int b200fft_malloc(void** d_ptr, size_t bytes);
B200FFT_API int b200fft_free(void* d_ptr);
B200FFT_API int b200fft_ipc_export(void* d_ptr, unsigned char handle[B200FFT_IPC_HANDLE_BYTES]);
B200FFT_API int b200fft_ipc_open(const unsigned char handle[B200FFT_IPC_HANDLE_BYTES], void** d_ptr);
B200FFT_API int b200fft_ipc_close(void* d_ptr);

/* ---- Slab decomposition as ONE kernel per rank (slab.cuh): X rows, Y columns with the exchange fused into
 * their stores, and the Z columns of the received slab, overlapped tile by tile; cross-GPU dependencies are
 * per-x-block arrival counters that every rank bumps on every peer over NVLink (no barrier, no all-to-all).
 * Cubic volumes n^3 with n in {64, 128, 256, 512}, n divisible by `ranks`. Every rank allocates TWO receive
 * buffers of b200fft_slab_recv_bytes() with b200fft_malloc, ZEROES them, shares them over CUDA IPC and
 * synchronises with its peers once before the first exec; calls alternate buffer = 0, 1, 0, ... and every rank
 * must make the same sequence of calls. peer_recv[h] = rank h's buffer `buffer` (peer_recv[rank] = the local
 * one); after the kernel the first n * (n/ranks) * n complex values of the local buffer hold out[z][y_local][x]. */
typedef struct b200fft_slab b200fft_slab;
B200FFT_API int b200fft_slab_create(b200fft_slab** slab, int64_t n, int ranks, int rank, int inverse, int device);
B200FFT_API size_t b200fft_slab_recv_bytes(const b200fft_slab* slab);
/* byte offset, inside a receive buffer, of a uint32 that counts Z tiles whose wait for the peers timed out (~2 s);
 * non-zero after a synchronise means the result of that call is invalid (a rank died or skipped a call) */
B200FFT_API size_t b200fft_slab_timeout_offset(const b200fft_slab* slab);
B200FFT_API int b200fft_slab_exec(b200fft_slab* slab, const void* d_in, void* d_work, void* const* peer_recv, int buffer,
                                  void* cu_stream);
B200FFT_API size_t b200fft_slab_describe(const b200fft_slab* slab, char* buf, size_t cap);
B200FFT_API int b200fft_slab_destroy(b200fft_slab* slab);

B200FFT_API int b200fft_plan_destroy(b200fft_plan* plan);

/* ---- Multi-device entry points: ONE host process drives several GPUs of a node (SURVEY.md 8b/8e). The reference has
 * no multi-GPU path; a Mojo host owns one DeviceContext per GPU and would otherwise have to re-implement the sharding
 * and the slab orchestration that python/b200fft/slab.py does over torch.distributed. Device slot g runs on CUDA
 * ordinal devices[g] (devices == NULL: ordinals 0..ngpu-1) on a plan-owned non-blocking stream.
 *
 *   B200FFT_MGPU_BATCH_SHARD  `desc` describes the WHOLE job; slot g owns the contiguous batch items
 *                             [first_g, first_g + count_g) (the first batch % ngpu slots hold one more). No
 *                             communication. d_in[g] / d_out[g] hold only that slot's items.
 *   B200FFT_MGPU_SLAB         one 3-D complex fp32 or fp64 transform (batch 1, dims (Z, Y, X), Z and Y divisible by ngpu,
 *                             the same type in and out). Slot g holds the input z planes [g Z/G, (g+1) Z/G) as
 *                             d_in[g][Z/G][Y][X]; after exec d_out[h] holds out[z][y_local][x] for y = h Y/G + y_local,
 *                             i.e. d_out[h][Z][Y/G][X] ("transposed out", as the slab decomposition of north_star leaves
 *                             it). Local (Y, X) transform with the exchange fused into the Y pass's stores (peer-to-peer
 *                             over NVLink, cudaDeviceEnablePeerAccess, no pack buffer, no all-to-all), device-side event
 *                             barrier, strided Z pass in place on d_out. The inverse keeps this orientation (z planes in,
 *                             Y-slabs out). d_out[] must be peer-accessible device memory (cudaMalloc / b200fft_malloc).
 *                             With real_mode = B200FFT_REAL_HALF (W = X/2+1, X even or odd):
 *                             forward (R2C): d_in[g][Z/G][Y][X] real (fp32 or fp64, cast on load) -> d_out[h]
 *                               [Z][Y/G][W] complex in out_dtype (fp32 or fp64): the same Y-slabs over the half spectrum,
 *                               which halves the bytes the exchange moves.
 *                             inverse (C2R): the OTHER orientation, so that forward then inverse round-trips on the device
 *                               buffers: d_in[g][Z][Y/G][W] is the Y-slab the forward leaves (rows y = g Y/G + y_local, in
 *                               the working precision) -> d_out[g][Z/G][Y][X] real z planes, scaled by 1 / (Z Y X). A Z
 *                               pass whose stores go to the owning peers' receive buffers (allocated by the plan),
 *                               the event barrier, then the local (Y, X) C2R. d_in is not written.
 *                             Refused with status 4: batch > 1, axis_mask != 0, real input with B200FFT_REAL_FULL, uint8
 *                             input (as by the single-device half-spectrum plans), and a
 *                             half-spectrum plan whose scattering axis (Y forward, Z inverse) is too long for one column
 *                             tile (checked at plan creation).
 *
 * exec enqueues on every slot's stream and returns; b200fft_mgpu_synchronize waits for all of them.
 * b200fft_mgpu_stream(plan, g) is that stream (a cudaStream_t) for callers that order their own work against it.
 * exec_host takes the WHOLE job in host memory, natural order (SLAB: h_in[Z][Y][X] -> h_out[Z][Y][X]; half spectrum:
 * real [Z][Y][X] -> complex [Z][Y][X/2+1], the inverse the reverse): every slot
 * copies its share in, runs, and copies its share out (one host thread per slot for BATCH_SHARD, each running the
 * chunked 3-stream pipeline of b200fft_exec_host); returns when h_out is complete. */
enum { B200FFT_MGPU_BATCH_SHARD = 0, B200FFT_MGPU_SLAB = 1 };
typedef struct b200fft_mgpu_plan b200fft_mgpu_plan;
B200FFT_API int b200fft_mgpu_plan_create(b200fft_mgpu_plan** plan, const b200fft_desc* desc, int ngpu, const int* devices,
                                         int mode);
B200FFT_API int b200fft_mgpu_plan_destroy(b200fft_mgpu_plan* plan);
B200FFT_API int b200fft_mgpu_ngpu(const b200fft_mgpu_plan* plan);
/* what slot g holds on input: batch items (BATCH_SHARD), z planes (SLAB) or, for the SLAB half-spectrum inverse, y rows
 * [*first, *first + *count). in_bytes / out_bytes: the sizes of slot g's d_in[g] / d_out[g]. */
B200FFT_API int b200fft_mgpu_shard(const b200fft_mgpu_plan* plan, int g, int64_t* first, int64_t* count);
B200FFT_API size_t b200fft_mgpu_in_bytes(const b200fft_mgpu_plan* plan, int g);
B200FFT_API size_t b200fft_mgpu_out_bytes(const b200fft_mgpu_plan* plan, int g);
B200FFT_API int b200fft_mgpu_exec(b200fft_mgpu_plan* plan, void* const* d_out, const void* const* d_in);
B200FFT_API int b200fft_mgpu_synchronize(b200fft_mgpu_plan* plan);
B200FFT_API void* b200fft_mgpu_stream(const b200fft_mgpu_plan* plan, int g);
B200FFT_API int b200fft_mgpu_exec_host(b200fft_mgpu_plan* plan, void* h_out, const void* h_in);
B200FFT_API size_t b200fft_mgpu_describe(const b200fft_mgpu_plan* plan, char* buf, size_t cap);
/* host-only: the batch split BATCH_SHARD uses (no CUDA call) */
B200FFT_API int b200fft_mgpu_split(int64_t batch, int ngpu, int g, int64_t* first, int64_t* count);

/* ---- introspection (tests, harness) */
B200FFT_API size_t b200fft_plan_workspace_bytes(const b200fft_plan* plan);
/* ordered stage list of an axis, the reference's `_get_ordered_bases_processed_list`
 * (_utils.mojo:186-221); returns the count or -1 */
B200FFT_API int b200fft_plan_get_bases(const b200fft_plan* plan, int axis, uint32_t* out, int cap);
/* human-readable list of the kernel passes the plan launches; returns bytes needed */
B200FFT_API size_t b200fft_plan_describe(const b200fft_plan* plan, char* buf, size_t cap);
/* number of kernel launches one b200fft_exec performs */
B200FFT_API int b200fft_plan_launches(const b200fft_plan* plan);
/* in/out buffer sizes in bytes for one exec */
B200FFT_API size_t b200fft_plan_in_bytes(const b200fft_plan* plan);
B200FFT_API size_t b200fft_plan_out_bytes(const b200fft_plan* plan);

/* ---- host-side planner rules, usable without a GPU */
/* `_build_ordered_bases` + validity asserts (_utils.mojo:163-221); count or -1 if rejected */
B200FFT_API int b200fft_ordered_bases(uint64_t length, const uint32_t* bases, int nbases, uint32_t* out, int cap);
/* `_estimate_best_bases` (fft.mojo:49-104); gpu_target != 0 selects the GPU rule */
B200FFT_API int b200fft_default_bases(uint64_t length, int gpu_target, uint32_t* out, int cap);
/* validate a descriptor and write the pass list it would produce, without touching CUDA */
B200FFT_API int b200fft_plan_dry_run(const b200fft_desc* desc, char* buf, size_t cap);

/* Plan-time specialisation (csrc/jit.cu): axis lengths without a hand-registered kernel variant get the compile-time
 * kernels instantiated through NVRTC when the plan is created — the run-time counterpart of the reference
 * specialising every (length, bases) at compile time (_ndim_fft_gpu.mojo:279-450). This probe compiles the kernel the
 * planner would pick for ONE axis (length n, element stride `inner`, user bases or NULL for the default rule) and
 * writes "<variant>: <template-id>, smem, cubin size, compile time, symbol" into buf. Needs libnvrtc but no GPU. */
B200FFT_API int b200fft_jit_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in,
                                  int half /* 0 complex, 1 half-spectrum R2C rows, 2 C2R rows, 3 the scattering Z pass of a
                                              half-spectrum slab inverse (B200FFT_MGPU_SLAB) over `inner` columns */,
                                  int in_dtype, int out_dtype,
                                  char* buf, size_t cap);
/* The same for the strided form of that kernel (b200fft_plan_create_strided; inner > 1: column tiles over `inner` columns).
 * Its variant name ends in "_str". No GPU needed. */
B200FFT_API int b200fft_jit_probe_strided(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in,
                                          int half, int in_dtype, int out_dtype, char* buf, size_t cap);
/* The same for an axis too long for one tile: compiles the two passes (pass A: N1-point strided transforms with the
 * twiddle fused into the store; pass B: N2-point rows with the natural-order, half-spectrum or real store) the
 * planner builds for it, and writes "<pass A report>; <pass B report>". Serves complex, real-input and half-spectrum
 * (R2C / C2R, even and odd n) axes; B200FFT_ERR_UNSUPPORTED when the stage list has no such split. No GPU needed. */
B200FFT_API int b200fft_jit_split_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in,
                                        int half, int in_dtype, int out_dtype, char* buf, size_t cap);
/* The same for a contiguous axis longer than 2^24 points: compiles the three passes (1: N1-point strided transforms of
 * the user's array, W_n twiddle from two tables of about sqrt(n) entries; 2: N2-point strided transforms in place on
 * the temporary, W_M twiddle likewise; 3: N3-point rows with the natural-order store) the planner builds for it, and
 * writes "<pass 1 report>; <pass 2 report>; <pass 3 report>". Complex input, or real input with the full spectrum;
 * B200FFT_ERR_UNSUPPORTED for n <= 2^24, half-spectrum rows, strided axes (inner > 1), a radix above 127, or a stage
 * list with no such split. No GPU needed. */
B200FFT_API int b200fft_jit_split3_probe(int64_t n, int64_t inner, const uint32_t* bases, int nbases, int inverse, int real_in,
                                         int half, int in_dtype, int out_dtype, char* buf, size_t cap);

/* Tile schedule of the fused N-d kernel (host logic, no CUDA): phases[p] = {tiles_per_transform,
 * tiles_per_group, dep_div, quota}; writes up to `cap` segments as {phase, first_item, first_tile, count}
 * and returns the number of segments (or -1). Tests use it to check that every tile appears once and
 * never before the tiles it depends on. */
B200FFT_API int b200fft_schedule_dry_run(int nphases, const int64_t* phases /* [nphases][4] */, int64_t batch,
                                         int64_t* segments /* [cap][4] */, int cap);

/* ---- errors / bookkeeping */
B200FFT_API const char* b200fft_strerror(int status);
B200FFT_API const char* b200fft_last_error(void); /* thread-local detail of the last failure */
B200FFT_API int b200fft_version(void);
/* total kernels launched by this library in this process (bench.py's gpu_launches) */
B200FFT_API uint64_t b200fft_launch_count(void);
/* number of compiled-in kernel variants: tier 0 = compile-time row / column variants, 1 = fused N-d kernels,
 * 2 = two-pass split kernels; -1 for an unknown tier. Host-only (no CUDA call); safe to call from several threads at
 * once, like plan creation: the variant tables are built exactly once. */
B200FFT_API int b200fft_variant_count(int tier);
/* One line describing variant `index` of `tier` (same tiers and order as b200fft_variant_count), fields separated
 * by spaces:
 *   name=<name> kind=<rows|rowsIP|cols|colsT|splitA|splitB_cols|splitB_rows|fused> n=<length> (fused: dims, "64x64x64")
 *   radices=<16x8> (fused: the phases' stage lists, "8x8;8x8|8x8") tile=<rows or columns per CTA> threads=<count>
 *   forms=<comma list> of what the variant instantiates: fwd, inv (complex input), real (real input, full spectrum),
 *   r2c, c2r (half spectrum of 2n points on this n-point variant), r2c-reg (R2C with the register unpack), r2c-odd,
 *   c2r-odd (half spectrum of odd n itself), scatter (slab exchange in the store); fused: mode=<c2c|real|r2c> and
 *   direction fwd or inv.
 * Writes at most `cap` bytes including the terminating NUL and returns the length of the whole line plus one, or
 * -1 for an unknown tier or index. Host-only (no CUDA call). */
B200FFT_API int b200fft_variant_info(int tier, int index, char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* B200FFT_H */

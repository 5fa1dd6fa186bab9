// Multi-device entry points of the C ABI (include/b200fft.h: b200fft_mgpu_*): one host process, several GPUs.
// Built entirely on the single-device entry points (plan_create / exec / exec_scatter / exec_host): a device slot is
// one b200fft_plan (two for the slab mode) + one non-blocking stream + a few events on its own CUDA device.
//
// BATCH_SHARD: independent transforms split by batch, no communication (north_star: "batched transforms are split by
// batch across the 8 GPUs with no communication").
// SLAB: one (Z, Y, X) volume, slot g owns z planes [g Z/G, (g+1) Z/G):
//   1. local (Y, X) transform; the Y pass stores row y straight into the slab of the slot that owns y
//      (b200fft_exec_scatter over peer-mapped pointers: the all-to-all is the kernel's own NVLink stores);
//   2. device-side barrier: every slot's stream waits for the "scatter done" event of every other slot;
//   3. strided Z pass in place on the received [Z][Y/G][X] slab.
// What python/b200fft/slab.py does with one process per GPU, CUDA IPC and a one-word all-reduce, done here with peer
// access and cross-device events: no NCCL, no host round trip between the steps.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.hpp"

using namespace b200fft;

namespace {

struct DevGuard {
  int prev = -1;
  DevGuard() { cudaGetDevice(&prev); }
  ~DevGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

struct Slot {
  int device = 0;
  int64_t first = 0, count = 0;  // batch items (BATCH_SHARD) / z planes (SLAB)
  b200fft_plan* plan = nullptr;  // BATCH_SHARD: the shard's plan; SLAB: local (Y, X) transform of the slot's planes
  b200fft_plan* planz = nullptr; // SLAB: Z pass over the received [Z][Y/G][X] slab
  cudaStream_t stream = nullptr;
  cudaEvent_t scattered = nullptr, done = nullptr;
  void* work = nullptr;          // SLAB: [Z/G][Y][X] intermediate of step 1
  void* h_in = nullptr;          // SLAB exec_host: device staging, allocated on first use
  void* h_out = nullptr;
  size_t in_bytes = 0, out_bytes = 0;
};

}  // namespace

struct MgpuPool {
  std::vector<std::thread> threads;
  std::mutex mu;
  std::condition_variable cv;
  std::atomic<uint64_t> gen{0};
  std::atomic<int> arrived{0};
  std::atomic<bool> stop{false};
  void* const* out_tab = nullptr;
  const void* const* in_tab = nullptr;
  std::vector<int> rc;
  std::vector<std::string> msg;
  void start(b200fft_mgpu_plan* plan, int n);
  int run(int n, void* const* d_out, const void* const* d_in);
  void shutdown();
};

struct b200fft_mgpu_plan {
  std::unique_ptr<MgpuPool> pool;  // enqueue workers (B200FFT_MGPU_THREADS=0: enqueue from the calling thread)
  int mode = 0;
  int64_t batch = 0;
  int64_t Z = 0, Y = 0, X = 0;
  size_t in_item = 0, out_item = 0;  // BATCH_SHARD: bytes per batch item
  bool executed = false;             // SLAB: `done` events have been recorded at least once
  std::vector<Slot> slots;
  std::string text;
};

namespace {

int split_batch(int64_t batch, int ngpu, int g, int64_t* first, int64_t* count) {
  if (batch < 0 || ngpu < 1 || g < 0 || g >= ngpu) return -1;
  const int64_t q = batch / ngpu, r = batch % ngpu;
  if (first) *first = (int64_t)g * q + std::min<int64_t>(g, r);
  if (count) *count = q + (g < r ? 1 : 0);
  return 0;
}

// the concatenated user bases of axes [a0, a1) of `desc` (empty = defaults everywhere)
void slice_bases(const b200fft_desc& d, int a0, int a1, std::vector<uint32_t>* bases, std::vector<int32_t>* counts) {
  bases->clear();
  counts->clear();
  if (!d.bases || !d.bases_count) return;
  size_t off = 0;
  for (int a = 0; a < d.rank; ++a) {
    const int32_t c = d.bases_count[a];
    if (a >= a0 && a < a1) {
      counts->push_back(c);
      for (int32_t i = 0; i < c; ++i) bases->push_back(d.bases[off + (size_t)i]);
    }
    off += (size_t)std::max<int32_t>(c, 0);
  }
}

int enable_peers(const std::vector<Slot>& slots) {
  for (const Slot& a : slots) {
    B200_CUDA_CHECK(cudaSetDevice(a.device));
    for (const Slot& b : slots) {
      if (a.device == b.device) continue;
      int can = 0;
      B200_CUDA_CHECK(cudaDeviceCanAccessPeer(&can, a.device, b.device));
      if (!can)
        return fail(B200FFT_ERR_UNSUPPORTED, "device %d cannot map device %d's memory: the slab exchange needs peer access",
                    a.device, b.device);
      cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess)
        return fail(B200FFT_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", a.device, b.device, cudaGetErrorString(e));
    }
  }
  return B200FFT_OK;
}

int describe_plan(const b200fft_plan* p, std::string* out) {
  const size_t need = b200fft_plan_describe(p, nullptr, 0);
  std::string s(need + 1, '\0');
  b200fft_plan_describe(p, &s[0], s.size());
  s.resize(strlen(s.c_str()));
  *out = s;
  return 0;
}

}  // namespace

extern "C" {

int b200fft_mgpu_split(int64_t batch, int ngpu, int g, int64_t* first, int64_t* count) {
  return split_batch(batch, ngpu, g, first, count);
}

int b200fft_mgpu_plan_destroy(b200fft_mgpu_plan* m) {
  if (!m) return B200FFT_OK;
  if (m->pool) m->pool->shutdown();
  DevGuard guard;
  for (Slot& s : m->slots) {
    cudaSetDevice(s.device);
    if (s.stream) cudaStreamSynchronize(s.stream);
  }
  for (Slot& s : m->slots) {
    cudaSetDevice(s.device);
    if (s.plan) b200fft_plan_destroy(s.plan);
    if (s.planz) b200fft_plan_destroy(s.planz);
    for (void* p : {s.work, s.h_in, s.h_out})
      if (p) cudaFree(p);
    if (s.scattered) cudaEventDestroy(s.scattered);
    if (s.done) cudaEventDestroy(s.done);
    if (s.stream) cudaStreamDestroy(s.stream);
  }
  cudaGetLastError();
  delete m;
  return B200FFT_OK;
}

int b200fft_mgpu_plan_create(b200fft_mgpu_plan** out, const b200fft_desc* desc, int ngpu, const int* devices, int mode) {
  if (!out) return fail(B200FFT_ERR_INVALID_ARG, "null plan pointer");
  *out = nullptr;
  if (!desc) return fail(B200FFT_ERR_INVALID_ARG, "null descriptor");
  if (ngpu < 1 || ngpu > 16) return fail(B200FFT_ERR_INVALID_ARG, "ngpu = %d (1..16)", ngpu);
  if (mode != B200FFT_MGPU_BATCH_SHARD && mode != B200FFT_MGPU_SLAB)
    return fail(B200FFT_ERR_INVALID_ARG, "unknown multi-device mode %d", mode);
  if (desc->rank < 1 || desc->rank > B200FFT_MAX_RANK) return fail(B200FFT_ERR_INVALID_ARG, "rank %d", desc->rank);
  int ndev = 0;
  B200_CUDA_CHECK(cudaGetDeviceCount(&ndev));
  std::vector<int> devs((size_t)ngpu);
  for (int g = 0; g < ngpu; ++g) {
    devs[(size_t)g] = devices ? devices[g] : g;
    if (devs[(size_t)g] < 0 || devs[(size_t)g] >= ndev)
      return fail(B200FFT_ERR_INVALID_ARG, "slot %d: CUDA device %d of %d", g, devs[(size_t)g], ndev);
    for (int h = 0; h < g; ++h)
      if (mode == B200FFT_MGPU_SLAB && devs[(size_t)h] == devs[(size_t)g] && ngpu > 1 && !getenv("B200FFT_MGPU_ALLOW_SAME_DEVICE"))
        return fail(B200FFT_ERR_INVALID_ARG, "slots %d and %d name the same device %d", h, g, devs[(size_t)g]);
  }

  DevGuard guard;
  std::unique_ptr<b200fft_mgpu_plan> m(new b200fft_mgpu_plan());
  m->mode = mode;
  m->slots.resize((size_t)ngpu);
  auto bail = [&](int rc) {
    b200fft_mgpu_plan_destroy(m.release());
    return rc;
  };
  for (int g = 0; g < ngpu; ++g) m->slots[(size_t)g].device = devs[(size_t)g];

  if (mode == B200FFT_MGPU_BATCH_SHARD) {
    if (desc->batch < ngpu) return bail(fail(B200FFT_ERR_INVALID_ARG, "batch %lld is smaller than %d devices", (long long)desc->batch, ngpu));
    m->batch = desc->batch;
    for (int g = 0; g < ngpu; ++g) {
      Slot& s = m->slots[(size_t)g];
      split_batch(desc->batch, ngpu, g, &s.first, &s.count);
      b200fft_desc d = *desc;
      d.batch = s.count;
      d.device = s.device;
      if (int rc = b200fft_plan_create(&s.plan, &d)) return bail(rc);
      s.in_bytes = b200fft_plan_in_bytes(s.plan);
      s.out_bytes = b200fft_plan_out_bytes(s.plan);
      if (g == 0) {
        m->in_item = s.in_bytes / (size_t)s.count;
        m->out_item = s.out_bytes / (size_t)s.count;
      }
    }
  } else {
    if (desc->rank != 3 || desc->batch != 1 || desc->in_components != 2 || desc->in_dtype != B200FFT_F32 ||
        desc->out_dtype != B200FFT_F32 || desc->real_mode != B200FFT_REAL_FULL || desc->axis_mask != 0)
      return bail(fail(B200FFT_ERR_UNSUPPORTED, "slab mode takes ONE 3-D complex fp32 transform (batch 1, rank 3, all axes)"));
    m->Z = desc->dims[0];
    m->Y = desc->dims[1];
    m->X = desc->dims[2];
    if (m->Z % ngpu || m->Y % ngpu)
      return bail(fail(B200FFT_ERR_INVALID_ARG, "slab decomposition needs Z = %lld and Y = %lld divisible by %d devices",
                       (long long)m->Z, (long long)m->Y, ngpu));
    const int64_t zl = m->Z / ngpu, yl = m->Y / ngpu;
    if (yl < 2 && ngpu > 1) return bail(fail(B200FFT_ERR_INVALID_ARG, "fewer than 2 y rows per device"));
    if (int rc = enable_peers(m->slots)) return bail(rc);
    std::vector<uint32_t> b_yx, b_z;
    std::vector<int32_t> c_yx, c_z;
    slice_bases(*desc, 1, 3, &b_yx, &c_yx);
    slice_bases(*desc, 0, 1, &b_z, &c_z);
    for (int g = 0; g < ngpu; ++g) {
      Slot& s = m->slots[(size_t)g];
      s.first = g * zl;
      s.count = zl;
      s.in_bytes = (size_t)zl * m->Y * m->X * 8;
      s.out_bytes = (size_t)m->Z * yl * m->X * 8;
      b200fft_desc d2 = *desc;  // local 2-D transform of zl planes; exec_scatter drives its per-axis passes
      d2.rank = 2;
      d2.dims[0] = m->Y;
      d2.dims[1] = m->X;
      d2.batch = zl;
      d2.device = s.device;
      d2.flags = (desc->flags | B200FFT_FLAG_NO_FUSED) & ~(uint32_t)B200FFT_FLAG_PREFER_FUSED;
      d2.bases = c_yx.empty() ? nullptr : b_yx.data();
      d2.bases_count = c_yx.empty() ? nullptr : c_yx.data();
      if (int rc = b200fft_plan_create(&s.plan, &d2)) return bail(rc);
      b200fft_desc dz = *desc;  // Z pass over [Z][yl][X], only axis 0 transformed
      dz.rank = 3;
      dz.dims[0] = m->Z;
      dz.dims[1] = yl;
      dz.dims[2] = m->X;
      dz.batch = 1;
      dz.axis_mask = 1;
      dz.device = s.device;
      std::vector<int32_t> cz3;
      if (!c_z.empty()) cz3 = {c_z[0], 0, 0};
      dz.bases = cz3.empty() ? nullptr : b_z.data();
      dz.bases_count = cz3.empty() ? nullptr : cz3.data();
      if (int rc = b200fft_plan_create(&s.planz, &dz)) return bail(rc);
      if (cudaSetDevice(s.device) != cudaSuccess || cudaMalloc(&s.work, s.in_bytes) != cudaSuccess) {
        cudaGetLastError();
        return bail(fail(B200FFT_ERR_ALLOC, "cannot allocate %zu B of slab workspace on device %d", s.in_bytes, s.device));
      }
    }
  }
  for (Slot& s : m->slots) {
    if (cudaSetDevice(s.device) != cudaSuccess || cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.scattered, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming) != cudaSuccess) {
      cudaError_t e = cudaGetLastError();
      return bail(fail(B200FFT_ERR_CUDA, "stream / event creation on device %d: %s", s.device, cudaGetErrorString(e)));
    }
  }
  char head[320];
  if (mode == B200FFT_MGPU_BATCH_SHARD)
    snprintf(head, sizeof head, "mgpu batch-shard over %d devices, batch %lld, no communication\n", ngpu, (long long)m->batch);
  else
    snprintf(head, sizeof head,
             "mgpu slab %lldx%lldx%lld over %d devices: local (Y,X) + peer-to-peer scattering Y stores -> event barrier -> Z pass\n",
             (long long)m->Z, (long long)m->Y, (long long)m->X, ngpu);
  m->text = head;
  for (int g = 0; g < ngpu; ++g) {
    const Slot& s = m->slots[(size_t)g];
    std::string t;
    describe_plan(s.plan, &t);
    char line[160];
    snprintf(line, sizeof line, " slot %d (device %d): %s [%lld, %lld)\n", g, s.device,
             mode == B200FFT_MGPU_SLAB ? "z planes" : "batch items", (long long)s.first, (long long)(s.first + s.count));
    m->text += line;
    if (g == 0) {
      m->text += t;
      if (s.planz) {
        describe_plan(s.planz, &t);
        m->text += t;
      }
    }
  }
  {
    const char* e = getenv("B200FFT_MGPU_THREADS");
    if (ngpu > 1 && !(e && atoi(e) == 0)) {
      m->pool.reset(new MgpuPool());
      m->pool->start(m.get(), ngpu);
    }
  }
  *out = m.release();
  return B200FFT_OK;
}

int b200fft_mgpu_ngpu(const b200fft_mgpu_plan* m) { return m ? (int)m->slots.size() : 0; }

int b200fft_mgpu_shard(const b200fft_mgpu_plan* m, int g, int64_t* first, int64_t* count) {
  if (!m || g < 0 || g >= (int)m->slots.size()) return fail(B200FFT_ERR_INVALID_ARG, "no such device slot");
  if (first) *first = m->slots[(size_t)g].first;
  if (count) *count = m->slots[(size_t)g].count;
  return B200FFT_OK;
}

size_t b200fft_mgpu_in_bytes(const b200fft_mgpu_plan* m, int g) {
  return m && g >= 0 && g < (int)m->slots.size() ? m->slots[(size_t)g].in_bytes : 0;
}
size_t b200fft_mgpu_out_bytes(const b200fft_mgpu_plan* m, int g) {
  return m && g >= 0 && g < (int)m->slots.size() ? m->slots[(size_t)g].out_bytes : 0;
}
void* b200fft_mgpu_stream(const b200fft_mgpu_plan* m, int g) {
  return m && g >= 0 && g < (int)m->slots.size() ? (void*)m->slots[(size_t)g].stream : nullptr;
}

size_t b200fft_mgpu_describe(const b200fft_mgpu_plan* m, char* buf, size_t cap) {
  if (!m) return 0;
  if (buf && cap) {
    strncpy(buf, m->text.c_str(), cap - 1);
    buf[cap - 1] = 0;
  }
  return m->text.size() + 1;
}

// One slot's share of an exec call. phase 0: everything up to (and including) the record of `scattered`; phase 1: the Z
// pass. Between the two every slot must have RECORDED its `scattered` event, or a wait on it would be a no-op.
static int slot_enqueue(b200fft_mgpu_plan* m, int g, int phase, void* const* d_out, const void* const* d_in) {
  const int G = (int)m->slots.size();
  Slot& s = m->slots[(size_t)g];
  B200_CUDA_CHECK(cudaSetDevice(s.device));
  if (m->mode == B200FFT_MGPU_BATCH_SHARD) return phase == 0 ? b200fft_exec(s.plan, d_out[g], d_in[g], s.stream) : B200FFT_OK;
  if (phase == 0) {
    // a slot may not start scattering call k+1 into a peer's slab while that peer still runs the Z pass of call k
    if (m->executed)
      for (int h = 0; h < G; ++h)
        if (h != g) B200_CUDA_CHECK(cudaStreamWaitEvent(s.stream, m->slots[(size_t)h].done, 0));
    if (int rc = b200fft_exec_scatter(s.plan, d_out, G, g, d_in[g], s.work, s.stream)) return rc;
    B200_CUDA_CHECK(cudaSetDevice(s.device));
    B200_CUDA_CHECK(cudaEventRecord(s.scattered, s.stream));
    return B200FFT_OK;
  }
  for (int h = 0; h < G; ++h)
    if (h != g) B200_CUDA_CHECK(cudaStreamWaitEvent(s.stream, m->slots[(size_t)h].scattered, 0));
  if (int rc = b200fft_exec(s.planz, d_out[g], d_out[g], s.stream)) return rc;
  B200_CUDA_CHECK(cudaSetDevice(s.device));
  B200_CUDA_CHECK(cudaEventRecord(s.done, s.stream));
  return B200FFT_OK;
}

// Enqueue workers: one persistent host thread per slot. Issuing one exec to 8 devices from ONE thread costs ~100 driver
// calls back to back (~0.3 ms: as long as the 512^3 slab transform itself takes on 8 GPUs); spread over the workers the
// host side takes the time of one slot. Workers spin briefly for the next call before they sleep.
void MgpuPool::start(b200fft_mgpu_plan* plan, int n) {
  for (int g = 0; g < n; ++g)
    threads.emplace_back([this, plan, g, n] {
      uint64_t seen = 0;
      for (;;) {
        uint64_t cur = seen;
        for (int spin = 0; spin < 20000 && (cur = gen.load(std::memory_order_acquire)) == seen; ++spin) {
        }
        if (cur == seen) {
          std::unique_lock<std::mutex> lk(mu);
          cv.wait(lk, [&] { return gen.load(std::memory_order_acquire) != seen; });
          cur = gen.load(std::memory_order_acquire);
        }
        seen = cur;
        if (stop.load()) return;
        for (int phase = 0; phase < 2; ++phase) {
          if (rc[(size_t)g] == B200FFT_OK) {
            const int r = slot_enqueue(plan, g, phase, out_tab, in_tab);
            if (r != B200FFT_OK) {
              rc[(size_t)g] = r;
              msg[(size_t)g] = last_error();
            }
          }
          // phase barrier (also the completion signal after phase 1)
          const int want = (phase + 1) * n;
          arrived.fetch_add(1, std::memory_order_acq_rel);
          if (phase == 0)
            while (arrived.load(std::memory_order_acquire) < want) {
            }
        }
      }
    });
}

void MgpuPool::shutdown() {
  if (threads.empty()) return;
  {
    std::lock_guard<std::mutex> lk(mu);
    stop.store(true);
    gen.fetch_add(1, std::memory_order_release);
  }
  cv.notify_all();
  for (auto& t : threads) t.join();
  threads.clear();
}

int MgpuPool::run(int n, void* const* d_out, const void* const* d_in) {
  out_tab = d_out;
  in_tab = d_in;
  rc.assign((size_t)n, B200FFT_OK);
  msg.assign((size_t)n, std::string());
  arrived.store(0, std::memory_order_release);
  {
    std::lock_guard<std::mutex> lk(mu);
    gen.fetch_add(1, std::memory_order_release);
  }
  cv.notify_all();
  while (arrived.load(std::memory_order_acquire) < 2 * n) {
  }
  for (int g = 0; g < n; ++g)
    if (rc[(size_t)g] != B200FFT_OK) return fail(rc[(size_t)g], "device slot %d: %s", g, msg[(size_t)g].c_str());
  return B200FFT_OK;
}

int b200fft_mgpu_exec(b200fft_mgpu_plan* m, void* const* d_out, const void* const* d_in) {
  if (!m || !d_out || !d_in) return fail(B200FFT_ERR_INVALID_ARG, "null plan or pointer table");
  const int G = (int)m->slots.size();
  for (int g = 0; g < G; ++g)
    if (!d_out[g] || !d_in[g]) return fail(B200FFT_ERR_INVALID_ARG, "null buffer for device slot %d", g);
  int rc = B200FFT_OK;
  if (m->pool && G > 1) {
    rc = m->pool->run(G, d_out, d_in);
  } else {
    DevGuard guard;
    for (int phase = 0; phase < 2 && rc == B200FFT_OK; ++phase)
      for (int g = 0; g < G && rc == B200FFT_OK; ++g) rc = slot_enqueue(m, g, phase, d_out, d_in);
  }
  if (rc == B200FFT_OK) m->executed = true;
  return rc;
}

int b200fft_mgpu_synchronize(b200fft_mgpu_plan* m) {
  if (!m) return fail(B200FFT_ERR_INVALID_ARG, "null plan");
  DevGuard guard;
  for (Slot& s : m->slots) {
    B200_CUDA_CHECK(cudaSetDevice(s.device));
    B200_CUDA_CHECK(cudaStreamSynchronize(s.stream));
  }
  return B200FFT_OK;
}

int b200fft_mgpu_exec_host(b200fft_mgpu_plan* m, void* h_out, const void* h_in) {
  if (!m || !h_out || !h_in) return fail(B200FFT_ERR_INVALID_ARG, "null plan or buffer");
  const int G = (int)m->slots.size();
  if (m->mode == B200FFT_MGPU_BATCH_SHARD) {
    // one host thread per device, each running the single-device chunked H2D -> kernels -> D2H pipeline on its shard
    std::vector<int> rc((size_t)G, B200FFT_OK);
    std::vector<std::string> msg((size_t)G);
    std::vector<std::thread> th;
    for (int g = 0; g < G; ++g)
      th.emplace_back([&, g] {
        Slot& s = m->slots[(size_t)g];
        cudaSetDevice(s.device);
        rc[(size_t)g] = b200fft_exec_host(s.plan, (char*)h_out + (size_t)s.first * m->out_item,
                                          (const char*)h_in + (size_t)s.first * m->in_item);
        if (rc[(size_t)g]) msg[(size_t)g] = b200fft_last_error();
      });
    for (auto& t : th) t.join();
    for (int g = 0; g < G; ++g)
      if (rc[(size_t)g]) return fail(rc[(size_t)g], "device slot %d: %s", g, msg[(size_t)g].c_str());
    return B200FFT_OK;
  }
  DevGuard guard;
  std::vector<void*> outs((size_t)G);
  std::vector<const void*> ins((size_t)G);
  for (int g = 0; g < G; ++g) {
    Slot& s = m->slots[(size_t)g];
    B200_CUDA_CHECK(cudaSetDevice(s.device));
    if (!s.h_in) B200_CUDA_CHECK(cudaMalloc(&s.h_in, s.in_bytes));
    if (!s.h_out) B200_CUDA_CHECK(cudaMalloc(&s.h_out, s.out_bytes));
    ins[(size_t)g] = s.h_in;
    outs[(size_t)g] = s.h_out;
    B200_CUDA_CHECK(cudaMemcpyAsync(s.h_in, (const char*)h_in + (size_t)g * s.in_bytes, s.in_bytes, cudaMemcpyHostToDevice, s.stream));
  }
  int rc = b200fft_mgpu_exec(m, outs.data(), ins.data());
  if (rc == B200FFT_OK) {
    // slot h's [Z][yl][X] slab -> rows y in [h yl, (h+1) yl) of every z plane of the natural-order host volume
    const size_t yl = (size_t)(m->Y / G), row = yl * (size_t)m->X * 8, pitch = (size_t)m->Y * (size_t)m->X * 8;
    for (int g = 0; g < G && rc == B200FFT_OK; ++g) {
      Slot& s = m->slots[(size_t)g];
      cudaSetDevice(s.device);
      cudaError_t e = cudaMemcpy2DAsync((char*)h_out + (size_t)g * row, pitch, s.h_out, row, row, (size_t)m->Z,
                                        cudaMemcpyDeviceToHost, s.stream);
      if (e != cudaSuccess) rc = fail(B200FFT_ERR_CUDA, "device-to-host copy of slot %d: %s", g, cudaGetErrorString(e));
    }
  }
  // the caller may free its host buffers once we return: wait for every copy, also after an error
  for (Slot& s : m->slots) {
    cudaSetDevice(s.device);
    cudaError_t e = cudaStreamSynchronize(s.stream);
    if (e != cudaSuccess && rc == B200FFT_OK) rc = fail(B200FFT_ERR_CUDA, "device %d: %s", s.device, cudaGetErrorString(e));
  }
  return rc;
}

}  // extern "C"

#!/usr/bin/env python3
"""bench.py — the driver's measurement contract for the batched N-d radix-n FFT hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-shapes] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one forward C2C transform of the primary workload (BASELINE.json configs[1]:
1-D C2C fp32, batch 100000 x 1024) through the C ABI (b200fft_exec). At N > 1 every rank
owns its own batch of that shape (batch sharding, no data-path collective, "weak"
scaling); the time is the max over ranks and `value` the whole-job GFLOP/s
(5*N*log2(N) per transform, the usual effective-flop model of FFT benchmarks). W warm-up
steps run first, then exactly K timed steps between CUDA events; NVML samples the clocks during them.

`--dump-outputs DIR` writes, after the timed steps, what the last step computed on rank 0: a fixed,
seeded sample of the output rows as DIR/out.npy (see dump_outputs). The input is generated from a
fixed seed, so two builds run with the same arguments can be compared output for output.

Printed on rank 0: ONE JSON line with value / ms_per_step, `roofline` (HBM, measured
peak from MEASURED_PEAKS.json), `cpu_baseline` (the oracle = C++ port of the
reference's CPU path, timed on the box's host cores), `e2e` (same metric through
b200fft_exec_host with pinned HOST buffers, copies inside the timed region),
`gpu_launches`, `clocks`, and `shapes`: every BASELINE.json single-GPU config timed
the same way next to cuFFT (same buffers, same stream, CUDA events).

`--impl reference` times the reference's CPU implementation of the path (the oracle
port; the Mojo original cannot run in this image) with all host threads.
"""
import argparse
import ctypes
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "hackathon-fft_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
os.environ.setdefault("B200FFT_JIT_CACHE", "0")  # no on-disk kernel cache outside the repository from this script

METRIC = "batched C2C FFT ms, GFLOP/s & HBM GB/s vs peak at 1/2/4/8 B200 vs cuFFT"
PRIMARY = {"name": "1D C2C fp32 100000x1024", "shape": (100000, 1024)}
# BASELINE.json single-GPU configs (shape = (batch, dims...)); r2c = real input
SHAPES = [
    ("1d_500000x128", (500000, 128), False),
    ("1d_100000x1024", (100000, 1024), False),
    ("1d_500000x93", (500000, 93), False),
    ("2d_100x640x480", (100, 640, 480), False),
    ("2d_100x640x480_r2c_full", (100, 640, 480), True),
    ("2d_100x640x480_r2c_half", (100, 640, 480), "half"),
    ("3d_100x64x64x64", (100, 64, 64, 64), False),
    ("3d_10x128x128x128", (10, 128, 128, 128), False),
    ("3d_1x256x256x256", (1, 256, 256, 256), False),
    ("3d_1x512x512x512", (1, 512, 512, 512), False),
    # half-spectrum R2C of the 1-D and 3-D configs (what cufft_benchmark.cu's R2C rows time, :34-46)
    ("1d_500000x128_r2c_half", (500000, 128), "half"),
    ("1d_100000x1024_r2c_half", (100000, 1024), "half"),
    ("1d_500000x93_r2c_half", (500000, 93), "half"),
    ("3d_100x64x64x64_r2c_half", (100, 64, 64, 64), "half"),
    ("3d_10x128x128x128_r2c_half", (10, 128, 128, 128), "half"),
    ("3d_1x256x256x256_r2c_half", (1, 256, 256, 256), "half"),
    # lengths WITHOUT a hand-registered kernel variant: specialised at plan time through NVRTC (csrc/jit.cu), the
    # counterpart of the reference specialising every shape at compile time (profiles/r2_jit_tier.md)
    ("1d_50000x1000_plan_time_specialised", (50000, 1000), False),
    ("3d_4x200x200x200_plan_time_specialised", (4, 200, 200, 200), False),
    # long contiguous rows: one launch, one shared exchange buffer (rows_ip_kernel; profiles/r2_long_rows.md). (100, 16384)
    # is the reference's published shape (fft/bench.mojo:111)
    ("1d_100x16384", (100, 16384), False),
    ("1d_25000x4096", (25000, 4096), False),
]


def flops_c2c(shape):
    n = int(np.prod(shape[1:]))
    return 5.0 * n * math.log2(n) * shape[0]


def algorithmic_bytes(shape, real_in=False):
    pts = int(np.prod(shape))
    return pts * (4 if real_in else 8) + pts * 8


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self.marks = {}
        self._stop = threading.Event()
        self._thr = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None
            return self
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def _run(self):
        nv = self._nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.001)

    def mark(self, name):
        self.marks[name] = len(self.samples)

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()
        s = sorted(self.samples)
        t0, t1 = self.marks.get("timed_start", 0), self.marks.get("timed_end", len(self.samples))
        timed = t1 - t0
        ts = sorted(self.samples[t0:t1])
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_mhz_timed_region": (ts[len(ts) // 2] if ts else None),
                "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s), "samples_in_timed_region": timed,
                "sampled": "NVML, back to back, over the timed steps"}


def physical_gpu_index(local_index):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_index])
        except Exception:
            return local_index
    return local_index


def bind_to_gpu_numa(index):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, so the pinned host buffers of
    the e2e leg are first-touched on the GPU's own NUMA node (one process per GPU: otherwise every
    rank's staging memory lands on one socket and the ranks share its memory / PCIe bandwidth)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return 0


class CuFFT:
    """cuFFT through baseline/libcufft_shim.so (same call as the reference's cufft_benchmark.cu)."""

    def __init__(self, shape, r2c=False):
        path = os.path.join(ROOT, "baseline", "libcufft_shim.so")
        self.lib = ctypes.CDLL(path)
        self.lib.cufft_shim_create.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                               ctypes.POINTER(ctypes.c_longlong), ctypes.c_longlong, ctypes.c_int,
                                               ctypes.POINTER(ctypes.c_size_t)]
        self.lib.cufft_shim_exec.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int]
        self.lib.cufft_shim_destroy.argtypes = [ctypes.c_void_p]
        dims = (ctypes.c_longlong * (len(shape) - 1))(*shape[1:])
        self.h = ctypes.c_void_p()
        ws = ctypes.c_size_t()
        rc = self.lib.cufft_shim_create(ctypes.byref(self.h), len(shape) - 1, dims, shape[0], int(r2c), ctypes.byref(ws))
        if rc:
            raise RuntimeError("cufft plan failed: %d" % rc)
        self.r2c, self.work = r2c, ws.value

    def exec(self, x, out, stream):
        rc = self.lib.cufft_shim_exec(self.h, x.data_ptr(), out.data_ptr(), stream, int(self.r2c), 0)
        if rc:
            raise RuntimeError("cufft exec failed: %d" % rc)

    def destroy(self):
        self.lib.cufft_shim_destroy(self.h)


def time_gpu(fn, warmup, steps, torch):
    """CUDA-event timing on the current stream (the stream the kernels are launched on)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


DUMP_ROWS = 4096  # 4096 transforms of 1024 complex fp32 points: 32 MB of the 819 MB output


def dump_rows(batch):
    """The batch items --dump-outputs writes: picked by a fixed seed, in increasing order, the same on every run."""
    return np.sort(np.random.default_rng(0).choice(batch, size=min(DUMP_ROWS, batch), replace=False))


def dump_outputs(dirname, out, torch):
    """Write the dump_rows() items of `out` (batch, length, 2) to dirname/out.npy as float32 (DUMP_ROWS, length, 2)."""
    sample = out.index_select(0, torch.from_numpy(dump_rows(out.shape[0])).to(out.device)).cpu().numpy()
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "out.npy"), sample)


def _to_complex(x):
    return x[..., 0] + 1j * x[..., 1] if x.shape[-1] == 2 else x[..., 0]


def scipy_time(x, threads, repeats=2):
    """Sanity CPU datapoint next to the port: scipy.fft.fftn (pocketfft, complex64) over all non-batch axes with
    workers=n, the call benchmark-cpu-others/benchmark.py:35-49 times. Returns seconds per call (best of `repeats`)."""
    import scipy.fft
    xc = np.ascontiguousarray(_to_complex(x).astype(np.complex64))
    axes = tuple(range(1, xc.ndim))
    scipy.fft.fftn(xc, axes=axes, workers=threads)
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        scipy.fft.fftn(xc, axes=axes, workers=threads)
        best = min(best, time.perf_counter() - t0)
    return best


def cpu_reference_time(shape, real_in, workers, budget_s=12.0, repeats=3):
    """Time the oracle (C++ port of the reference CPU path, workers=n) on a bounded sample of the workload's batch.
    Like the reference's own CPU bench (fft/bench.mojo:83-90) the plan — stage lists, twiddles, calc_buf — is built
    OUTSIDE the timed region and only `fft(out, x, plan=plan)` into a preallocated output is timed.
    Returns (ms for the FULL batch extrapolated linearly, sample batch, threads, scipy ms for the full batch)."""
    import oracle
    threads = workers or oracle.hardware_threads()
    per = int(np.prod(shape[1:]))
    comps = 1 if real_in else 2
    rng = np.random.default_rng(0)

    def timed(batch, reps):
        x = rng.standard_normal((batch,) + tuple(shape[1:]) + (comps,)).astype(np.float32)
        plan = oracle.RefPlan(x.shape, np.float32)
        out = np.empty(plan.out_shape, np.float32)
        plan.exec(out, x, workers=threads)  # warm-up: first touch of out / calc_buf, pool start
        best = float("inf")
        for _ in range(reps):
            t0 = time.perf_counter()
            plan.exec(out, x, workers=threads)
            best = min(best, time.perf_counter() - t0)
        plan.destroy()
        return best, x

    probe_b = max(1, min(shape[0], max(threads * 8, 400000 // per)))
    t_probe, x = timed(probe_b, 1)
    sample_b = int(max(1, min(shape[0], probe_b * (budget_s / (repeats + 1)) / max(t_probe, 1e-5))))
    best, x = timed(sample_b, repeats) if sample_b != probe_b else (t_probe, x)
    sp_ms = None
    try:
        sp_ms = scipy_time(x, threads) * 1e3 * shape[0] / sample_b
    except Exception:
        pass
    return best * 1e3 * shape[0] / sample_b, sample_b, threads, sp_ms


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port, all host threads) on the same
    config / metric / unit, timed the way the reference's bench_cpu_radix_n_rfft does (fft/bench.mojo:60-96): plan
    built once outside the loop, each step = one fft(out, x, plan=plan) on a bounded sample. Rank 0 only under torchrun."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import oracle
    oracle.build()
    shape = PRIMARY["shape"]
    threads = oracle.hardware_threads()
    per = int(np.prod(shape[1:]))
    rng = np.random.default_rng(0)

    def make(batch):
        x = rng.standard_normal((batch,) + tuple(shape[1:]) + (2,)).astype(np.float32)
        plan = oracle.RefPlan(x.shape, np.float32)
        out = np.empty(plan.out_shape, np.float32)
        plan.exec(out, x, workers=threads)
        return x, out, plan

    x, out, plan = make(max(threads * 8, 512))
    t0 = time.perf_counter()
    plan.exec(out, x, workers=threads)
    t_probe = time.perf_counter() - t0
    total_steps = max(1, args.steps + args.warmup)
    # seconds of CPU work per step: bounded so the whole run ends within ~2 minutes (B200FFT_BENCH_REF_SECONDS
    # overrides it; the CPU test-suite uses a fraction of a second)
    target_s = min(20.0, 120.0 / total_steps)
    if os.environ.get("B200FFT_BENCH_REF_SECONDS"):
        target_s = float(os.environ["B200FFT_BENCH_REF_SECONDS"])
    sample_b = int(max(1, min(shape[0], x.shape[0] * target_s / max(t_probe, 1e-5))))
    if sample_b != x.shape[0]:
        plan.destroy()
        x, out, plan = make(sample_b)
    for _ in range(args.warmup):
        plan.exec(out, x, workers=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        plan.exec(out, x, workers=threads)
    dt = (time.perf_counter() - t0) / args.steps
    plan.destroy()
    gflops = flops_c2c((sample_b,) + tuple(shape[1:])) / dt / 1e9
    ms_full = dt * 1e3 * shape[0] / sample_b
    scipy_gflops = None
    try:
        scipy_gflops = flops_c2c((sample_b,) + tuple(shape[1:])) / scipy_time(x, threads) / 1e9
    except Exception:
        pass
    line = {
        "impl": "reference", "metric": METRIC, "value": gflops, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_full, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": PRIMARY["name"], "note": "CPU reference path (workers=n): C++ port of the Mojo "
                   "radix-n implementation (oracle/ref_fft.cpp), plan built once outside the timed loop like "
                   "fft/bench.mojo:83-90; ms_per_step extrapolated to the full batch"},
        "cpu_baseline": {"value": gflops, "unit": "GFLOP/s", "cores": threads, "kind": "port",
                         "sample": "%d of %d transforms of length %d per step" % (sample_b, shape[0], per),
                         "scipy_fft_workers_n_gflops": scipy_gflops},
        "e2e": {"value": gflops, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


_TRAFFIC = None


def _plan_traffic():
    global _TRAFFIC
    if _TRAFFIC is None:
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                _TRAFFIC = json.load(f)
        except Exception:
            _TRAFFIC = {}
    return _TRAFFIC


def bench_shape(name, shape, real_in, torch, b200fft, steps, warmup, peak):
    """ours vs cuFFT on one shape, same buffers, same stream, CUDA events."""
    comps = 1 if real_in else 2
    half = real_in == "half"
    row = {"name": name, "shape": list(shape), "real_in": bool(real_in), "half_spectrum": half}
    try:
        g = torch.Generator(device="cuda").manual_seed(1234)
        x = torch.randn(tuple(shape) + (comps,), generator=g, device="cuda", dtype=torch.float32)
        oshape = tuple(shape[:-1]) + (shape[-1] // 2 + 1, 2) if half else tuple(shape) + (2,)
        out = torch.empty(oshape, device="cuda", dtype=torch.float32)
        plan = b200fft.plan_fft("float32", "float32", x.shape, out.shape,
                                real_mode=b200fft.REAL_HALF if half else b200fft.REAL_FULL)
        stream = torch.cuda.current_stream().cuda_stream
        ms = time_gpu(lambda: plan.exec(out, x, stream), warmup, steps, torch)
        ab = algorithmic_bytes(shape, real_in) if not half else int(np.prod(shape)) * 4 + int(np.prod(oshape)) * 4
        row.update({"ms": ms, "gflops": flops_c2c(shape) * (0.5 if real_in else 1.0) / ms / 1e6,
                    "gbs": ab / ms / 1e6, "hbm_frac": ab / ms / 1e6 / peak, "launches": plan.launches,
                    "kernels": plan.describe().strip().split("\n")})
        # DRAM bytes of one exec of this plan (all its launches) from a committed ncu capture, over the algorithmic bytes:
        # > 1 = passes re-reading what did not stay in L2 (profiles/traffic.json, tools/ncu_summary.py "plan:" entries)
        tr = _plan_traffic().get("plan:" + name)
        if tr and tr.get("dram_bytes_per_exec"):
            row["traffic_over_algorithmic"] = tr["dram_bytes_per_exec"] / ab
            row["traffic_source"] = tr.get("source")
        # parity on one batch item against numpy f64
        ref_in = x[0].double().cpu().numpy()
        want = np.fft.rfftn(ref_in[..., 0]) if half else np.fft.fftn(ref_in[..., 0] + (1j * ref_in[..., 1] if comps == 2 else 0))
        got = out[0].double().cpu().numpy()
        got = got[..., 0] + 1j * got[..., 1]
        row["rel_l2_vs_numpy_f64"] = float(np.linalg.norm(got - want) / np.linalg.norm(want))
        plan.destroy()
        try:
            if real_in:
                # cuFFT R2C writes the half spectrum (cufft_benchmark.cu:34-46)
                half = tuple(shape[:-1]) + (shape[-1] // 2 + 1, 2)
                cout = torch.empty(half, device="cuda", dtype=torch.float32)
            else:
                cout = torch.empty_like(out)
            cf = CuFFT(shape, r2c=bool(real_in))
            cms = time_gpu(lambda: cf.exec(x, cout, stream), warmup, steps, torch)
            row["cufft_note"] = "cuFFT R2C writes the half spectrum" if real_in else ""
            cf.destroy()
            row.update({"cufft_ms": cms, "ours_over_cufft": ms / cms})
            del cout
        except Exception as e:  # cuFFT shim missing or plan failure: report, do not hide
            row["cufft_error"] = str(e)
        del x, out
        torch.cuda.empty_cache()
    except Exception as e:
        row["error"] = "%s: %s" % (type(e).__name__, e)
    return row


def bench_slab(n, world, rank, torch, dist, steps=10, warmup=3):
    """Single n^3 C2C transform slab-decomposed over the ranks (b200fft.slab.SlabFFT3D): local 2-D FFTs,
    exchange (fused into the Y pass's stores over NVLink = "p2p", or pack + NCCL all-to-all = "nccl"), Z pass.
    Timed with CUDA events between barriers, max over ranks, exchange included; output stays Y-slab distributed."""
    from b200fft.slab import SlabFFT3D
    res = {"n": n, "ranks": world, "output": "Y-slab distributed (transposed out)", "timed": "2-D pass + exchange + Z pass"}
    if n % world:
        res["error"] = "%d not divisible by %d ranks" % (n, world)
        return res
    zl = n // world
    g = torch.Generator(device="cuda").manual_seed(77 + rank)
    x = torch.randn((zl, n, n, 2), generator=g, device="cuda")
    for mode in ("fused", "p2p", "nccl"):
        try:
            sl = SlabFFT3D((n, n, n), exchange=mode)
            for _ in range(warmup):
                sl.forward(x)
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = sl.forward(x)
            e1.record()
            torch.cuda.synchronize()
            dist.barrier()
            t = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            # parity of the DISTRIBUTED result (b200fft.verify): (1) sampled bins — every rank's float64 share of the
            # direct DFT sum, all-reduced, against the element the owning rank holds: sees accuracy and any systematic
            # misplacement; (2) an impulse per source rank, exact spectrum compared at EVERY element of every slab: sees a
            # single row in the wrong peer slot. Parseval (blind to permutations) is kept as a third figure.
            from b200fft import verify
            out = sl.forward(x).clone()
            torch.cuda.synchronize()
            bins_err = verify.sampled_bins_check(x, out, (n, n, n), rank, world)
            dout = sl.forward(verify.delta_input((n, n, n), rank, world, x.device)).clone()
            torch.cuda.synchronize()
            delta_err = verify.delta_volume_check(dout, (n, n, n), rank, world)
            del dout
            e = torch.stack([out.double().pow(2).sum(), x.double().pow(2).sum()])
            dist.all_reduce(e)
            res[mode] = {"ms": ms, "gflops": 5.0 * n ** 3 * math.log2(n ** 3) / ms / 1e6,
                         "sampled_bins_max_rel_err": bins_err, "sampled_bins": 32,
                         "delta_volume_max_rel_err": delta_err,
                         "parity_ok": bool(bins_err < 2e-6 and delta_err < 2e-6),
                         "parseval_rel_err": abs(float(e[0] / (e[1] * n ** 3)) - 1.0)}
            if mode == "fused":
                res[mode]["peer_wait_timeouts"] = sl.timeouts()
            sl.close()
            del out
        except Exception as ex:  # report, keep the bench line
            res[mode] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    return res


def bench_mgpu(world, shape, torch, b200fft):
    """N > 1, rank 0 only (the other ranks idle at a barrier): the SAME job through the C ABI's single-process multi-device
    entry points (b200fft_mgpu_*, include/b200fft.h) — what a Mojo / C host without torch.distributed would call.
    (a) end to end: world x per-GPU batch from ONE pinned host array, one host thread + 3-stream pipeline per device;
    (b) the 512^3 slab transform with device-resident slabs (peer-to-peer scattering stores + event barrier)."""
    res = {"api": "b200fft_mgpu_plan_create / exec / exec_host, one process driving %d devices" % world}
    try:
        devs = list(range(world))
        B = shape[0] * world
        lay = (B,) + tuple(shape[1:]) + (2,)
        plan = b200fft.MgpuPlan("float32", "float32", lay, lay, devices=devs, mode=b200fft.MGPU_BATCH_SHARD)
        h_in = torch.empty(lay, dtype=torch.float32).pin_memory()
        h_in[:shape[0]].normal_()
        for g in range(1, world):
            h_in[g * shape[0]:(g + 1) * shape[0]].copy_(h_in[:shape[0]])
        h_out = torch.empty(lay, dtype=torch.float32).pin_memory()
        plan.exec_host(h_out.numpy(), h_in.numpy())
        best = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            plan.exec_host(h_out.numpy(), h_in.numpy())
            best = min(best, (time.perf_counter() - t0) * 1e3)
        k = 4
        want = torch.fft.fft(torch.view_as_complex(h_in[-k:].double().contiguous()), dim=1)
        got = torch.view_as_complex(h_out[-k:].double().contiguous())
        res["e2e_batch_shard"] = {"ms_per_step": best, "value": world * flops_c2c(shape) / best / 1e6, "unit": "GFLOP/s",
                                  "h2d_bytes_per_step": int(h_in.numel() * 4), "d2h_bytes_per_step": int(h_out.numel() * 4),
                                  "rel_l2_vs_torch_f64_last_rows": float((got - want).norm() / want.norm())}
        plan.destroy()
        del h_in, h_out
    except Exception as ex:
        res["e2e_batch_shard"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    try:
        n = 512
        zl = yl = n // world
        lay = (1, n, n, n, 2)
        plan = b200fft.MgpuPlan("float32", "float32", lay, lay, devices=devs, mode=b200fft.MGPU_SLAB)
        ins = [torch.randn((zl, n, n, 2), device="cuda:%d" % d) for d in devs]
        outs = [torch.empty((n, yl, n, 2), device="cuda:%d" % d) for d in devs]
        streams = [torch.cuda.ExternalStream(plan.stream(i), device="cuda:%d" % d) for i, d in enumerate(devs)]
        for _ in range(3):
            plan.exec(outs, ins)
        plan.synchronize()
        ev = []
        for i, d in enumerate(devs):
            with torch.cuda.device(d):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(streams[i])
                ev.append((e0, e1))
        steps = 10
        for _ in range(steps):
            plan.exec(outs, ins)
        for i, d in enumerate(devs):
            with torch.cuda.device(d):
                ev[i][1].record(streams[i])
        plan.synchronize()
        ms = max(a.elapsed_time(b) for a, b in ev) / steps
        # parity: Parseval over all devices + one sampled output bin by direct summation in float64
        e_in = sum(float(t.double().pow(2).sum()) for t in ins)
        e_out = sum(float(t.double().pow(2).sum()) for t in outs)
        res["slab_512"] = {"ms": ms, "gflops": 5.0 * n ** 3 * math.log2(n ** 3) / ms / 1e6,
                           "parseval_rel_err": abs(e_out / (e_in * n ** 3) - 1.0)}
        plan.destroy()
    except Exception as ex:
        res["slab_512"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-shapes", action="store_true", help="skip the per-shape table vs cuFFT")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of the last step's output to DIR/out.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import b200fft

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa(physical_gpu_index(local))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    peak, peak_src = measured_peak()
    shape = PRIMARY["shape"]
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    x = torch.randn(shape + (2,), generator=g, device="cuda", dtype=torch.float32)
    out = torch.empty_like(x)
    plan = b200fft.plan_fft("float32", "float32", x.shape, out.shape)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        plan.exec(out, x, stream)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    # The timed region: exactly K steps after the W warm-up steps, bracketed by CUDA events on the launching stream with
    # a synchronise on both sides -> ms_per_step / value. An NVML query takes ~1 ms, so a short K yields few clock samples.
    sampler = ClockSampler(physical_gpu_index(local)).start()
    sampler.mark("timed_start")
    launches0 = b200fft.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    sampler.mark("timed_end")
    launches = b200fft.launch_count() - launches0
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, torch)
    if dist:
        dist.barrier()
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    gflops_total = world * flops_c2c(shape) / ms / 1e6

    # ---- e2e: the same transform through b200fft_exec_host with pinned HOST buffers
    h_in = torch.empty(shape + (2,), dtype=torch.float32).pin_memory()
    h_in.copy_(x.cpu())
    h_out = torch.empty(shape + (2,), dtype=torch.float32).pin_memory()
    e2e_steps = max(2, min(args.steps, 5))
    plan.exec_host(h_out.numpy(), h_in.numpy())  # warm-up (allocates the staging buffers)
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        plan.exec_host(h_out.numpy(), h_in.numpy())
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    if dist:
        t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_ok = bool(torch.allclose(h_out[:4], out[:4].cpu(), rtol=0, atol=0))
    e2e = {"value": world * flops_c2c(shape) / e2e_ms / 1e6, "unit": "GFLOP/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": plan.in_bytes, "d2h_bytes_per_step": plan.out_bytes,
           "matches_device_path": e2e_ok, "api": "b200fft_exec_host (pinned host buffers, chunked 3-stream pipeline)",
           "host_cpus_bound": numa_cpus}

    # ---- N > 1: the single 512^3 transform, slab-decomposed over the ranks (exchange inside the timed region)
    slab = None
    if dist:
        del h_in, h_out
        slab = bench_slab(512, world, rank, torch, dist)

    if rank != 0:
        if dist:
            dist.barrier()
            dist.destroy_process_group()
        return

    ab = algorithmic_bytes(shape)
    kernel_ms = ms / max(1, plan.launches)
    traffic = None  # ncu dram__bytes_read.sum + dram__bytes_write.sum of this kernel, per launch
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(PRIMARY["name"], {}).get("dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": ab / plan.launches / kernel_ms / 1e6, "peak": peak, "unit": "GB/s",
                "frac": ab / plan.launches / kernel_ms / 1e6 / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel": plan.describe().strip().split("\n")[0],
                "algorithmic_bytes_per_launch": ab // plan.launches}

    cpu = None
    if not args.no_cpu:
        import oracle
        oracle.build()
        cpu_ms, sample_b, threads, sp_ms = cpu_reference_time(shape, False, 0)
        cpu = {"value": flops_c2c(shape) / cpu_ms / 1e6, "unit": "GFLOP/s", "cores": threads, "kind": "port",
               "ms_full_batch_extrapolated": cpu_ms,
               "sample": "%d of %d transforms of length %d (oracle/ref_fft.cpp, workers=%d; plan built outside the "
                         "timed region, exec into a preallocated output, best of 3)" % (sample_b, shape[0], shape[1], threads),
               "scipy_fft_workers_n": {"value": (flops_c2c(shape) / sp_ms / 1e6) if sp_ms else None, "unit": "GFLOP/s",
                                       "ms_full_batch_extrapolated": sp_ms,
                                       "note": "scipy.fft.fftn complex64 workers=n on the same sample (sanity datapoint, "
                                               "benchmark-cpu-others/benchmark.py:35-49)"}}

    line = {
        "metric": METRIC, "value": gflops_total, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": PRIMARY["name"], "per_gpu_batch": shape[0], "length": shape[1],
                   "sharding": "batch-sharded, no collective" if world > 1 else "single GPU",
                   "l2": "inputs+outputs %.0f MB per step > 126 MB L2 (no flush needed)" % (2 * ab / 2 / 1e6),
                   "flop_model": "5*N*log2(N) per transform",
                   "timing": "exactly %d steps after %d warm-up steps (CUDA events)" % (args.steps, args.warmup)},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
    }
    if slab is not None:
        line["slab_3d_1x512x512x512"] = slab
    del x, out
    plan.destroy()
    torch.cuda.empty_cache()
    if dist and world > 1:
        line["mgpu_single_process"] = bench_mgpu(world, shape, torch, b200fft)

    if not args.no_shapes and world == 1:
        line["shapes"] = [bench_shape(n, s, r, torch, b200fft, max(5, min(args.steps, 20)), 3, peak)
                          for n, s, r in SHAPES]
    print(json.dumps(line))
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Timing of contiguous axes longer than 2^24 points (the three-pass form of csrc/jit.cu: make_jit_split3_pass) next to
torch.fft (cuFFT) on the same device tensors.

For every shape: warm-up, then CUDA-event timing over windows of at least 0.2 s. Every array is 256 MB or more, so
nothing stays in the 126 MB L2 between passes. Bandwidth is quoted against the one-read-one-write bytes of the
transform (16 n per complex fp32 row, 32 n fp64): the three passes themselves move three times that (each reads and
writes every point once). rel-err is the rel-L2 distance to torch.fft in float64 on the same input, for both ours and
cuFFT. The GPU name, power limit and max SM clock are read in the same run and written beside the table.

    python tools/very_long_shapes.py [--out profiles/r3_very_long_axes.md] [--window 0.2]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hackathon-fft_b200", "python"))
import b200fft  # noqa: E402

# (label, batch, n, dtype): complex input and output of that dtype, forward
SHAPES = [("1 x 2^25", 1, 1 << 25, "float32"), ("1 x 2^27", 1, 1 << 27, "float32"), ("1 x 2^28", 1, 1 << 28, "float32"),
          ("4 x 2^26", 4, 1 << 26, "float32"), ("1 x 10^8", 1, 10 ** 8, "float32"), ("1 x 2^26 fp64", 1, 1 << 26, "float64")]


def time_ms(fn, window):
    """Mean ms per call over a window of at least `window` seconds, after a warm-up."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 1
    while True:
        start.record()
        for _ in range(reps):
            fn()
        stop.record()
        stop.synchronize()
        ms = start.elapsed_time(stop)
        if ms >= window * 1e3:
            return ms / reps
        reps = max(reps * 2, int(reps * window * 1e3 / max(ms, 1e-3) * 1.2) + 1)


def gpu_facts():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q or "unknown"


def rel_err(got, want):
    return float((got - want).norm() / want.norm())


def one(label, batch, n, dtype, window):
    tdt = torch.float32 if dtype == "float32" else torch.float64
    g = torch.Generator(device="cuda").manual_seed(n % 100003)
    x = torch.randn((batch, n, 2), generator=g, device="cuda", dtype=tdt)
    out = torch.empty_like(x)
    plan = b200fft.plan_fft(dtype, dtype, x.shape, out.shape)
    stream = torch.cuda.current_stream().cuda_stream
    xc = torch.view_as_complex(x)
    ours = lambda: plan.exec(out, x, stream)  # noqa: E731
    ref = lambda: torch.fft.fft(xc, dim=-1)  # noqa: E731
    ours()
    want = torch.fft.fft(xc.to(torch.complex128), dim=-1)
    err = rel_err(torch.view_as_complex(out).to(torch.complex128), want)
    err_ref = rel_err(ref().to(torch.complex128), want)
    del want
    torch.cuda.empty_cache()
    t_ours, t_ref = time_ms(ours, window), time_ms(ref, window)
    desc, launches = plan.describe().strip(), plan.launches
    plan.destroy()
    io_bytes = 2 * batch * n * x.element_size() * 2  # one read and one write of every complex point
    return dict(label=label, n=n, ours=t_ours, cufft=t_ref, err=err, err_ref=err_ref, launches=launches, desc=desc,
                io_bytes=io_bytes)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_very_long_axes.md"))
    ap.add_argument("--window", type=float, default=0.2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("very_long_shapes.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    name, facts = gpu_facts()
    print("%s, power limit / max SM clock: %s" % (name, facts), flush=True)
    rows = []
    for s in SHAPES:
        r = one(*s, window=args.window)
        rows.append(r)
        print("%-14s ours %.3f ms (%.0f GB/s)  cuFFT %.3f ms (%.0f GB/s)  ours/cuFFT %.2f  rel-err %.1e / %.1e" %
              (r["label"], r["ours"], r["io_bytes"] / r["ours"] / 1e6, r["cufft"], r["io_bytes"] / r["cufft"] / 1e6,
               r["ours"] / r["cufft"], r["err"], r["err_ref"]), flush=True)
    lines = ["# Contiguous axes longer than 2^24 points (round 3)", "",
             "Measured on %s, power limit / max SM clock: %s." % (name, facts),
             "`tools/very_long_shapes.py`, CUDA events, windows of at least %.1f s after warm-up; every array exceeds the "
             "126 MB L2. Complex input and output, forward. GB/s = one-read-one-write bytes (16 n per fp32 row, 32 n fp64) "
             "over the time; the three passes move 3 x those bytes (48 n fp32, 96 n fp64), so three-pass traffic in GB/s is "
             "3 x the figure shown. rel-err = rel-L2 against torch.fft in float64 on the same input. Kernel-level numbers "
             "(per-pass time, achieved DRAM bandwidth from counters): not measured." % args.window,
             "", "| shape | ours (ms) | torch.fft / cuFFT (ms) | ours / cuFFT | ours GB/s (1R1W) | cuFFT GB/s (1R1W) | launches "
             "| rel-err ours | rel-err cuFFT |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append("| %s | %.3f | %.3f | %.2f | %.0f | %.0f | %d | %.1e | %.1e |" %
                     (r["label"], r["ours"], r["cufft"], r["ours"] / r["cufft"], r["io_bytes"] / r["ours"] / 1e6,
                      r["io_bytes"] / r["cufft"] / 1e6, r["launches"], r["err"], r["err_ref"]))
    lines += ["", "Plans:", ""]
    for r in rows:
        lines.append("- %s: `%s`" % (r["label"], r["desc"].replace("\n", " | ")))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()

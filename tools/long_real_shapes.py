"""Timing of long real-input and half-spectrum axes (the two-pass forms of csrc/jit.cu: make_jit_split_pass) next to
torch.fft (cuFFT) on the same device tensors and next to our own complex split of the same bytes.

For every shape: warm-up, then CUDA-event timing over windows of at least 0.2 s. Input, temporary and output
together exceed the 126 MB L2 (every real or half-spectrum array is 64-125 MB), so the passes stream from HBM. The third column is the floor this
design can reach: the complex two-pass transform of H = n/2 points on the same bytes (even n), or of n points (odd n
and the full spectrum of real input, which run the full n-point split). The GPU name and power limit are read in
the same run and written beside the table.

    python tools/long_real_shapes.py [--out profiles/r3_long_real.md] [--window 0.2]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hackathon-fft_b200", "python"))
import b200fft  # noqa: E402

# (label, mode, batch, n, input dtype); mode: r2c / c2r = REAL_HALF, full = REAL_FULL forward
SHAPES = [("256 x 2^16", "r2c", 256, 1 << 16, "float32"), ("256 x 2^16", "c2r", 256, 1 << 16, "float32"),
          ("64 x 2^18", "r2c", 64, 1 << 18, "float32"), ("64 x 2^18", "c2r", 64, 1 << 18, "float32"),
          ("16 x 2^20", "r2c", 16, 1 << 20, "float32"), ("16 x 2^20", "c2r", 16, 1 << 20, "float32"),
          ("320 x 100000", "r2c", 320, 100000, "float32"), ("320 x 100000", "c2r", 320, 100000, "float32"),
          ("400 x 5^7 (odd)", "r2c", 400, 5 ** 7, "float32"), ("400 x 5^7 (odd)", "c2r", 400, 5 ** 7, "float32"),
          ("64 x 2^18 uint8", "full", 64, 1 << 18, "uint8")]


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
    return name, q


def one(label, mode, batch, n, dtype, window):
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(n)
    bins = n // 2 + 1
    if mode == "c2r":
        x = torch.randn((batch, bins, 2), generator=g, device=dev)
        x[:, 0, 1] = 0
        if n % 2 == 0:
            x[:, -1, 1] = 0
        out = torch.empty((batch, n, 1), device=dev)
        plan = b200fft.plan_fft("float32", "float32", x.shape, out.shape, real_mode=b200fft.REAL_HALF, inverse=True)
        xc = torch.view_as_complex(x)
        ref = lambda: torch.fft.irfft(xc, n=n, dim=-1)  # noqa: E731
    else:
        if dtype == "uint8":
            x = torch.randint(0, 256, (batch, n, 1), generator=g, device=dev, dtype=torch.uint8)
        else:
            x = torch.randn((batch, n, 1), generator=g, device=dev)
        if mode == "r2c":
            out = torch.empty((batch, bins, 2), device=dev)
            plan = b200fft.plan_fft(dtype, "float32", x.shape, out.shape, real_mode=b200fft.REAL_HALF)
            ref = lambda: torch.fft.rfft(x[..., 0], dim=-1)  # noqa: E731
        else:
            out = torch.empty((batch, n, 2), device=dev)
            plan = b200fft.plan_fft(dtype, "float32", x.shape, out.shape)
            xf = x[..., 0]
            ref = lambda: torch.fft.fft(xf.float(), dim=-1)  # noqa: E731  (cuFFT has no uint8 input: the cast is part of it)
    stream = torch.cuda.current_stream().cuda_stream
    ours = lambda: plan.exec(out, x, stream)  # noqa: E731
    # correctness on the timed tensors, against cuFFT
    ours()
    want = ref()
    got = torch.view_as_complex(out) if mode != "c2r" else out[..., 0]
    want = torch.view_as_real(want) if want.is_complex() else want
    got = torch.view_as_real(got) if got.is_complex() else got
    err = float((got.double() - want.double()).norm() / want.double().norm())
    # the floor: our complex split on the same bytes (H points) or on n points
    m = n // 2 if (mode != "full" and n % 2 == 0) else n
    cx = torch.randn((batch, m, 2), generator=g, device=dev)
    cout = torch.empty_like(cx)
    cplan = b200fft.plan_fft("float32", "float32", cx.shape, cx.shape, inverse=(mode == "c2r"))
    floor = lambda: cplan.exec(cout, cx, stream)  # noqa: E731
    t_ours, t_ref, t_floor = time_ms(ours, window), time_ms(ref, window), time_ms(floor, window)
    desc, cdesc, launches = plan.describe().strip(), cplan.describe().strip(), plan.launches
    plan.destroy()
    cplan.destroy()
    return dict(label=label, mode=mode, n=n, ours=t_ours, cufft=t_ref, floor=t_floor, floor_n=m, err=err, launches=launches,
                desc=desc, cdesc=cdesc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_long_real.md"))
    ap.add_argument("--window", type=float, default=0.2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("long_real_shapes.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    name, power = gpu_facts()
    rows = []
    for s in SHAPES:
        r = one(*s, window=args.window)
        rows.append(r)
        print("%-18s %-4s ours %.4f ms  cuFFT %.4f ms  floor %.4f ms  ours/floor %.2f  rel-err %.1e" %
              (r["label"], r["mode"], r["ours"], r["cufft"], r["floor"], r["ours"] / r["floor"], r["err"]), flush=True)
    lines = ["# Long real-input and half-spectrum axes (round 3)", "",
             "Measured on %s, power limit / max SM clock: %s." % (name, power),
             "`tools/long_real_shapes.py`, CUDA events, windows of at least %.1f s after warm-up; every working set exceeds the "
             "126 MB L2. fp32 output. \"floor\" = our complex two-pass split of the same bytes (H = n/2 points for even n; n points "
             "for odd n and real input with the full spectrum). rel-err = rel-L2 against torch.fft on the same tensors." % args.window,
             "", "| shape | mode | ours (ms) | torch.fft / cuFFT (ms) | complex split floor (ms) | ours / cuFFT | ours / floor | launches | rel-err |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append("| %s | %s | %.4f | %.4f | %.4f (n=%d) | %.2f | %.2f | %d | %.1e |" %
                     (r["label"], r["mode"], r["ours"], r["cufft"], r["floor"], r["floor_n"], r["ours"] / r["cufft"],
                      r["ours"] / r["floor"], r["launches"], r["err"]))
    lines += ["", "Plans:", ""]
    for r in rows:
        lines.append("- %s %s: `%s`" % (r["label"], r["mode"], r["desc"].replace("\n", " | ")))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()

"""B200 time of strided plans (b200fft_plan_create_strided) against what a caller with a strided array does without them.

For each shape three things are timed with CUDA events after a warm-up, every working set larger than the 126 MB L2 (the
16 x 128^3 C2R, at 136 MB, is the smallest):
  strided     the strided plan on the view, no copy;
  copy+dense  view.contiguous() followed by the dense plan (the extra HBM round trip a caller pays today);
  dense       the dense plan alone on dense data (the floor a strided layout can reach).
Writes a markdown table (default profiles/r3_strided.md) that names the card and its power limit read in the same run.

    python tools/strided_shapes.py [--out FILE] [--iters N]
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hackathon-fft_b200", "python"))
import b200fft  # noqa: E402


def dense(shape):
    out, s = [], 1
    for v in reversed(shape):
        out.append(s)
        s *= v
    return list(reversed(out))


def time_ms(fn, iters, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def view(buf, shape, strides, comps):
    return buf.as_strided(tuple(shape) + (comps,), tuple(s * comps for s in strides) + (1,))


def c2c_case(shape, in_strides, span):
    """complex input through in_strides, dense complex output"""
    buf = torch.randn(span * 2, device="cuda")
    x = view(buf, shape, in_strides, 2)
    y = torch.empty(tuple(shape) + (2,), device="cuda")
    lay = tuple(shape) + (2,)
    sp = b200fft.plan_fft("float32", "float32", lay, lay, in_strides=in_strides)
    dp = b200fft.plan_fft("float32", "float32", lay, lay)
    xd = x.contiguous()
    return sp, dp, x, y, xd, lay


def run(iters):
    rows = []

    def record(name, sp, fn_s, fn_c, fn_d):
        ts, tc, td = time_ms(fn_s, iters), time_ms(fn_c, iters), time_ms(fn_d, iters)
        kern = "; ".join(ln.split(":")[1].split()[0] for ln in sp.describe().strip().split("\n"))
        rows.append((name, ts, tc, td, kern))
        print("%-46s strided %.4f  copy+dense %.4f  dense %.4f ms  [%s]" % (name, ts, tc, td, kern), flush=True)

    # 1. in-place padded R2C, 100000 x 1024 (real pitch 1026 = 2 x 513)
    B, n = 100000, 1024
    hb = n // 2 + 1
    buf = torch.randn(B * hb * 2, device="cuda")
    real = view(buf, (B, n), [2 * hb, 1], 1)
    cplx = view(buf, (B, hb), [hb, 1], 2)
    sp = b200fft.plan_fft("float32", "float32", (B, n, 1), (B, hb, 2), real_mode=b200fft.REAL_HALF, in_strides=[2 * hb, 1],
                          out_strides=[hb, 1])
    dp = b200fft.plan_fft("float32", "float32", (B, n, 1), (B, hb, 2), real_mode=b200fft.REAL_HALF)
    xd = real.contiguous()
    yd = torch.empty((B, hb, 2), device="cuda")
    record("R2C 100000 x 1024, in place, padded rows", sp, lambda: b200fft.fft(cplx, real, plan=sp),
           lambda: b200fft.fft(yd, real.contiguous(), plan=dp), lambda: b200fft.fft(yd, xd, plan=dp))
    del buf, real, cplx, xd, yd, sp, dp

    # 2. C2C 100000 x 1024 inside rows of pitch 1040, pitched output too
    B, n, pitch = 100000, 1024, 1040
    bi = torch.randn(B * pitch * 2, device="cuda")
    bo = torch.empty(B * pitch * 2, device="cuda")
    x, y = view(bi, (B, n), [pitch, 1], 2), view(bo, (B, n), [pitch, 1], 2)
    sp = b200fft.plan_fft("float32", "float32", (B, n, 2), (B, n, 2), in_strides=[pitch, 1], out_strides=[pitch, 1])
    dp = b200fft.plan_fft("float32", "float32", (B, n, 2), (B, n, 2))
    xd, yd = x.contiguous(), torch.empty((B, n, 2), device="cuda")
    record("C2C 100000 x 1024, rows of pitch 1040", sp, lambda: b200fft.fft(y, x, plan=sp),
           lambda: b200fft.fft(yd, x.contiguous(), plan=dp), lambda: b200fft.fft(yd, xd, plan=dp))
    del bi, bo, x, y, xd, yd, sp, dp

    # 3. 100 x 640 x 480 C2C of a transposed view (storage 100 x 480 x 640)
    shape = (100, 640, 480)
    sp, dp, x, y, xd, lay = c2c_case(shape, [480 * 640, 1, 640], 100 * 480 * 640)
    record("C2C 100 x 640 x 480, transposed view", sp, lambda: b200fft.fft(y, x, plan=sp),
           lambda: b200fft.fft(y, x.contiguous(), plan=dp), lambda: b200fft.fft(y, xd, plan=dp))
    del sp, dp, x, y, xd

    # 4. element stride 3 on 1024-point rows (one channel of three interleaved)
    B, n = 40000, 1024
    sp, dp, x, y, xd, lay = c2c_case((B, n), [3 * n, 3], B * n * 3)
    record("C2C 40000 x 1024, element stride 3", sp, lambda: b200fft.fft(y, x, plan=sp),
           lambda: b200fft.fft(y, x.contiguous(), plan=dp), lambda: b200fft.fft(y, xd, plan=dp))
    del sp, dp, x, y, xd

    # 5. in-place padded C2R 16 x 128^3
    shape = (16, 128, 128, 128)
    cshape = (16, 128, 128, 65)
    cst = dense(cshape)
    rst = [2 * s for s in cst[:-1]] + [1]
    buf = torch.randn(16 * 128 * 128 * 65 * 2, device="cuda")
    cplx, real = view(buf, cshape, cst, 2), view(buf, shape, rst, 1)
    sp = b200fft.plan_fft("float32", "float32", cshape + (2,), shape + (1,), real_mode=b200fft.REAL_HALF, inverse=True,
                          in_strides=cst, out_strides=rst)
    dp = b200fft.plan_fft("float32", "float32", cshape + (2,), shape + (1,), real_mode=b200fft.REAL_HALF, inverse=True)
    xd, yd = cplx.contiguous(), torch.empty(shape + (1,), device="cuda")
    # the in-place C2R overwrites its own input: the timed calls transform whatever the previous call left (same cost)
    record("C2R 16 x 128^3, in place, padded rows", sp, lambda: b200fft.fft(real, cplx, plan=sp),
           lambda: b200fft.fft(yd, cplx.contiguous(), plan=dp), lambda: b200fft.fft(yd, xd, plan=dp))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_strided.md"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().split("\n")[0]
    rows = run(args.iters)
    with open(args.out, "w") as f:
        f.write("# Strided layouts: strided plan vs copy + dense plan vs dense plan (tools/strided_shapes.py)\n\n")
        f.write("Card: %s (name, power limit, max SM clock as nvidia-smi reports them in the same run). fp32, CUDA events, "
                "%d timed calls after 5 warm-up calls; ms per call.\n\n" % (card, args.iters))
        f.write("| shape | strided | copy + dense | dense on dense data | strided / dense | kernels of the strided plan |\n")
        f.write("|---|---|---|---|---|---|\n")
        for name, ts, tc, td, kern in rows:
            f.write("| %s | %.4f | %.4f | %.4f | %.2f | %s |\n" % (name, ts, tc, td, ts / td, kern))
    print("wrote", args.out)


if __name__ == "__main__":
    main()

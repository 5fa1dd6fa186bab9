#!/usr/bin/env python3
"""Half-spectrum slab decomposition through MgpuPlan (b200fft_mgpu_*, MGPU_SLAB, REAL_HALF), device-resident:
    python tools/mgpu_half_shapes.py [--out profiles/r3_mgpu_half.md] [--sizes 256 512] [--steps 20] [--warmup 5]
For each n^3 in fp32 and each G in {1, 2, 4, 8} the machine has GPUs for: the R2C forward and the C2R inverse, next to the
complex slab of the same dims (forward / inverse) and to torch.fft.rfftn / irfftn (cuFFT) on one GPU. Timing: CUDA events
on every slot's stream, max over slots, per call, after a warm-up; the input volumes are larger than the L2 at 512^3 only.
Each timed plan is first checked against torch float64 on the same input. Rows for a G the machine lacks say "not
measured". Writes a markdown table with the card name and power limit read in the same run, and one JSON line per row to
stdout."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "hackathon-fft_b200", "python")]
import torch

import b200fft


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def time_slots(plan, devs, outs, ins, steps, warmup):
    """ms per call: CUDA events on every slot's stream, max over slots."""
    G = len(devs)
    streams = [torch.cuda.ExternalStream(plan.stream(i), device="cuda:%d" % devs[i]) for i in range(G)]
    for _ in range(warmup):
        plan.exec(outs, ins)
    plan.synchronize()
    ev = []
    for i, d in enumerate(devs):
        with torch.cuda.device(d):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(streams[i])
            ev.append((e0, e1))
    for _ in range(steps):
        plan.exec(outs, ins)
    for i, d in enumerate(devs):
        with torch.cuda.device(d):
            ev[i][1].record(streams[i])
    plan.synchronize()
    return max(e0.elapsed_time(e1) for e0, e1 in ev) / steps


def time_torch(fn, steps, warmup):
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


def rel(got, want):
    return float((got - want).norm() / want.norm())


def half_rows(n, G, steps, warmup):
    devs = list(range(G))
    dev0 = torch.device("cuda", 0)
    zl, yl, W = n // G, n // G, n // 2 + 1
    real_lay, cplx_lay, c_lay = (1, n, n, n, 1), (1, n, n, W, 2), (1, n, n, n, 2)
    gen = torch.Generator().manual_seed(n + G)
    vol = torch.randn((n, n, n), generator=gen)
    rows = {}

    # R2C forward: real z planes -> half-spectrum Y-slabs
    fwd = b200fft.MgpuPlan("float32", "float32", real_lay, cplx_lay, devices=devs, mode=b200fft.MGPU_SLAB,
                           real_mode=b200fft.REAL_HALF)
    ins = [vol[g * zl:(g + 1) * zl].to("cuda:%d" % g) for g in range(G)]
    outs = [torch.full((n, yl, W, 2), float("nan"), device="cuda:%d" % g) for g in range(G)]
    fwd.exec(outs, ins)
    fwd.synchronize()
    want = torch.fft.rfftn(vol.to(dev0, torch.float64))
    err = max(rel(torch.view_as_complex(outs[h].to(dev0, torch.float64)), want[:, h * yl:(h + 1) * yl]) for h in range(G))
    rows["r2c"] = (time_slots(fwd, devs, outs, ins, steps, warmup), err)
    fwd.destroy()

    # C2R inverse: those Y-slabs -> real z planes
    inv = b200fft.MgpuPlan("float32", "float32", cplx_lay, real_lay, devices=devs, mode=b200fft.MGPU_SLAB,
                           real_mode=b200fft.REAL_HALF, inverse=True)
    back = [torch.full((zl, n, n), float("nan"), device="cuda:%d" % g) for g in range(G)]
    inv.exec(back, outs)
    inv.synchronize()
    err = max(rel(back[g].to(dev0, torch.float64), vol[g * zl:(g + 1) * zl].to(dev0, torch.float64)) for g in range(G))
    rows["c2r"] = (time_slots(inv, devs, back, outs, steps, warmup), err)
    inv.destroy()
    del ins, outs, back, want

    # the complex slab of the same dims, both directions
    cvol = torch.randn((n, n, n, 2), generator=gen)
    for inverse in (False, True):
        plan = b200fft.MgpuPlan("float32", "float32", c_lay, c_lay, devices=devs, mode=b200fft.MGPU_SLAB, inverse=inverse)
        ins = [cvol[g * zl:(g + 1) * zl].to("cuda:%d" % g) for g in range(G)]
        outs = [torch.full((n, yl, n, 2), float("nan"), device="cuda:%d" % g) for g in range(G)]
        plan.exec(outs, ins)
        plan.synchronize()
        xc = torch.view_as_complex(cvol.to(dev0, torch.float64))
        want = torch.fft.ifftn(xc) if inverse else torch.fft.fftn(xc)
        err = max(rel(torch.view_as_complex(outs[h].to(dev0, torch.float64)), want[:, h * yl:(h + 1) * yl]) for h in range(G))
        rows["c2c_inv" if inverse else "c2c_fwd"] = (time_slots(plan, devs, outs, ins, steps, warmup), err)
        plan.destroy()
        del ins, outs, want, xc
    torch.cuda.empty_cache()
    return rows


def torch_rows(n, steps, warmup):
    x = torch.randn((n, n, n), device="cuda:0")
    spec = torch.fft.rfftn(x)
    return {"rfftn": time_torch(lambda: torch.fft.rfftn(x), steps, warmup),
            "irfftn": time_torch(lambda: torch.fft.irfftn(spec, s=(n, n, n)), steps, warmup)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_mgpu_half.md"))
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 512])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    have = torch.cuda.device_count()
    if have < 1:
        sys.exit("mgpu_half_shapes: no CUDA device; nothing is measured without one")
    name = card()
    lines = ["# Half-spectrum slab decomposition (MGPU_SLAB, REAL_HALF), device-resident, fp32", "",
             "Measured by `tools/mgpu_half_shapes.py` on %d visible GPU(s): %s (name, power limit, max SM clock)." % (have, name),
             "Milliseconds per call: CUDA events on every slot's stream, max over slots, %d calls after %d warm-up calls. "
             "The complex slab is the same dims through the same entry point; torch (cuFFT) runs on one GPU. "
             "rel L2: the timed plan's output against torch float64 on the same input, before timing "
             "(C2R: forward then inverse, against the original volume)." % (args.steps, args.warmup), "",
             "| volume | G | R2C fwd ms | complex fwd ms | torch rfftn ms (1 GPU) | C2R inv ms | complex inv ms | "
             "torch irfftn ms (1 GPU) | rel L2 R2C / C2R |",
             "|---|---|---|---|---|---|---|---|---|"]
    for n in args.sizes:
        tr = torch_rows(n, args.steps, args.warmup)
        for G in (1, 2, 4, 8):
            if G > have:
                lines.append("| %d^3 | %d | not measured | not measured | %.4f | not measured | not measured | %.4f | - |"
                             % (n, G, tr["rfftn"], tr["irfftn"]))
                print(json.dumps({"n": n, "gpus": G, "measured": False}), flush=True)
                continue
            r = half_rows(n, G, args.steps, args.warmup)
            rec = {"n": n, "gpus": G, "card": name, **{k: round(v[0], 4) for k, v in r.items()},
                   "rel_l2": {k: v[1] for k, v in r.items()}, **{"torch_" + k: round(v, 4) for k, v in tr.items()}}
            print(json.dumps(rec), flush=True)
            lines.append("| %d^3 | %d | %.4f | %.4f | %.4f | %.4f | %.4f | %.4f | %.1e / %.1e |"
                         % (n, G, r["r2c"][0], r["c2c_fwd"][0], tr["rfftn"], r["c2r"][0], r["c2c_inv"][0], tr["irfftn"],
                            r["r2c"][1], r["c2r"][1]))
    lines += ["", "G above the number of visible GPUs: not measured. Virtual slots on one GPU (the test suite's) say nothing "
              "about NVLink, so no such rows are given. That an R2C slab moves about half the bytes of the complex slab "
              "across the exchange (n/2+1 of every n bins) is arithmetic, not a measurement.", ""]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines))
    print("wrote", args.out)


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""Time one shape under a list of environment settings (kernel-variant knobs): one JSON line per setting.
    python tools/variant_sweep.py <mode: c2c|real|half> <batch,d0,d1,..> "K=V,K=V;K=V;..."   (';' separates settings)"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "hackathon-fft_b200", "python")]
import torch

import b200fft
from bench import time_gpu

KNOBS = ("B200FFT_PDL", "B200FFT_PLANE_PREFER", "B200FFT_PLANE", "B200FFT_PLANE_C2R", "B200FFT_SERPENTINE", "B200FFT_JIT", "B200FFT_JIT_MAX_RADIX", "B200FFT_FUSED", "B200FFT_CHUNK_MB", "B200FFT_FUSED_PREFER", "B200FFT_PREFER")


def main():
    mode, shape = sys.argv[1], tuple(int(v) for v in sys.argv[2].split(","))
    settings = [dict(kv.split("=", 1) for kv in s.split(",") if kv) for s in sys.argv[3].split(";")]
    comps = 2 if mode == "c2c" else 1
    x = torch.randn(shape + (comps,), device="cuda")
    oshape = shape[:-1] + (shape[-1] // 2 + 1, 2) if mode == "half" else shape + (2,)
    out = torch.empty(oshape, device="cuda")
    rm = b200fft.REAL_HALF if mode == "half" else b200fft.REAL_FULL
    st = torch.cuda.current_stream().cuda_stream
    want = None
    for env in settings:
        for k in KNOBS:
            os.environ.pop(k, None)
        os.environ.update(env)
        try:
            plan = b200fft.plan_fft("float32", "float32", x.shape, oshape, real_mode=rm)
            ms = min(time_gpu(lambda: plan.exec(out, x, st), 5, 20, torch) for _ in range(3))
            if want is None:
                want = out.clone()
            err = float((out - want).norm() / want.norm())
            print(json.dumps({"shape": list(shape), "mode": mode, "env": env, "ms": round(ms, 5), "rel_vs_first": err,
                              "plan": plan.describe().strip().split("\n")[0][:150]}), flush=True)
            plan.destroy()
        except Exception as e:
            print(json.dumps({"env": env, "error": str(e)}), flush=True)


if __name__ == "__main__":
    main()

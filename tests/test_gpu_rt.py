"""Runtime-length tier (csrc/rt.cu): which stage lists stay on the generic kernel, and that the tier is much faster than
it. The transforms of both kernels are checked against float64 by the form table (tests/_rt_generic_forms.py,
tests/test_gpu_rt_generic_forms.py)."""
import pytest

import b200fft

pytestmark = pytest.mark.gpu


def test_radix_above_64_stays_generic():
    p = b200fft.plan_fft("float32", "float32", (4, 74, 2), (4, 74, 2), flags=b200fft.FLAG_FORCE_RT)   # 74 = 37 * 2
    assert "generic" in p.describe()                                      # the rt tier's codelets stop at radix 32
    p = b200fft.plan_fft("float32", "float32", (4, 262, 2), (4, 262, 2), bases=[[131, 2]])   # above the specialised tier's 127 too
    assert "generic" in p.describe()
    p = b200fft.plan_fft("float32", "float32", (4, 64, 2), (4, 64, 2), _test="generic")
    assert "generic" in p.describe()


def test_rt_is_much_faster_than_generic():
    import torch
    x = torch.randn((20000, 1000, 2), device="cuda")
    out = torch.empty_like(x)
    st = torch.cuda.current_stream().cuda_stream
    times = {}
    for name, kw in (("rt", {"flags": b200fft.FLAG_FORCE_RT}), ("generic", {"_test": "generic"})):
        plan = b200fft.plan_fft("float32", "float32", x.shape, x.shape, **kw)
        for _ in range(3):
            plan.exec(out, x, st)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            plan.exec(out, x, st)
        e1.record()
        torch.cuda.synchronize()
        times[name] = e0.elapsed_time(e1) / 5
        plan.destroy()
    print("20000 x 1000: rt %.3f ms, generic %.3f ms" % (times["rt"], times["generic"]))
    assert times["rt"] * 3 < times["generic"]

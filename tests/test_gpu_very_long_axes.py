"""Contiguous axes longer than 2^24 points: three passes specialised at plan time (csrc/jit.cu: jit_split3_plan /
make_jit_split3_pass; kernels cols_split_a_kernel<..., TW2> and rows_split_c_kernel in csrc/fast.cuh), against
torch.fft in float64 on the same tensors.

Tolerances: fp32 rel-L2 2.5e-6 and max-abs 1e-5 * max|X| (test_gpu_long_axes.py); fp64 rel-L2 1e-13."""
import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu

N25 = 1 << 25


def _tdt(name):
    import torch
    return {"float32": torch.float32, "float64": torch.float64, "uint8": torch.uint8}[name]


def _input(shape, comps, dtype, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    if dtype == "uint8":
        return torch.randint(0, 256, shape + (comps,), generator=g, device="cuda", dtype=torch.uint8)
    return torch.randn(shape + (comps,), generator=g, device="cuda", dtype=_tdt(dtype))


def _reference(x, inverse):
    """torch.fft in float64 over the last transformed axis of a (batch, ..., n, comps) tensor."""
    import torch
    xd = x.to(torch.float64)
    z = torch.complex(xd[..., 0], xd[..., 1]) if x.shape[-1] == 2 else xd[..., 0].to(torch.complex128)
    return z


def _check(got, want, f64=False):
    import torch
    g = torch.complex(got[..., 0].to(torch.float64), got[..., 1].to(torch.float64))
    d = g - want
    rel = (torch.linalg.vector_norm(d) / torch.linalg.vector_norm(want)).item()
    mx = (d.abs().max() / want.abs().max()).item()
    if f64:
        assert rel <= 1e-13, rel
    else:
        assert rel <= 2.5e-6 and mx <= 1e-5, (rel, mx)


def _run(x, out_dtype="float32", inverse=False, in_place=False, **kw):
    """Plan, run once, check the input is untouched (unless in place); returns (output, plan facts)."""
    import torch
    shape = tuple(x.shape[:-1])
    keep = x.clone()
    out = x if in_place else torch.full(shape + (2,), float("nan"), dtype=_tdt(out_dtype), device="cuda")
    plan = b200fft.plan_fft(str(x.dtype).replace("torch.", ""), out_dtype, x.shape, shape + (2,), inverse=inverse, **kw)
    before = b200fft.launch_count()
    b200fft.fft(out, x, plan=plan)
    torch.cuda.synchronize()
    facts = dict(desc=plan.describe(), launches=plan.launches, ws=plan.workspace_bytes,
                 launched=b200fft.launch_count() - before)
    plan.destroy()
    if not in_place:
        assert torch.equal(x, keep)
    return out, facts, keep


def _fft(z, inverse, dims=(-1,)):
    import torch
    return torch.fft.ifftn(z, dim=dims) if inverse else torch.fft.fftn(z, dim=dims)


@pytest.mark.parametrize("shape,inverse", [((1, N25), False), ((1, N25), True), ((3, N25), False), ((1, 1 << 27), False),
                                           ((1, 3 ** 16), False), ((1, 10 ** 8), False)])
def test_complex_fp32(shape, inverse):
    x = _input(shape, 2, "float32", shape[1] % 1000 + shape[0])
    got, f, _ = _run(x, inverse=inverse)
    _check(got, _fft(_reference(x, inverse), inverse))
    assert "split3 n=%d" % shape[1] in f["desc"] and "jitsplit3C" in f["desc"], f["desc"]
    assert f["launches"] == 3 and f["launched"] == 3, f


def test_complex_fp64():
    x = _input((1, N25), 2, "float64", 5)
    got, f, _ = _run(x, "float64")
    _check(got, _fft(_reference(x, False), False), f64=True)
    assert "split3" in f["desc"] and "_f64" in f["desc"], f["desc"]


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_real_full_spectrum(dtype):
    x = _input((1, N25), 1, dtype, 6)
    got, f, _ = _run(x)
    _check(got, _fft(_reference(x, False), False))
    assert "split3 n=%d real-in" % N25 in f["desc"] and "_realin" in f["desc"], f["desc"]
    if dtype == "uint8":
        assert "_inu8" in f["desc"], f["desc"]


def test_nd_long_last_axis():
    """The last axis takes the three-pass split, then the axis of length 2 runs as a strided pass over its output."""
    x = _input((1, 2, N25), 2, "float32", 7)
    got, f, _ = _run(x)
    _check(got, _fft(_reference(x, False), False, dims=(1, 2)))
    assert "axis 1: split3 n=%d" % N25 in f["desc"] and f["launches"] >= 4, f["desc"]


def test_in_place():
    x = _input((1, N25), 2, "float32", 8)
    got, f, keep = _run(x, in_place=True)
    _check(got, _fft(_reference(keep, False), False))
    assert "split3" in f["desc"], f["desc"]


def test_exec_host():
    import torch
    x = _input((1, N25), 2, "float32", 9)
    h_in = x.cpu().numpy()
    h_out = np.full(h_in.shape, np.nan, dtype=np.float32)
    plan = b200fft.plan_fft("float32", "float32", h_in.shape, h_in.shape)
    plan.exec_host(h_out, h_in)
    desc = plan.describe()
    plan.destroy()
    _check(torch.from_numpy(h_out).cuda(), _fft(_reference(x, False), False))
    assert "split3" in desc, desc


def test_plan_properties():
    import torch
    shape = (2, N25)
    plan = b200fft.plan_fft("float32", "float32", shape + (2,), shape + (2,))
    try:
        assert plan.launches == 3
        assert "split3 n=%d" % N25 in plan.describe()
        assert plan.workspace_bytes == shape[0] * N25 * 8
        x = _input(shape, 2, "float32", 10)
        out = torch.empty_like(x)
        for _ in range(2):
            before = b200fft.launch_count()
            b200fft.fft(out, x, plan=plan)
            torch.cuda.synchronize()
            assert b200fft.launch_count() - before == 3
    finally:
        plan.destroy()


def test_two_pass_up_to_2_24():
    """Lengths up to 2^24 keep the plans they had: 2^23 its two-pass split. 2^24 has none (its stages do not split into
    two tiles that fit) and the three-pass form does not take it either: still status 4."""
    x = _input((1, 1 << 23), 2, "float32", 11)
    got, f, _ = _run(x)
    _check(got, _fft(_reference(x, False), False))
    assert "split n=8388608" in f["desc"] and "split3" not in f["desc"] and f["launches"] == 2, f["desc"]
    shape = (1, 1 << 24, 2)
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft("float32", "float32", shape, shape)
    assert e.value.status == 4 and "split3" not in str(e.value), str(e.value)


@pytest.mark.parametrize("in_shape,out_shape,kw,why", [
    ((1, 1 << 26, 1), (1, (1 << 25) + 1, 2), dict(real_mode=b200fft.REAL_HALF), "half-spectrum"),
    ((1, N25, 2, 2), (1, N25, 2, 2), {}, "strided"),
    ((1, N25, 2), (1, N25, 2), dict(flags=b200fft.FLAG_FORCE_GENERIC), "FORCE_GENERIC"),
])
def test_refusals(in_shape, out_shape, kw, why):
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft("float32", "float32", in_shape, out_shape, **kw)
    assert e.value.status == 4
    assert why in str(e.value), str(e.value)

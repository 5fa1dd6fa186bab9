"""Strided layouts on a B200 (b200fft_plan_create_strided), against torch.fft in float64 of the actual input.

Every case reads its input through a view of a larger random buffer and writes its output through a view of a larger
NaN-filled buffer: afterwards the input buffer is unchanged and every output element outside the view is still NaN. The
plan has one launch per transformed axis, names only plan-time `_str` kernels, and a second plan of the same problem
gives the same bits."""
import numpy as np
import pytest
import torch

import b200fft

pytestmark = pytest.mark.gpu

DT = {"float32": torch.float32, "float64": torch.float64, "uint8": torch.uint8}


def dense(shape):
    out, s = [], 1
    for v in reversed(shape):
        out.append(s)
        s *= v
    return list(reversed(out))


def buffer_view(shape, strides, comps, dtype, fill, gen=None):
    """A view of logical `shape` (batch, dims...) with element `strides` into a fresh buffer one element longer than
    the span (so the view never ends at the buffer's end); `fill`: "rand" or "nan"."""
    span = sum((n - 1) * s for n, s in zip(shape, strides)) + 2
    dt = DT[dtype]
    if fill == "nan":
        buf = torch.full((span * comps,), float("nan"), dtype=dt, device="cuda")
    elif dt == torch.uint8:
        buf = torch.randint(0, 256, (span * comps,), dtype=dt, device="cuda", generator=gen)
    else:
        buf = torch.randn(span * comps, dtype=dt, device="cuda", generator=gen)
    view = buf.as_strided(tuple(shape) + (comps,), tuple(s * comps for s in strides) + (1,))
    return buf, view


def as_complex64(t, comps):
    t = t.double()
    return torch.complex(t[..., 0], t[..., 1]) if comps == 2 else t[..., 0].to(torch.complex128)


def check(got, ref, out_dtype):
    got, ref = got.cpu(), ref.cpu()
    err = (torch.linalg.vector_norm(got - ref) / torch.linalg.vector_norm(ref)).item()
    if out_dtype == "float64":
        assert err <= 1e-13, err
    else:
        assert err <= 2e-6, err
        assert (got - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


def run_case(shape, in_strides, out_strides, *, in_dtype="float32", out_dtype="float32", comps=2, half=False, inverse=False,
             axis_mask=0):
    """shape: logical (batch, dims...) of the real side for half-spectrum plans, of both sides otherwise."""
    gen = torch.Generator(device="cuda").manual_seed(sum(shape))
    rank = len(shape) - 1
    axes = [a for a in range(rank) if not axis_mask or axis_mask >> a & 1]
    cshape = list(shape[:-1]) + [shape[-1] // 2 + 1] if half else list(shape)
    ishape, oshape = (cshape, shape) if half and inverse else (shape, cshape) if half else (shape, shape)
    icomps = 2 if half and inverse else 1 if half else comps
    ocomps = 1 if half and inverse else 2
    in_buf, x = buffer_view(ishape, in_strides, icomps, in_dtype, "rand", gen)
    if half and inverse:  # a Hermitian spectrum: the half spectrum of a real signal
        real = torch.randn(tuple(shape), dtype=torch.float64, device="cuda", generator=gen)
        spec = torch.fft.rfftn(real, dim=[a + 1 for a in axes])
        x[..., 0].copy_(spec.real)
        x[..., 1].copy_(spec.imag)
    in_copy = in_buf.clone()
    out_buf, y = buffer_view(oshape, out_strides, ocomps, out_dtype, "nan")
    kw = dict(inverse=inverse, axis_mask=axis_mask, real_mode=b200fft.REAL_HALF if half else b200fft.REAL_FULL,
              in_strides=in_strides, out_strides=out_strides)
    plan = b200fft.plan_fft(in_dtype, out_dtype, tuple(ishape) + (icomps,), tuple(oshape) + (ocomps,), **kw)
    assert plan.launches == len(axes), plan.describe()
    lines = plan.describe().strip().split("\n")
    assert len(lines) == len(axes) and all("_str" in ln and "NVRTC" in ln for ln in lines), lines
    b200fft.fft(y, x, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(in_buf, in_copy), "the input was modified"
    mask = torch.ones(out_buf.shape, dtype=torch.bool, device="cuda")
    mask.as_strided(y.shape, y.stride()).fill_(False)
    assert out_buf[mask].isnan().all(), "an element outside the output view was written"
    assert not y.isnan().any(), "an output element was not written"
    dims = [a + 1 for a in axes]
    xd = as_complex64(x, icomps)
    if half and inverse:
        ref = torch.fft.irfftn(xd, s=[shape[a] for a in dims], dim=dims)
        got = y[..., 0].double()
    elif half:
        ref = torch.fft.rfftn(x[..., 0].double(), dim=dims)
        got = as_complex64(y, 2)
    else:
        ref = (torch.fft.ifftn if inverse else torch.fft.fftn)(xd, dim=dims)
        got = as_complex64(y, 2)
    check(got, ref, out_dtype)
    # a second plan of the same problem: the same bits
    out2_buf, y2 = buffer_view(oshape, out_strides, ocomps, out_dtype, "nan")
    plan2 = b200fft.plan_fft(in_dtype, out_dtype, tuple(ishape) + (icomps,), tuple(oshape) + (ocomps,), **kw)
    b200fft.fft(y2, x, plan=plan2)
    torch.cuda.synchronize()
    assert torch.equal(y, y2)


def t2(shape, perm):
    """element strides of a dense array of `shape` seen through the axis permutation `perm` (batch stays first)"""
    st = dense(shape)
    return [st[p] for p in perm]


CASES = [
    # (id, logical shape, in strides, out strides, options)
    ("c2c-batch-slice-1024", (64, 1024), [2048, 1], [2048, 1], {}),
    ("c2c-pitch-1000-inverse", (300, 1000), [1040, 1], [1040, 1], dict(inverse=True)),
    ("c2c-elem-stride3-1024", (200, 1024), [3 * 1024, 3], dense((200, 1024)), {}),
    ("c2c-elem-stride3-93", (500, 93), [3 * 93, 3], [3 * 93, 3], {}),
    ("c2c-pitch-2187", (40, 2187), [2200, 1], [2200, 1], dict(inverse=True)),
    ("c2c-rowsIP-16384", (8, 16384), [16400, 1], [16400, 1], {}),
    ("c2c-2d-transposed", (20, 48, 64), t2((20, 64, 48), [0, 2, 1]), dense((20, 48, 64)), {}),
    ("c2c-3d-transposed", (6, 24, 16, 20), t2((6, 16, 20, 24), [0, 3, 1, 2]), dense((6, 24, 16, 20)), dict(inverse=True)),
    ("c2c-3d-axis-mask", (6, 24, 16, 20), t2((6, 16, 20, 24), [0, 3, 1, 2]), t2((6, 20, 16, 24), [0, 3, 2, 1]),
     dict(axis_mask=0b101)),
    ("c2c-f64-pitch", (100, 1000), [1010, 1], [1020, 1], dict(in_dtype="float64", out_dtype="float64")),
    ("c2c-f32-in-f64-out", (20, 48, 64), t2((20, 64, 48), [0, 2, 1]), dense((20, 48, 64)), dict(out_dtype="float64")),
    ("real-f32-pitch", (300, 1000), [1040, 1], dense((300, 1000)), dict(comps=1)),
    ("real-u8-transposed", (20, 48, 64), t2((20, 64, 48), [0, 2, 1]), dense((20, 48, 64)), dict(comps=1, in_dtype="uint8")),
    ("real-f64-stride3", (200, 1024), [3 * 1024, 3], dense((200, 1024)), dict(comps=1, in_dtype="float64", out_dtype="float64")),
    ("r2c-even-pitch", (300, 1000), [1040, 1], [520, 1], dict(half=True)),
    ("r2c-1024-padded", (200, 1024), [1026, 1], [513, 1], dict(half=True)),
    ("r2c-odd-93", (500, 93), [100, 1], [50, 1], dict(half=True)),
    ("r2c-nd", (4, 24, 20, 64), [24 * 20 * 66, 20 * 66, 66, 1], [24 * 20 * 40, 20 * 40, 40, 1], dict(half=True)),
    ("r2c-f64", (100, 1000), [1040, 1], [520, 1], dict(half=True, in_dtype="float64", out_dtype="float64")),
    ("c2r-even-pitch", (300, 1000), [520, 1], [1040, 1], dict(half=True, inverse=True)),
    ("c2r-odd-2187", (40, 2187), [1100, 1], [2200, 1], dict(half=True, inverse=True)),
    ("c2r-nd", (4, 24, 20, 64), [24 * 20 * 40, 20 * 40, 40, 1], [24 * 20 * 66, 20 * 66, 66, 1], dict(half=True, inverse=True)),
    ("c2r-nd-f64", (4, 16, 93), [16 * 50, 50, 1], [16 * 100, 100, 1],
     dict(half=True, inverse=True, in_dtype="float64", out_dtype="float64")),
]


@pytest.mark.parametrize("shape,in_strides,out_strides,opts", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_strided_view_matches_torch(shape, in_strides, out_strides, opts):
    run_case(shape, in_strides, out_strides, **opts)


@pytest.mark.parametrize("shape", [(100000, 1024), (16, 128, 128, 128)], ids=["1d", "3d"])
def test_in_place_padded_round_trip(shape):
    """The classic in-place layout: real rows of pitch 2(n/2+1) sharing their bytes with the n/2+1 complex bins."""
    n = shape[-1]
    hb = n // 2 + 1
    cshape = shape[:-1] + (hb,)
    cst = dense(cshape)
    rst = [2 * s for s in cst[:-1]] + [1]
    gen = torch.Generator(device="cuda").manual_seed(1)
    buf = torch.empty(int(np.prod(cshape)) * 2, dtype=torch.float32, device="cuda")
    real = buf.as_strided(shape + (1,), tuple(rst) + (1,))
    real.copy_(torch.randn(shape + (1,), generator=gen, device="cuda"))
    x0 = real.clone()
    cplx = buf.as_strided(cshape + (2,), tuple(2 * s for s in cst) + (1,))
    fwd = b200fft.plan_fft("float32", "float32", shape + (1,), cshape + (2,), real_mode=b200fft.REAL_HALF,
                           in_strides=rst, out_strides=cst)
    inv = b200fft.plan_fft("float32", "float32", cshape + (2,), shape + (1,), real_mode=b200fft.REAL_HALF, inverse=True,
                           in_strides=cst, out_strides=rst)
    # out of place through the same layouts first
    sep = torch.full_like(buf, float("nan"))
    sep_c = sep.as_strided(cplx.shape, cplx.stride())
    b200fft.fft(sep_c, real, plan=fwd)
    b200fft.fft(cplx, real, plan=fwd)  # in place
    torch.cuda.synchronize()
    assert torch.equal(cplx, sep_c), "in-place R2C differs from the out-of-place result"
    dims = list(range(1, len(shape)))
    ref = torch.fft.rfftn(x0[..., 0].double(), dim=dims)
    check(torch.complex(cplx[..., 0].double(), cplx[..., 1].double()), ref, "float32")
    back = torch.full_like(buf, float("nan"))
    back_r = back.as_strided(real.shape, real.stride())
    b200fft.fft(back_r, cplx, plan=inv)
    b200fft.fft(real, cplx, plan=inv)  # in place
    torch.cuda.synchronize()
    assert torch.equal(real, back_r), "in-place C2R differs from the out-of-place result"
    check(real[..., 0].double(), x0[..., 0].double(), "float32")


def test_dense_strides_make_the_dense_plan():
    for shape, kw in (((64, 1024, 2), {}), ((10, 48, 64, 2), dict(inverse=True)), ((8, 96, 1), dict(real_mode=b200fft.REAL_HALF))):
        out = (8, 49, 2) if kw.get("real_mode") else shape
        a = b200fft.plan_fft("float32", "float32", shape, out, **kw)
        b = b200fft.plan_fft("float32", "float32", shape, out, in_strides=dense(shape[:-1]), out_strides=dense(out[:-1]), **kw)
        c = b200fft.plan_fft("float32", "float32", shape, out, out_strides=dense(out[:-1]), **kw)
        assert a.describe() == b.describe() == c.describe()
        assert a.launches == b.launches and "_str" not in a.describe()


def test_refusals_on_the_device():
    shape = (64, 1000, 2)
    plan = b200fft.plan_fft("float32", "float32", shape, shape, in_strides=[1040, 1], out_strides=[1000, 1])
    assert plan.in_bytes == (63 * 1040 + 1000) * 8 and plan.out_bytes == 64 * 1000 * 8
    host = np.zeros((64 * 1040 * 2,), dtype=np.float32)
    with pytest.raises(b200fft.B200FFTError) as e:
        plan.exec_host(host, host)
    assert e.value.status == 4
    buf = torch.zeros(64 * 1040 * 2, device="cuda")
    with pytest.raises(b200fft.B200FFTError) as e:  # in place, but input and output strides differ
        plan.exec(buf, buf)
    assert e.value.status == 1
    # equal strides: in place is exact
    same = b200fft.plan_fft("float32", "float32", shape, shape, in_strides=[1040, 1], out_strides=[1040, 1])
    same.exec(buf, buf)
    torch.cuda.synchronize()

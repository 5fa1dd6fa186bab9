"""Strided layouts on a B200 (b200fft_plan_create_strided), against torch.fft in float64 of the actual input.

Every case reads its input through a view of a larger random buffer and writes its output through a view of a larger
NaN-filled buffer: afterwards the input buffer is unchanged and every output element outside the view is still NaN. The
plan has one launch per transformed axis, names only plan-time `_str` kernels, and a second plan of the same problem
gives the same bits (tests/_strided_forms.py: run_case; tests/test_gpu_strided_forms.py runs its table of every
strided kernel form)."""
import numpy as np
import pytest
import torch

import b200fft
from _strided_forms import check, dense, run_case, t2

pytestmark = pytest.mark.gpu

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


@pytest.mark.parametrize("shape,axis_mask", [((100000, 1024), 0), ((16, 128, 128, 128), 0), ((1, 64, 64, 64), 0),
                                              ((4, 1, 64), 0b10)], ids=["1d", "3d", "3d-batch-1", "masked-axis-of-1"])
def test_in_place_padded_round_trip(shape, axis_mask):
    """The classic in-place layout: real rows of pitch 2(n/2+1) sharing their bytes with the n/2+1 complex bins. A
    dimension of extent 1 (a batch of 1, a masked axis of one point) runs in place whatever its strides."""
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
                           in_strides=rst, out_strides=cst, axis_mask=axis_mask)
    inv = b200fft.plan_fft("float32", "float32", cshape + (2,), shape + (1,), real_mode=b200fft.REAL_HALF, inverse=True,
                           in_strides=cst, out_strides=rst, axis_mask=axis_mask)
    # out of place through the same layouts first
    sep = torch.full_like(buf, float("nan"))
    sep_c = sep.as_strided(cplx.shape, cplx.stride())
    b200fft.fft(sep_c, real, plan=fwd)
    b200fft.fft(cplx, real, plan=fwd)  # in place
    torch.cuda.synchronize()
    assert torch.equal(cplx, sep_c), "in-place R2C differs from the out-of-place result"
    dims = [a + 1 for a in range(len(shape) - 1) if not axis_mask or axis_mask >> a & 1]
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
    # equal strides: in place is exact, the same bits as out of place, and the pitch padding is left alone
    same = b200fft.plan_fft("float32", "float32", shape, shape, in_strides=[1040, 1], out_strides=[1040, 1])
    buf.copy_(torch.randn(buf.shape, generator=torch.Generator(device="cuda").manual_seed(2), device="cuda"))
    sep = torch.full_like(buf, float("nan"))
    same.exec(sep, buf)
    before = buf.clone()
    same.exec(buf, buf)
    torch.cuda.synchronize()
    rows = buf.view(64, 1040, 2)
    assert torch.equal(rows[:, :1000], sep.view(64, 1040, 2)[:, :1000]), "in place differs from out of place"
    assert torch.equal(rows[:, 1000:], before.view(64, 1040, 2)[:, 1000:]), "in place wrote into the pitch padding"

"""Every row of the strided kernel table (tests/_strided_forms.py) on a B200, against torch.fft in float64, and the
layouts views produce that the table's pitched and permuted rows do not: broadcast and overlapping input, views at an
element offset, offsets beyond 2^31 elements, and strides of extent-1 dimensions.

For each table row, run_case checks the float64 reference (fp32: relative L2 <= 2e-6 and max-abs <= 1e-5 * max|X|; fp64:
relative L2 <= 1e-13), that every output element inside the view is written and none outside it, that the input is
unchanged, that the plan has one launch per transformed axis and names the row's kernels in launch order, and that a
second plan gives the same bits. A complex-to-complex row also runs in place on its input layout, bit-identical to the
same plan out of place.

B200FFT_STRIDED_REPORT=<file> appends one JSON line per row (kernel names, peak device memory)."""
import json
import os

import pytest
import torch

import b200fft
from _strided_forms import F32, F64, FORMS, KINDS, U8, buffer_view, check, names_in, result, run_case, sides

pytestmark = pytest.mark.gpu


def _report(**rec):
    path = os.environ.get("B200FFT_STRIDED_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")


def _in_place(form):
    """the row's transform on its input layout, in place and out of place: the same bits"""
    kw = form.kwargs()
    shape, st, off = kw["shape"], kw["in_strides"], kw["offset"][0]
    dt = form.in_dtype
    layout = tuple(shape) + (2,)
    plan = b200fft.plan_fft(dt, dt, layout, layout, bases=form.bases, inverse=form.inverse, axis_mask=form.axis_mask,
                            in_strides=st, out_strides=st)
    gen = torch.Generator(device="cuda").manual_seed(7)
    buf, x = buffer_view(shape, st, 2, dt, "rand", gen, off)
    _, y = buffer_view(shape, st, 2, dt, "nan", None, off)
    b200fft.fft(y, x, plan=plan)
    outside = buf.clone()
    b200fft.fft(x, x, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(x, y), "in place differs from out of place"
    mask = torch.ones(buf.shape, dtype=torch.bool, device="cuda")
    mask.as_strided(x.shape, x.stride(), x.storage_offset()).fill_(False)
    assert torch.equal(buf[mask], outside[mask]), "in place wrote outside the view"


@pytest.mark.parametrize("form", FORMS, ids=[f.id for f in FORMS])
def test_strided_form(form):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    desc, _, _ = run_case(**form.kwargs())
    if form.c2c:
        _in_place(form)
    _report(id=form.id, kernels=names_in(desc), peak_bytes=torch.cuda.max_memory_allocated())


# ---- broadcast and overlapping input ------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,in_strides,out_strides,opts", [
    ((8, 1000), [0, 1], [1008, 1], {}),                                  # the batch: one row, transformed 8 times
    ((4, 6, 64), [70, 0, 1], [6 * 64, 64, 1], {}),                      # an outer axis: 6 equal rows per batch
    ((3, 6, 64), [0, 0, 1], [6 * 72, 72, 1], dict(comps=1, in_dtype=U8)),
    ((3, 6, 64), [70, 0, 1], [6 * 64, 64, 1], dict(axis_mask=0b10, in_dtype=F64, out_dtype=F64)),
], ids=["batch", "outer-axis", "batch-and-axis-u8-real", "masked-outer-f64"])
def test_broadcast_input(shape, in_strides, out_strides, opts):
    run_case(shape, in_strides, out_strides, **opts)


@pytest.mark.parametrize("dtype", [F32, F64])
def test_constant_signal_along_a_stride_0_axis(dtype):
    """stride 0 along the transformed axis: every row is one value repeated, all its energy lands in bin 0"""
    _, x, y = run_case((5, 256), [1, 0], [264, 1], in_dtype=dtype, out_dtype=dtype)
    z = result(y, False, False)
    x0 = torch.complex(x[:, 0, 0].double(), x[:, 0, 1].double())
    torch.testing.assert_close(z[:, 0], 256 * x0, rtol=1e-6 if dtype == F32 else 1e-14, atol=0)
    assert z[:, 1:].abs().max().item() <= (1e-5 if dtype == F32 else 1e-13) * z[:, 0].abs().max().item()


@pytest.mark.parametrize("hop", [256, 1000])
def test_sliding_window_frames(hop):
    """overlapping frames of one real fp32 signal (an STFT without the window): n = 1024, the hop below n, through R2C"""
    n, frames = 1024, 60
    gen = torch.Generator(device="cuda").manual_seed(hop)
    sig = torch.randn((frames - 1) * hop + n + 1, device="cuda", generator=gen)
    x = sig.as_strided((frames, n, 1), (hop, 1, 1))
    out = torch.full((frames * (n // 2 + 8) * 2,), float("nan"), device="cuda")
    y = out.as_strided((frames, n // 2 + 1, 2), ((n // 2 + 8) * 2, 2, 1))
    plan = b200fft.plan_fft(F32, F32, (frames, n, 1), (frames, n // 2 + 1, 2), real_mode=b200fft.REAL_HALF,
                            in_strides=[hop, 1], out_strides=[n // 2 + 8, 1])
    assert plan.launches == 1 and "_str" in plan.describe()
    before = sig.clone()
    b200fft.fft(y, x, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(sig, before)
    frames_d = sig.double().as_strided((frames, n), (hop, 1))
    check(result(y, True, False), torch.fft.rfft(frames_d, dim=1), F32)


def test_odd_hop_with_even_length_is_refused():
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft(F32, F32, (60, 1024, 1), (60, 513, 2), real_mode=b200fft.REAL_HALF, in_strides=[255, 1],
                         out_strides=[520, 1])
    assert e.value.status == 4 and "odd" in str(e.value)


# ---- element offsets ----------------------------------------------------------------------------------------------------
def _first(kind, f64):
    return next(f for f in FORMS if f.kinds[0] == kind and f.f64 == f64)


@pytest.mark.parametrize("f64", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("kind", KINDS)
def test_views_one_element_in(kind, f64):
    """both views start one element into their buffers (8 B in fp32 complex, 16 B in fp64 complex; a pair of real
    scalars on the real side of an even half spectrum, which the kernels read and write as pairs)"""
    form = _first(kind, f64)
    kw = form.kwargs()
    n = kw["shape"][-1]
    pair = 2 if form.half and n % 2 == 0 else 1
    kw["offset"] = (pair if form.half and not form.inverse else 1, pair if form.half and form.inverse else 1)
    run_case(**kw)


@pytest.mark.parametrize("inverse", [False, True], ids=["r2c", "c2r"])
def test_real_view_one_scalar_in_is_refused(inverse):
    """an even half spectrum moves real rows as pairs of scalars: a real view one fp32 scalar into its buffer is
    misaligned, and b200fft_exec refuses it with B200FFT_ERR_INVALID_ARG before any launch"""
    real, cplx = (4, 1000, 1), (4, 501, 2)
    ilay, olay = (cplx, real) if inverse else (real, cplx)
    rst, cst = [1008, 1], [510, 1]
    plan = b200fft.plan_fft(F32, F32, ilay, olay, real_mode=b200fft.REAL_HALF, inverse=inverse,
                            in_strides=cst if inverse else rst, out_strides=rst if inverse else cst)
    rbuf = torch.zeros(4 * 1008 + 8, device="cuda")
    cbuf = torch.zeros(4 * 510 * 2 + 8, device="cuda")
    r = rbuf[1:]  # one scalar in: 4 B past an aligned base
    before = b200fft.launch_count()
    with pytest.raises(b200fft.B200FFTError) as e:
        if inverse:
            plan.exec(r, cbuf)
        else:
            plan.exec(cbuf, r)
    assert e.value.status == 1 and "aligned" in str(e.value), str(e.value)
    assert b200fft.launch_count() == before
    if inverse:  # a whole pair in: served
        plan.exec(rbuf[2:], cbuf)
    else:
        plan.exec(cbuf, rbuf[2:])
    torch.cuda.synchronize()


# ---- element offsets beyond 2^31 ----------------------------------------------------------------------------------------
GB = 2 ** 30


def _need(free_bytes):
    free, _ = torch.cuda.mem_get_info()
    if free < free_bytes:
        pytest.skip("needs %.0f GB of free device memory, %.1f GB free" % (free_bytes / GB, free / GB))


def test_input_rows_beyond_2_to_32_bytes():
    """uint8 real input, 2 rows of 1024 points 2^32 + 2 elements apart: the second row lies past every 32-bit offset"""
    _need(24 * GB)
    torch.cuda.reset_peak_memory_stats()
    n, stride, g = 1024, 2 ** 32 + 2, 64
    gen = torch.Generator(device="cuda").manual_seed(3)
    rows = torch.randint(0, 256, (2, n), dtype=torch.uint8, device="cuda", generator=gen)
    buf = x = None  # every name that holds the 4 GB buffer, released in `finally` whatever the outcome
    try:
        buf = torch.zeros(stride + n + g, dtype=torch.uint8, device="cuda")
        buf[:n].copy_(rows[0])
        buf[stride:stride + n].copy_(rows[1])
        x = buf.as_strided((2, n, 1), (stride, 1, 1))
        out = torch.full((2, n + 16, 2), float("nan"), device="cuda")
        y = out[:, :n]
        plan = b200fft.plan_fft(U8, F32, (2, n, 1), (2, n, 2), in_strides=[stride, 1], out_strides=[n + 16, 1])
        b200fft.fft(y, x, plan=plan)
        torch.cuda.synchronize()
        assert out[:, n:].isnan().all()
        assert not buf[n:n + g].any() and not buf[stride - g:stride].any() and not buf[stride + n:].any()
        assert torch.equal(buf[:n], rows[0]) and torch.equal(buf[stride:stride + n], rows[1])
        check(result(y, False, False), torch.fft.fft(rows.double(), dim=1), F32)
        _report(id="offset-input-2^32", peak_bytes=torch.cuda.max_memory_allocated())
    finally:
        buf = x = None
        torch.cuda.empty_cache()


def test_output_rows_beyond_2_to_31_elements():
    """fp32 complex output, 2 rows of 1024 points 2^31 + 64 elements (16 GB) apart, the guard bands around each row
    left as they were"""
    _need(24 * GB)
    torch.cuda.reset_peak_memory_stats()
    n, stride, g = 1024, 2 ** 31 + 64, 64
    gen = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn((2, n, 2), device="cuda", generator=gen)
    xs = torch.zeros((2, n + 8, 2), device="cuda")
    xs[:, :n] = x
    xv = xs[:, :n]
    out = y = None  # every name that holds the 16 GB buffer, released in `finally` whatever the outcome
    try:
        out = torch.full((stride + n + g, 2), float("nan"), device="cuda")
        y = out.as_strided((2, n, 2), (2 * stride, 2, 1))
        plan = b200fft.plan_fft(F32, F32, (2, n, 2), (2, n, 2), in_strides=[n + 8, 1], out_strides=[stride, 1],
                                inverse=True)
        b200fft.fft(y, xv, plan=plan)
        torch.cuda.synchronize()
        for lo, hi in ((n, n + g), (stride - g, stride), (stride + n, stride + n + g)):
            assert out[lo:hi].isnan().all(), "a store outside the rows, elements %d..%d" % (lo, hi)
        assert not y.isnan().any()
        ref = torch.fft.ifft(torch.complex(x[..., 0].double(), x[..., 1].double()), dim=1)
        check(result(y, False, False), ref, F32)
        _report(id="offset-output-2^31", peak_bytes=torch.cuda.max_memory_allocated())
    finally:
        out = y = None
        torch.cuda.empty_cache()


# ---- strides of extent-1 dimensions -------------------------------------------------------------------------------------
ODD_STRIDES = [0, 7, 2 ** 40]


@pytest.mark.parametrize("case", ["rows-1000", "rows-65536", "2d", "r2c-odd-pitch"])
def test_batch_of_one_with_any_stride_is_the_dense_plan(case):
    """a batch of 1, dense but for its batch stride: b200fft_plan_create's plan, whatever that stride is"""
    shape, half = {"rows-1000": ((1, 1000), False), "rows-65536": ((1, 65536), False), "2d": ((1, 48, 64), False),
                   "r2c-odd-pitch": ((1, 1000), True)}[case]
    ishape, oshape = sides(shape, half, False)
    ilay, olay = tuple(ishape) + (1 if half else 2,), tuple(oshape) + (2,)
    mode = b200fft.REAL_HALF if half else b200fft.REAL_FULL
    dense_plan = b200fft.plan_fft(F32, F32, ilay, olay, real_mode=mode)
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(ilay, device="cuda", generator=gen)
    want = torch.full(olay, float("nan"), device="cuda")
    b200fft.fft(want, x, plan=dense_plan)
    for s in ODD_STRIDES + [1001]:
        ist = [s] + [v // ilay[-1] for v in x.stride()[1:-1]]
        ost = [s + 1] + [v // 2 for v in want.stride()[1:-1]]
        plan = b200fft.plan_fft(F32, F32, ilay, olay, real_mode=mode, in_strides=ist, out_strides=ost)
        assert plan.describe() == dense_plan.describe(), (s, plan.describe())
        got = torch.full(olay, float("nan"), device="cuda")
        b200fft.fft(got, x, plan=plan)
        torch.cuda.synchronize()
        assert torch.equal(got, want), s


def test_extent_1_strides_leave_a_strided_plan_unchanged():
    """a masked axis of extent 1 inside strided layouts, and a batch of 1: their strides change neither the plan nor
    the bits"""
    for shape, ist, ost, mask in (((6, 1, 100), [108, 108, 1], [110, 110, 1], 0b10),
                                  ((1, 37, 1, 24), [0, 30, 7, 1], [37 * 24, 1, 5, 37], 0b101)):
        base = run_case(shape, ist, ost, axis_mask=mask)
        for s in ODD_STRIDES:
            i2 = [s if n == 1 else v for n, v in zip(shape, ist)]
            o2 = [s + 1 if n == 1 else v for n, v in zip(shape, ost)]
            desc, _, y = run_case(shape, i2, o2, axis_mask=mask)
            assert desc == base[0], (s, desc)
            assert torch.equal(y, base[2]), s


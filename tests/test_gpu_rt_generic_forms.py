"""Every row of the runtime-length / generic kernel table (tests/_rt_generic_forms.py) on the GPU, against float64.

For each row:
  * plan.describe() has one line per pass with the row's kinds; every rt and generic line is exactly the one the rule
    copies predict from the dry_run stage lists (tile, shared memory, super-stages, suffix), so no plan-time or
    compiled-in kernel stands where the row expects an rt or generic pass;
  * fp32 output: relative L2 <= 2e-6 * sqrt(axes) and max-abs <= 1e-5 * max|X|, also at the radix-14519 stage; fp64
    output: relative L2 <= 1e-13 * sqrt(axes). The reference is the float64 transform of the actual input (numpy, or
    torch.fft in float64 on the device above 2^22 points);
  * the output is NaN-prefilled between 4 KB sentinel guard bands that must come back unchanged, an out-of-place run
    leaves its input unchanged, and the launch counter moves by plan.launches;
  * a complex-to-complex row run in place gives the same bits as the out-of-place run.
Rows marked refused must fail at plan creation with status 4 and the row's message.

B200FFT_FORMS_REPORT=<file> appends one JSON line per row (error, device memory) for the suite's statistics."""
import json
import os
import zlib

import numpy as np
import pytest

import b200fft
from _rt_generic_forms import REFUSED, RUNS, U8, expected_lines

pytestmark = pytest.mark.gpu

GUARD = 4096
SENTINEL = 0xA5
BIG = 2 ** 22  # points above which the reference runs on the device
_ENV = ("B200FFT_PREFER", "B200FFT_R2C_SMEM", "B200FFT_FUSED", "B200FFT_PLANE", "B200FFT_FUSED_PREFER",
        "B200FFT_ROWS_INPLACE", "B200FFT_JIT_MAX_RADIX", "B200FFT_JIT_PLANE", "B200FFT_JIT")


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in _ENV:
        monkeypatch.delenv(k, raising=False)


class Buf:
    """A device buffer of `nbytes` between two guard bands of SENTINEL bytes."""

    def __init__(self, nbytes, fill_nan=True):
        import torch
        self.nbytes = nbytes
        self.raw = torch.full((GUARD + nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        if fill_nan:
            self.body().view(torch.float32).fill_(float("nan"))
        self.ptr = self.raw.data_ptr() + GUARD

    def body(self):
        return self.raw[GUARD:GUARD + self.nbytes]

    def guards_intact(self):
        return bool((self.raw[:GUARD] == SENTINEL).all().item()) and bool((self.raw[GUARD + self.nbytes:] == SENTINEL).all().item())


def _axes(form):
    ndim = len(form.shape) - 1
    if form.axis_mask:
        return tuple(1 + a for a in range(ndim) if form.axis_mask >> a & 1)
    return tuple(range(1, ndim + 1))


def _input(form, in_layout, axes, rng):
    if form.half and form.inverse:
        # the half spectrum of real data, scaled to unit variance; DC and Nyquist bins of the last axis exactly real
        z = np.fft.rfftn(rng.standard_normal(form.shape), axes=axes) / np.sqrt(np.prod([form.shape[a] for a in axes]))
        z[..., 0] = z[..., 0].real
        if form.shape[-1] % 2 == 0:
            z[..., -1] = z[..., -1].real
        return np.stack([z.real, z.imag], axis=-1).astype(form.in_dtype)
    if form.in_dtype == U8:
        return rng.integers(0, 256, size=in_layout, dtype=np.uint8)
    return rng.standard_normal(in_layout).astype(form.in_dtype)


def _reference(form, xt, axes):
    """torch complex128 / float64 on the device: the float64 transform of the input xt (a device tensor)."""
    import torch
    xd = xt.to(torch.float64)
    if xd.numel() > BIG:
        if form.half and form.inverse:
            return torch.fft.irfftn(torch.view_as_complex(xd), s=[form.shape[a] for a in axes], dim=axes)
        if form.half:
            return torch.fft.rfftn(xd[..., 0], dim=axes)
        z = xd[..., 0].to(torch.complex128) if form.comps == 1 else torch.view_as_complex(xd)
        return (torch.fft.ifftn if form.inverse else torch.fft.fftn)(z, dim=axes)
    x = xd.cpu().numpy()
    if form.half and form.inverse:
        r = np.fft.irfftn(x[..., 0] + 1j * x[..., 1], s=[form.shape[a] for a in axes], axes=axes)
    elif form.half:
        r = np.fft.rfftn(x[..., 0], axes=axes)
    else:
        z = x[..., 0] if form.comps == 1 else x[..., 0] + 1j * x[..., 1]
        r = (np.fft.ifftn if form.inverse else np.fft.fftn)(z, axes=axes)
    return torch.from_numpy(r).cuda()


def _errors(form, got, want):
    """(relative L2, max-abs over max|X|) of the device output `got` (raw dtype view) against `want`."""
    import torch
    g = got.to(torch.float64)
    g = g[..., 0] if form.half and form.inverse else torch.view_as_complex(g)
    assert bool(torch.isfinite(g).all()), "non-finite output (unwritten elements or NaN arithmetic)"
    d = g - want
    l2 = (torch.linalg.vector_norm(d) / torch.linalg.vector_norm(want)).item()
    mx = (d.abs().max() / want.abs().max()).item()
    return l2, mx


def _plan(form):
    in_layout, out_layout = form.layouts()
    return b200fft.plan_fft(form.in_dtype, form.out_dtype, in_layout, out_layout, bases=form.bases, inverse=form.inverse,
                            real_mode=b200fft.REAL_HALF if form.half else b200fft.REAL_FULL, axis_mask=form.axis_mask,
                            flags=form.flags)


def _report(form, **kw):
    path = os.environ.get("B200FFT_FORMS_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(dict(id=form.id, **kw)) + "\n")


@pytest.mark.parametrize("form", RUNS, ids=[f.id for f in RUNS])
def test_rt_generic_form(monkeypatch, form):
    import torch
    for k, v in form.env.items():
        monkeypatch.setenv(k, v)
    expected = expected_lines(form)
    axes = _axes(form)
    in_layout, out_layout = form.layouts()
    odt = getattr(torch, form.out_dtype)
    out_numel = int(np.prod(out_layout))
    rng = np.random.default_rng(zlib.crc32(form.id.encode()))
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()

    plan = _plan(form)
    bufs = {}
    try:
        desc = plan.describe()
        lines = desc.strip().split("\n")
        assert len(lines) == len(expected), "%s: %d passes, the row has %s" % (desc, len(lines), form.kinds)
        for line, (kind, want_line) in zip(lines, expected):
            if want_line is None:
                assert "[NVRTC" in line, "%s: not a plan-time kernel: %s" % (kind, line)
            else:
                assert line == want_line, "plan: %s\nrules: %s" % (line, want_line)

        bufs["x"] = torch.from_numpy(_input(form, in_layout, axes, rng)).cuda()
        bufs["x0"] = bufs["x"].clone()
        bufs["out"] = Buf(out_numel * odt.itemsize)
        before = b200fft.launch_count()
        plan.exec(bufs["out"].ptr, bufs["x"])
        torch.cuda.synchronize()
        assert b200fft.launch_count() - before == plan.launches, desc
        assert bufs["out"].guards_intact(), "store outside the output array: %s" % desc
        assert torch.equal(bufs["x"], bufs["x0"]), "an out-of-place run changed its input: %s" % desc
        del bufs["x0"]
        got = bufs["out"].body().view(odt).view(out_layout)
        bufs["want"] = _reference(form, bufs["x"], axes)
        l2, mx = _errors(form, got, bufs["want"])
        del bufs["want"]
        peak = torch.cuda.max_memory_allocated()
        _report(form, rel_l2=l2, max_abs=mx, peak_bytes=peak, passes=lines)
        naxes = len(axes)
        if form.f64:
            assert l2 <= 1e-13 * np.sqrt(naxes), "rel-L2 %.2e vs float64: %s" % (l2, desc)
        else:
            assert l2 <= 2e-6 * np.sqrt(naxes) and mx <= 1e-5, "rel-L2 %.2e, max-abs %.2e vs float64: %s" % (l2, mx, desc)

        if not form.half and in_layout == out_layout and form.in_dtype == form.out_dtype:
            bufs["io"] = Buf(out_numel * odt.itemsize, fill_nan=False)
            bufs["io"].body().copy_(bufs["x"].view(-1).view(torch.uint8))
            plan.exec(bufs["io"].ptr, bufs["io"].ptr)
            torch.cuda.synchronize()
            assert bufs["io"].guards_intact(), "in place: store outside the array: %s" % desc
            assert torch.equal(bufs["io"].body(), bufs["out"].body()), "in place differs: %s" % desc
    finally:
        plan.destroy()
        bufs.clear()
        torch.cuda.empty_cache()


@pytest.mark.parametrize("form", REFUSED, ids=[f.id for f in REFUSED])
def test_refused_at_plan_creation(form):
    with pytest.raises(b200fft.B200FFTError) as e:
        _plan(form)
    assert e.value.status == 4 and form.refused in str(e.value), str(e.value)

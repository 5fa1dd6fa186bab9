"""Every row of the plan-time kernel table (tests/_jit_forms.py) on the GPU, against float64.

For each row:
  * the plan names the row's NVRTC kernels and no runtime-length or generic kernel; a probed row's full kernel names
    are what the host probe reports for the same axis (tests/test_host_jit_forms.py), so probe and planner agree;
  * fp32 output: relative L2 <= 2e-6 (two-pass and three-pass splits: 2.5e-6, as tests/test_gpu_long_axes.py) and
    max-abs <= 1e-5 * max|X|; fp64 output: relative L2 <= 1e-13. N-d rows multiply the relative L2 bound by
    sqrt(axes): each axis pass adds its own independent rounding. The reference is the float64 value of the actual
    input (numpy, or torch.fft in float64 on the device above 2^22 points);
  * the output is NaN-prefilled between 4 KB sentinel guard bands that must come back unchanged, an out-of-place run
    leaves its input unchanged, and the launch counter moves by plan.launches;
  * where the input and output layouts and dtypes match, an in-place run is bit-identical to the out-of-place one;
  * a second plan of the same problem has the same description and gives bit-identical output;
  * rows marked exec_host also run through exec_host, which cuts the batch into chunks;
  * scatter rows run b200fft_exec_scatter_at with virtual ranks on one GPU, bit-identical to the plain plan's output.

B200FFT_FORMS_REPORT=<file> appends one JSON line per row (kernel names, device memory) for the suite's statistics."""
import ctypes
import json
import os
import re
import zlib

import numpy as np
import pytest

import b200fft
from _jit_forms import FORMS, U8, logical_shape

pytestmark = pytest.mark.gpu

GUARD = 4096
SENTINEL = 0xA5
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

    def load(self, data):
        import torch
        self.body().copy_(torch.from_numpy(np.ascontiguousarray(data).reshape(-1).view(np.uint8)).cuda())

    def numpy(self, dtype):
        return self.body().cpu().numpy().view(dtype)

    def guards_intact(self):
        return bool((self.raw[:GUARD] == SENTINEL).all().item()) and bool((self.raw[GUARD + self.nbytes:] == SENTINEL).all().item())


def _layouts(shape, comps, half, inverse):
    if half:
        cplx = tuple(shape[:-1]) + (shape[-1] // 2 + 1, 2)
        real = tuple(shape) + (1,)
        return (cplx, real) if inverse else (real, cplx)
    return tuple(shape) + (comps,), tuple(shape) + (2,)


def _axes(form, shape):
    ndim = len(shape) - 1
    if form.axis_mask:
        return tuple(1 + a for a in range(ndim) if form.axis_mask >> a & 1)
    return tuple(range(1, ndim + 1))


def _input(form, shape, in_layout, axes, rng):
    if form.half and form.inverse:  # a Hermitian half spectrum: the transform of real data, scaled to unit variance
        z = np.fft.rfftn(rng.standard_normal(shape), axes=axes) / np.sqrt(np.prod([shape[a] for a in axes]))
        return np.stack([z.real, z.imag], axis=-1).astype(form.in_dtype)
    if form.in_dtype == U8:
        return rng.integers(0, 256, size=in_layout, dtype=np.uint8)
    return rng.standard_normal(in_layout).astype(form.in_dtype)


def _reference(form, x, axes, n_last):
    """float64 transform of the float64 value of the input x (in its own layout)."""
    xd = x.astype(np.float64)
    if xd.size > 2 ** 22 and not form.half:
        import torch
        t = torch.from_numpy(xd).cuda()
        z = t[..., 0].to(torch.complex128) if form.comps == 1 else torch.view_as_complex(t)
        del t
        r = (torch.fft.ifftn if form.inverse else torch.fft.fftn)(z, dim=axes)
        del z
        out = r.cpu().numpy()
        del r
        torch.cuda.empty_cache()
        return out
    if form.half and form.inverse:
        return np.fft.irfftn(xd[..., 0] + 1j * xd[..., 1], s=[n_last] if len(axes) == 1 else None, axes=axes)
    if form.half:
        return np.fft.rfftn(xd[..., 0], axes=axes)
    z = xd[..., 0] if form.comps == 1 else xd[..., 0] + 1j * xd[..., 1]
    return (np.fft.ifftn if form.inverse else np.fft.fftn)(z, axes=axes)


def _result(form, got):
    if form.half and form.inverse:
        return got[..., 0].astype(np.float64)
    return got[..., 0].astype(np.float64) + 1j * got[..., 1]


def _check_close(form, got, want, naxes, desc):
    assert np.isfinite(got).all(), "non-finite output (unwritten elements or NaN arithmetic): %s" % desc
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    split = any(k.startswith("jitsplit") for k in form.kinds)
    if form.f64:
        tol = 1e-13 * np.sqrt(naxes)
        assert err <= tol, "rel-L2 %.2e > %.1e vs float64: %s" % (err, tol, desc)
        return
    tol = (2.5e-6 if split else 2e-6) * np.sqrt(naxes)
    mx = np.abs(got - want).max() / np.abs(want).max()
    assert err <= tol and mx <= 1e-5, "rel-L2 %.2e (<= %.1e), max-abs %.2e vs float64: %s" % (err, tol, mx, desc)


def _names_kernels(desc, tag):
    if tag.endswith(("_", "(")):  # the leading part of a name
        return tag in desc
    return re.search(re.escape(tag) + r"(?![\w])", desc) is not None


def _plan(form, in_layout, out_layout):
    return b200fft.plan_fft(form.in_dtype, form.out_dtype, in_layout, out_layout, bases=form.bases, inverse=form.inverse,
                            real_mode=b200fft.REAL_HALF if form.half else b200fft.REAL_FULL, axis_mask=form.axis_mask,
                            flags=form.flags)


def _report(form, desc, peak):
    path = os.environ.get("B200FFT_FORMS_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps({"id": form.id, "kernels": sorted(set(re.findall(r"\bjit\w+", desc))), "peak_bytes": peak}) + "\n")


@pytest.mark.parametrize("form", FORMS, ids=[f.id for f in FORMS])
def test_jit_form(monkeypatch, form):
    import torch
    for k, v in form.env.items():
        monkeypatch.setenv(k, v)
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    shape = logical_shape(form)
    axes = _axes(form, shape)
    in_layout, out_layout = _layouts(shape, form.comps, form.half, form.inverse)
    rng = np.random.default_rng(zlib.crc32(form.id.encode()))
    x = _input(form, shape, in_layout, axes, rng)
    want = _reference(form, x, axes, shape[-1])
    odt = np.dtype(form.out_dtype)
    out_bytes = int(np.prod(out_layout)) * odt.itemsize

    plan = _plan(form, in_layout, out_layout)
    desc = plan.describe()
    try:
        assert "NVRTC" in desc and "rt_" not in desc and "generic" not in desc, desc
        for tag in form.tags:
            if not tag.startswith("jitscatter"):  # built on first exec_scatter; the description names the column pass
                assert _names_kernels(desc, tag), "%s is not in the plan: %s" % (tag, desc)
        xin = torch.from_numpy(x).cuda()
        x_before = xin.clone()
        out = Buf(out_bytes)
        before = b200fft.launch_count()
        plan.exec(out.ptr, xin)
        torch.cuda.synchronize()
        assert b200fft.launch_count() - before == plan.launches, desc
        assert out.guards_intact(), "store outside the output array: %s" % desc
        assert torch.equal(xin, x_before), "an out-of-place run changed its input: %s" % desc
        del x_before
        got = out.numpy(odt).reshape(out_layout)
        _check_close(form, _result(form, got), want, len(axes), desc)
        del want
        peak = torch.cuda.max_memory_allocated() + plan.workspace_bytes

        if in_layout == out_layout and np.dtype(form.in_dtype) == odt:
            io = Buf(out_bytes, fill_nan=False)
            io.load(x)
            plan.exec(io.ptr, io.ptr)
            torch.cuda.synchronize()
            assert io.guards_intact(), "in place: store outside the array: %s" % desc
            assert np.array_equal(io.numpy(odt).reshape(out_layout), got, equal_nan=False), "in place differs: %s" % desc
            del io
            peak = max(peak, torch.cuda.max_memory_allocated() + plan.workspace_bytes)

        if form.exec_host:
            h_out = np.full(out_layout, np.nan, dtype=odt)
            plan.exec_host(h_out, np.ascontiguousarray(x))
            assert np.array_equal(h_out, got), "exec_host differs from exec: %s" % desc

        if form.scatter:
            _check_scatter(form, plan, x, shape, got)
    finally:
        plan.destroy()

    again = _plan(form, in_layout, out_layout)  # the first plan is gone: its temporary does not add to this one's
    try:
        assert again.describe() == desc
        out2 = Buf(out_bytes)
        again.exec(out2.ptr, xin)
        torch.cuda.synchronize()
        assert np.array_equal(out2.numpy(odt).reshape(out_layout), got), "a second plan of the same problem differs: %s" % desc
    finally:
        again.destroy()
    _report(form, desc, peak)


def _check_scatter(form, plan, x, shape, got, G=2):
    """Virtual ranks on one GPU: the same slab `x` taken as each rank's planes in turn, scattered with z_first = r * zl,
    must land bit for bit where the plain plan's output has it (rows h * yl .. of the split axis on peer h)."""
    import torch
    zl, Y = shape[0], shape[1]
    yl = Y // G
    recv = [Buf(G * zl * yl * int(np.prod(shape[2:])) * 2 * np.dtype(form.out_dtype).itemsize) for _ in range(G)]
    xin = torch.from_numpy(x).cuda()
    work = Buf(got.nbytes, fill_nan=False)
    peers = (ctypes.c_void_p * G)(*[b.ptr for b in recv])
    for r in range(G):
        before = b200fft.launch_count()
        rc = b200fft.lib().b200fft_exec_scatter_at(plan._h, peers, G, r * zl, xin.data_ptr(), work.ptr, None)
        torch.cuda.synchronize()
        assert rc == 0, b200fft.lib().b200fft_last_error().decode()
        assert b200fft.launch_count() - before == 1
    for h in range(G):
        assert recv[h].guards_intact()
        slab = recv[h].numpy(np.dtype(form.out_dtype)).reshape((G * zl, yl) + tuple(shape[2:]) + (2,))
        for r in range(G):
            assert np.array_equal(slab[r * zl:(r + 1) * zl], got[:, h * yl:(h + 1) * yl]), "peer %d, rank %d" % (h, r)

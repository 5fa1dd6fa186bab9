"""Real-input and half-spectrum transforms of axes too long for one tile: two passes specialised at plan time
(csrc/jit.cu: jit_split_plan / make_jit_split_pass; kernels in csrc/fast.cuh), against numpy float64.

Forms: even-n R2C with the Hermitian unpack fused into pass B (rows_split_b_r2c_kernel), even-n C2R with the pack
fused into pass A (cols_split_a_c2r_kernel), odd-n R2C / C2R on the full n-point split, and real or dtype-cast input
with the full spectrum (cols_split_a_kernel<..., REAL>).
Tolerances: fp32 rel-L2 2.5e-6 and max-abs 1e-5 * max|X| (test_gpu_long_axes.py); fp64 rel-L2 1e-13."""
import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu

EVEN = [(3, 26000), (2, 30000), (2, 32768), (64, 65536), (1, 1 << 18), (1, 1 << 20), (2, 100000)]
ODD = [(2, 13125), (2, 15625), (1, 59049), (1, 78125)]


def _tdt(name):
    import torch
    return {"float32": torch.float32, "float64": torch.float64, "uint8": torch.uint8}[name]


def _check(got, want, f64=False):
    got = np.asarray(got, dtype=np.complex128 if np.iscomplexobj(got) else np.float64)
    rel = np.linalg.norm(got - want) / np.linalg.norm(want)
    mx = np.abs(got - want).max() / np.abs(want).max()
    if f64:
        assert rel <= 1e-13, rel
    else:
        assert rel <= 2.5e-6 and mx <= 1e-5, (rel, mx)


def _cplx(a):
    return a[..., 0].astype(np.float64) + 1j * a[..., 1].astype(np.float64)


def _run(x, out_shape, out_dtype="float32", **kw):
    """Plan, run once on the GPU, check the input is untouched; returns (output as numpy, plan facts)."""
    import torch
    xt = torch.from_numpy(x).cuda()
    keep = xt.clone()
    out = torch.full(out_shape, float("nan"), dtype=_tdt(out_dtype), device="cuda")
    plan = b200fft.plan_fft(str(x.dtype), out_dtype, x.shape, out_shape, **kw)
    b200fft.fft(out, xt, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(xt, keep)
    facts = dict(desc=plan.describe(), launches=plan.launches, ws=plan.workspace_bytes, bases=plan.bases(0))
    plan.destroy()
    return out.cpu().numpy(), facts


def _r2c(x, out_dtype="float32", **kw):
    shape = x.shape[:-1]
    return _run(x, shape[:-1] + (shape[-1] // 2 + 1, 2), out_dtype, real_mode=b200fft.REAL_HALF, **kw)


def _c2r(X, n, out_dtype="float32", **kw):
    return _run(X, X.shape[:-2] + (n, 1), out_dtype, real_mode=b200fft.REAL_HALF, inverse=True, **kw)


def _half_spectrum(rng, shape, dtype=np.float32):
    """A valid half spectrum: rfft of a random real signal (DC and Nyquist bins real)."""
    X = np.fft.rfft(rng.standard_normal(shape), axis=-1)
    return np.stack([X.real, X.imag], axis=-1).astype(dtype)


@pytest.mark.parametrize("shape", EVEN)
def test_r2c_even(shape):
    rng = np.random.default_rng(shape[1])
    x = rng.standard_normal(shape + (1,)).astype(np.float32)
    got, f = _r2c(x)
    _check(_cplx(got), np.fft.rfft(x[..., 0].astype(np.float64), axis=-1))
    assert "split n=%d r2c" % shape[1] in f["desc"] and "jitsplitBr2c" in f["desc"] and "generic" not in f["desc"], f["desc"]
    assert f["launches"] == 2
    assert f["ws"] >= shape[0] * (shape[1] // 2) * 8  # the temporary of H complex values per transform


@pytest.mark.parametrize("shape", EVEN)
def test_c2r_even(shape):
    rng = np.random.default_rng(shape[1] + 1)
    X = _half_spectrum(rng, shape)
    got, f = _c2r(X, shape[1])
    _check(got[..., 0], np.fft.irfft(_cplx(X), n=shape[1], axis=-1))
    assert "split n=%d c2r" % shape[1] in f["desc"] and "jitsplitAc2r" in f["desc"] and "generic" not in f["desc"], f["desc"]
    assert f["launches"] == 2
    assert f["ws"] >= shape[0] * (shape[1] // 2) * 8


@pytest.mark.parametrize("shape", ODD)
def test_r2c_c2r_odd(shape):
    """13125 used to fall through to the runtime-length / generic kernels; the others were refused."""
    rng = np.random.default_rng(shape[1])
    x = rng.standard_normal(shape + (1,)).astype(np.float32)
    got, f = _r2c(x)
    _check(_cplx(got), np.fft.rfft(x[..., 0].astype(np.float64), axis=-1))
    assert "jitsplitBhalf" in f["desc"] and "generic" not in f["desc"] and f["launches"] == 2, f["desc"]
    X = _half_spectrum(rng, shape)
    got, f = _c2r(X, shape[1])
    _check(got[..., 0], np.fft.irfft(_cplx(X), n=shape[1], axis=-1))
    assert "jitsplitAc2rodd" in f["desc"] and "jitsplitBreal" in f["desc"] and f["launches"] == 2, f["desc"]


@pytest.mark.parametrize("shape", [(2, 12000), (1, 1 << 18)])
def test_f64(shape):
    rng = np.random.default_rng(7)
    x = rng.standard_normal(shape + (1,))
    got, f = _r2c(x, "float64")
    _check(_cplx(got), np.fft.rfft(x[..., 0], axis=-1), f64=True)
    assert "jitsplitBr2c" in f["desc"] and "_f64" in f["desc"], f["desc"]
    X = _half_spectrum(rng, shape, np.float64)
    got, f = _c2r(X, shape[1], "float64")
    _check(got[..., 0], np.fft.irfft(_cplx(X), n=shape[1], axis=-1), f64=True)
    assert "jitsplitAc2r" in f["desc"] and "_f64" in f["desc"], f["desc"]


def test_f64_input_f32_output_r2c():
    rng = np.random.default_rng(8)
    x = rng.standard_normal((2, 1 << 18, 1))
    got, f = _r2c(x, "float32")
    _check(_cplx(got), np.fft.rfft(x[..., 0], axis=-1))
    assert "_inf64" in f["desc"] and "jitsplitBr2c" in f["desc"], f["desc"]


@pytest.mark.parametrize("dtype", ["float32", "uint8", "float64"])
@pytest.mark.parametrize("inverse", [False, True])
def test_real_full(dtype, inverse):
    rng = np.random.default_rng(9)
    shape = (2, 1 << 18)
    x = (rng.integers(0, 256, size=shape + (1,)) if dtype == "uint8" else rng.standard_normal(shape + (1,))).astype(dtype)
    got, f = _run(x, shape + (2,), inverse=inverse)
    xd = x[..., 0].astype(np.float64)
    _check(_cplx(got), np.fft.ifft(xd, axis=-1) if inverse else np.fft.fft(xd, axis=-1))
    assert "real-in" in f["desc"] and "_realin" in f["desc"] and f["launches"] == 2, f["desc"]


def test_complex_uint8_input():
    rng = np.random.default_rng(10)
    x = rng.integers(0, 256, size=(3, 30000, 2), dtype=np.uint8)
    got, f = _run(x, x.shape)
    _check(_cplx(got), np.fft.fft(_cplx(x), axis=-1))
    assert "split n=30000" in f["desc"] and "_inu8" in f["desc"], f["desc"]


def test_nd_long_last_axis():
    """R2C: the strided passes run over the half spectrum the split wrote; C2R: they fill the workspace it reads."""
    rng = np.random.default_rng(11)
    shape = (2, 3, 1 << 16)
    x = rng.standard_normal(shape + (1,)).astype(np.float32)
    got, f = _r2c(x)
    _check(_cplx(got), np.fft.rfftn(x[..., 0].astype(np.float64), axes=(1, 2)))
    assert "jitsplitBr2c" in f["desc"], f["desc"]
    X = np.fft.rfftn(rng.standard_normal(shape), axes=(1, 2))
    Xs = np.stack([X.real, X.imag], axis=-1).astype(np.float32)
    got, f = _c2r(Xs, shape[-1])
    _check(got[..., 0], np.fft.irfftn(_cplx(Xs), s=shape[1:], axes=(1, 2)))
    assert "jitsplitAc2r" in f["desc"] and f["ws"] >= 2 * 3 * (shape[-1] // 2 + 1) * 8, f["desc"]


def test_nd_real_full():
    rng = np.random.default_rng(12)
    shape = (2, 4, 40000)
    x = rng.standard_normal(shape + (1,)).astype(np.float32)
    got, f = _run(x, shape + (2,))
    _check(_cplx(got), np.fft.fftn(x[..., 0].astype(np.float64), axes=(1, 2)))
    assert "split n=40000 real-in" in f["desc"], f["desc"]


def test_round_trip():
    rng = np.random.default_rng(13)
    n = 1 << 20
    x = rng.standard_normal((2, n, 1)).astype(np.float32)
    X, _ = _r2c(x)
    y, _ = _c2r(X, n)
    rel = np.linalg.norm(y - x) / np.linalg.norm(x)
    assert rel < 2.5e-6, rel


def test_user_bases_honoured():
    rng = np.random.default_rng(14)
    n = 1 << 20
    bases = [8] * 6 + [4]
    x = rng.standard_normal((1, n, 1)).astype(np.float32)
    got, f = _r2c(x, bases=[bases])
    _check(_cplx(got), np.fft.rfft(x[..., 0].astype(np.float64), axis=-1))
    assert f["bases"] == b200fft.ordered_bases(n, bases), (f["bases"], bases)
    assert "user stages=[%s]" % ",".join(str(b) for b in f["bases"]) in f["desc"], f["desc"]
    assert "jitsplitBr2c512_8x8x8" in f["desc"], f["desc"]


def test_exec_host_long_r2c():
    rng = np.random.default_rng(15)
    n = 1 << 18
    x = rng.standard_normal((3, n, 1)).astype(np.float32)
    out_shape = (3, n // 2 + 1, 2)
    h_out = np.full(out_shape, np.nan, dtype=np.float32)
    plan = b200fft.plan_fft("float32", "float32", x.shape, out_shape, real_mode=b200fft.REAL_HALF)
    plan.exec_host(h_out, x)
    desc = plan.describe()
    plan.destroy()
    _check(_cplx(h_out), np.fft.rfft(x[..., 0].astype(np.float64), axis=-1))
    assert "jitsplitBr2c" in desc, desc


@pytest.mark.parametrize("n,kw,out_dtype", [(24000, dict(real_mode=1), "float32"),    # R2C on one tile
                                            (22000, dict(real_mode=0), "float32"),    # real input, full spectrum
                                            (12005, dict(real_mode=1), "float32"),    # odd R2C
                                            (10000, dict(real_mode=1), "float64")])   # fp64 R2C
def test_single_tile_plans_unchanged(n, kw, out_dtype):
    """Lengths a single-tile kernel serves keep that kernel: the split only takes what no tile can."""
    rng = np.random.default_rng(n)
    x = rng.standard_normal((2, n, 1)).astype(out_dtype)
    if kw["real_mode"] == 1:
        got, f = _r2c(x, out_dtype)
        want = np.fft.rfft(x[..., 0].astype(np.float64), axis=-1)
    else:
        got, f = _run(x, (2, n, 2), out_dtype)
        want = np.fft.fft(x[..., 0].astype(np.float64), axis=-1)
    _check(_cplx(got), want, f64=out_dtype == "float64")
    assert "split" not in f["desc"] and "generic" not in f["desc"] and f["launches"] == 1, f["desc"]

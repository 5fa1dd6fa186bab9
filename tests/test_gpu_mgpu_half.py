"""Half-spectrum (REAL_HALF) and fp64 forms of the slab decomposition (b200fft_mgpu_*, MGPU_SLAB) and the per-rank
scattering store of forward half-spectrum plans (b200fft_exec_scatter / _at).

The forward R2C takes real z planes and leaves Y-slabs of the X/2+1-bin spectrum; the inverse C2R takes exactly those
Y-slabs and returns real z planes, so the two round-trip on the device buffers. The inverse's Z pass stores into the
owning peers' receive buffers (the reverse exchange, a kernel form only the plan-time tier builds: "jitscatterZ").

On a one-GPU box the slots are virtual (all on cuda:0; B200FFT_MGPU_ALLOW_SAME_DEVICE lets the slab mode name a device
twice); with more GPUs visible the same cases run on distinct devices over peer access. Checked against numpy float64:
relative L2 <= 2e-6 in fp32 (DESIGN.md section 2), <= 1e-13 x sqrt(3) in fp64."""
import ctypes

import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu


def _tol(work):
    return 2e-6 if work == "float32" else 1e-13 * np.sqrt(3)


def _devices(n, monkeypatch):
    import torch
    have = torch.cuda.device_count()
    if have < n:
        monkeypatch.setenv("B200FFT_MGPU_ALLOW_SAME_DEVICE", "1")
    return [g % have for g in range(n)]


def _rel(got, want):
    return float(np.linalg.norm(got - want) / np.linalg.norm(want))


def _c(a):
    a = np.asarray(a, dtype=np.float64)
    return a[..., 0] + 1j * a[..., 1]


def _pairs(z, dtype):
    return np.stack([z.real, z.imag], axis=-1).astype(dtype)


def _dev(a, d):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda", d))


def _nan(shape, dtype, d):
    import torch
    return torch.full(shape, float("nan"), dtype=getattr(torch, dtype), device=torch.device("cuda", d))


def _volume(dims, dtype, seed):
    return np.random.default_rng(seed).standard_normal(dims).astype(dtype)


HALF_CASES = [
    ((64, 64, 64), 1, "float32", "float32"),
    ((64, 64, 64), 2, "float32", "float32"),
    ((128, 128, 64), 4, "float32", "float32"),
    ((64, 128, 256), 8, "float32", "float32"),
    ((48, 40, 100), 2, "float32", "float32"),   # Y = 40 and the 50-point R2C core of X = 100 have no registered variant
    ((24, 40, 45), 4, "float32", "float32"),    # odd X
    ((256, 256, 256), 4, "float32", "float32"),
    ((64, 64, 64), 2, "float64", "float32"),    # fp64 input cast on load
    ((64, 64, 64), 2, "float64", "float64"),
    ((48, 40, 100), 2, "float64", "float64"),
]


@pytest.mark.parametrize("dims,G,in_dtype,work", HALF_CASES)
def test_half_slab_forward_inverse_roundtrip(dims, G, in_dtype, work, monkeypatch):
    devs = _devices(G, monkeypatch)
    Z, Y, X = dims
    W, zl, yl = X // 2 + 1, Z // G, Y // G
    real_lay, cplx_lay = (1, Z, Y, X, 1), (1, Z, Y, W, 2)
    isz, wsz = np.dtype(in_dtype).itemsize, np.dtype(work).itemsize
    tol = _tol(work)
    x = _volume(dims, in_dtype, 3)
    want = np.fft.rfftn(x.astype(np.float64))

    # ---- forward: real z planes -> Y-slabs of the half spectrum
    fwd = b200fft.MgpuPlan(in_dtype, work, real_lay, cplx_lay, devices=devs, mode=b200fft.MGPU_SLAB,
                           real_mode=b200fft.REAL_HALF)
    text = fwd.describe()
    assert "half spectrum" in text and "R2C" in text and "scattering Y stores" in text and "event barrier" in text, text
    ins = [_dev(x[g * zl:(g + 1) * zl], devs[g]) for g in range(G)]
    outs = [_nan((Z, yl, W, 2), work, devs[g]) for g in range(G)]
    for g in range(G):
        assert fwd.shard(g) == (g * zl, zl)
        assert fwd.in_bytes(g) == zl * Y * X * isz and fwd.out_bytes(g) == Z * yl * W * 2 * wsz
    import torch
    torch.cuda.synchronize()
    for _ in range(3):  # back-to-back calls: the `done` events keep call k+1's stores out of call k's Z pass
        fwd.exec(outs, ins)
    fwd.synchronize()
    for h in range(G):
        got = outs[h].cpu().numpy()
        assert np.isfinite(got).all()
        assert _rel(_c(got), want[:, h * yl:(h + 1) * yl]) <= tol, h
        assert np.array_equal(ins[h].cpu().numpy(), x[h * zl:(h + 1) * zl])  # inputs untouched
    h_out = np.full((Z, Y, W, 2), np.nan, dtype=work)
    fwd.exec_host(h_out, x)  # natural order in, natural order out
    assert _rel(_c(h_out), want) <= tol

    # ---- inverse: the Y-slabs of a spectrum -> real z planes, scaled by 1 / (Z Y X)
    inv = b200fft.MgpuPlan(work, work, cplx_lay, real_lay, devices=devs, mode=b200fft.MGPU_SLAB,
                           real_mode=b200fft.REAL_HALF, inverse=True)
    text = inv.describe()
    assert "half spectrum inverse" in text and "C2R" in text and "jitscatterZ" in text and "event barrier" in text, text
    spec = _pairs(want, work)
    want_inv = np.fft.irfftn(_c(spec), s=dims, axes=(0, 1, 2))
    sin = [_dev(spec[:, g * yl:(g + 1) * yl], devs[g]) for g in range(G)]
    sout = [_nan((zl, Y, X), work, devs[g]) for g in range(G)]
    for g in range(G):
        assert inv.shard(g) == (g * yl, yl)
        assert inv.in_bytes(g) == Z * yl * W * 2 * wsz and inv.out_bytes(g) == zl * Y * X * wsz
    torch.cuda.synchronize()
    for _ in range(3):
        inv.exec(sout, sin)
    inv.synchronize()
    for g in range(G):
        got = sout[g].cpu().numpy().astype(np.float64)
        assert np.isfinite(got).all()
        assert _rel(got, want_inv[g * zl:(g + 1) * zl]) <= tol, g
        assert np.array_equal(sin[g].cpu().numpy(), spec[:, g * yl:(g + 1) * yl])  # the inverse never writes its input
    h_back = np.full(dims, np.nan, dtype=work)
    inv.exec_host(h_back, spec)
    assert _rel(h_back.astype(np.float64), want_inv) <= tol

    # ---- forward then inverse on the device buffers: no redistribution in between
    for g in range(G):
        sout[g].fill_(float("nan"))
    torch.cuda.synchronize()
    inv.exec(sout, outs)
    inv.synchronize()
    back = np.concatenate([t.cpu().numpy().astype(np.float64) for t in sout])
    assert _rel(back, x.astype(np.float64)) <= tol
    fwd.destroy()
    inv.destroy()


@pytest.mark.parametrize("inverse", [False, True])
def test_complex_fp64_slab(inverse, monkeypatch):
    import torch
    G, (Z, Y, X) = 2, (64, 48, 40)
    devs = _devices(G, monkeypatch)
    zl, yl = Z // G, Y // G
    lay = (1, Z, Y, X, 2)
    plan = b200fft.MgpuPlan("float64", "float64", lay, lay, devices=devs, mode=b200fft.MGPU_SLAB, inverse=inverse)
    x = np.random.default_rng(7).standard_normal((Z, Y, X, 2))
    want = np.fft.ifftn(_c(x)) if inverse else np.fft.fftn(_c(x))
    ins = [_dev(x[g * zl:(g + 1) * zl], devs[g]) for g in range(G)]
    outs = [_nan((Z, yl, X, 2), "float64", devs[g]) for g in range(G)]
    for g in range(G):
        assert plan.shard(g) == (g * zl, zl)
        assert plan.in_bytes(g) == zl * Y * X * 16 and plan.out_bytes(g) == Z * yl * X * 16
    torch.cuda.synchronize()
    for _ in range(3):
        plan.exec(outs, ins)
    plan.synchronize()
    for h in range(G):
        assert _rel(_c(outs[h].cpu().numpy()), want[:, h * yl:(h + 1) * yl]) <= _tol("float64")
        assert np.array_equal(ins[h].cpu().numpy(), x[h * zl:(h + 1) * zl])
    h_out = np.full((Z, Y, X, 2), np.nan)
    plan.exec_host(h_out, x)
    assert _rel(_c(h_out), want) <= _tol("float64")
    plan.destroy()


def _create_status(in_dtype, out_dtype, in_lay, out_lay, ngpu, *, inverse=False, real_mode=b200fft.REAL_HALF, axis_mask=0):
    d, keep = b200fft._make_desc(in_dtype, out_dtype, in_lay, out_lay, None, inverse, real_mode, axis_mask, None, 0)
    h = ctypes.c_void_p()
    devs = (ctypes.c_int * ngpu)(*([0] * ngpu))
    rc = b200fft.lib().b200fft_mgpu_plan_create(ctypes.byref(h), ctypes.byref(d), ngpu, devs, b200fft.MGPU_SLAB)
    if rc == 0:
        b200fft.lib().b200fft_mgpu_plan_destroy(h)
    return rc, b200fft.lib().b200fft_last_error().decode()


def test_half_slab_refusals(monkeypatch):
    monkeypatch.setenv("B200FFT_MGPU_ALLOW_SAME_DEVICE", "1")
    real, cplx = (1, 64, 64, 64, 1), (1, 64, 64, 33, 2)
    assert _create_status("float32", "float32", (2,) + real[1:], (2,) + cplx[1:], 1)[0] == 4      # batch 2
    assert _create_status("float32", "float32", real, cplx, 1, axis_mask=3)[0] == 4                # not all axes
    assert _create_status("float32", "float32", real, (1, 64, 64, 64, 2), 1,
                          real_mode=b200fft.REAL_FULL)[0] == 4                                      # real, full spectrum
    assert _create_status("uint8", "float32", real, cplx, 1)[0] == 4           # uint8: as the single-device R2C plan
    rc, why = _create_status("float32", "float32", (1, 2, 8192, 4, 1), (1, 2, 8192, 3, 2), 2)     # Y longer than a tile
    assert rc == 4, why
    rc, why = _create_status("float32", "float32", (1, 4096, 4, 3, 2), (1, 4096, 4, 4, 1), 2, inverse=True)  # Z too long
    assert rc == 4 and "column tile" in why, why
    for inverse in (False, True):
        for dims in ((66, 64, 64), (64, 66, 64)):  # Z, then Y, not divisible by 4 devices
            r, c = (1,) + dims + (1,), (1, dims[0], dims[1], dims[2] // 2 + 1, 2)
            lay = (c, r) if inverse else (r, c)
            assert _create_status("float32", "float32", *lay, 4, inverse=inverse)[0] == 1, (dims, inverse)


def _r2c_plan(dims, dtype):
    zl, Y, X = dims
    return b200fft.plan_fft(dtype, dtype, (zl, Y, X, 1), (zl, Y, X // 2 + 1, 2), real_mode=b200fft.REAL_HALF,
                            flags=b200fft.FLAG_NO_FUSED)


def test_exec_scatter_half_refusals():
    import torch
    plan = _r2c_plan((2, 64, 64), "float32")
    x = torch.zeros((2, 64, 64), device="cuda")
    work = torch.zeros((2, 64, 33, 2), device="cuda")
    peers = [torch.zeros((2, 32, 33, 2), device="cuda") for _ in range(2)]
    with pytest.raises(b200fft.B200FFTError) as e:  # d_work receives the half spectrum: it cannot be the real input
        plan.exec_scatter(peers, 0, x, x)
    assert e.value.status == 1
    plan.exec_scatter(peers, 0, x, work)
    torch.cuda.synchronize()
    plan.destroy()
    c2r = b200fft.plan_fft("float32", "float32", (2, 64, 33, 2), (2, 64, 64, 1), real_mode=b200fft.REAL_HALF, inverse=True,
                           flags=b200fft.FLAG_NO_FUSED)
    with pytest.raises(b200fft.B200FFTError) as e:
        c2r.exec_scatter(peers, 0, work, work)
    assert e.value.status == 4
    c2r.destroy()


@pytest.mark.parametrize("dims,dtype", [((3, 64, 64), "float32"), ((3, 40, 45), "float32"), ((2, 48, 100), "float32"),
                                        ((3, 64, 64), "float64")])
def test_exec_scatter_at_r2c_matches_plain_plan(dims, dtype):
    """Virtual ranks on one GPU: the same real slab taken as each rank's planes in turn, scattered with z_first = r * zl,
    must land bit for bit where the plain R2C plan's output has it (rows h * yl .. of the split axis on peer h)."""
    import torch
    G = 2
    zl, Y, X = dims
    W, yl = X // 2 + 1, Y // 2
    plan = _r2c_plan(dims, dtype)
    x = _volume(dims, dtype, 11)
    xin = _dev(x, 0)
    plain = _nan((zl, Y, W, 2), dtype, 0)
    plan.exec(plain, xin)
    torch.cuda.synchronize()
    got = plain.cpu().numpy()
    assert _rel(_c(got), np.fft.rfftn(x.astype(np.float64), axes=(1, 2))) <= _tol(dtype)
    recv = [_nan((G * zl, yl, W, 2), dtype, 0) for _ in range(G)]
    work = _nan((zl, Y, W, 2), dtype, 0)
    peers = (ctypes.c_void_p * G)(*[t.data_ptr() for t in recv])
    for r in range(G):
        before = b200fft.launch_count()
        rc = b200fft.lib().b200fft_exec_scatter_at(plan._h, peers, G, r * zl, xin.data_ptr(), work.data_ptr(), None)
        torch.cuda.synchronize()
        assert rc == 0, b200fft.lib().b200fft_last_error().decode()
        assert b200fft.launch_count() - before == plan.launches
    for h in range(G):
        slab = recv[h].cpu().numpy()
        for r in range(G):
            assert np.array_equal(slab[r * zl:(r + 1) * zl], got[:, h * yl:(h + 1) * yl]), "peer %d, rank %d" % (h, r)
    assert np.array_equal(xin.cpu().numpy(), x)
    plan.destroy()

"""Multi-device entry points of the C ABI (b200fft_mgpu_*, include/b200fft.h): one process drives several device
slots. On a one-GPU box the slots are virtual (all on cuda:0; B200FFT_MGPU_ALLOW_SAME_DEVICE lets the slab mode name
a device twice), which exercises the sharding, the peer indexing of the scattering stores, the cross-stream event
barrier and the host gather; with more GPUs visible the same cases run on distinct devices over peer access.
Checked against numpy float64 at the stated fp32 tolerance (DESIGN.md section 2: relative L2 <= 2e-6)."""
import os

import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu
TOL = 2e-6


def _devices(n):
    import torch
    have = torch.cuda.device_count()
    return [g % have for g in range(n)], have >= n


def _rel(got, want):
    return float(np.linalg.norm(got - want) / np.linalg.norm(want))


@pytest.mark.parametrize("shape,ngpu", [((10, 1024), 1), ((10, 1024), 4), ((7, 93), 3), ((13, 64, 64, 64), 2),
                                        ((6, 640, 480), 4), ((100, 128), 8)])
def test_batch_shard_device_and_host(shape, ngpu):
    import torch
    devs, real = _devices(ngpu)
    layout = shape + (2,)
    plan = b200fft.MgpuPlan("float32", "float32", layout, layout, devices=devs, mode=b200fft.MGPU_BATCH_SHARD)
    assert plan.ngpu == ngpu and "no communication" in plan.describe()
    rng = np.random.default_rng(5)
    x = rng.standard_normal(layout).astype(np.float32)
    want = np.fft.fftn(x[..., 0].astype(np.float64) + 1j * x[..., 1], axes=tuple(range(1, len(shape))))
    # device path: each slot gets its own share of the batch
    ins, outs, covered = [], [], 0
    for g in range(ngpu):
        first, count = plan.shard(g)
        assert (first, count) == b200fft.mgpu_split(shape[0], ngpu, g) and first == covered
        covered += count
        dev = torch.device("cuda", devs[g])
        ins.append(torch.from_numpy(x[first:first + count]).to(dev))
        outs.append(torch.full_like(ins[-1], float("nan")))
        assert plan.in_bytes(g) == ins[-1].numel() * 4 and plan.out_bytes(g) == outs[-1].numel() * 4
    assert covered == shape[0]
    torch.cuda.synchronize()
    before = b200fft.launch_count()
    plan.exec(outs, ins)
    plan.synchronize()
    assert b200fft.launch_count() >= before + ngpu
    got = np.concatenate([o.cpu().numpy() for o in outs]).astype(np.float64)
    assert _rel(got[..., 0] + 1j * got[..., 1], want) < TOL
    # host path: the whole job in one host array
    h_out = np.full(layout, np.nan, dtype=np.float32)
    plan.exec_host(h_out, x)
    assert _rel(h_out[..., 0].astype(np.float64) + 1j * h_out[..., 1], want) < TOL
    plan.destroy()


@pytest.mark.parametrize("dims,ngpu,inverse", [((64, 64, 64), 1, False), ((64, 64, 64), 2, False), ((128, 128, 64), 4, False),
                                               ((64, 128, 256), 8, False), ((128, 64, 96), 2, True), ((256, 256, 256), 4, False)])
def test_slab_device_and_host(dims, ngpu, inverse, monkeypatch):
    import torch
    devs, real = _devices(ngpu)
    if not real:
        monkeypatch.setenv("B200FFT_MGPU_ALLOW_SAME_DEVICE", "1")
    Z, Y, X = dims
    zl, yl = Z // ngpu, Y // ngpu
    layout = (1, Z, Y, X, 2)
    plan = b200fft.MgpuPlan("float32", "float32", layout, layout, devices=devs, mode=b200fft.MGPU_SLAB, inverse=inverse)
    assert "event barrier" in plan.describe()
    rng = np.random.default_rng(11)
    x = rng.standard_normal((Z, Y, X, 2)).astype(np.float32)
    xc = x[..., 0].astype(np.float64) + 1j * x[..., 1]
    want = np.fft.ifftn(xc) if inverse else np.fft.fftn(xc)
    ins = [torch.from_numpy(x[g * zl:(g + 1) * zl]).to(torch.device("cuda", devs[g])) for g in range(ngpu)]
    outs = [torch.full((Z, yl, X, 2), float("nan"), device=torch.device("cuda", devs[g])) for g in range(ngpu)]
    for g in range(ngpu):
        assert plan.shard(g) == (g * zl, zl)
        assert plan.in_bytes(g) == ins[g].numel() * 4 and plan.out_bytes(g) == outs[g].numel() * 4
    torch.cuda.synchronize()
    for rep in range(3):  # back-to-back calls: the `done` events keep call k+1's stores out of call k's Z pass
        plan.exec(outs, ins)
    plan.synchronize()
    for h in range(ngpu):
        got = outs[h].cpu().numpy().astype(np.float64)
        assert np.isfinite(got).all()
        assert _rel(got[..., 0] + 1j * got[..., 1], want[:, h * yl:(h + 1) * yl, :]) < TOL
        assert np.array_equal(ins[h].cpu().numpy(), x[h * zl:(h + 1) * zl])  # inputs untouched
    h_out = np.full((Z, Y, X, 2), np.nan, dtype=np.float32)
    plan.exec_host(h_out, x)  # natural order in, natural order out
    assert _rel(h_out[..., 0].astype(np.float64) + 1j * h_out[..., 1], want) < TOL
    plan.destroy()


def test_mgpu_user_bases_reach_every_axis():
    devs, real = _devices(2)
    if not real:
        os.environ["B200FFT_MGPU_ALLOW_SAME_DEVICE"] = "1"
    try:
        plan = b200fft.MgpuPlan("float32", "float32", (1, 64, 64, 64, 2), (1, 64, 64, 64, 2), devices=devs,
                                mode=b200fft.MGPU_SLAB, bases=[[4], [8], [2]])
        text = plan.describe()
        assert "2,2,2,2,2,2" in text and "8,8" in text and "4,4,4" in text, text
        plan.destroy()
    finally:
        os.environ.pop("B200FFT_MGPU_ALLOW_SAME_DEVICE", None)


def test_mgpu_errors():
    import torch
    lay = (1, 64, 64, 64, 2)
    with pytest.raises(b200fft.B200FFTError):   # 64 planes do not split over 3 devices
        b200fft.MgpuPlan("float32", "float32", lay, lay, devices=[0, 0, 0], mode=b200fft.MGPU_SLAB)
    with pytest.raises(b200fft.B200FFTError) as e:   # slab mode is one complex transform
        b200fft.MgpuPlan("float32", "float32", (2, 64, 64, 64, 2), (2, 64, 64, 64, 2), devices=[0], mode=b200fft.MGPU_SLAB)
    assert e.value.status == 4
    with pytest.raises(b200fft.B200FFTError):   # no such device
        b200fft.MgpuPlan("float32", "float32", (8, 64, 2), (8, 64, 2), devices=[torch.cuda.device_count()])
    with pytest.raises(b200fft.B200FFTError):   # more devices than batch items
        b200fft.MgpuPlan("float32", "float32", (2, 64, 2), (2, 64, 2), devices=[0, 0, 0])
    with pytest.raises(b200fft.B200FFTError) as e:   # the single-device layout rules still apply
        b200fft.MgpuPlan("float32", "float32", (8, 64, 3), (8, 64, 2), devices=[0])
    assert e.value.status == 2
    if torch.cuda.device_count() < 2:
        os.environ.pop("B200FFT_MGPU_ALLOW_SAME_DEVICE", None)
        with pytest.raises(b200fft.B200FFTError):   # the same device named twice in slab mode
            b200fft.MgpuPlan("float32", "float32", lay, lay, devices=[0, 0], mode=b200fft.MGPU_SLAB)

"""Slab decomposition on ONE GPU: G virtual ranks emulated in one process (their slabs all live on
cuda:0), exercising b200fft_exec_scatter's peer indexing for G > 1 and the Z pass, against numpy.
The real multi-process / multi-GPU run is tools/slab_check.py (torchrun, NCCL + CUDA IPC)."""
import ctypes

import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dims,G", [((64, 64, 64), 2), ((128, 128, 64), 4), ((64, 128, 128), 8), ((512, 512, 16), 2),
                                    ((64, 64, 64), 1)])
def test_exec_scatter_virtual_ranks(dims, G):
    import torch
    Z, Y, X = dims
    zl, yl = Z // G, Y // G
    g = torch.Generator(device="cuda").manual_seed(3)
    full = torch.randn((Z, Y, X, 2), generator=g, device="cuda")
    recv = [torch.full((Z, yl, X, 2), float("nan"), device="cuda") for _ in range(G)]
    plan2d = b200fft.plan_fft("float32", "float32", (zl, Y, X, 2), (zl, Y, X, 2),
                              flags=b200fft.FLAG_NO_FUSED)      # exec_scatter drives per-axis passes (include/b200fft.h)
    planz = b200fft.plan_fft("float32", "float32", (1, Z, yl, X, 2), (1, Z, yl, X, 2), axis_mask=1)
    work = torch.empty((zl, Y, X, 2), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for r in range(G):
        x_local = full[r * zl:(r + 1) * zl].contiguous()
        keep = x_local.clone()
        plan2d.exec_scatter(recv, r, x_local, work, st)
        assert torch.equal(x_local, keep)          # input untouched when d_work != d_in
    for r in range(G):
        b200fft.fft(recv[r].unsqueeze(0), recv[r].unsqueeze(0), plan=planz)
    torch.cuda.synchronize()
    want = torch.fft.fftn(torch.view_as_complex(full.double().contiguous()))
    for r in range(G):
        got = torch.view_as_complex(recv[r].double().contiguous())
        ref = want[:, r * yl:(r + 1) * yl, :]
        assert torch.isfinite(recv[r]).all()
        assert float((got - ref).norm() / ref.norm()) < 2e-6


def _scatter_at(plan, recv, z_first, x, work, st):
    arr = (ctypes.c_void_p * len(recv))(*[t.data_ptr() for t in recv])
    return b200fft.lib().b200fft_exec_scatter_at(plan._h, arr, len(recv), z_first, x.data_ptr(), work.data_ptr(), st)


@pytest.mark.parametrize("dims,G,pieces", [((64, 64, 64), 2, 4), ((128, 128, 64), 4, 2), ((64, 128, 256), 8, 8),
                                           ((96, 64, 64), 1, 3)])
@pytest.mark.parametrize("axis_mask", [0, 1])  # 1: only the split axis Y, a one-pass plan that scatters from its input
def test_exec_scatter_at_virtual_ranks(dims, G, pieces, axis_mask):
    """b200fft_exec_scatter_at with z_first = r * zl stores bit for bit what exec_scatter with my_rank = r stores, and
    so does the same rank's slab cut into `pieces` sub-ranges of planes, each scattered at its own z_first."""
    import torch
    Z, Y, X = dims
    zl, yl, zc = Z // G, Y // G, Z // G // pieces
    g = torch.Generator(device="cuda").manual_seed(5)
    full = torch.randn((Z, Y, X, 2), generator=g, device="cuda")
    flags = b200fft.FLAG_NO_FUSED
    plan = b200fft.plan_fft("float32", "float32", (zl, Y, X, 2), (zl, Y, X, 2), axis_mask=axis_mask, flags=flags)
    plan_c = b200fft.plan_fft("float32", "float32", (zc, Y, X, 2), (zc, Y, X, 2), axis_mask=axis_mask, flags=flags)
    work = torch.empty((zl, Y, X, 2), device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    recv = {k: [torch.full((Z, yl, X, 2), float("nan"), device="cuda") for _ in range(G)] for k in ("rank", "at", "pieces")}
    for r in range(G):
        x_local = full[r * zl:(r + 1) * zl].contiguous()
        keep = x_local.clone()
        plan.exec_scatter(recv["rank"], r, x_local, work, st)
        assert _scatter_at(plan, recv["at"], r * zl, x_local, work, st) == 0
        for c in range(pieces):
            x_c = x_local[c * zc:(c + 1) * zc]
            assert _scatter_at(plan_c, recv["pieces"], r * zl + c * zc, x_c, work[c * zc:(c + 1) * zc], st) == 0
        assert torch.equal(x_local, keep)
    torch.cuda.synchronize()
    xc = torch.view_as_complex(full.double().contiguous())
    want = torch.fft.fft(xc, dim=1) if axis_mask == 1 else torch.fft.fftn(xc, dim=(1, 2))
    for h in range(G):
        assert torch.equal(recv["at"][h], recv["rank"][h])
        assert torch.equal(recv["pieces"][h], recv["rank"][h])
        got = torch.view_as_complex(recv["rank"][h].double().contiguous())
        ref = want[:, h * yl:(h + 1) * yl, :]
        assert float((got - ref).norm() / ref.norm()) < 2e-6
    assert _scatter_at(plan, recv["at"], -1, full[:zl].contiguous(), work, st) == 1  # B200FFT_ERR_INVALID_ARG
    plan.destroy()
    plan_c.destroy()


def test_exec_scatter_errors():
    import torch
    plan = b200fft.plan_fft("float32", "float32", (4, 64, 64, 2), (4, 64, 64, 2))
    x = torch.zeros((4, 64, 64, 2), device="cuda")
    w = torch.zeros_like(x)
    with pytest.raises(b200fft.B200FFTError):            # 64 rows cannot be split over 3 peers
        plan.exec_scatter([x, x, x], 0, x, w)
    with pytest.raises(b200fft.B200FFTError):            # rank outside the peer list
        plan.exec_scatter([x, x], 2, x, w)
    rows = b200fft.plan_fft("float32", "float32", (4, 64, 2), (4, 64, 2))
    x1 = torch.zeros((4, 64, 2), device="cuda")
    with pytest.raises(b200fft.B200FFTError) as e:       # contiguous-axis pass has no scattering store
        rows.exec_scatter([x1, x1], 0, x1, torch.zeros_like(x1))
    assert e.value.status == 4


@pytest.mark.parametrize("n", [64, 128, 256])
@pytest.mark.parametrize("inverse", [False, True])
def test_fused_slab_kernel_single_rank(n, inverse):
    """b200fft_slab_exec with one rank: all three phases, the x-block arrival counters and the alternating
    receive buffers on one GPU (the multi-rank run over NVLink is tools/slab_check.py under torchrun)."""
    import torch
    plan = b200fft.SlabPlan(n, 1, 0, inverse)
    assert "slab_fused" in plan.describe()
    nfloat = plan.recv_bytes // 4
    bufs = [torch.zeros(nfloat, device="cuda") for _ in range(2)]
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.randn((n, n, n, 2), generator=g, device="cuda")
    keep = x.clone()
    work = torch.empty_like(x)
    xc = torch.view_as_complex(x.double().contiguous())
    want = torch.fft.ifftn(xc) if inverse else torch.fft.fftn(xc)
    for call in range(5):                      # counters keep growing across calls; buffers alternate
        k = call & 1
        plan.exec(x, work, [bufs[k]], k)
        torch.cuda.synchronize()
        got = torch.view_as_complex(bufs[k][:n * n * n * 2].view(n, n, n, 2).double().contiguous())
        assert float((got - want).norm() / want.norm()) < 2e-6
    assert torch.equal(x, keep)
    plan.destroy()


def test_fused_slab_rejects_unsupported():
    with pytest.raises(b200fft.B200FFTError):
        b200fft.SlabPlan(100, 1, 0)            # not a registered cubic size
    with pytest.raises(b200fft.B200FFTError):
        b200fft.SlabPlan(128, 3, 0)            # 128 planes cannot be split over 3 ranks


def test_pencil_and_slab_restore_single_rank_nccl():
    """The product engines behind PencilFFT3D and SlabFFT3D.restore() on one GPU (a 1-rank NCCL group; the block
    order over 2 and 4 ranks is covered on CPU by tests/test_pencil_gloo.py): X / Y / Z passes through axis-masked
    plans, pack / exchange / unpack, natural-order output and the forward -> inverse round trip."""
    import os
    import socket
    import torch
    import torch.distributed as dist
    from b200fft.pencil import PencilFFT3D
    from b200fft.slab import SlabFFT3D
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        g = torch.Generator(device="cuda").manual_seed(21)
        for dims, inverse in (((64, 96, 128), False), ((32, 64, 100), True)):
            x = torch.randn(dims + (2,), generator=g, device="cuda")
            keep = x.clone()
            pen = PencilFFT3D(dims, (1, 1), inverse=inverse)
            got = torch.view_as_complex(pen.forward(x).double().contiguous())
            xc = torch.view_as_complex(x.double().contiguous())
            want = torch.fft.ifftn(xc) if inverse else torch.fft.fftn(xc)
            assert float((got - want).norm() / want.norm()) < 2e-6
            assert torch.equal(x, keep)
            pen.close()
        dims = (64, 64, 64)
        x = torch.randn(dims + (2,), generator=g, device="cuda")
        xc = torch.view_as_complex(x.double().contiguous())
        for mode in ("nccl", "p2p", "fused"):
            fwd = SlabFFT3D(dims, exchange=mode)
            inv = SlabFFT3D(dims, exchange=mode, inverse=True)
            spec = fwd.forward(x, natural=True)
            want = torch.fft.fftn(xc)
            assert float((torch.view_as_complex(spec.double().contiguous()) - want).norm() / want.norm()) < 2e-6
            back = inv.forward(spec, natural=True)
            assert float((back - x).norm() / x.norm()) < 2e-6
            fwd.close()
            inv.close()
    finally:
        dist.destroy_process_group()

"""bench.py's reference arm (`--impl reference`: the reference's CPU path = the oracle port, all host threads) runs
without a GPU; check the JSON line it prints against the driver's contract. The GPU arm is exercised on the B200."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, B200FFT_BENCH_REF_SECONDS="0.2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == baseline["metric"]
    assert d["unit"] == "GFLOP/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 2 and d["warmup"] >= 1 and d["n_gpus"] == 1
    assert d["config"]["workload"] == "1D C2C fp32 100000x1024"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "transforms" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1", B200FFT_BENCH_REF_SECONDS="0.2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_repeat_and_match_numpy(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same bits, a sample of the primary workload's output
    that matches numpy float64 on the same seeded input; the timed region launches the plan exactly --steps times."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import b200fft
    batch, length = bench.PRIMARY["shape"]
    plan = b200fft.plan_fft("float32", "float32", (batch, length, 2), (batch, length, 2))
    launches_per_step = plan.launches
    plan.destroy()
    steps = 3
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--no-shapes",
                              "--no-cpu", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps and line["gpu_launches"] == steps * launches_per_step
        assert os.listdir(d) == ["out.npy"]
        dumps.append(np.load(d / "out.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (bench.DUMP_ROWS, length, 2) and dumps[0].nbytes <= 64 << 20
    assert np.array_equal(dumps[0], dumps[1])
    g = torch.Generator(device="cuda").manual_seed(1234)            # bench.py's rank-0 input
    x = torch.randn((batch, length, 2), generator=g, device="cuda", dtype=torch.float32)
    rows = bench.dump_rows(batch)
    xs = x.index_select(0, torch.from_numpy(rows).cuda()).double().cpu().numpy()
    want = np.fft.fft(xs[..., 0] + 1j * xs[..., 1], axis=1)
    got = dumps[0][..., 0].astype(np.float64) + 1j * dumps[0][..., 1]
    assert np.linalg.norm(got - want) <= 2e-6 * np.linalg.norm(want)


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_shape_rows_find_their_plan_traffic():
    """bench.py's shapes[] rows report DRAM traffic / algorithmic bytes from profiles/traffic.json "plan:<row name>" entries
    (ncu captures of one exec of the whole plan): every multi-pass BASELINE row must have one, with the kernels of the plan
    the planner picks today."""
    sys.path.insert(0, ROOT)
    import bench
    traffic = bench._plan_traffic()
    names = {n for n, _, _ in bench.SHAPES}
    for row in ("2d_100x640x480", "2d_100x640x480_r2c_half", "3d_100x64x64x64", "3d_100x64x64x64_r2c_half", "3d_10x128x128x128",
                "3d_1x256x256x256", "3d_1x512x512x512"):
        assert row in names
        e = traffic["plan:" + row]
        assert e["dram_bytes_per_exec"] > 0.9 * e["algorithmic_bytes_per_exec"] and e["launches"] == len(e["kernels"]) >= 1
    assert "plane_kernel" in traffic["plan:3d_100x64x64x64"]["kernels"][0]          # the default plan, not the fused kernel's capture
    assert "nd_async_kernel" in traffic["fused-plan:3d_100x64x64x64"]["kernels"][0]

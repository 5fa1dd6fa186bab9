"""Strided layouts (b200fft_plan_create_strided), checked without a GPU: the stride rules refuse before any CUDA call, and
the strided form of every kernel kind a strided plan runs compiles for sm_100a through NVRTC under a name of its own."""
import os
import subprocess

import pytest

import b200fft

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C2C = ((8, 64, 2), (8, 64, 2))


def status_of(*args, **kw):
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft(*args, **kw)
    return e.value.status, str(e.value)


def test_entry_points_are_bound():
    names = [s[0] for s in b200fft.SYMBOLS]
    assert "b200fft_plan_create_strided" in names and "b200fft_jit_probe_strided" in names
    assert b200fft.lib().b200fft_plan_create_strided(None, None, None, None) == 1


@pytest.mark.parametrize("case,kw,want", [
    ("overlapping output", dict(out_strides=(64, 2)), 2),                 # batch stride 64 < 2 * 64: rows collide
    ("output stride 0", dict(out_strides=(0, 1)), 2),
    ("negative input stride", dict(in_strides=(64, -1)), 2),
    ("offset beyond int64", dict(out_strides=(2 ** 61, 1)), 1),
    ("wrong stride count", dict(in_strides=(64,)), 2),
])
def test_bad_strides_refuse_before_the_device(case, kw, want):
    status, msg = status_of("float32", "float32", *C2C, **kw)
    assert status == want, (case, msg)


def test_half_spectrum_layout_rules():
    real, cplx = (4, 6, 64, 1), (4, 6, 33, 2)
    # the last axis must have stride 1 on both sides
    status, msg = status_of("float32", "float32", real, cplx, real_mode=b200fft.REAL_HALF, in_strides=(768, 128, 2))
    assert status == 4 and "stride 1 along the last axis" in msg, msg
    # even n: the real rows move as pairs, so every other real-side stride is even
    status, msg = status_of("float32", "float32", real, cplx, real_mode=b200fft.REAL_HALF, in_strides=(6 * 65, 65, 1))
    assert status == 4 and "odd" in msg, msg
    status, msg = status_of("float32", "float32", cplx, real, real_mode=b200fft.REAL_HALF, inverse=True, out_strides=(6 * 65, 65, 1))
    assert status == 4 and "odd" in msg, msg


@pytest.mark.parametrize("flags,name", [(b200fft.FLAG_FORCE_GENERIC, "FORCE_GENERIC"), (b200fft.FLAG_FORCE_RT, "FORCE_RT")])
def test_strided_plans_refuse_the_other_tiers(flags, name):
    status, msg = status_of("float32", "float32", *C2C, out_strides=(128, 2), flags=flags)
    assert status == 4 and name in msg, msg


def test_strided_plans_refuse_without_the_plan_time_tier(monkeypatch):
    monkeypatch.setenv("B200FFT_JIT", "0")
    status, msg = status_of("float32", "float32", *C2C, out_strides=(128, 2))
    assert status == 4 and "B200FFT_JIT=0" in msg, msg


def test_axes_longer_than_one_tile_refuse():
    # far beyond one tile's shared memory (fp32 columns: 1024 points; rows: 16384), read across a transposed view and
    # along pitched rows; tests/test_host_strided_forms.py pins the boundaries themselves
    shape = (1, 32768, 4, 2)
    status, msg = status_of("float32", "float32", shape, shape, in_strides=(4 * 32768, 1, 32768))
    assert status == 4 and "one tile" in msg, msg
    shape = (2, 65536, 2)
    status, msg = status_of("float32", "float32", shape, shape, out_strides=(65536 * 2, 2))
    assert status == 4 and "one tile" in msg, msg


# (kind, probe arguments): every kind a strided plan runs, with the input types each accepts
PROBES = [
    ("jitrows", dict(n=600)),
    ("jitrows", dict(n=600, real_in=True)),
    ("jitrows", dict(n=600, real_in=True, in_dtype="uint8")),
    ("jitrows", dict(n=600, in_dtype="float64")),
    ("jitrowsIP", dict(n=8192)),
    ("jitrowsIP", dict(n=8192, real_in=True, in_dtype="uint8")),
    ("jitcols", dict(n=600, inner=64)),
    ("jitcols", dict(n=93, inner=64, real_in=True)),
    ("jitcols", dict(n=600, inner=64, inverse=True, in_dtype="float64")),
    ("jitr2c", dict(n=1000, half=1)),
    ("jitr2creg", dict(n=1024, half=1)),
    ("jitr2codd", dict(n=93, half=1)),
    ("jitc2r", dict(n=1000, half=2)),
    ("jitc2rodd", dict(n=2187, half=2)),
]


@pytest.mark.parametrize("out_dtype", ["float32", "float64"])
@pytest.mark.parametrize("kind,kw", PROBES, ids=["%s-%d" % (k, i) for i, (k, _) in enumerate(PROBES)])
def test_strided_forms_compile_under_their_own_names(kind, kw, out_dtype):
    kw = dict(kw, out_dtype=out_dtype)
    if kw.get("half") == 2:
        kw["in_dtype"] = out_dtype  # the C2R kernels read the half spectrum in the working precision
    strided = b200fft.jit_probe(strided=True, **kw)
    dense = b200fft.jit_probe(**kw)
    name, dense_name = strided.split(":")[0], dense.split(":")[0]
    assert name == dense_name + "_str", (strided, dense)
    if out_dtype == "float32":  # (fp64 1024-point R2C rows have no register-unpack shape: they take jitr2c)
        assert name.startswith(kind) and not name[len(kind)].isalpha(), name
    assert "b200fft::StrLay>" in strided and "StrLay" not in dense, strided
    assert ("_f64" in name) == (out_dtype == "float64"), name


def test_cpp_host_layer_takes_strides(tmp_path):
    """include/b200fft.hpp: PlanOptions::in_strides / out_strides reach b200fft_plan_create_strided; compiled with the same
    -Wall -Wextra -Werror as the header's own test."""
    src = tmp_path / "strided.cpp"
    src.write_text(r'''
#include "b200fft.hpp"
int main() {
  using namespace b200fft;
  Layout x{{8, 64, 2}};
  PlanOptions o;
  o.out_strides = {64, 2};  // overlapping rows
  try { plan_fft(f32, f32, x, x, o); return 1; } catch (const Error& e) { if (e.status() != B200FFT_ERR_LAYOUT) return 2; }
  o.out_strides = {128, 2};
  o.in_strides = {64};      // one stride short
  try { plan_fft(f32, f32, x, x, o); return 3; } catch (const Error& e) { if (e.status() != B200FFT_ERR_LAYOUT) return 4; }
  o.in_strides = {64, -1};
  try { plan_fft(f32, f32, x, x, o); return 5; } catch (const Error& e) { if (e.status() != B200FFT_ERR_LAYOUT) return 6; }
  PlanOptions h;
  h.real_mode = real_half;
  h.in_strides = {130, 65, 1};  // odd pitch for an even length
  try { plan_fft(f32, f32, Layout{{4, 6, 64, 1}}, Layout{{4, 6, 33, 2}}, h); return 7; }
  catch (const Error& e) { if (e.status() != B200FFT_ERR_UNSUPPORTED) return 8; }
  return 0;
}
''')
    exe = tmp_path / "strided"
    libdir = os.path.dirname(b200fft.lib_path())
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), "-L", libdir, "-lb200fft", "-Wl,-rpath," + libdir])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)

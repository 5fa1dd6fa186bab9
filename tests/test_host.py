"""CPU-only checks of the boundary: the C-ABI library loads, exports every symbol
include/b200fft.h declares, and its host planner reproduces the reference's
compile-time plan rules (compared with the oracle's independent restatement)."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest

import b200fft

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200fft.h")).read()
    return sorted(set(re.findall(r"B200FFT_API[^;]*?\b(b200fft_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    declared = _declared_symbols()
    assert len(declared) >= 18
    L = ctypes.CDLL(b200fft.lib_path())
    missing = [s for s in declared if not hasattr(L, s)]
    assert not missing, missing
    assert sorted(s[0] for s in b200fft.SYMBOLS) == declared  # the shim binds exactly the header
    assert b200fft.lib().b200fft_version() >= 100


def test_strerror():
    assert b200fft.lib().b200fft_strerror(0) == b"ok"
    assert b"bases" in b200fft.lib().b200fft_strerror(3)


LENGTHS = [2, 3, 4, 5, 6, 7, 8, 10, 16, 20, 21, 30, 32, 35, 48, 60, 64, 93, 100, 128, 194, 480, 512, 640, 1024, 4096]


@pytest.mark.parametrize("n", LENGTHS)
def test_default_bases_match_oracle(oracle, n):
    for target in ("cpu", "gpu"):
        assert b200fft.default_bases(n, target) == oracle.default_bases(n, target)


def test_ordered_bases_golden_cases(oracle, golden):
    for case in golden["cases_1d"]:
        got = b200fft.ordered_bases(case["length"], case["bases"])
        assert got == oracle.ordered_bases(case["length"], case["bases"])
        assert int(np.prod(got)) == case["length"]
        assert got == sorted(got, reverse=True)


def test_ordered_bases_random_match_oracle(oracle):
    rng = np.random.default_rng(0)
    pool = [2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 16, 20, 31, 32, 97]
    for _ in range(400):
        k = int(rng.integers(1, 4))
        bases = [int(b) for b in rng.choice(pool, size=k, replace=False)]
        n = 1
        for b in bases:
            n *= b ** int(rng.integers(0, 3))
        n = max(n, 2)
        assert b200fft.ordered_bases(n, bases) == oracle.ordered_bases(n, bases), (n, bases)


def test_rejected_bases():
    assert b200fft.ordered_bases(60, [7, 2]) is None
    assert b200fft.ordered_bases(8, [1, 2]) is None
    assert b200fft.ordered_bases(93, [3]) is None


def test_dry_run_layout_conditions():
    """_check_layout_conditions_nd (fft.mojo:20-46) as runtime errors."""
    ok = b200fft.dry_run("float32", "float32", (4, 128, 2), (4, 128, 2))
    assert "stages=[2,2,2,2,2,2,2]" in ok
    txt = b200fft.dry_run("uint8", "float64", (1, 6, 4, 8, 1), (1, 6, 4, 8, 2))
    assert txt.splitlines()[0].startswith("axis 2") and "reads input" in txt.splitlines()[0]
    assert txt.splitlines()[-1].startswith("axis 0")
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.dry_run("float32", "float32", (4, 2), (4, 2))
    assert e.value.status == 2
    with pytest.raises(b200fft.B200FFTError):
        b200fft.dry_run("float32", "float32", (4, 8, 3), (4, 8, 2))       # in last dim must be 1|2
    with pytest.raises(b200fft.B200FFTError):
        b200fft.dry_run("float32", "float32", (4, 8, 2), (4, 8, 1))       # out last dim must be 2
    with pytest.raises(b200fft.B200FFTError):
        b200fft.dry_run("float32", "float32", (4, 8, 2), (4, 9, 2))       # equal leading shape
    with pytest.raises(b200fft.B200FFTError):
        b200fft.dry_run("float32", "float32", (4, 1, 8, 2), (4, 1, 8, 2))  # no inner dim of size 1
    with pytest.raises(b200fft.B200FFTError):
        b200fft.dry_run("float32", "uint8", (4, 8, 2), (4, 8, 2))         # out dtype must be float
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.dry_run("float32", "float32", (4, 60, 2), (4, 60, 2), bases=[[7, 2]])
    assert e.value.status == 3 and "only able to produce" in str(e.value)
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.dry_run("float32", "float32", (4, 8, 8, 2), (4, 8, 8, 2), bases=[[2]])
    assert e.value.status == 3                                            # one bases list per axis


def test_user_bases_reach_the_plan():
    txt = b200fft.dry_run("float32", "float32", (2, 93, 2), (2, 93, 2), bases=[[3, 31]])
    assert "stages=[31,3]" in txt
    txt = b200fft.dry_run("float32", "float32", (2, 128, 2), (2, 128, 2), bases=[[16, 8]])
    assert "stages=[16,8]" in txt
    txt = b200fft.dry_run("float32", "float32", (2, 60, 48, 2), (2, 60, 48, 2), bases=[[6, 5, 2], [3, 2]])
    assert "stages=[6,5,2]" in txt and "stages=[3,2,2,2,2]" in txt


def test_no_cpu_fallback():
    """Without a GPU the product must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft("float32", "float32", (2, 8, 2), (2, 8, 2))
    assert e.value.status == 5


def test_header_is_plain_c_and_links(tmp_path):
    """include/b200fft.h must be consumable from C (the Mojo / cgo-style FFI boundary): compile a C99 program against
    it with gcc -pedantic, link it with the built library and call two entry points that need no GPU."""
    import subprocess
    src = tmp_path / "abi.c"
    src.write_text('#include "b200fft.h"\n#include <string.h>\n'
                   "int main(void) {\n"
                   "  uint32_t out[16]; uint32_t bases[1] = {2};\n"
                   "  b200fft_desc d; memset(&d, 0, sizeof d);\n"
                   "  if (sizeof(b200fft_desc) != 128) return 2;\n"
                   "  if (b200fft_version() <= 0) return 3;\n"
                   "  if (b200fft_ordered_bases(8, bases, 1, out, 16) != 3) return 4;\n"
                   "  return strcmp(b200fft_strerror(B200FFT_OK), \"ok\") != 0;\n}\n")
    exe = tmp_path / "abi"
    libdir = os.path.dirname(b200fft.lib_path())
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), "-L", libdir, "-lb200fft", "-Wl,-rpath," + libdir])
    assert subprocess.run([str(exe)]).returncode == 0


@pytest.mark.parametrize("H,R", [(512, 16), (64, 8), (128, 8), (256, 16), (240, 15), (160, 10), (48, 3), (640, 20), (1024, 32)])
def test_r2c_register_unpack_index_algebra(H, R):
    """The lane algebra behind R2CRegDst (csrc/fast.cuh), restated in numpy: in the last stage of an H-point transform
    (radix R, P = H / R butterflies per row) butterfly p holds Z[p + k P]; the mirrored bins Z[H - p - k P] are
    butterfly (P - p) mod P's outputs R-1-k (butterfly 0: its own outputs (R - k) mod R), and
    X[k] = ((Z[k] + conj Z[H-k]) - i W_n^k (Z[k] - conj Z[H-k])) / 2, X[H] = Re Z[0] - Im Z[0], is the real transform."""
    P = H // R
    assert P * R == H and 8 <= P <= 32 and 32 % P == 0          # the eligibility rule r2c_reg_ok() applies
    rng = np.random.default_rng(H)
    x = rng.standard_normal(2 * H)
    Z = np.fft.fft(x[0::2] + 1j * x[1::2])
    held = np.array([[Z[p + k * P] for k in range(R)] for p in range(P)])     # held[p][k]: registers of butterfly p
    X = np.empty(H + 1, dtype=complex)
    for p in range(P):
        partner = (P - p) % P
        for k in range(R):
            zm = held[p][(R - k) % R] if p == 0 else held[partner][R - 1 - k]
            assert zm == Z[(H - (p + k * P)) % H]
            zk = held[p][k]
            s, d = zk + np.conj(zm), zk - np.conj(zm)
            X[p + k * P] = 0.5 * (s - 1j * np.exp(-2j * np.pi * (p + k * P) / (2 * H)) * d)
    X[H] = Z[0].real - Z[0].imag
    np.testing.assert_allclose(X, np.fft.rfft(x), atol=1e-10)


def test_cpp_host_layer_mirrors_the_reference_api(tmp_path):
    """include/b200fft.hpp: the header-only C++ host layer (plan_fft / fft with the reference's names over the C ABI).
    Compile a C++17 program against it with -Wall -Wextra -Werror, link the built library and exercise everything
    that needs no GPU: base rules, dry run, the layout / bases errors with the C ABI's status codes, and the loud
    failure of plan_fft without an sm_100 device (no CPU fallback)."""
    import subprocess
    src = tmp_path / "host.cpp"
    src.write_text(r'''
#include "b200fft.hpp"
#include <cstdio>
#include <cstring>
int main() {
  using namespace b200fft;
  if (ordered_bases(60, {5, 3, 2}) != std::vector<uint32_t>({5, 3, 2, 2})) return 1;   // _utils.mojo:163-183
  if (!ordered_bases(60, {7}).empty()) return 2;                                       // rejected like the reference
  if (default_bases(93) != std::vector<uint32_t>({31, 3})) return 3;                   // fft.mojo:49-104
  Layout img{{100, 640, 480, 2}};
  PlanOptions o;
  o.bases = {{5, 2}, {5, 3, 2}};
  const std::string txt = dry_run(f32, f32, img, img, o);
  if (txt.find("stages=[5,2,2,2,2,2,2,2]") == std::string::npos || txt.find("stages=[5,3,2,2,2,2,2]") == std::string::npos) return 4;
  try { dry_run(f32, f32, Layout{{8, 2}}, Layout{{8, 2}}); return 5; } catch (const Error& e) { if (e.status() != B200FFT_ERR_LAYOUT) return 6; }
  try { o.bases = {{7}, {5, 3, 2}}; dry_run(f32, f32, img, img, o); return 7; } catch (const Error& e) { if (e.status() != B200FFT_ERR_BASES) return 8; }
  try { o.bases = {{5, 2}}; dry_run(f32, f32, img, img, o); return 9; } catch (const Error& e) { if (e.status() != B200FFT_ERR_BASES) return 10; }
  PlanOptions h;
  h.real_mode = real_half;
  const std::string half = dry_run(f32, f32, Layout{{100, 640, 480, 1}}, Layout{{100, 640, 241, 2}}, h);
  if (half.find("r2c") == std::string::npos) return 11;
  try { dry_run(f32, f32, Layout{{100, 640, 480, 1}}, Layout{{100, 640, 240, 2}}, h); return 12; } catch (const Error& e) { if (e.status() != B200FFT_ERR_LAYOUT) return 13; }
  try {
    Plan p = plan_fft(f32, f32, Layout{{4, 128, 2}}, Layout{{4, 128, 2}});
    Plan q = std::move(p);                       // move-only handle
    if (p || !q || q.launches() < 1) return 14;  // a GPU box: the plan exists and describes its kernels
  } catch (const Error& e) {
    if (e.status() != B200FFT_ERR_CUDA) return 15;   // no sm_100 device: loud failure, never a CPU path
    std::printf("no-gpu: %s\n", e.what());
  }
  try {   // the multi-device layer: same loud failure without GPUs, a working plan with them
    MultiGpuPlan mp(f32, f32, Layout{{8, 128, 2}}, Layout{{8, 128, 2}}, {0}, MultiGpuMode::batch_shard);
    MultiGpuPlan mq = std::move(mp);
    if (mp || !mq || mq.ngpu() != 1 || mq.shard(0) != std::pair<int64_t, int64_t>(0, 8) || mq.in_bytes(0) != 8 * 128 * 8) return 16;
  } catch (const Error& e) {
    if (e.status() != B200FFT_ERR_CUDA) return 17;
  }
  return 0;
}
''')
    exe = tmp_path / "host"
    libdir = os.path.dirname(b200fft.lib_path())
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           str(src), "-o", str(exe), "-L", libdir, "-lb200fft", "-Wl,-rpath," + libdir])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)


def test_variant_tables_are_built_once_under_concurrent_first_use():
    """include/b200fft.h promises that distinct plans may be created from distinct threads: the kernel-variant tables
    behind plan creation must be built exactly once even when the FIRST calls race. A fresh process starts 16 threads
    that all ask for the table sizes at the same moment (ctypes releases the GIL during the call)."""
    import subprocess
    import sys
    code = r'''
import ctypes, sys, threading
L = ctypes.CDLL(sys.argv[1])
L.b200fft_variant_count.restype = ctypes.c_int
L.b200fft_variant_count.argtypes = [ctypes.c_int]
start = threading.Barrier(16)
seen = []
def work():
    start.wait()
    seen.append(tuple(L.b200fft_variant_count(t) for t in (0, 1, 2)))
ts = [threading.Thread(target=work) for _ in range(16)]
[t.start() for t in ts]
[t.join() for t in ts]
assert len(set(seen)) == 1 and len(seen) == 16, seen
print(*seen[0], L.b200fft_variant_count(7))
'''
    for _ in range(3):
        r = subprocess.run([sys.executable, "-c", code, b200fft.lib_path()], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        fast, fused, split, unknown = (int(v) for v in r.stdout.split())
        assert fast >= 40 and fused >= 10 and split >= 8 and unknown == -1, r.stdout
    # and the in-process view agrees (tables are per process, sizes are a property of the build)
    assert b200fft.lib().b200fft_variant_count(0) == fast


def test_mgpu_batch_split_rule():
    """BATCH_SHARD's split (b200fft_mgpu_split, host-only): contiguous, covers the batch, sizes differ by at most one,
    the larger shares first (SURVEY.md 8e: 10 items over 4 devices -> 3/3/2/2, 100 over 8 -> 13 x 4 + 12 x 4)."""
    for batch, n in ((10, 4), (100, 8), (500000, 8), (7, 7), (1, 1), (9, 2)):
        nxt, sizes = 0, []
        for g in range(n):
            first, count = b200fft.mgpu_split(batch, n, g)
            assert first == nxt
            nxt += count
            sizes.append(count)
        assert nxt == batch and max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
    assert [b200fft.mgpu_split(10, 4, g)[1] for g in range(4)] == [3, 3, 2, 2]
    with pytest.raises(b200fft.B200FFTError):
        b200fft.mgpu_split(10, 4, 4)


def test_mgpu_needs_cuda_no_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.MgpuPlan("float32", "float32", (8, 64, 2), (8, 64, 2), devices=[0])
    assert e.value.status == 5


def test_jit_sources_compile_with_nvrtc_for_sm100a():
    """The plan-time specialisation tier's sources (the device headers embedded in the library) compile for sm_100a
    with NVRTC in this container: rows and strided kernels, forward / inverse, real input, a prime radix above 32."""
    for kw, want in ((dict(n=1000), "rows_ip_kernel<1000, b200fft::Radices<10, 10, 10>"),  # three narrow stages in one buffer beat 40 x 25
                     (dict(n=1296), "rows_kernel<1296, b200fft::Radices<36, 36>"),      # wide codelets save a stage
                     (dict(n=16384, inverse=True), "rows_ip_kernel<16384, b200fft::Radices<32, 32, 16>, 1, 512, true, false>"),
                     (dict(n=10000, in_dtype="float64", out_dtype="float64"), "rows_ip_kernel<10000, b200fft::Radices<10, 10, 10, 10>"),
                     (dict(n=1000, half=1), "rows_r2c_kernel<500, b200fft::Radices<25, 20>"),
                     (dict(n=1000, half=2), "rows_c2r_kernel<500, b200fft::Radices<25, 20>"),
                     (dict(n=243, half=1), "rows_r2c_odd_kernel<243, b200fft::Radices<27, 9>"),
                     (dict(n=360, inner=360, inverse=True), "cols_kernel<360, b200fft::Radices<20, 18>, 16, 288, true, false>"),
                     (dict(n=200, real_in=True), "false, true>"),
                     (dict(n=74), "Radices<37, 2>"),
                     (dict(n=194, bases=[97, 2]), "Radices<97, 2>")):          # looped prime codelet: compiles in under a second
        rep = b200fft.jit_probe(**kw)
        assert want in rep and "cubin=" in rep, rep
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_probe(n=262, bases=[131, 2])       # a prime above 127: left to the generic kernel
    assert e.value.status == 4
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_probe(n=100, bases=[3])
    assert e.value.status == 3


def test_row_planner_one_buffer_rules(monkeypatch):
    """Which contiguous rows the plan-time tier gives to the one-buffer kernel (csrc/jit.cu: jit_plan_axis,
    jit_rows_ip_geometry; measured in profiles/r2_long_rows.md). Host-only: the planner + an NVRTC compile."""
    def kernel(n, **kw):
        return b200fft.jit_probe(n, **kw).split(":")[0]
    assert kernel(1800).startswith("jitrows1800_")            # under 16 KB per row: two buffers, several rows per CTA
    assert kernel(2187) == "jitrowsIP2187_27x9x9_c1_t128"     # 3 stages from 2048 points: one buffer, one row per CTA
    assert kernel(1536) == "jitrows1536_48x32_c3_t96"         # two wide stages that measured faster stay
    assert kernel(2000) == "jitrowsIP2000_20x10x10_c1_t128"   # ... a radix-40/50 codelet does not (50 x 40)
    assert kernel(20000) == "jitrowsIP20000_20x40x25_c1_t512"  # order permuted: 25 in the middle would hold 50 values at 512 threads
    assert kernel(3000) == "jitrowsIP3000_20x15x10_c1_t160"   # ... and is left alone when it fits
    assert kernel(1024, in_dtype="float64", out_dtype="float64").startswith("jitrowsIP1024_16x8x8_c1_t128_f64")  # the rule is in bytes
    with pytest.raises(b200fft.B200FFTError):                  # no stage order fits the register budget: two passes
        b200fft.jit_probe(24000)
    monkeypatch.setenv("B200FFT_ROWS_INPLACE", "0")            # A/B knob, read per plan
    assert kernel(2187).startswith("jitrows2187_27x9x9_c3_")
    with pytest.raises(b200fft.B200FFTError):
        b200fft.jit_probe(20000)


def test_jit_disk_cache(tmp_path):
    """A kernel compiled by one process is loaded from the on-disk cache by the next (fresh processes: the cache
    directory is read once per process); a rebuilt library (different header text) or another key never matches."""
    import subprocess
    code = ("import sys; sys.path.insert(0, %r); import b200fft; print(b200fft.jit_probe(n=%%d))"
            % os.path.join(ROOT, "hackathon-fft_b200", "python"))
    env = dict(os.environ, B200FFT_JIT_CACHE="1", B200FFT_JIT_CACHE_DIR=str(tmp_path / "cache"))
    first = subprocess.run([sys.executable, "-c", code % 1000], env=env, capture_output=True, text=True, check=True).stdout
    assert "disk cache" not in first and "cubin=" in first
    files = os.listdir(tmp_path / "cache")
    assert len(files) == 1 and files[0].endswith(".cubin")
    second = subprocess.run([sys.executable, "-c", code % 1000], env=env, capture_output=True, text=True, check=True).stdout
    assert "(disk cache)" in second and second.split("symbol ")[1] == first.split("symbol ")[1]
    other = subprocess.run([sys.executable, "-c", code % 100], env=env, capture_output=True, text=True, check=True).stdout
    assert "disk cache" not in other and len(os.listdir(tmp_path / "cache")) == 2
    off = subprocess.run([sys.executable, "-c", code % 1000], env=dict(env, B200FFT_JIT_CACHE="0"), capture_output=True, text=True,
                         check=True).stdout
    assert "disk cache" not in off


@pytest.mark.parametrize("tier", [0, 1, 2])
def test_variant_info_describes_every_registered_variant(tier):
    """b200fft_variant_info lists each tier's registry (what tests/test_gpu_variants.py forces one variant at a time),
    and the lines agree with what the planner relies on: unique names, radices that multiply to n, and the forms
    a variant instantiates."""
    info = b200fft.variant_info(tier)
    assert len(info) == b200fft.lib().b200fft_variant_count(tier)
    names = [v["name"] for v in info]
    assert len(set(names)) == len(names)
    L = b200fft.lib()
    assert L.b200fft_variant_info(tier, len(info), None, 0) == -1
    assert L.b200fft_variant_info(tier, -1, None, 0) == -1
    assert L.b200fft_variant_info(3, 0, None, 0) == -1
    small = ctypes.create_string_buffer(8)  # a short buffer is truncated, the return value is the full length
    need = L.b200fft_variant_info(tier, 0, small, len(small))
    assert need > len(small) and small.value.decode() == ("name=" + names[0])[:7]
    for v in info:
        if tier == 1:
            assert v["kind"] == "fused" and v["mode"] in ("c2c", "real", "r2c") and v["forms"] in (["fwd"], ["inv"])
            assert v["async"] == v["name"].startswith("ndA")
            dims = [int(d) for d in v["n"].split("x")]
            assert v["name"].startswith(("ndA" if v["async"] else "nd") + v["n"] + ("_inv" if v["forms"] == ["inv"] else ""))
            # one stage list per axis (a plane phase carries two: y; x), together the whole transform (R2C: n/2 on x)
            stages = [s for ph in v["radices"].split("|") for s in ph.split(";")]
            assert len(stages) == len(dims), v["name"]
            prod = int(np.prod([int(r) for s in stages for r in s.split("x")]))
            assert prod == int(np.prod(dims)) // (2 if v["mode"] == "r2c" else 1), v["name"]
            continue
        assert int(np.prod(v["radices"])) == v["n"], v["name"]
        assert v["tile"] >= 1 and v["threads"] >= 32
        if tier == 2:
            assert v["kind"] in ("splitA", "splitB_cols", "splitB_rows") and v["forms"] == ["fwd", "inv"]
            assert v["name"].startswith({"splitA": "splitA_cols", "splitB_cols": "splitB_cols", "splitB_rows": "splitB_rows"}
                                        [v["kind"]] + str(v["n"]) + "_")
            continue
        assert v["kind"] in ("rows", "rowsIP", "cols", "colsT")
        assert v["name"].startswith({"rows": "rows", "rowsIP": "rowsIP", "cols": "cols", "colsT": "colsT"}[v["kind"]])
        forms = v["forms"]
        assert forms[0] == "fwd"
        if v["kind"] == "rowsIP":  # one-buffer rows: every direction and input, no half-spectrum forms
            assert forms == ["fwd", "inv", "real"] and v["full"] == 0
        elif v["kind"] == "colsT":
            assert forms == ["fwd", "inv"]
        elif not v["full"]:  # tuning candidates: forward complex only
            assert forms == ["fwd"]
        else:
            assert forms[:3] == ["fwd", "inv", "real"]
        if v["kind"] == "rows" and v["full"]:
            fits = v["smem_r2c"] <= 227 * 1024 and v["smem_c2r"] <= 227 * 1024
            assert ("r2c" in forms) == fits and ("c2r" in forms) == fits, v
            assert ("r2c-reg" not in forms) or fits
            assert ("r2c-odd" in forms) == ("c2r-odd" in forms) == (v["n"] % 2 == 1)
        else:
            assert not {"r2c", "c2r", "r2c-reg", "r2c-odd", "c2r-odd"} & set(forms)
        assert ("scatter" in forms) == (v["kind"] == "cols" and bool(v["full"]))
    if tier == 0:
        # B200FFT_PREFER matches substrings: each name must select exactly one variant
        clash = [(a, b) for a in names for b in names if a != b and a in b]
        assert not clash, clash
        kinds = {v["kind"] for v in info}
        assert kinds == {"rows", "rowsIP", "cols", "colsT"}

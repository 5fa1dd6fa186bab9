"""Host-only (no GPU): the scattering Z pass of the half-spectrum slab inverse (MGPU_SLAB with REAL_HALF, inverse) is a
kernel form only the plan-time tier builds. b200fft_jit_probe with half = 3 compiles it for sm_100a through NVRTC, as the
plan would at creation, in both working precisions, and refuses the axes the plan refuses with status 4."""
import re

import pytest

import b200fft


@pytest.mark.parametrize("n,inner,dtype", [(64, 16 * 33, "float32"), (64, 16 * 33, "float64"), (48, 20 * 51, "float32"),
                                           (48, 20 * 51, "float64"), (24, 10 * 23, "float32"), (256, 64 * 129, "float32")])
def test_scatter_z_form_compiles(n, inner, dtype):
    report = b200fft.jit_probe(n, inner=inner, inverse=True, half=3, in_dtype=dtype, out_dtype=dtype)
    name = report.split(":")[0]
    assert re.fullmatch(r"jitscatterZ%d_[0-9x]+_w\d+_t\d+%s" % (n, "_f64" if dtype == "float64" else ""), name), report
    assert "cols_scatter_kernel<%d, " % n in report and ", true, b200fft::ScatterZArgs>" in report, report


def test_scatter_z_form_refusals():
    with pytest.raises(b200fft.B200FFTError) as e:  # 4096 points of 6 columns: no column tile fits shared memory
        b200fft.jit_probe(4096, inner=6, inverse=True, half=3)
    assert e.value.status == 4 and "column tile" in str(e.value)
    with pytest.raises(b200fft.B200FFTError) as e:  # longer than any column tile
        b200fft.jit_probe(20000, inner=64, inverse=True, half=3)
    assert e.value.status == 4
    with pytest.raises(b200fft.B200FFTError) as e:  # only the plain probe has the form
        b200fft.jit_probe(64, inner=64, inverse=True, half=3, strided=True)
    assert e.value.status == 1

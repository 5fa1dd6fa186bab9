"""The two-pass forms of long real-input and half-spectrum axes compile for sm_100a through NVRTC on a machine
without a GPU (b200fft_jit_split_probe: the same host-side choice make_jit_split_pass makes, csrc/jit.cu)."""
import pytest

import b200fft


def _passes(**kw):
    a, b = b200fft.jit_split_probe(**kw).split("; ")
    assert "cubin=" in a and "cubin=" in b, (a, b)
    return a, b


@pytest.mark.parametrize("kw,want_a,want_b", [
    (dict(n=1 << 20, half=1), "cols_split_a_kernel<1024, b200fft::Radices<32, 32>, 8, 256, false>",
     "rows_split_b_r2c_kernel<512, b200fft::Radices<32, 16>, "),                                        # even R2C: H = 2^19
    (dict(n=1 << 20, half=2), "cols_split_a_c2r_kernel<1024, b200fft::Radices<32, 32>, 8, 256, false>",
     "rows_split_b_kernel<512, b200fft::Radices<32, 16>, 8, 128, true>"),                               # even C2R
    (dict(n=13125, half=1), "cols_split_a_kernel<25, b200fft::Radices<25>, 64, 64, false, true>",
     "rows_split_b_kernel<525, b200fft::Radices<25, 21>, 5, 128, false, 1>"),                           # odd R2C
    (dict(n=78125, half=2), "cols_split_a_c2r_kernel<625, b200fft::Radices<25, 25>, 8, 224, true>",
     "rows_split_b_kernel<125, b200fft::Radices<25, 5>, 25, 128, true, 2>"),                            # odd C2R
    (dict(n=1 << 18, real_in=True, in_dtype="uint8"), "cols_split_a_kernel<512, b200fft::Radices<32, 16>, 16, 256, false, true>",
     "rows_split_b_kernel<512, b200fft::Radices<32, 16>, 8, 128, false>"),                              # real uint8 input
    (dict(n=1 << 18, real_in=True, in_dtype="float64", inverse=True), "cols_split_a_kernel<512, b200fft::Radices<32, 16>, 16, 256, true, true>",
     "rows_split_b_kernel<512, b200fft::Radices<32, 16>, 8, 128, true>"),                               # real fp64 input, fp32 out
    (dict(n=1 << 18, half=1, in_dtype="float64", out_dtype="float64"), "cols_split_a_kernel<256, b200fft::Radices<16, 16>, 16, 256, false>",
     "rows_split_b_r2c_kernel<512, b200fft::Radices<8, 8, 8>, 4, 256>"),                                # fp64 R2C
    (dict(n=12000, half=2, in_dtype="float64", out_dtype="float64"), "cols_split_a_c2r_kernel<100, b200fft::Radices<10, 10>, 16, 160, false>",
     "rows_split_b_kernel<60, b200fft::Radices<10, 6>, 50, 320, true>"),                                # fp64 C2R
    (dict(n=20000, inner=6), "cols_split_a_kernel<", "cols_split_b_kernel<"),                            # complex strided axis
])
def test_split_forms_compile(kw, want_a, want_b):
    a, b = _passes(**kw)
    assert want_a in a, a
    assert want_b in b, b


def test_split_names_distinguish_forms():
    """Each form has its own variant name (and template id, the on-disk cache key)."""
    names = {}
    for kw in (dict(n=1 << 18), dict(n=1 << 18, real_in=True), dict(n=1 << 18, half=1), dict(n=1 << 18, half=2),
               dict(n=59049, half=1), dict(n=59049, half=2)):
        a, b = _passes(**kw)
        names[str(kw)] = (a.split(":")[0], b.split(":")[0])
    tags = [t for pair in names.values() for t in pair]
    for want in ("jitsplitA512", "_realin", "jitsplitBr2c", "jitsplitAc2r", "jitsplitBhalf", "jitsplitAc2rodd", "jitsplitBreal"):
        assert any(want in t for t in tags), (want, names)
    assert len(set(names.values())) == len(names), names


def test_split_probe_refusals():
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_split_probe(n=131 * 512, half=1, bases=[131, 512])   # a prime above 127: no split
    assert e.value.status == 4
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_split_probe(n=1 << 18, half=1, in_dtype="uint8")     # uint8 half spectrum: as on one tile, not served
    assert e.value.status == 4
    with pytest.raises(b200fft.B200FFTError):
        b200fft.jit_probe(26000, half=1)                                 # the single-tile probe keeps its meaning

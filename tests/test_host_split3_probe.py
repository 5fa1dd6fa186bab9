"""The three passes of contiguous axes longer than 2^24 points compile for sm_100a through NVRTC on a machine without a
GPU (b200fft_jit_split3_probe: the same host-side choice make_jit_split3_pass makes, csrc/jit.cu)."""
import re

import pytest

import b200fft


def _passes(n, **kw):
    parts = b200fft.jit_split3_probe(n=n, **kw).split("; ")
    assert len(parts) == 3, parts
    ids = []
    for p in parts:
        assert "cubin=" in p, p
        m = re.search(r": (b200fft::\w+<(\d+), )", p)
        assert m, p
        ids.append((m.group(1), int(m.group(2))))
    sizes = [s for _, s in ids]
    assert sizes[0] * sizes[1] * sizes[2] == n and max(sizes) <= 8192, (n, sizes)
    assert ids[0][0].startswith("b200fft::cols_split_a_kernel<") and ids[1][0].startswith("b200fft::cols_split_a_kernel<")
    assert ids[2][0].startswith("b200fft::rows_split_c_kernel<")
    return parts


@pytest.mark.parametrize("n,kw", [
    (1 << 25, {}),
    (1 << 28, {}),
    (1 << 31, {}),
    (3 ** 16, {}),
    (10 ** 8, {}),
    (1 << 26, dict(in_dtype="float64", out_dtype="float64")),
    (1 << 25, dict(real_in=True, in_dtype="uint8")),
    (1 << 25, dict(inverse=True)),
])
def test_split3_compiles(n, kw):
    a, b, c = _passes(n, **kw)
    # the two-table twiddle form of pass A (its last template argument), pass 3 with its own kernel
    assert re.search(r"cols_split_a_kernel<[^>]*>, \d+, \d+, (true|false), (true|false), true>", a), a
    assert re.search(r"cols_split_a_kernel<[^>]*>, \d+, \d+, (true|false), false, true>", b), b
    inv = "true" if kw.get("inverse") else "false"
    assert ", %s>" % inv in c.split(",  smem")[0].split(", smem")[0], c
    if kw.get("real_in"):
        assert "_realin_inu8" in a.split(":")[0] and ", false, true, true>" in a, a
    if kw.get("out_dtype") == "float64":
        assert all(p.split(":")[0].endswith("_f64") for p in (a, b, c)), (a, b, c)


def test_split3_names():
    """Each pass has a variant name of its own (the template id is the on-disk cache key)."""
    a, b, c = _passes(1 << 25)
    assert a.split(":")[0].startswith("jitsplit3A") and b.split(":")[0].startswith("jitsplit3A")
    assert c.split(":")[0].startswith("jitsplit3C")


@pytest.mark.parametrize("n,kw", [
    (1 << 24, {}),                                 # two passes serve it
    (1 << 26, dict(half=1)),                       # half-spectrum rows above 2^24 split points
    (131 << 18, dict(bases=[131] + [8] * 6)),      # a radix above 127
    (1 << 25, dict(inner=2)),                      # strided axis
])
def test_split3_refusals(n, kw):
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_split3_probe(n=n, **kw)
    assert e.value.status == 4


def test_two_pass_probe_unchanged():
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.jit_split_probe(n=1 << 25)
    assert e.value.status == 4

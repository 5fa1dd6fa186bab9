"""The strided kernel table (tests/_strided_forms.py) and the limits of strided plans, checked without a GPU.

Every probed row compiles its first pass for sm_100a through NVRTC and must report exactly the row's first tag. The
completeness tests fail when the table loses a kind, the fp64 half of a kind, an input type a kind accepts, the few-rows
or many-rows regime of a row kind, a few-rows / many-rows pair, a column-tile shape or a layout. The boundary tests pin
the longest axes one tile serves (the limits include/b200fft.h and INTEGRATION.md state), and the extent-1 tests that no
stride rule applies to a dimension no kernel reads.

Without a device a plan the layout rules accept fails at its first CUDA call, after the strided planner has chosen every
pass: a refusal of the planner is status 4 before that."""
import re

import pytest

import b200fft
from _strided_forms import ACCEPTED, F32, F64, FEW, FORMS, FP64_EXCEPTIONS, KINDS, MANY, logical_shape, strides_of

PROBED = [f for f in FORMS if f.probe]
ROW_KINDS = ("jitrows", "jitrowsIP")


@pytest.mark.parametrize("form", PROBED, ids=[f.id for f in PROBED])
def test_probe_names_the_first_kernel_of_the_row(form):
    report = b200fft.jit_probe(strided=True, **form.probe)
    name = report.split(":")[0]
    assert name == form.tags[0], (form.id, report)
    assert name.endswith("_str") and ("_f64" in name) == form.f64, name
    if form.kinds[0] in ROW_KINDS:
        assert form.rows() >= MANY, "%s: the probe plans for many rows, the row runs %d" % (form.id, form.rows())


def test_every_tag_is_a_strided_kernel():
    for f in FORMS:
        assert f.tags and all(t.endswith("_str") for t in f.tags), (f.id, f.tags)
        assert len(f.tags) == bin(f.axis_mask).count("1") if f.axis_mask else len(f.tags) == len(f.shape) - 1, f.id


def test_table_reaches_every_kind_in_both_precisions():
    seen = {}
    for f in FORMS:
        for k in f.kinds:
            seen.setdefault(k, set()).add(f.f64)
    for k in KINDS:
        want = {False} if (k, True) in FP64_EXCEPTIONS else {False, True}
        assert seen.get(k) == want, "%s in %s, wants %s" % (k, seen.get(k), want)
    assert len(KINDS) == 8 and not FP64_EXCEPTIONS


def test_table_reads_every_input_type_each_kind_accepts():
    seen = {}
    for f in FORMS:
        seen.setdefault(f.kinds[0], set()).add(f.reads())
    for k, want in ACCEPTED.items():
        assert seen.get(k, set()) == want, "%s reads %s, accepts %s" % (k, sorted(seen.get(k, set())), sorted(want))
    assert set(seen) <= set(ACCEPTED)


def test_row_kinds_run_at_few_and_many_rows():
    for k in ROW_KINDS:
        for prec in (False, True):
            rows = [f.rows() for f in FORMS if f.kinds[0] == k and f.f64 == prec and len(f.shape) == 2]
            assert any(r <= FEW for r in rows) and any(r >= MANY for r in rows), (k, prec, rows)


def test_few_and_many_rows_pairs_name_different_kernels():
    pairs = {}
    for f in FORMS:
        if f.pair:
            pairs.setdefault(f.pair, []).append(f)
    assert sorted(pairs) == ["10000", "2000", "3000", "f64-1024"], sorted(pairs)
    for key, (a, b) in pairs.items():
        few, many = (a, b) if a.rows() <= FEW else (b, a)
        assert few.rows() <= FEW and many.rows() >= MANY, key
        assert logical_shape(few)[1:] == logical_shape(many)[1:] and few.out_dtype == many.out_dtype, key
        assert many.probe and few.tags[0] != many.tags[0], (key, few.tags, many.tags)


def _w(tag):
    return int(re.search(r"_w(\d+)_", tag).group(1))


def test_column_tiles():
    cols = [f for f in FORMS if f.kinds[0] == "jitcols" and f.axis_mask == 1 and len(f.shape) == 3]
    widths = {(_w(f.tags[0]), f.shape[2]) for f in cols}
    assert any(w < 8 and w == c for w, c in widths), "no tile narrower than 8 columns"
    assert any(c % w for w, c in widths), "no ragged last tile"
    assert any(w == 64 for w, _ in widths), "no 64-wide tile"
    assert any("127x" in f.tags[0] or "x127_" in f.tags[0] for f in cols), "no looped prime 127"
    longest = {(f.shape[1], f.f64) for f in cols}
    assert (1024, False) in longest and (512, True) in longest, "the longest column axes of each precision"
    # an odd n/2 + 1 column count in the pass after the R2C rows / before the C2R rows
    assert any(f.half and len(f.shape) == 3 and (f.shape[-1] // 2 + 1) % 2 == 1 and "jitcols" in f.kinds for f in FORMS)


def test_layouts():
    st = {f.id: strides_of(f) for f in FORMS}
    assert any(s[0][-1] > 1 and s[1][-1] > 1 for s in st.values()), "element stride > 1 along the axis"
    assert any(s[0][0] == 1 for s in st.values()), "batch-interleaved (batch stride 1)"
    assert any(len(f.shape) == 9 and f.axis_mask and sorted(st[f.id][0]) != st[f.id][0][::-1] for f in FORMS), "rank 8"
    assert any(f.half and len(f.shape) == 3 for f in FORMS), "N-d half spectrum in the padded layout"
    for k in KINDS:
        assert any(f.kinds[0] == k and any(f.offset) for f in FORMS), "%s never reads a view at an element offset" % k


# ---- the longest axes one tile serves -------------------------------------------------------------------------------
def _served(dt, shape, in_strides, **kw):
    """True when the strided planner builds every pass (status 0 on a device, a CUDA error without one); False on its
    status-4 refusal, which must name the shared-memory budget"""
    try:
        b200fft.plan_fft(dt, dt, shape, shape, in_strides=in_strides, **kw).destroy()
        return True
    except b200fft.B200FFTError as e:
        if e.status == 4:
            msg = str(e)
            assert "200 KB shared-memory budget" in msg and ("fp64" if dt == F64 else "fp32") in msg, msg
            return False
        assert e.status == 5, str(e)  # no device
        return True


def _rows(dt, n, count):
    return _served(dt, (count, n, 2), [n + 16, 1])


def _cols(dt, n, cols=16):
    return _served(dt, (2, n, cols, 2), [n * cols + 3, cols, 1], axis_mask=1)  # axis 0 alone, across `cols` columns


# `beyond`: a length served past the longest power of two. Only fp32 columns serve one past the refused power of two too
# (2304 = 48 x 48 > 2048: two stages need one exchange buffer, not two). Rows and fp64 columns cannot: a rowsIP tile holds
# n points plus padding (200 KB: 25600 fp32 / 12800 fp64 points), and an fp64 column axis above 256 points has 3+ stages
# (radices up to 16), two buffers of n x 8 columns x 16 B (800 points: exactly 200 KB). So for those `beyond` lies between
# the longest power of two served and the refused one.
@pytest.mark.parametrize("what,dt,longest,beyond", [
    ("rows", F32, 16384, 20000),
    ("rows", F64, 8192, 12500),
    ("columns", F32, 1024, 2304),
    ("columns", F64, 512, 800),
], ids=["rows-fp32", "rows-fp64", "columns-fp32", "columns-fp64"])
def test_tile_boundary(what, dt, longest, beyond):
    # rows at few and at many rows (the planner's rows_hint picks a different row kernel); column tiles take no rows_hint
    checks = [lambda n: _rows(dt, n, 2), lambda n: _rows(dt, n, MANY)] if what == "rows" else [lambda n: _cols(dt, n)]
    for fn in checks:
        assert fn(longest), "%s of %d points (%s) are not served" % (what, longest, dt)
        assert not fn(2 * longest), "%s of %d points (%s) are served" % (what, 2 * longest, dt)
        assert fn(beyond), "%s of %d points (%s) are not served" % (what, beyond, dt)
    if what == "columns":
        # a tile of 5 columns (fewer than 8: the tile is the column count) takes the axis a wider tile cannot
        assert _cols(dt, 2 * longest, 5)


def test_refusal_names_the_stage_list_and_the_dtype():
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft(F32, F32, (4, 100, 2), (4, 100, 2), bases=[[100]], in_strides=[300, 1])
    assert e.value.status == 4 and "codelets" in str(e.value), str(e.value)
    with pytest.raises(b200fft.B200FFTError) as e:
        b200fft.plan_fft(F32, F64, (4, 33, 2), (4, 64, 1), real_mode=b200fft.REAL_HALF, inverse=True, in_strides=[40, 1])
    assert e.value.status == 4 and "working precision" in str(e.value), str(e.value)
    with pytest.raises(b200fft.B200FFTError) as e:  # (plan_fft refuses uint8 half spectra before the planner)
        b200fft.jit_probe(64, half=1, in_dtype="uint8", strided=True)
    assert e.value.status == 4 and "floating-point input" in str(e.value), str(e.value)


# ---- strides of extent-1 dimensions -----------------------------------------------------------------------------------
def _no_stride_error(*args, **kw):
    try:
        b200fft.plan_fft(*args, **kw).destroy()
    except b200fft.B200FFTError as e:
        assert "stride" not in str(e) and e.status == 5, str(e)  # no device: the first CUDA call


@pytest.mark.parametrize("s", [0, 7, -3, 2 ** 40])
def test_batch_of_one_takes_any_stride(s):
    _no_stride_error(F32, F32, (1, 1024, 2), (1, 1024, 2), in_strides=[s, 1], out_strides=[s, 1])
    _no_stride_error(F32, F32, (1, 1024, 1), (1, 513, 2), real_mode=b200fft.REAL_HALF, in_strides=[s, 1],
                     out_strides=[520, 1])
    _no_stride_error(F32, F32, (1, 513, 2), (1, 1024, 1), real_mode=b200fft.REAL_HALF, inverse=True,
                     in_strides=[520, 1], out_strides=[s, 1])
    # a single 65536-point row sliced from a wider buffer: the dense plan, not a refusal
    _no_stride_error(F32, F32, (1, 65536, 2), (1, 65536, 2), in_strides=[2 * 65536 + s, 1])


@pytest.mark.parametrize("s", [0, 7, -3, 2 ** 40])
def test_masked_axis_of_one_point_takes_any_stride(s):
    shape = (4, 1, 100, 2)
    _no_stride_error(F32, F32, shape, shape, axis_mask=0b10, in_strides=[108, s, 1], out_strides=[110, s, 1])
    real, cplx = (4, 1, 64, 1), (4, 1, 33, 2)
    _no_stride_error(F32, F32, real, cplx, real_mode=b200fft.REAL_HALF, axis_mask=0b10, in_strides=[66, s, 1],
                     out_strides=[40, s, 1])

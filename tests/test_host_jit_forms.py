"""The table of plan-time kernel forms (tests/_jit_forms.py), checked without a GPU.

Every row with a host probe compiles the axis for sm_100a through NVRTC and must report exactly the kernels the row
names, suffixes included (_f64, _inu8, _inf64, _inf32, _realin). The probes plan as for many rows, so a planner change
that silently moves a large-batch case off its kind fails here. tests/test_gpu_jit_forms.py runs the same rows on a
B200 and asserts that the plans name the same kernels.

The completeness tests fail when the table loses a kind, the fp64 half of a kind, an input type a kind accepts, or one
half of a few-rows / many-rows pair."""
import re

import pytest

import b200fft
from _jit_forms import ACCEPTED, FEW, FORMS, FP32_ONLY, KINDS, MANY, F64, logical_shape, readers

PROBES = {"jit": b200fft.jit_probe, "split": b200fft.jit_split_probe, "split3": b200fft.jit_split3_probe}
PROBED = [f for f in FORMS if f.probe]
ROW_KINDS = ("jitrows", "jitrowsIP")  # the kinds whose kernel depends on the number of rows (jit_plan_axis: rows_hint)


@pytest.mark.parametrize("form", PROBED, ids=[f.id for f in PROBED])
def test_probe_names_the_kernels_of_the_row(form):
    fn, kw = form.probe
    report = PROBES[fn](**kw)
    names = [part.split(":")[0].strip() for part in report.split("; ")]
    assert names == form.tags, (form.id, report)
    for name in names:
        assert name.endswith("_f64") or "_f64_" in name if form.f64 else "_f64" not in name, name
    if form.kinds[0] in ROW_KINDS:
        assert form.rows() >= MANY, "%s: the probe plans for many rows, the row runs %d" % (form.id, form.rows())


def test_table_reaches_every_kind_in_both_precisions():
    seen = {}
    for f in FORMS:
        for k in f.kinds:
            seen.setdefault(k, set()).add(f.f64)
    missing = [k for k in KINDS if k not in seen]
    assert not missing, "kinds no row reaches: %s" % missing
    for k in KINDS:
        want = {False} if k in FP32_ONLY else {False, True}
        assert seen[k] == want, "%s appears in %s, wants %s" % (k, sorted("fp64" if p else "fp32" for p in seen[k]),
                                                               sorted("fp64" if p else "fp32" for p in want))
    assert len(KINDS) == 21 and len(set(KINDS)) == 21


def test_table_reads_every_input_type_each_kind_accepts():
    seen = {}
    for f in FORMS:
        for k in readers(f):
            seen.setdefault(k, set()).add(f.reads())
    for k, want in ACCEPTED.items():
        assert seen.get(k, set()) == want, "%s reads %s, accepts %s" % (k, sorted(seen.get(k, set())), sorted(want))
    assert set(seen) <= set(ACCEPTED), "kinds reading the user's array without an ACCEPTED entry: %s" % (set(seen) - set(ACCEPTED))


def test_row_kinds_run_at_few_and_many_rows():
    for k in ROW_KINDS:
        rows = [f.rows() for f in FORMS if f.kinds[0] == k]
        for regime, ok in (("few", lambda r: r <= FEW), ("many", lambda r: r >= MANY)):
            for prec in (False, True):
                assert any(ok(f.rows()) for f in FORMS if f.kinds[0] == k and f.f64 == prec), (
                    "no %s row of %s at %s rows" % ("fp64" if prec else "fp32", k, regime))
        assert rows


def test_few_and_many_rows_pairs_name_different_kernels():
    pairs = {}
    for f in FORMS:
        if f.pair:
            pairs.setdefault(f.pair, []).append(f)
    assert len(pairs) >= 4, sorted(pairs)
    for key, forms in pairs.items():
        assert len(forms) == 2, (key, forms)
        few = [f for f in forms if f.rows() <= FEW]
        many = [f for f in forms if f.rows() >= MANY]
        assert len(few) == 1 and len(many) == 1, (key, [(f.id, f.rows()) for f in forms])
        a, b = few[0], many[0]
        assert logical_shape(a)[1:] == logical_shape(b)[1:] and a.bases == b.bases, key
        assert (a.in_dtype, a.out_dtype, a.comps, a.inverse) == (b.in_dtype, b.out_dtype, b.comps, b.inverse), key
        assert b.probe, "%s: the many-rows row must be probed" % key
        ta, tb = a.tags[0], b.tags[0]
        assert not tb.startswith(ta) and not ta.startswith(tb), "%s: %s at few rows, %s at many" % (key, ta, tb)


def _radices(tag):
    return [int(r) for r in re.match(r"jit[A-Za-z0-9]*?\d+_([0-9x]+)_", tag).group(1).split("x")]


def test_rows_ip_stage_order():
    """rows_ip keeps the descending stage order where its middle stages fit the register budget and permutes it
    otherwise; a looped prime (more than 64 values per thread) is never a middle stage."""
    marked = [f for f in FORMS if f.permuted is not None]
    assert any(f.permuted for f in marked) and any(not f.permuted for f in marked)
    for f in marked:
        r = _radices(f.tags[0])
        assert (r != sorted(r, reverse=True)) == f.permuted, (f.id, r)
        assert all(x <= 64 for x in r[1:-1]), (f.id, r)

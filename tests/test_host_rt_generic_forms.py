"""The table of runtime-length and generic kernel forms (tests/_rt_generic_forms.py), checked without a GPU.

For every row, the dry_run stage lists put through the rule copies must route each pass to the row's kind: an rt pass
must fit the rt tier, a generic pass behind FORCE_RT, B200FFT_JIT=0 or no switch must be one the rt tier (and, with no
switch, the plan-time tier) refuses, and a refused row must fit no kernel. tests/test_gpu_rt_generic_forms.py asserts on
a B200 that the plans print exactly the lines these rules predict.

The completeness test fails when the table stops reaching a codelet of one of the four rt kernels, a stage count, an
input type, a tile width of the generic kernel, a wrapping grid or one of the routes that reach these kernels with no
switch set."""
import pytest

from _rt_generic_forms import (F32, F64, FLAG_FORCE_GENERIC, FLAG_FORCE_RT, FORMS, GEN_MAX_STAGES, RT_GRID_PER_SM,
                               SM_COUNT, U8, by_id, dry_passes, expected_lines, generic_geometry, group_stages,
                               rt_geometry, tiles)

JIT_MAX_RADIX = 127  # jit.cu: the plan-time tier's codelets stop at prime 127


def _rt_forced(form):
    return bool(form.flags & FLAG_FORCE_RT) or form.env.get("B200FFT_JIT") == "0"


def _jit_refuses(form, p):
    """jit.cu jit_plan_axis, the two refusals the table relies on."""
    c2r_other_precision = p["half"] == "c2r" and p["reads_input"] and form.in_dtype != form.out_dtype
    return any(r > JIT_MAX_RADIX for r in p["stages"]) or c2r_other_precision


@pytest.mark.parametrize("form", FORMS, ids=[f.id for f in FORMS])
def test_rules_route_the_row_to_its_kinds(form):
    passes = dry_passes(form)
    assert len(passes) == len(form.kinds), (form.id, passes)
    for p, kind in zip(passes, form.kinds):
        rt = rt_geometry(p["n"], p["inner"], p["stages"], f64_out=form.f64, half=p["half"])
        gen = generic_geometry(p["n"], p["inner"], f64_out=form.f64, nstages=len(p["stages"]))
        if form.refused:
            assert rt is None and gen is None, (form.id, p)
            continue
        if kind.startswith("rt_"):
            assert not form.flags & FLAG_FORCE_GENERIC
            assert rt is not None and rt["row"] == (kind == "rt_rows"), (form.id, p, rt)
            if not _rt_forced(form):
                assert _jit_refuses(form, p), (form.id, p)
        elif kind.startswith("generic_"):
            assert gen is not None and gen["row"] == (kind == "generic_rows"), (form.id, p, gen)
            if not form.flags & FLAG_FORCE_GENERIC:
                assert rt is None, "%s: the rt tier would serve %s" % (form.id, p)
            if not form.flags and not form.env:
                assert _jit_refuses(form, p), "%s: the plan-time tier would serve %s" % (form.id, p)
        else:
            assert kind == "jit" and not form.flags and not _jit_refuses(form, p), (form.id, p)
    if not form.refused:
        assert len(expected_lines(form)) == len(form.kinds)


def _reached():
    """Everything the table reaches, as a set of tuples."""
    got = set()
    for f in FORMS:
        if f.refused:
            continue
        for i, (p, kind) in enumerate(zip(dry_passes(f), f.kinds)):
            if kind.startswith("rt_"):
                g = rt_geometry(p["n"], p["inner"], p["stages"], f64_out=f.f64, half=p["half"])
                for R in g["radices"]:
                    got.add(("codelet", g["rmaxk"], f.inverse, R))
                if g["rmaxk"] == 32 and min(g["radices"]) <= 16:
                    got.add(("small in large",))
                got.add(("S", g["S"]))
                if g["row"] and any(g["padded"]):
                    got.add(("rows exchange", "padded"))
                if g["row"] and any(g["dense_odd"]):
                    got.add(("rows exchange", "dense"))
                if not g["row"]:
                    got.add(("rt cols", "inner < 8")) if p["inner"] < 8 else None
                    got.add(("rt cols", "ragged")) if p["inner"] > g["tile"] and p["inner"] % g["tile"] else None
                    got.add(("rt cols", "in place")) if not p["reads_input"] else None
                if p["reads_input"]:
                    mode = p["half"] or "full"
                    got.add(("rt reads", mode, f.reads()))
                if p["half"]:
                    got.add(("rt half", p["half"], p["n"] % 2))
                nt = tiles(f, p, g["tile"])
                if g["row"] and nt > SM_COUNT * RT_GRID_PER_SM and tiles(f, p, 1) % g["tile"]:
                    got.add(("rt wraps", f.inverse))
            elif kind.startswith("generic_"):
                g = generic_geometry(p["n"], p["inner"], f64_out=f.f64, nstages=len(p["stages"]))
                got.add(("generic", f.f64, kind))
                got.add(("generic reads", p["half"] or "c2c", f.f64, f.reads())) if p["reads_input"] else None
                got.add(("generic C", f.f64, kind, g["C"]))
                if not g["row"] and p["inner"] < (8 if f.f64 else 16):
                    got.add(("generic cols inner < C", f.f64))
                big = [r for r in p["stages"] if r > JIT_MAX_RADIX]
                if big:
                    assert p["stages"].index(big[0]) == 0 and len(big) == 1, (f.id, p)
                    got.add(("prime > 127", "alone" if len(p["stages"]) == 1 else "with small stages", kind))
                    if any(k == "jit" for k in f.kinds):
                        got.add(("prime > 127", "outer axis after plan-time passes", kind))
                nt = tiles(f, p, g["C"])
                if g["row"] and nt > SM_COUNT * g["per_sm"] and tiles(f, p, 1) % g["C"]:
                    got.add(("generic wraps", f.f64))
                if f.flags == 0 and not f.env:
                    got.add(("no switch", kind, p["half"]))
    return got


def test_table_reaches_every_form():
    got = _reached()
    missing = []

    def want(item):
        if item not in got:
            missing.append(item)

    # rt tier: every codelet in each of the four kernels
    for inverse in (False, True):
        for R in range(2, 17):
            want(("codelet", 16, inverse, R))
        for R in range(17, 33):
            want(("codelet", 32, inverse, R))
        want(("rt wraps", inverse))
    want(("small in large",))
    for S in range(1, 6):  # S = 1: no exchange buffer, S = 2: one, S >= 3: two
        want(("S", S))
    want(("rows exchange", "padded"))
    want(("rows exchange", "dense"))
    for what in ("inner < 8", "ragged", "in place"):
        want(("rt cols", what))
    for d in (U8, F32, F64):
        for c in (1, 2):
            want(("rt reads", "full", (d, c)))
    for d in (F32, F64):
        want(("rt reads", "r2c", (d, 1)))
        want(("rt reads", "c2r", (d, 2)))
    for half in ("r2c", "c2r"):
        for odd in (0, 1):
            want(("rt half", half, odd))

    # generic kernel
    for f64 in (False, True):
        for kind in ("generic_rows", "generic_cols"):
            want(("generic", f64, kind))
        for d in (U8, F32, F64):
            for c in (1, 2):
                want(("generic reads", "c2c", f64, (d, c)))
        for d in (F32, F64):
            want(("generic reads", "r2c", f64, (d, 1)))
            want(("generic reads", "c2r", f64, (d, 2)))
        want(("generic C", f64, "generic_rows", 64))
        want(("generic C", f64, "generic_rows", 1))
        for C in ((8, 4, 2, 1) if f64 else (16, 8, 4, 2, 1)):
            want(("generic C", f64, "generic_cols", C))
        want(("generic cols inner < C", f64))
        want(("generic wraps", f64))
    want(("prime > 127", "alone", "generic_rows"))
    want(("prime > 127", "with small stages", "generic_rows"))
    want(("prime > 127", "outer axis after plan-time passes", "generic_cols"))
    for kind, half in (("generic_rows", ""), ("generic_cols", ""), ("generic_rows", "r2c"), ("generic_rows", "c2r")):
        want(("no switch", kind, half))
    assert not missing, "the table does not reach: %s" % missing


def test_named_rows():
    """The rows the issue of these kernels names: the accuracy primes, the longest lengths, the no-switch routes."""
    f = by_id()
    for id, n, f64 in (("prime-14519", 14519, False), ("prime-7253-f64", 7253, True), ("longest-14528", 14528, False),
                       ("longest-7264-f64", 7264, True), ("refused-14529", 14529, False), ("refused-7265-f64", 7265, True)):
        p = dry_passes(f[id])[0]
        assert p["n"] == n and f[id].f64 == f64
        assert (generic_geometry(n, 1, f64_out=f64) is None) == bool(f[id].refused)
    for n in range(14519 + 1, 14528):  # 14519 is the largest prime that fits in fp32, 7253 in fp64
        assert any(n % d == 0 for d in range(2, 121)), n
    for n in range(7253 + 1, 7264):
        assert any(n % d == 0 for d in range(2, 86)), n
    assert generic_geometry(14528, 1)["smem"] == 227 * 1024 == generic_geometry(7264, 1, f64_out=True)["smem"]
    for id in ("prime-131", "prime-1009", "prime-8191", "prime-131x2", "prime-131-r2c", "prime-131-c2r"):
        assert f[id].flags == 0 and not f[id].env
    assert f["c2r-f32-to-f64"].kinds == ["generic_rows"] and f["c2r-f32-to-f64"].flags == 0
    assert f["c2r-f64-to-f32"].kinds == ["rt_rows"] and f["c2r-f64-to-f32"].flags == 0
    assert f["force-rt-f64-out"].flags == FLAG_FORCE_RT and f["force-rt-f64-out"].out_dtype == F64
    assert f["force-rt-radix37"].flags == FLAG_FORCE_RT and 37 in dry_passes(f["force-rt-radix37"])[0]["stages"]
    assert f["rt-s5-7776"].in_dtype == F32 and rt_geometry(7776, 1, [6] * 5)["smem"] > 140 * 1024


def test_rule_copies_on_known_cases():
    """A few values worked out by hand from rt.cu and generic.cu."""
    assert group_stages([5, 5, 2, 2]) == [10, 10]
    assert group_stages([5, 5, 5, 2, 2, 2]) == [10, 10, 10]
    assert group_stages([3] * 5) == [27, 9]
    assert group_stages([3] * 7) == [27, 9, 9]  # balanced over the fewest groups, not greedy
    assert group_stages([37, 2]) is None and group_stages([6] * 7) is None
    # S = 6 needs six groups of at least 6 (a group of 5 or less merges with a 6): 6^6 points, more than one tile holds
    assert group_stages([6] * 6) == [6] * 6 and rt_geometry(6 ** 6, 1, [6] * 6) is None
    g = rt_geometry(1000, 1, [5, 5, 5, 2, 2, 2])
    assert (g["tile"], g["S"], g["padded"], g["rmaxk"]) == (6, 3, [True, True], 16)
    assert g["smem"] == 2 * 6 * (1000 + 100) * 8
    g = rt_geometry(992, 870, [32, 31])
    assert (g["row"], g["tile"], g["smem"], g["rmaxk"]) == (False, 12, 992 * 12 * 8, 32)
    assert rt_geometry(1000, 1, [10, 10, 10], f64_out=True) is None
    assert generic_geometry(100, 1) == dict(C=64, smem=64 * 1600, per_sm=2, row=True)
    assert generic_geometry(14519, 1)["C"] == 1 and generic_geometry(14529, 1) is None
    assert generic_geometry(20, 36, f64_out=True)["C"] == 8 and generic_geometry(100, 5)["C"] == 5
    assert generic_geometry(10, 1, nstages=GEN_MAX_STAGES + 1) is None

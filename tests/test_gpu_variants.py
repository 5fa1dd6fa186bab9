"""Every compiled-in kernel variant, forced one at a time, against numpy float64.

The planner launches the first registered variant that matches an axis, so most variants only run when a base list
excludes the earlier ones or B200FFT_PREFER / B200FFT_FUSED_PREFER moves them to the front. This sweep enumerates the
three registries with b200fft.variant_info (0: row / column kernels, 1: fused N-d kernels, 2: two-pass split kernels)
and runs each (variant, form) pair the variant instantiates:

  * it forces the variant and asserts that plan.describe() names it, so a silent fallback fails;
  * shapes hit the ragged edges: one row and 2 * tile + 3 rows, strided axes whose inner extent is not a multiple of
    the tile (odd for the LDG column kernels, tile + 6 for the TMA ones, which need an even extent);
  * fp32 tolerance vs numpy float64 (tests/test_gpu_parity.py): relative L2 <= 2e-6, max-abs <= 1e-5 * max|X|;
  * the output is prefilled with NaN and lies between 4 KB guard bands that must come back untouched (stores past
    the end or before the start of the output would change them);
  * the input is unchanged by an out-of-place run, an in-place run gives the identical result, the launch counter
    moves by plan.launches, and the default plan of the same problem agrees to 1e-6.

It also checks the pointer-alignment rule of b200fft_exec (include/b200fft.h): 16-byte offsets work everywhere,
pointers less aligned than a plan's kernels need are refused before any launch, and kernels declared 8-byte-safe
run at an 8-byte offset."""
import os

import numpy as np
import pytest

import b200fft

pytestmark = pytest.mark.gpu

RTOL_L2, RTOL_MAX = 2e-6, 1e-5
GUARD = 4096
SENTINEL = 0xA5

_ENV = ("B200FFT_PREFER", "B200FFT_R2C_SMEM", "B200FFT_FUSED", "B200FFT_PLANE", "B200FFT_FUSED_PREFER",
        "B200FFT_ROWS_INPLACE", "B200FFT_PLANE_C2R")


def _info(tier):
    # collected on machines without a GPU too (the ids come from the host-only registry listing)
    try:
        return b200fft.variant_info(tier)
    except b200fft.B200FFTError:
        return []


FAST, FUSED, SPLIT = _info(0), _info(1), _info(2)


def _primes(n):
    out, p = [], 2
    while n > 1:
        if n % p == 0:
            out.append(p)
            while n % p == 0:
                n //= p
        p += 1
    return out


@pytest.fixture(autouse=True)
def _clean_env(monkeypatch):
    for k in _ENV:
        monkeypatch.delenv(k, raising=False)


# ---- running one plan ------------------------------------------------------------------------------------------------

class Buf:
    """A device buffer of `nbytes` between two guard bands of SENTINEL bytes; `ptr` is the first byte after the front
    band (plus `offset`, for the alignment tests)."""

    def __init__(self, nbytes, fill_nan=True, offset=0):
        import torch
        self.nbytes, self.offset = nbytes, offset
        self.raw = torch.full((GUARD + offset + nbytes + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        if fill_nan:
            assert nbytes % 4 == 0
            self.body().view(torch.float32).fill_(float("nan"))
        self.ptr = self.raw.data_ptr() + GUARD + offset

    def body(self):
        return self.raw[GUARD + self.offset:GUARD + self.offset + self.nbytes]

    def load(self, data):
        import torch
        self.body().copy_(torch.from_numpy(np.ascontiguousarray(data).view(np.uint8).reshape(-1)).cuda())

    def numpy(self, dtype):
        return self.body().cpu().numpy().view(dtype)

    def guards_intact(self):
        front = self.raw[:GUARD + self.offset]
        back = self.raw[GUARD + self.offset + self.nbytes:]
        return bool((front == SENTINEL).all().item()) and bool((back == SENTINEL).all().item())


def _layouts(shape, real_in, half, inverse):
    """(in_layout, out_layout) of a plan over the logical array `shape` = (batch, dims...)."""
    if half:
        cplx = tuple(shape[:-1]) + (shape[-1] // 2 + 1, 2)
        real = tuple(shape) + (1,)
        return (cplx, real) if inverse else (real, cplx)
    return tuple(shape) + ((1,) if real_in else (2,)), tuple(shape) + (2,)


def _reference(x, axes, real_in, half, inverse, n_last):
    """numpy float64 of the same transform; x is the float64 input array in its own layout. Arrays of more than 2^25
    points (the 512^3 fused variants) take torch.fft in float64 on the device instead, which is much faster there."""
    if x.size > 2 ** 25 and not half:
        import torch
        t = torch.from_numpy(x).cuda()
        z = t[..., 0].to(torch.complex128) if real_in else torch.view_as_complex(t.contiguous())
        r = (torch.fft.ifftn if inverse else torch.fft.fftn)(z, dim=axes)
        return r.cpu().numpy()
    if half and inverse:
        z = x[..., 0] + 1j * x[..., 1]
        return np.fft.irfftn(z, s=[n_last] if len(axes) == 1 else None, axes=axes)
    z = x[..., 0] if (real_in or half) else x[..., 0] + 1j * x[..., 1]
    if half:
        return np.fft.rfftn(z, axes=axes)
    return np.fft.ifftn(z, axes=axes) if inverse else np.fft.fftn(z, axes=axes)


def _as_complex(a):
    return a[..., 0].astype(np.float64) + 1j * a[..., 1]


def _check_close(got, want, what):
    assert np.isfinite(got).all(), "%s: non-finite output (unwritten elements or NaN arithmetic)" % what
    err = np.linalg.norm(got - want) / np.linalg.norm(want)
    mx = np.abs(got - want).max() / np.abs(want).max()
    assert err <= RTOL_L2 and mx <= RTOL_MAX, "%s: rel-L2 %.2e, max-abs %.2e vs float64" % (what, err, mx)


def run_case(shape, *, axes, real_in=False, half=False, inverse=False, bases=None, axis_mask=0, expect=None,
             launches=None, in_place=None, seed=0):
    """Plan + exec with guard bands around the output, checked against float64. Returns (result, describe text)."""
    import torch
    rng = np.random.default_rng(seed)
    in_layout, out_layout = _layouts(shape, real_in, half, inverse)
    x = rng.standard_normal(in_layout).astype(np.float32)
    if half and inverse:  # a Hermitian half spectrum: the transform of real data
        xr = rng.standard_normal(shape)
        z = np.fft.rfftn(xr, axes=axes) / np.sqrt(np.prod([shape[a] for a in axes]))
        x = np.stack([z.real, z.imag], axis=-1).astype(np.float32)
    plan = b200fft.plan_fft("float32", "float32", in_layout, out_layout, bases=bases, inverse=inverse,
                            real_mode=b200fft.REAL_HALF if half else b200fft.REAL_FULL, axis_mask=axis_mask)
    try:
        desc = plan.describe()
        if expect is not None:
            for name in ([expect] if isinstance(expect, str) else expect):
                assert name in desc, "%s was not used: %s" % (name, desc)
        if launches is not None:
            assert plan.launches == launches, desc
        xin = torch.from_numpy(x).cuda()
        x_before = xin.clone()
        out = Buf(int(np.prod(out_layout)) * 4)
        before = b200fft.launch_count()
        plan.exec(out.ptr, xin)
        torch.cuda.synchronize()
        assert b200fft.launch_count() - before == plan.launches
        assert out.guards_intact(), "store outside the output array: %s" % desc
        assert torch.equal(xin, x_before), "an out-of-place run changed its input: %s" % desc
        got = out.numpy(np.float32).reshape(out_layout)
        want = _reference(x.astype(np.float64), axes, real_in, half, inverse, shape[-1])
        got_c = got[..., 0].astype(np.float64) if (half and inverse) else _as_complex(got)
        _check_close(got_c, want, desc.strip())
        if in_place if in_place is not None else (not real_in and not half):
            io = Buf(int(np.prod(out_layout)) * 4, fill_nan=False)
            io.load(x)
            plan.exec(io.ptr, io.ptr)
            torch.cuda.synchronize()
            assert io.guards_intact(), "in place: store outside the array: %s" % desc
            assert np.array_equal(io.numpy(np.float32).reshape(out_layout), got), "in place differs: %s" % desc
        return got, desc
    finally:
        plan.destroy()


def run_default(shape, **kw):
    """The same problem on the default plan (no forced variant, default bases)."""
    for k in _ENV:
        os.environ.pop(k, None)
    kw = dict(kw, bases=None, expect=None, launches=None)
    return run_case(shape, **kw)[0]


def agree(a, b, what):
    a, b = a.astype(np.float64), b.astype(np.float64)
    err = np.linalg.norm(a - b) / np.linalg.norm(b)
    assert err <= 1e-6, "%s: %.2e from the default plan" % (what, err)


# ---- tier 0: row / column variants -----------------------------------------------------------------------------------

def _fast_cases():
    out = []
    for v in FAST:
        for f in v["forms"]:
            out.append(pytest.param(v, f, id="%s-%s" % (v["name"], f)))
    return out


@pytest.mark.parametrize("v,form", _fast_cases())
def test_fast_variant(monkeypatch, v, form):
    name, n, rad, tile = v["name"], v["n"], v["radices"], v["tile"]
    monkeypatch.setenv("B200FFT_PREFER", name)
    if form in ("r2c", "c2r", "r2c-reg"):
        if form == "r2c" and "r2c-reg" in v["forms"]:
            monkeypatch.setenv("B200FFT_R2C_SMEM", "1")
        tag = {"r2c": "r2c[", "c2r": "c2r[", "r2c-reg": "r2c-reg["}[form] + name + "]"
        for batch in (1, 2 * tile + 3):
            kw = dict(axes=(1,), half=True, inverse=form == "c2r", bases=[[2] + rad], expect=tag, launches=1)
            got, _ = run_case((batch, 2 * n), **kw)
            agree(got, run_default((batch, 2 * n), **kw), name)
            monkeypatch.setenv("B200FFT_PREFER", name)
            if form == "r2c" and "r2c-reg" in v["forms"]:
                monkeypatch.setenv("B200FFT_R2C_SMEM", "1")
        return
    if form in ("r2c-odd", "c2r-odd"):
        tag = form + "[" + name + "]"
        for batch in (1, 2 * tile + 3):
            kw = dict(axes=(1,), half=True, inverse=form == "c2r-odd", bases=[rad], expect=tag, launches=1)
            got, _ = run_case((batch, n), **kw)
            agree(got, run_default((batch, n), **kw), name)
            monkeypatch.setenv("B200FFT_PREFER", name)
        return
    if v["kind"] in ("rows", "rowsIP"):
        shapes = [(1, n), (2 * tile + 3, n)]
        kw = dict(axes=(1,), bases=[rad])
    else:
        inner = tile + 6 if v["kind"] == "colsT" else tile + 5  # a ragged last column tile; TMA needs an even extent
        shapes = [(1, n, inner), (3, n, inner)]
        kw = dict(axes=(1,), bases=[rad, [inner]], axis_mask=1)
    if form == "scatter":
        for shape in shapes:
            _run_scatter(shape, name, rad)
            _run_scatter(shape, name, rad, inverse=True)
        return
    directions = [(False, True), (True, True)] if form == "real" else [(form == "inv", False)]
    for inverse, real_in in directions:
        for shape in shapes:
            c = dict(kw, inverse=inverse, real_in=real_in)
            got, desc = run_case(shape, expect=name + " ", launches=1, **c)
            assert ("real-in" in desc) == real_in, desc
            agree(got, run_default(shape, **c), name)
            monkeypatch.setenv("B200FFT_PREFER", name)


def _run_scatter(shape, name, rad, inverse=False):
    """exec_scatter with one peer: the scattering store of the column kernel writes the natural layout."""
    import torch
    rng = np.random.default_rng(1)
    layout = tuple(shape) + (2,)
    x = rng.standard_normal(layout).astype(np.float32)
    plan = b200fft.plan_fft("float32", "float32", layout, layout, bases=[rad, [shape[2]]], inverse=inverse, axis_mask=1)
    try:
        assert name + " " in plan.describe()
        xin = torch.from_numpy(x).cuda()
        out = Buf(x.nbytes)
        work = Buf(x.nbytes)
        before = b200fft.launch_count()
        plan.exec_scatter([out.ptr], 0, xin, work.ptr)
        torch.cuda.synchronize()
        assert b200fft.launch_count() - before == 1
        assert out.guards_intact() and work.guards_intact()
        want = (np.fft.ifft if inverse else np.fft.fft)(_as_complex(x.astype(np.float64)), axis=1)
        _check_close(_as_complex(out.numpy(np.float32).reshape(layout)), want, "scatter " + name)
    finally:
        plan.destroy()


NOT_FULL = [v for v in FAST if v["kind"] in ("rows", "cols") and not v["full"]]


@pytest.mark.parametrize("v", NOT_FULL, ids=[v["name"] for v in NOT_FULL])
def test_tuning_variant_is_skipped_where_it_has_no_kernel(monkeypatch, v):
    """A variant registered for forward complex only must not be picked for an inverse or real-input request even
    when B200FFT_PREFER names it: the planner takes another variant and the result is still right."""
    monkeypatch.setenv("B200FFT_PREFER", v["name"])
    n, tile = v["n"], v["tile"]
    if v["kind"] == "rows":
        shape, kw = (2 * tile + 3, n), dict(axes=(1,), bases=[_primes(n)])
    else:
        inner = tile + 5
        shape, kw = (3, n, inner), dict(axes=(1,), bases=[_primes(n), [inner]], axis_mask=1)
    _, desc = run_case(shape, **kw)
    assert v["name"] + " " in desc  # forward complex: the preferred variant itself
    for inverse, real_in in ((True, False), (False, True), (True, True)):
        _, desc = run_case(shape, inverse=inverse, real_in=real_in, **kw)
        assert v["name"] not in desc, desc


# ---- tier 1: fused N-d variants --------------------------------------------------------------------------------------

@pytest.mark.parametrize("v", FUSED, ids=[v["name"] for v in FUSED])
def test_fused_variant(monkeypatch, v):
    dims = [int(d) for d in v["n"].split("x")]
    mode, inverse = v["mode"], v["forms"] == ["inv"]
    big = int(np.prod(dims)) >= 512 ** 3
    for batch in ((1,) if big else (1, 2)):
        for k in _ENV:
            monkeypatch.delenv(k, raising=False)
        monkeypatch.setenv("B200FFT_FUSED", "1")
        monkeypatch.setenv("B200FFT_PLANE", "0")
        monkeypatch.setenv("B200FFT_FUSED_PREFER", v["name"] + ":")
        shape = (batch,) + tuple(dims)
        kw = dict(axes=tuple(range(1, len(dims) + 1)), real_in=mode == "real", half=mode == "r2c", inverse=inverse,
                  bases=[_primes(d) for d in dims])
        got, _ = run_case(shape, expect="fused " + v["name"] + ":", launches=1, **kw)
        if not big:
            agree(got, run_default(shape, **kw), v["name"])


# ---- tier 2: two-pass split pairs ------------------------------------------------------------------------------------

def _can_group(ordered, target):
    """fast_registry.cu: can_group — partition the stage list into groups with exactly the target products."""
    if not target:
        return not ordered
    want, rest_t = target[-1], target[:-1]

    def rec(i, prod, chosen):
        if prod == want:
            remaining = [o for j, o in enumerate(ordered) if j not in chosen]
            return _can_group(remaining, rest_t)
        if i >= len(ordered) or prod > want:
            return False
        if want % (prod * ordered[i]) == 0 and rec(i + 1, prod * ordered[i], chosen | {i}):
            return True
        return rec(i + 1, prod, chosen)
    return rec(0, 1, frozenset())


def _split_pairs():
    a_side = [k for k in SPLIT if k["kind"] == "splitA"]
    b_side = [k for k in SPLIT if k["kind"] != "splitA"]
    return [(a, b) for a in a_side for b in b_side if b["kind"] == "splitB_cols" or a["n"] % b["tile"] == 0]


def _split_winner(ordered, n, rows):
    """The pair make_split_pass picks for this stage list (first A, then first B, in registration order)."""
    for a, b in _split_pairs():
        if a["n"] * b["n"] == n and (b["kind"] == "splitB_rows") == rows and _can_group(ordered, a["radices"] + b["radices"]):
            return a, b
    return None


# Pairs no base list reaches: an earlier pair has the same multiset of stages, so every stage list that groups into
# the listed pair groups into the earlier one first (make_split_pass takes the first match in registration order).
SAME_STAGES = "an earlier pair with the same stages (%s) is picked for every base list"
UNREACHABLE = {
    ("splitA_cols256_16x16_w16_t256", "splitB_rows128_16x8_c32_t256"):
        SAME_STAGES % "splitA_cols128_16x8 + splitB_rows256_16x16",
    ("splitA_cols256_16x16_w16_t256", "splitB_rows64_8x8_c32_t256"):
        SAME_STAGES % "splitA_cols128_16x8 + splitB_rows128_16x8",
    ("splitA_cols64_8x8_w16_t128", "splitB_rows128_16x8_c32_t256"):
        SAME_STAGES % "splitA_cols128_16x8 + splitB_rows64_8x8",
    ("splitA_cols64_8x8_w16_t128", "splitB_rows256_16x16_c16_t256"):
        SAME_STAGES % "splitA_cols128_16x8 + splitB_rows128_16x8",
}


def _split_cases():
    out = []
    for a, b in _split_pairs():
        out.append(pytest.param(a, b, id="%s+%s" % (a["name"], b["name"])))
    return out


def _fast_preempts(ordered, n, rows):
    for v in FAST:
        if v["n"] != n or not _can_group(ordered, v["radices"]):
            continue
        if rows and v["kind"] in ("rows", "rowsIP"):
            return v["name"]
        if not rows and v["kind"] == "cols":
            return v["name"]
    return None


def split_reachable(a, b):
    """(True, bases) when the pair's own radices as bases select it; (False, reason) otherwise."""
    n, rows = a["n"] * b["n"], b["kind"] == "splitB_rows"
    bases = a["radices"] + b["radices"]
    ordered = sorted(bases, reverse=True)
    pre = _fast_preempts(ordered, n, rows)
    if pre:
        return False, "single-tile variant %s groups the same stage list" % pre
    win = _split_winner(ordered, n, rows)
    if win != (a, b):
        return False, "%s + %s comes first for the same stage list" % (win[0]["name"], win[1]["name"])
    return True, bases


@pytest.mark.parametrize("a,b", _split_cases())
def test_split_pair(a, b):
    n, rows = a["n"] * b["n"], b["kind"] == "splitB_rows"
    ok, why = split_reachable(a, b)
    key = (a["name"], b["name"])
    if key in UNREACHABLE:
        # listed as unreachable: the pair's own stages select the earlier pair, on the host rule and on the device
        assert not ok, "%s + %s is reachable with bases %s: remove it from UNREACHABLE" % (key + (why,))
        bases = a["radices"] + b["radices"]
        shape = (1, n) if rows else (1, n, 3)
        kw = dict(axes=(1,), bases=[bases] if rows else [bases, [3]], axis_mask=0 if rows else 1)
        _, desc = run_case(shape, **kw)
        assert not (a["name"] in desc and b["name"] in desc), desc
        return
    assert ok, "%s + %s cannot be reached (%s): list it in UNREACHABLE with the reason" % (key + (why,))
    for inverse in (False, True):
        if rows:
            shapes = [(1, n), (3, n)]
            kw = dict(axes=(1,), bases=[why])
        else:
            inner = b["tile"] + 5
            shapes = [(1, n, inner), (2, n, inner)]
            kw = dict(axes=(1,), bases=[why, [inner]], axis_mask=1)
        for shape in shapes:
            c = dict(kw, inverse=inverse)
            got, _ = run_case(shape, expect=[a["name"] + " ", b["name"] + " "], launches=2, **c)
            agree(got, run_default(shape, **c), a["name"] + " + " + b["name"])


# ---- pointer alignment -----------------------------------------------------------------------------------------------

# one plan of every kind: (label, logical shape, run_case keywords, environment)
PLAN_KINDS = [
    ("rowsV (128-bit rows)", (37, 128), dict(axes=(1,)), {}),
    ("rows (LDG rows)", (19, 1024), dict(axes=(1,)), {}),
    ("rowsIP", (3, 4096), dict(axes=(1,)), {}),
    ("cols (LDG)", (2, 64, 21), dict(axes=(1,), axis_mask=1), {}),
    ("colsT (TMA)", (2, 64, 22), dict(axes=(1,), axis_mask=1), {"B200FFT_PREFER": "colsT64_"}),
    ("real-input rows", (5, 256), dict(axes=(1,), real_in=True), {}),
    ("r2c", (9, 1024), dict(axes=(1,), half=True), {}),
    ("c2r", (9, 1024), dict(axes=(1,), half=True, inverse=True), {}),
    ("r2c odd", (9, 93), dict(axes=(1,), half=True, bases=[[31, 3]]), {}),
    ("split", (2, 1920), dict(axes=(1,)), {}),
    ("plane + cols 3-D", (2, 64, 64, 64), dict(axes=(1, 2, 3)), {}),
    ("plane r2c 3-D", (2, 64, 64, 64), dict(axes=(1, 2, 3), half=True), {}),
    ("plane c2r 2-D", (3, 64, 64), dict(axes=(1, 2), half=True, inverse=True), {}),
    ("fused v2 (bulk-async)", (1, 64, 64, 64), dict(axes=(1, 2, 3)), {"B200FFT_FUSED": "1", "B200FFT_PLANE": "0"}),
    ("specialised at plan time", (7, 96), dict(axes=(1,)), {}),
    ("specialised r2c", (7, 200), dict(axes=(1,), half=True), {}),
]


def run_offset(shape, in_offset, out_offset, *, axes, real_in=False, half=False, inverse=False, bases=None, axis_mask=0):
    """Plan + exec with input and output at the given byte offsets past a 16-byte aligned address. Returns (status,
    result, reference, launches counted, plan description)."""
    import torch
    rng = np.random.default_rng(3)
    in_layout, out_layout = _layouts(shape, real_in, half, inverse)
    x = rng.standard_normal(in_layout).astype(np.float32)
    if half and inverse:
        z = np.fft.rfftn(rng.standard_normal(shape), axes=axes)
        x = np.stack([z.real, z.imag], axis=-1).astype(np.float32)
    plan = b200fft.plan_fft("float32", "float32", in_layout, out_layout, bases=bases, inverse=inverse,
                            real_mode=b200fft.REAL_HALF if half else b200fft.REAL_FULL, axis_mask=axis_mask)
    try:
        src = Buf(x.nbytes, fill_nan=False, offset=in_offset)
        src.load(x)
        out = Buf(int(np.prod(out_layout)) * 4, offset=out_offset)
        before = b200fft.launch_count()
        status = b200fft.lib().b200fft_exec(plan._h, out.ptr, src.ptr, None)
        torch.cuda.synchronize()
        counted = b200fft.launch_count() - before
        assert out.guards_intact() and src.guards_intact()
        got = out.numpy(np.float32).reshape(out_layout)
        got = got[..., 0].astype(np.float64) if (half and inverse) else _as_complex(got)
        return status, got, _reference(x.astype(np.float64), axes, real_in, half, inverse, shape[-1]), counted, plan.describe()
    finally:
        plan.destroy()


@pytest.mark.parametrize("label,shape,kw,env", PLAN_KINDS, ids=[p[0] for p in PLAN_KINDS])
def test_every_plan_kind_accepts_16_byte_offsets(monkeypatch, label, shape, kw, env):
    """16 bytes is the most any kernel needs: an allocation offset by 16 must work on every plan kind (and catches any
    assumption of 128- or 256-byte aligned buffers)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    status, got, want, counted, desc = run_offset(shape, 16, 16, **kw)
    assert status == 0, b200fft.lib().b200fft_last_error().decode()
    assert counted >= 1
    _check_close(got, want, label + ": " + desc)
    if "B200FFT_PREFER" in env:
        assert env["B200FFT_PREFER"] in desc


@pytest.mark.parametrize("label,shape,kw,env,offsets,pointer", [
    ("rowsV (float4 loads)", (37, 128), dict(axes=(1,)), {}, (8, 0), "d_in"),
    ("rowsV (float4 stores)", (37, 128), dict(axes=(1,)), {}, (0, 8), "d_out"),
    ("colsT (tensor maps)", (2, 64, 22), dict(axes=(1,), axis_mask=1), {"B200FFT_PREFER": "colsT64_"}, (8, 8), "d_in"),
    ("fused v2 (bulk copies)", (1, 64, 64, 64), dict(axes=(1, 2, 3)), {"B200FFT_FUSED": "1", "B200FFT_PLANE": "0"}, (0, 8),
     "d_out"),
    ("r2c (real rows read as float2 pairs)", (9, 1024), dict(axes=(1,), half=True), {}, (4, 0), "d_in"),
    ("c2r (real rows stored as float2 pairs)", (9, 1024), dict(axes=(1,), half=True, inverse=True), {}, (0, 4), "d_out"),
])
def test_underaligned_pointers_are_refused_before_any_launch(monkeypatch, label, shape, kw, env, offsets, pointer):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    status, got, _, counted, desc = run_offset(shape, *offsets, **kw)
    assert status == 1, (label, status, desc)
    assert counted == 0, "a refused exec launched %d kernels" % counted
    msg = b200fft.lib().b200fft_last_error().decode()
    assert "aligned to" in msg and msg.startswith(pointer), msg
    assert np.isnan(got.real).all(), "a refused exec wrote its output"


@pytest.mark.parametrize("label,shape,kw,env", [
    ("rows1024 (8-byte loads)", (19, 1024), dict(axes=(1,)), {}),
    ("rows64 without 128-bit accesses", (37, 64), dict(axes=(1,)), {"B200FFT_PREFER": "rows64_8x8_"}),
    ("cols (LDG)", (2, 64, 21), dict(axes=(1,), axis_mask=1), {}),
    ("split", (2, 1920), dict(axes=(1,)), {}),
    ("r2c odd (scalar loads)", (9, 93), dict(axes=(1,), half=True, bases=[[31, 3]]), {}),
])
def test_8_byte_safe_plans_run_at_8_byte_offsets(monkeypatch, label, shape, kw, env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    status, got, want, counted, desc = run_offset(shape, 8, 8, **kw)
    assert status == 0, b200fft.lib().b200fft_last_error().decode()
    _check_close(got, want, label + ": " + desc)
    if "B200FFT_PREFER" in env:
        assert env["B200FFT_PREFER"] in desc

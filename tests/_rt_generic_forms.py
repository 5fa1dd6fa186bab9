"""One table of problems that reach every form of the runtime-length kernel (csrc/rt.cu, rt_axis_kernel) and of the
generic kernel (csrc/generic.cu, gen_fft_kernel), with plain-Python copies of the host rules that decide what each
problem reaches.

Each row is a problem (logical shape, dtypes, input components, half spectrum, direction, bases, axis mask, flags and
environment) and the kinds of its passes in launch order: "rt_rows" / "rt_cols" (runtime-length tier),
"generic_rows" / "generic_cols" (generic kernel) and "jit" (a plan-time NVRTC kernel). A row with `refused` set must be
refused at plan creation with status 4 and that text in the message.

The rule copies take the per-axis stage lists of b200fft.dry_run, which needs no GPU:
  * group_stages (rt.cu: group_stages) gives the super-stages, hence the codelets and the kernel: RMAXK = 16 when the
    largest super-stage is at most 16, else 32;
  * rt_geometry (rt.cu: make_rt_pass) gives the tile, which exchanges are padded, the stage count S and the shared
    memory;
  * generic_geometry (generic.cu: make_generic_pass) gives the tile C and the shared memory, hence per_sm and the grid.
From them `expected_lines` builds the exact plan.describe() line of every rt and generic pass.
tests/test_gpu_rt_generic_forms.py asserts that the plan prints those lines, so the copies cannot drift from the planner
unnoticed; tests/test_host_rt_generic_forms.py checks, without a GPU, that the rules route every row to its kinds and
that the table reaches every form.

Shapes are logical: (batch, dims...) of the real-side array."""
import re
from math import prod

F32, F64, U8 = "float32", "float64", "uint8"
FLAG_FORCE_GENERIC, FLAG_FORCE_RT = 1, 16  # b200fft.FLAG_*
JIT_OFF = {"B200FFT_JIT": "0"}             # the plan-time tier off: what it would serve goes to the rt tier

SM_COUNT = 148                             # B200
RT_MAX_RADIX, RT_MAX_STAGES, RT_THREADS = 32, 6, 256
MAX_SMEM = 227 * 1024
GEN_MAX_STAGES = 40
RT_GRID_PER_SM = 32                        # rt grid = min(tiles, SMs x 32)


# ---- rule copies -------------------------------------------------------------------------------------------------

def parse_dry_run(text):
    """The passes of a dry_run text, in launch order."""
    out = []
    for line in text.strip().split("\n"):
        m = re.match(r"axis (\d+): n=(\d+) inner=(\d+) stages=\[([\d,]*)\]( r2c| c2r)? \((reads input|in place)\)$", line)
        assert m, line
        out.append(dict(axis=int(m.group(1)), n=int(m.group(2)), inner=int(m.group(3)),
                        stages=[int(v) for v in m.group(4).split(",")], half=(m.group(5) or "").strip(),
                        reads_input=m.group(6) == "reads input"))
    return out


def group_stages(ordered):
    """rt.cu group_stages: the fewest super-stages of product <= 32, largest first; None when a base is above 32 or no
    grouping into RT_MAX_STAGES exists."""
    if any(r > RT_MAX_RADIX for r in ordered):
        return None
    bases = sorted(ordered, reverse=True)
    for want in range(1, RT_MAX_STAGES + 1):
        g = [1] * want
        ok = True
        for b in bases:
            best = -1
            for i in range(want):
                if g[i] * b <= RT_MAX_RADIX and (best < 0 or g[i] < g[best]):
                    best = i
            if best < 0:
                ok = False
                break
            g[best] *= b
        if not ok:
            continue
        out = [v for v in sorted(g, reverse=True) if v > 1]
        return out or [1]
    return None


def rt_geometry(n, inner, stages, *, f64_out=False, half=""):
    """rt.cu make_rt_pass: the pass's geometry, or None when the rt tier refuses the axis."""
    if f64_out or n > (1 << 20) or (half and inner != 1):
        return None
    radices = group_stages(stages)
    if radices is None:
        return None
    S, row = len(radices), inner == 1
    rmax = max(radices)
    tile = (2 * RT_THREADS * rmax + n - 1) // n
    if row:
        tile = max(1, tile)
    else:
        tile = max(16, (tile + 7) // 8 * 8)
        tile = min(tile, (inner + 7) // 8 * 8)
        tile = max(1, tile)
    P, max_stride, padded, Qs = 1, n, [], []
    for s, R in enumerate(radices):
        Q = P * R
        pad = row and P < 16 and Q % 2 == 0 and Q < n
        padded.append(pad)
        Qs.append(Q)
        stride = n + (n // Q * P if pad else 0)
        if s + 1 < S:
            max_stride = max(max_stride, stride)
        P = Q
    nbuf = 2 if S > 2 else (1 if S > 1 else 0)

    def smem_for(t):
        return nbuf * (t * max_stride if row else n * t) * 8

    min_tile = 1 if row else min(8, inner)
    while tile > min_tile and smem_for(tile) > 112 * 1024:
        tile = max(min_tile, (tile + 1) // 2)
    if smem_for(tile) > MAX_SMEM:
        return None
    # the exchanges are those written by stages 0..S-2; padded only on rows (P < 16 and Q even)
    return dict(radices=radices, S=S, row=row, tile=tile, smem=smem_for(tile), rmaxk=16 if rmax <= 16 else 32,
                padded=padded[:-1], dense_odd=[Q % 2 == 1 for Q in Qs[:-1]], nbuf=nbuf)


def generic_geometry(n, inner, *, f64_out=False, nstages=1):
    """generic.cu make_generic_pass: tile C and shared memory, or None (status 4) when one transform does not fit."""
    sz = 16 if f64_out else 8
    per_transform = 2 * n * sz
    if nstages > GEN_MAX_STAGES or per_transform > MAX_SMEM:
        return None
    row = inner == 1
    if row:
        C = max(1, min(64, 100 * 1024 // per_transform))
        while C > 1 and C * n > 8192:
            C //= 2
        C = max(C, 1)
    else:
        C = 8 if f64_out else 16
        while C > 1 and C * per_transform > MAX_SMEM:
            C //= 2
        while C > 1 and C * per_transform > 100 * 1024 and C * sz > 64:
            C //= 2
        C = min(C, inner)
    smem = C * per_transform
    per_sm = max(1, min(8, MAX_SMEM // max(smem, 1)))
    return dict(C=C, smem=smem, per_sm=per_sm, row=row)


def tiles(form, p, tile):
    """Tiles of pass p (a parse_dry_run entry) at `tile` rows / columns per CTA."""
    batch, dims = form.shape[0], form.shape[1:]
    if p["half"]:
        outer = batch * prod(dims[:-1])
    else:
        count = batch * (prod(dims[:-1]) * (dims[-1] // 2 + 1) if form.half else prod(dims))
        outer = count // (p["n"] * p["inner"])
    if p["inner"] == 1:
        return -(-outer // tile)
    return outer * -(-p["inner"] // tile)


# ---- the table ---------------------------------------------------------------------------------------------------

class Form:
    def __init__(self, id, shape, kinds, *, in_dtype=F32, out_dtype=F32, comps=2, half=False, inverse=False, bases=None,
                 axis_mask=0, flags=0, env=None, refused=None, note=""):
        self.id, self.shape, self.kinds = id, tuple(shape), list(kinds)
        self.in_dtype, self.out_dtype, self.comps, self.half, self.inverse = in_dtype, out_dtype, comps, half, inverse
        self.bases, self.axis_mask, self.flags, self.env = bases, axis_mask, flags, dict(env or {})
        self.refused, self.note = refused, note

    @property
    def f64(self):
        return self.out_dtype == F64

    def reads(self):
        """(input dtype, components) of the user's array as the first pass reads it."""
        return (self.in_dtype, 1 if (self.half and not self.inverse) else self.comps)

    def layouts(self):
        """(in_layout, out_layout) of the plan."""
        if self.half:
            cplx = self.shape[:-1] + (self.shape[-1] // 2 + 1, 2)
            real = self.shape + (1,)
            return (cplx, real) if self.inverse else (real, cplx)
        return self.shape + (self.comps,), self.shape + (2,)

    def __repr__(self):
        return self.id


def _rt(id, shape, kinds=None, **kw):
    kw.setdefault("flags", FLAG_FORCE_RT)
    if kinds is None:
        kinds = ["rt_rows"] + ["rt_cols"] * (len(shape) - 2)
    return Form(id, shape, kinds, **kw)


def _gen(id, shape, kinds=None, **kw):
    kw.setdefault("flags", FLAG_FORCE_GENERIC)
    if kinds is None:
        kinds = ["generic_rows"] + ["generic_cols"] * (len(shape) - 2)
    return Form(id, shape, kinds, **kw)


def _gcols(id, n, inner, **kw):
    """The strided axis of (2, n, inner) alone on the generic kernel."""
    return _gen(id, (2, n, inner), ["generic_cols"], axis_mask=1, **kw)


WRAP_RT_ROWS = RT_GRID_PER_SM * SM_COUNT * 6 + 1     # 1000-point rows, tile 6: one tile more than the grid, ragged
WRAP_GEN_ROWS = 2 * SM_COUNT * 64 + 1                # C = 64 at two CTAs per SM: one tile more than the grid, ragged

FORMS = [
    # ---- rt tier: the cases of the earlier hand-picked list, with their ids ---------------------------------------
    _rt("shape0-None-False-float32-2", (50, 1000)),
    _rt("shape1-bases1-True-float32-2", (50, 1000), bases=[[10, 10, 10]], inverse=True),
    _rt("shape2-bases2-False-float32-2", (33, 100), bases=[[5, 2]]),
    _rt("shape3-None-False-float32-2", (9, 343), note="7^3: Q odd, dense exchanges"),
    _rt("shape4-None-False-float32-2", (6, 31 * 29), note="two large primes, one stage each"),
    _rt("shape5-bases5-True-float32-2", (4, 2187), bases=[[3]], inverse=True, note="3^7 -> (27)(9)(9)"),
    _rt("shape6-None-False-float32-2", (3, 30, 21)),
    _rt("shape7-None-True-float32-2", (2, 12, 100, 18), inverse=True),
    _rt("shape8-None-False-float32-1", (5, 600), comps=1, note="real input, full spectrum"),
    _rt("shape9-None-False-uint8-1", (3, 50, 36), in_dtype=U8, comps=1),
    _rt("shape10-None-False-float64-2", (4, 225), in_dtype=F64, note="f64 in, f32 out"),
    _rt("shape11-None-False-float32-2", (2, 4000)),
    _rt("shape12-None-False-float32-2", (1, 10000)),
    _rt("shape13-None-False-float32-2", (7, 17, 1000), note="long strided axis next to a long contiguous one; ragged"),

    # ---- rt tier: every codelet in each of the four kernels -------------------------------------------------------
    # one axis per codelet R = 2..9, S = 1 each: rows, then columns at inner 9 .. 181440
    _rt("rt-codelets-2to9", (1, 2, 3, 4, 5, 6, 7, 8, 9)),
    _rt("rt-codelets-2to9-inv", (1, 2, 3, 4, 5, 6, 7, 8, 9), inverse=True),
    # bases whose pairwise products exceed 32 stay one super-stage each
    _rt("rt-codelets-16x15x14", (3, 3360), bases=[[16, 15, 14]]),
    _rt("rt-codelets-16x15x14-inv", (3, 3360), bases=[[16, 15, 14]], inverse=True),
    _rt("rt-codelets-13x12x11", (3, 1716), bases=[[13, 12, 11]]),
    _rt("rt-codelets-13x12x11-inv", (3, 1716), bases=[[13, 12, 11]], inverse=True),
    _rt("rt-s4-10x9x8x7", (2, 5040), bases=[[10, 9, 8, 7]]),
    _rt("rt-s4-10x9x8x7-inv", (2, 5040), bases=[[10, 9, 8, 7]], inverse=True),
    # the RMAXK = 32 kernel: R = 17..32, and radix 2 as the smaller stage of (17)(2)
    _rt("rt-codelets-32x31-30x29", (2, 992, 870), bases=[[32, 31], [30, 29]]),
    _rt("rt-codelets-32x31-30x29-inv", (2, 992, 870), bases=[[32, 31], [30, 29]], inverse=True),
    _rt("rt-codelets-28x27-26x25", (2, 756, 650), bases=[[28, 27], [26, 25]]),
    _rt("rt-codelets-28x27-26x25-inv", (2, 756, 650), bases=[[28, 27], [26, 25]], inverse=True),
    _rt("rt-codelets-24x23-22x21", (2, 552, 462), bases=[[24, 23], [22, 21]]),
    _rt("rt-codelets-24x23-22x21-inv", (2, 552, 462), bases=[[24, 23], [22, 21]], inverse=True),
    _rt("rt-codelets-20x19x18", (3, 6840), bases=[[20, 19, 18]]),
    _rt("rt-codelets-20x19x18-inv", (3, 6840), bases=[[20, 19, 18]], inverse=True),
    _rt("rt-codelets-17x2", (9, 34), bases=[[17, 2]]),
    _rt("rt-codelets-17x2-inv", (9, 34), bases=[[17, 2]], inverse=True),
    # S = 5: no two 6s fit under 32; the rows tile needs about 145 KB. S = 6 (RT_MAX_STAGES) needs six super-stages of
    # at least 6 (one of 5 or less would merge with another), so at least 6^6 points: more than one tile of two exchange
    # buffers holds, so no axis reaches it
    _rt("rt-s5-7776", (2, 7776), bases=[[6]]),

    # ---- rt tier: input types of the pass that reads the user's array -----------------------------------------------
    _rt("rt-u8-complex", (3, 50, 36), in_dtype=U8),
    _rt("rt-f64-real", (5, 600), in_dtype=F64, comps=1, inverse=True),
    _rt("rt-cols-inner5", (3, 100, 5), ["rt_cols"], axis_mask=1, note="inner < 8: the tile is the inner extent"),
    _rt("rt-cols-ragged", (2, 1000, 35), ["rt_cols"], axis_mask=1, inverse=True, note="tile 16 over 35 columns"),
    # half spectrum: R2C and C2R rows at even and odd lengths, fp32 and fp64 on the user's side
    _rt("rt-r2c-even", (6, 600), half=True, comps=1),
    _rt("rt-r2c-odd-f64", (6, 243), half=True, comps=1, in_dtype=F64),
    _rt("rt-c2r-even-f64", (6, 600), half=True, inverse=True, in_dtype=F64),
    _rt("rt-c2r-odd", (6, 243), half=True, inverse=True),
    _rt("rt-r2c-2d", (3, 30, 200), half=True, comps=1, note="columns over the 101-bin half spectrum"),
    _rt("rt-c2r-2d", (3, 30, 200), ["rt_cols", "rt_rows"], half=True, inverse=True),
    # more tiles than SMs x 32: the grid-stride loop wraps, and the last tile is ragged
    _rt("rt-wrap", (WRAP_RT_ROWS, 1000)),
    _rt("rt-wrap-inv", (WRAP_RT_ROWS, 1000), bases=[[10, 10, 10]], inverse=True),
    # B200FFT_JIT=0 instead of the flag
    _rt("rt-jit-off", (4, 1000), flags=0, env=JIT_OFF),
    _rt("rt-jit-off-f64-out", (4, 600), ["generic_rows"], flags=0, env=JIT_OFF, out_dtype=F64,
        note="the rt tier writes fp32 only"),

    # ---- forced routes that land on the generic kernel ----------------------------------------------------------
    _rt("force-rt-f64-out", (4, 1000), ["generic_rows"], out_dtype=F64),
    _rt("force-rt-radix37", (4, 74), ["generic_rows"], note="37 x 2: the rt codelets stop at 32"),

    # ---- generic kernel: every input type, rows (C = 64) then columns (C = 16 / 8), fp32 and fp64 out ----------------
    *[_gen("gen-2d-%s-c%d-to-f%s" % (d, c, o[5:]), (3, 20, 36), in_dtype=d, comps=c, out_dtype=o, inverse=(c == 1))
      for o in (F32, F64) for d in (U8, F32, F64) for c in (1, 2)],
    # half spectrum on rows, with fp32 and fp64 on each side
    *[_gen("gen-r2c-%s-to-%s" % (d[5:], o[5:]), (5, 200 if d == o else 243), half=True, comps=1, in_dtype=d, out_dtype=o)
      for d in (F32, F64) for o in (F32, F64)],
    *[_gen("gen-c2r-%s-to-%s" % (d[5:], o[5:]), (5, 243 if d == o else 200), half=True, inverse=True, in_dtype=d, out_dtype=o)
      for d in (F32, F64) for o in (F32, F64)],
    _gen("gen-r2c-2d", (3, 30, 200), half=True, comps=1, out_dtype=F64),
    _gen("gen-c2r-2d", (3, 30, 200), ["generic_cols", "generic_rows"], half=True, inverse=True),
    # column tiles halved from 16 (fp32) / 8 (fp64) down to 1 as the axis grows, and an inner extent below C
    _gcols("gen-cols-c16", 100, 19),
    _gcols("gen-cols-c8", 1000, 19, inverse=True),
    _gcols("gen-cols-c4", 2000, 19),
    _gcols("gen-cols-c2", 5000, 19),
    _gcols("gen-cols-c1", 10000, 3, inverse=True),
    _gcols("gen-cols-inner5", 100, 5),
    _gcols("gen-cols-c8-f64", 100, 11, in_dtype=F64, out_dtype=F64),
    _gcols("gen-cols-c4-f64", 1000, 11, in_dtype=F64, out_dtype=F64, inverse=True),
    _gcols("gen-cols-c2-f64", 2000, 11, in_dtype=F64, out_dtype=F64),
    _gcols("gen-cols-c1-f64", 5000, 3, in_dtype=F64, out_dtype=F64),
    _gcols("gen-cols-inner3-f64", 100, 3, in_dtype=F64, out_dtype=F64),
    # rows at C = 1, and more tiles than SMs x per_sm (C = 64, two CTAs per SM) with a ragged last tile
    _gen("gen-rows-c1", (3, 5000)),
    _gen("gen-wrap", (WRAP_GEN_ROWS, 100)),
    _gen("gen-wrap-f64", (WRAP_GEN_ROWS, 50), in_dtype=F64, out_dtype=F64, inverse=True),

    # ---- generic kernel without a switch: prime radices above the plan-time tier's 127 ---------------------------------
    # stages run in descending order and any two factors of 128 or more exceed one tile, so within a tile such a
    # prime is always stage 0
    _gen("prime-131", (16, 131), bases=[[131]], flags=0),
    _gen("prime-131x2", (16, 262), bases=[[131, 2]], flags=0),
    _gen("prime-1009", (8, 1009), bases=[[1009]], flags=0, inverse=True),
    _gen("prime-8191", (8, 8191), bases=[[8191]], flags=0),
    _gen("prime-257-outer", (2, 257, 36, 20), ["jit", "jit", "generic_cols"], bases=[[257], [6, 6], [5, 4]], flags=0,
         in_dtype=F64, note="fp64 input keeps the plane kernels off: one pass per axis"),
    _gen("prime-131-r2c", (6, 131), half=True, comps=1, bases=[[131]], flags=0),
    _gen("prime-131-c2r", (6, 131), half=True, inverse=True, bases=[[131]], flags=0),
    _gen("c2r-f32-to-f64", (5, 600), half=True, inverse=True, out_dtype=F64, flags=0,
         note="the plan-time tier reads a C2R input in the working precision only, the rt tier writes fp32 only"),
    _rt("c2r-f64-to-f32", (5, 600), half=True, inverse=True, in_dtype=F64, flags=0,
        note="the plan-time tier refuses the fp64 input, the compiled-in kernels want fp32: the rt tier serves it"),
    # the largest primes one tile holds: the accuracy rows
    _gen("prime-14519", (8, 14519), bases=[[14519]], flags=0),
    _gen("prime-7253-f64", (8, 7253), bases=[[7253]], flags=0, in_dtype=F64, out_dtype=F64),
    # the longest lengths one tile holds (exactly 227 KB), and the next lengths, refused
    _gen("longest-14528", (3, 14528), bases=[[227, 2]], flags=0, inverse=True),
    _gen("longest-7264-f64", (3, 7264), bases=[[227, 2]], flags=0, in_dtype=F64, out_dtype=F64),
    _gen("refused-14529", (2, 14529), bases=[[167, 29, 3]], flags=0, refused="shared-memory tile"),
    _gen("refused-7265-f64", (2, 7265), bases=[[1453, 5]], flags=0, in_dtype=F64, out_dtype=F64,
         refused="shared-memory tile"),
]

RUNS = [f for f in FORMS if not f.refused]
REFUSED = [f for f in FORMS if f.refused]


def by_id():
    return {f.id: f for f in FORMS}


def dry_passes(form):
    import b200fft
    in_layout, out_layout = form.layouts()
    return parse_dry_run(b200fft.dry_run(form.in_dtype, form.out_dtype, in_layout, out_layout, bases=form.bases,
                                         inverse=form.inverse, real_mode=b200fft.REAL_HALF if form.half else b200fft.REAL_FULL,
                                         axis_mask=form.axis_mask, flags=form.flags))


def rt_line(form, p, g):
    """The plan.describe() line of rt pass p with geometry g (rt.cu: make_rt_pass)."""
    suffix = {"r2c": " r2c (n-point, bins 0..n/2 stored)", "c2r": " c2r (Hermitian load)"}.get(p["half"], "")
    if not suffix and p["reads_input"] and form.comps == 1:
        suffix = " real-in"
    return "axis %d: rt_%s n=%d inner=%d tile=%d smem=%dB user stages=[%s] fused as (%s)%s" % (
        p["axis"], "rows" if g["row"] else "cols", p["n"], p["inner"], g["tile"], g["smem"],
        ",".join(map(str, p["stages"])), "x".join(map(str, g["radices"])), suffix)


def generic_line(form, p, g):
    """The plan.describe() line of generic pass p with geometry g (generic.cu: make_generic_pass)."""
    return "axis %d: generic<%s>%s n=%d inner=%d tile=%d smem=%dB stages=[%s]" % (
        p["axis"], "f64" if form.f64 else "f32", (" " + p["half"]) if p["half"] else "", p["n"], p["inner"], g["C"],
        g["smem"], ",".join(map(str, p["stages"])))


def geometry(form, p, kind):
    if kind.startswith("rt_"):
        return rt_geometry(p["n"], p["inner"], p["stages"], f64_out=form.f64, half=p["half"])
    if kind.startswith("generic_"):
        return generic_geometry(p["n"], p["inner"], f64_out=form.f64, nstages=len(p["stages"]))
    return None


def expected_lines(form):
    """(kind, exact describe line or None for a plan-time pass) per pass, in launch order."""
    passes = dry_passes(form)
    assert len(passes) == len(form.kinds), (form.id, passes)
    out = []
    for p, kind in zip(passes, form.kinds):
        g = geometry(form, p, kind)
        if kind.startswith("rt_"):
            out.append((kind, rt_line(form, p, g)))
        elif kind.startswith("generic_"):
            out.append((kind, generic_line(form, p, g)))
        else:
            out.append((kind, None))
    return out

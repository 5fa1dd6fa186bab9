"""One table of strided problems (b200fft_plan_create_strided) that reach every kernel form a strided plan builds, and
the helpers that run a strided case on a B200 against torch.fft in float64.

Every transformed axis of a strided plan is one plan-time tile kernel in its StrLay form (csrc/fast.cuh, csrc/strided.cu):
8 kinds, each in both working precisions. Each row of FORMS is a problem (logical shape, the element strides of both
buffers, the element offsets at which both views start, dtypes, input components, half spectrum, direction, bases, axis
mask) and the NVRTC kernel names its plan must launch, in launch order, every one ending in `_str`. `probe` holds the
b200fft.jit_probe(strided=True, ...) arguments that compile the first pass (the one that reads the user's array) without
a GPU: tests/test_host_strided_forms.py asserts that the probe reports tags[0], tests/test_gpu_strided_forms.py that the
plan names all the tags. The probes plan for many rows (rows_hint = 0), so a probed row kind has at least MANY rows.

Shapes are logical: (batch, dims...) of the real-side array. A batch of None is filled in from the tile of tags[0] as
k * tile + 1 with k * tile >= MANY: a ragged last tile at many rows. Strides are in elements (complex pairs or real
scalars) over (batch, dims...) of each buffer's own layout; the complex side of a half-spectrum problem has n/2 + 1
elements along the last axis. Strides of None are pitched rows (strides_of), and `offset` counts elements of each
buffer before its view starts.

tests/test_host_strided_forms.py checks that the table is complete: every kind in both working precisions, every kind
that reads the user's array with every (input dtype, components) the planner accepts for it, the row kinds at few and
many rows, the few-rows / many-rows pairs, the column-tile shapes and the layouts."""
import re

import torch

import b200fft

F32, F64, U8 = "float32", "float64", "uint8"
FEW, MANY = 2 * 148, 2 * 148 + 1  # rows_hint bounds of jit_plan_axis's few-rows rules

# the 8 kinds a strided plan runs (csrc/jit.cu: jit_name; every name ends in "_str")
KINDS = ["jitrows", "jitrowsIP", "jitcols", "jitr2c", "jitr2creg", "jitr2codd", "jitc2r", "jitc2rodd"]
# (kind, precision) pairs the tier cannot build: none. Every kind has an fp64 form (rows_r2c_reg_kernel too: 144 = 16 x 9
# keeps whole warps per row group at fp64's narrower stages)
FP64_EXCEPTIONS = set()

_ANY = {(d, c) for d in (U8, F32, F64) for c in (1, 2)}
_REAL = {(F32, 1), (F64, 1)}
ACCEPTED = {  # (input dtype, components) the planner accepts for the kinds that read the user's array
    "jitrows": _ANY, "jitrowsIP": _ANY, "jitcols": _ANY,
    "jitr2c": _REAL, "jitr2creg": _REAL, "jitr2codd": _REAL,
    "jitc2r": {(F32, 2), (F64, 2)}, "jitc2rodd": {(F32, 2), (F64, 2)},  # complex in the working precision (per row)
}

DT = {F32: torch.float32, F64: torch.float64, U8: torch.uint8}


def dense(shape):
    out, s = [], 1
    for v in reversed(shape):
        out.append(s)
        s *= v
    return list(reversed(out))


def t2(shape, perm):
    """element strides of a dense array of `shape` seen through the axis permutation `perm` (batch stays first)"""
    st = dense(shape)
    return [st[p] for p in perm]


def pitched(shape, pad):
    """strides of rows of shape[-1] elements at a pitch of shape[-1] + pad, the outer dimensions dense over them"""
    return dense(list(shape[:-1]) + [shape[-1] + pad])


def kind_of(tag):
    best = None
    for k in KINDS:
        if tag.startswith(k) and tag[len(k)].isdigit() and (best is None or len(k) > len(best)):
            best = k
    assert best, tag
    return best


class Form:
    def __init__(self, id, shape, in_strides, out_strides, tags, *, in_dtype=F32, out_dtype=F32, comps=2, half=False,
                 inverse=False, bases=None, axis_mask=0, offset=(0, 0), probe=None, pair=None, layout=""):
        self.id, self.shape, self.tags = id, tuple(shape), list(tags)
        self.in_strides, self.out_strides, self.offset = in_strides, out_strides, tuple(offset)
        self.in_dtype, self.out_dtype, self.comps, self.half, self.inverse = in_dtype, out_dtype, comps, half, inverse
        self.bases, self.axis_mask, self.probe, self.pair, self.layout = bases, axis_mask, probe, pair, layout

    @property
    def kinds(self):
        return [kind_of(t) for t in self.tags]

    @property
    def f64(self):
        return self.out_dtype == F64

    @property
    def c2c(self):
        return not self.half and self.comps == 2 and self.in_dtype == self.out_dtype

    def reads(self):
        """(input dtype, components) of the user's array as tags[0] reads it"""
        return (self.in_dtype, 1 if (self.half and not self.inverse) else self.comps)

    def rows(self):
        """rows per call of a first pass along the last axis (rows_hint = every other extent)"""
        n = 1
        for d in logical_shape(self)[:-1]:
            n *= d
        return n

    def kwargs(self):
        """run_case's arguments"""
        shape = logical_shape(self)
        ist, ost = strides_of(self)
        return dict(shape=shape, in_strides=ist, out_strides=ost, in_dtype=self.in_dtype, out_dtype=self.out_dtype,
                    comps=self.comps, half=self.half, inverse=self.inverse, axis_mask=self.axis_mask, bases=self.bases,
                    tags=self.tags, offset=self.offset)

    def __repr__(self):
        return self.id


def logical_shape(form):
    if form.shape[0] is not None:
        return form.shape
    tile = int(re.search(r"_c(\d+)_t", form.tags[0]).group(1))
    k = -(-MANY // tile)
    return (k * tile + 1,) + form.shape[1:]


def sides(shape, half, inverse):
    """logical shapes (batch, dims...) of the input and the output buffer"""
    if not half:
        return list(shape), list(shape)
    cshape = list(shape[:-1]) + [shape[-1] // 2 + 1]
    return (cshape, list(shape)) if inverse else (list(shape), cshape)


def strides_of(form):
    """the row's strides, pitched rows (input pad 6, output pad 10 elements) where the row gives None"""
    ishape, oshape = sides(logical_shape(form), form.half, form.inverse)
    ist = form.in_strides if form.in_strides is not None else pitched(ishape, 6)
    ost = form.out_strides if form.out_strides is not None else pitched(oshape, 10)
    return list(ist), list(ost)


def _rows(id, n, tags, *, batch=None, probe=True, **kw):
    """rows of n points (1-D), pitched on both sides unless strides are given"""
    in_st, out_st = kw.pop("in_strides", None), kw.pop("out_strides", None)
    half = kw.get("half", False)
    pr = None
    if probe:
        bases = kw.get("bases")
        pr = dict(n=n, bases=bases[0] if bases else None, inverse=kw.get("inverse", False),
                  real_in=kw.get("comps", 2) == 1 and not half, half=(2 if kw.get("inverse") else 1) if half else 0,
                  in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    return Form(id, (batch, n), in_st, out_st, tags, probe=pr, **kw)


def _cols(id, n, cols, tags, *, batch=2, **kw):
    """axis 0 of (batch, n, cols) alone (axis_mask = 1), read as column tiles over `cols` columns of a pitched batch"""
    bases = kw.pop("bases", None)
    pr = dict(n=n, inner=cols, bases=bases, inverse=kw.get("inverse", False), real_in=kw.get("comps", 2) == 1,
              in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    st_in = [n * cols + 3, cols, 1]
    st_out = kw.pop("out_strides", [n * cols + 5, cols, 1])
    return Form(id, (batch, n, cols), kw.pop("in_strides", st_in), st_out, tags, axis_mask=1,
                bases=[bases, [cols]] if bases else None, probe=pr, **kw)


# rank 8 (batch + 8 axes): a permuted dense buffer in, another permutation out, axes 1, 3 and 6 not transformed
R8 = (2, 3, 2, 4, 2, 3, 2, 5, 4)
R8_IN = [0, 8, 3, 1, 6, 2, 7, 4, 5]
R8_OUT = [0, 2, 5, 8, 1, 7, 3, 6, 4]


def _perm_strides(shape, perm):
    """strides of `shape` inside a dense buffer whose dimensions are `shape` reordered by `perm` (perm[0] = 0)"""
    st = dense([shape[p] for p in perm])
    out = [0] * len(shape)
    for j, p in enumerate(perm):
        out[p] = st[j]
    return out


FORMS = [
    # ---- jitrows: `tile` rows per CTA, two exchange buffers ---------------------------------------------------------------
    _rows("rows-c2c", 600, ["jitrows600_30x20_c8_t160_str"], layout="pitched rows"),
    _rows("rows-real", 600, ["jitrows600_30x20_c8_t160_str"], comps=1),
    _rows("rows-u8-real", 600, ["jitrows600_30x20_c8_t160_inu8_str"], in_dtype=U8, comps=1),
    _rows("rows-u8-complex", 600, ["jitrows600_30x20_c8_t160_inu8_str"], in_dtype=U8, inverse=True, offset=(1, 1)),
    _rows("rows-f64-in", 600, ["jitrows600_30x20_c8_t160_inf64_str"], in_dtype=F64),
    _rows("rows-f64-in-real", 600, ["jitrows600_30x20_c8_t160_inf64_str"], in_dtype=F64, comps=1),
    _rows("rows-f64", 600, ["jitrows600_10x10x6_c3_t192_f64_str"], in_dtype=F64, out_dtype=F64, inverse=True,
          offset=(1, 1)),
    _rows("rows-u8-to-f64", 600, ["jitrows600_10x10x6_c3_t192_f64_inu8_str"], in_dtype=U8, out_dtype=F64, comps=1),
    _rows("rows-f32-to-f64", 600, ["jitrows600_10x10x6_c3_t192_f64_inf32_str"], out_dtype=F64),
    # an element stride of 3 along the axis on both sides, the batch at a pitch of its own
    Form("rows-elem-stride3", (50, 93), [3 * 93 + 2, 3], [3 * 93 + 1, 3], ["jitrows93_31x3_c53_t160_str"], bases=[[31, 3]],
         layout="element stride 3"),
    # a looped prime (127) as the first stage
    _rows("rows-prime127", 254, ["jitrows254_127x2_c16_t32_str"], bases=[[127, 2]], batch=40, probe=False),

    # ---- few rows / many rows: the same axis, a different kernel ----------------------------------------------------------
    _rows("rows-2000-many", 2000, ["jitrowsIP2000_20x10x10_c1_t128_str"], pair="2000"),
    _rows("rows-2000-few", 2000, ["jitrows2000_50x40_c4_t160_str"], batch=3, probe=False, pair="2000"),
    _rows("rows-3000-many", 3000, ["jitrowsIP3000_20x15x10_c1_t160_str"], pair="3000"),
    _rows("rows-3000-few", 3000, ["jitrows3000_20x15x10_c1_t160_str"], batch=FEW, probe=False, pair="3000"),
    _rows("rowsIP-10000-few", 10000, ["jitrowsIP10000_10x10x10x10_c1_t512_str"], batch=5, probe=False, pair="10000"),
    _rows("rowsIP-10000-many", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_str"], pair="10000"),
    _rows("rows-f64-1024-few", 1024, ["jitrows1024_16x8x8_c2_t128_f64_str"], batch=7, probe=False, in_dtype=F64,
          out_dtype=F64, pair="f64-1024"),
    _rows("rowsIP-f64-1024-many", 1024, ["jitrowsIP1024_16x8x8_c1_t128_f64_str"], in_dtype=F64, out_dtype=F64,
          pair="f64-1024", offset=(1, 1)),

    # ---- jitrowsIP: one row per CTA in one shared buffer ------------------------------------------------------------------
    _rows("rowsIP-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_str"], comps=1, batch=MANY),
    _rows("rowsIP-u8-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inu8_str"], in_dtype=U8, comps=1, batch=MANY),
    _rows("rowsIP-u8-complex", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inu8_str"], in_dtype=U8, inverse=True,
          batch=MANY, offset=(1, 1)),
    _rows("rowsIP-f64-in", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inf64_str"], in_dtype=F64, batch=MANY),
    _rows("rowsIP-f64-in-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inf64_str"], in_dtype=F64, comps=1, batch=MANY),
    _rows("rowsIP-f32-to-f64-real", 8192, ["jitrowsIP8192_16x8x8x8_c1_t256_f64_inf32_str"], out_dtype=F64, comps=1,
          batch=MANY),
    # the longest power-of-two rows one tile serves (tests/test_host_strided_forms.py: the next one is refused)
    _rows("rowsIP-16384", 16384, ["jitrowsIP16384_32x32x16_c1_t512_str"], batch=MANY, layout="longest fp32 rows"),
    _rows("rowsIP-f64-few", 8192, ["jitrowsIP8192_16x8x8x8_c1_t512_f64_str"], batch=3, probe=False, in_dtype=F64,
          out_dtype=F64),
    _rows("rowsIP-f64-8192", 8192, ["jitrowsIP8192_16x8x8x8_c1_t256_f64_str"], in_dtype=F64, out_dtype=F64, batch=MANY,
          inverse=True, layout="longest fp64 rows"),

    # ---- jitcols: column tiles along the dimension of the smallest stride ------------------------------------------------
    _cols("cols-5-columns", 90, 5, ["jitcols90_10x9_w5_t64_str"], layout="5 columns: the tile is the column count"),
    _cols("cols-ragged", 100, 35, ["jitcols100_10x10_w32_t320_str"], batch=3, offset=(1, 1), layout="ragged last tile"),
    _cols("cols-w64", 36, 200, ["jitcols36_6x6_w64_t384_str"], layout="64-wide tiles"),
    _cols("cols-real", 100, 35, ["jitcols100_10x10_w32_t320_str"], comps=1),
    _cols("cols-u8-real", 100, 35, ["jitcols100_10x10_w32_t320_inu8_str"], in_dtype=U8, comps=1),
    _cols("cols-u8-complex", 100, 35, ["jitcols100_10x10_w32_t320_inu8_str"], in_dtype=U8, inverse=True),
    _cols("cols-f64-in", 100, 35, ["jitcols100_10x10_w32_t320_inf64_str"], in_dtype=F64),
    _cols("cols-f64-in-real", 100, 35, ["jitcols100_10x10_w32_t320_inf64_str"], in_dtype=F64, comps=1, inverse=True),
    _cols("cols-f64", 100, 35, ["jitcols100_10x10_w16_t160_f64_str"], in_dtype=F64, out_dtype=F64, offset=(1, 1)),
    _cols("cols-u8-to-f64-real", 100, 35, ["jitcols100_10x10_w16_t160_f64_inu8_str"], in_dtype=U8, out_dtype=F64, comps=1),
    _cols("cols-f32-to-f64", 100, 35, ["jitcols100_10x10_w16_t160_f64_inf32_str"], out_dtype=F64, inverse=True),
    _cols("cols-prime127", 254, 20, ["jitcols254_127x2_w16_t32_str"], bases=[127, 2], layout="looped prime 127"),
    # the longest power-of-two column axes one tile of 8 or more columns serves
    _cols("cols-1024", 1024, 16, ["jitcols1024_32x32_w8_t256_str"], layout="longest fp32 columns"),
    _cols("cols-f64-512", 512, 8, ["jitcols512_8x8x8_w8_t256_f64_str"], in_dtype=F64, out_dtype=F64, inverse=True,
          layout="longest fp64 columns"),
    # batch-interleaved (batch stride 1, cuFFT's idist = 1): columns along the batch
    Form("cols-batch-interleaved", (40, 1000), [1, 40], [1, 40], ["jitcols1000_40x25_w8_t224_str"], layout="batch stride 1"),
    Form("cols-batch-interleaved-f64", (24, 243), [1, 24], [1, 30], ["jitcols243_9x9x3_w8_t224_f64_str"], in_dtype=F64,
         out_dtype=F64, inverse=True, layout="batch stride 1"),

    # ---- N-d C2C: transposed, permuted, rank 8 -----------------------------------------------------------------------------
    Form("c2c-2d-transposed", (20, 48, 64), t2((20, 64, 48), [0, 2, 1]), dense((20, 48, 64)),
         ["jitcols64_8x8_w32_t256_str", "jitcols48_8x6_w64_t384_str"], offset=(1, 0), layout="transposed"),
    Form("c2c-3d-permuted-f64", (6, 24, 16, 20), t2((6, 16, 20, 24), [0, 3, 1, 2]), dense((6, 24, 16, 20)),
         ["jitcols20_5x4_w16_t64_f64_str", "jitcols16_16_w16_t32_f64_str", "jitcols24_6x4_w16_t64_f64_str"],
         in_dtype=F64, out_dtype=F64, inverse=True, layout="permuted"),
    Form("c2c-rank8", R8, _perm_strides(R8, R8_IN), _perm_strides(R8, R8_OUT),
         ["jitcols4_4_w3_t32_str", "jitcols2_2_w2_t32_str", "jitcols3_3_w2_t32_str", "jitcols4_4_w2_t32_str",
          "jitcols3_3_w2_t32_str"], axis_mask=0b10110101, offset=(1, 1), layout="rank 8, permuted, axes 1, 3, 6 masked"),

    # ---- half spectrum -------------------------------------------------------------------------------------------------------
    _rows("r2c", 200, ["jitr2c100_10x10_c35_t352_str"], half=True, comps=1, offset=(2, 1)),
    _rows("r2c-f64", 200, ["jitr2c100_10x10_c16_t160_f64_str"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _rows("r2c-f64-in", 200, ["jitr2c100_10x10_c35_t352_inf64_str"], half=True, comps=1, in_dtype=F64),
    _rows("r2c-f32-to-f64", 200, ["jitr2c100_10x10_c16_t160_f64_inf32_str"], half=True, comps=1, out_dtype=F64),
    _rows("r2creg", 288, ["jitr2creg144_16x9_c28_t256_str"], bases=[[32, 9]], half=True, comps=1),
    _rows("r2creg-f64", 288, ["jitr2creg144_16x9_c14_t128_f64_str"], bases=[[32, 9]], half=True, comps=1, in_dtype=F64,
          out_dtype=F64, offset=(2, 1)),
    _rows("r2creg-f64-in", 288, ["jitr2creg144_16x9_c28_t256_inf64_str"], bases=[[32, 9]], half=True, comps=1, in_dtype=F64),
    _rows("r2codd", 243, ["jitr2codd243_27x9_c21_t192_str"], half=True, comps=1, offset=(1, 1)),
    _rows("r2codd-f64", 243, ["jitr2codd243_9x9x3_c8_t224_f64_str"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _rows("r2codd-f64-in", 243, ["jitr2codd243_27x9_c21_t192_inf64_str"], half=True, comps=1, in_dtype=F64),
    _rows("c2r", 200, ["jitc2r100_10x10_c41_t416_str"], half=True, inverse=True, offset=(1, 2)),
    _rows("c2r-f64", 200, ["jitc2r100_10x10_c22_t224_f64_str"], half=True, inverse=True, in_dtype=F64, out_dtype=F64),
    _rows("c2rodd", 243, ["jitc2rodd243_27x9_c21_t192_str"], half=True, inverse=True),
    _rows("c2rodd-f64", 243, ["jitc2rodd243_9x9x3_c8_t224_f64_str"], half=True, inverse=True, in_dtype=F64, out_dtype=F64,
          offset=(1, 1)),
    # N-d, the padded layout: the column pass after the R2C rows (before the C2R rows) has n/2 + 1 = 101 columns, odd,
    # and a ragged last tile
    Form("r2c-2d-odd-columns", (3, 37, 200), [37 * 202, 202, 1], [37 * 101, 101, 1],
         ["jitr2c100_10x10_c35_t352_str", "jitcols37_37_w64_t64_str"], half=True, comps=1, layout="padded, 101 columns"),
    Form("c2r-2d-odd-columns", (3, 37, 200), [37 * 101, 101, 1], [37 * 202, 202, 1],
         ["jitcols37_37_w64_t64_str", "jitc2r100_10x10_c41_t416_str"], half=True, inverse=True,
         layout="padded, 101 columns"),
    Form("r2c-2d-odd-columns-f64", (3, 37, 200), [37 * 202, 202, 1], [37 * 101, 101, 1],
         ["jitr2c100_10x10_c16_t160_f64_str", "jitcols37_37_w64_t64_f64_str"], half=True, comps=1, in_dtype=F64,
         out_dtype=F64, layout="padded, 101 columns"),
    Form("c2r-2d-odd-columns-f64", (3, 37, 200), [37 * 101, 101, 1], [37 * 202, 202, 1],
         ["jitcols37_37_w64_t64_f64_str", "jitc2r100_10x10_c22_t224_f64_str"], half=True, inverse=True, in_dtype=F64,
         out_dtype=F64, layout="padded, 101 columns"),
]


def by_id():
    return {f.id: f for f in FORMS}


# ---- running a case on the GPU ------------------------------------------------------------------------------------------
def span_of(shape, strides):
    return sum((n - 1) * s for n, s in zip(shape, strides)) + 1


def buffer_view(shape, strides, comps, dtype, fill, gen=None, offset=0):
    """A view of logical `shape` (batch, dims...) with element `strides` into a fresh buffer, starting `offset` elements
    in and ending one element before the buffer's end; `fill`: "rand" or "nan"."""
    span = offset + span_of(shape, strides) + 1
    dt = DT[dtype]
    if fill == "nan":
        buf = torch.full((span * comps,), float("nan"), dtype=dt, device="cuda")
    elif dt == torch.uint8:
        buf = torch.randint(0, 256, (span * comps,), dtype=dt, device="cuda", generator=gen)
    else:
        buf = torch.randn(span * comps, dtype=dt, device="cuda", generator=gen)
    view = buf.as_strided(tuple(shape) + (comps,), tuple(s * comps for s in strides) + (1,), offset * comps)
    return buf, view


def as_complex128(t, comps):
    t = t.double()
    return torch.complex(t[..., 0], t[..., 1]) if comps == 2 else t[..., 0].to(torch.complex128)


def check(got, ref, out_dtype):
    got, ref = got.cpu(), ref.cpu()
    err = (torch.linalg.vector_norm(got - ref) / torch.linalg.vector_norm(ref)).item()
    if out_dtype == F64:
        assert err <= 1e-13, err
    else:
        assert err <= 2e-6, err
        assert (got - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


def reference(x, shape, axes, icomps, half, inverse):
    """float64 transform of the float64 value of the input view x"""
    dims = [a + 1 for a in axes]
    if half and inverse:
        return torch.fft.irfftn(as_complex128(x, 2), s=[shape[a] for a in dims], dim=dims)
    if half:
        return torch.fft.rfftn(x[..., 0].double(), dim=dims)
    return (torch.fft.ifftn if inverse else torch.fft.fftn)(as_complex128(x, icomps), dim=dims)


def result(y, half, inverse):
    return y[..., 0].double() if half and inverse else as_complex128(y, 2)


def names_in(desc):
    """the kernel names a plan description lists, in launch order"""
    return [ln.split(": ")[1].split(" ")[0] for ln in desc.strip().split("\n")]


def run_case(shape, in_strides, out_strides, *, in_dtype=F32, out_dtype=F32, comps=2, half=False, inverse=False,
             axis_mask=0, bases=None, tags=None, offset=(0, 0)):
    """shape: logical (batch, dims...) of the real side for half-spectrum plans, of both sides otherwise. offset: the
    elements of each buffer before its view starts. tags: the kernel names the plan must launch, in order. Returns the
    plan's description, the input view and the output view."""
    gen = torch.Generator(device="cuda").manual_seed(sum(shape))
    rank = len(shape) - 1
    axes = [a for a in range(rank) if not axis_mask or axis_mask >> a & 1]
    ishape, oshape = sides(shape, half, inverse)
    icomps = 2 if half and inverse else 1 if half else comps
    ocomps = 1 if half and inverse else 2
    in_buf, x = buffer_view(ishape, in_strides, icomps, in_dtype, "rand", gen, offset[0])
    if half and inverse:  # a Hermitian spectrum: the half spectrum of a real signal
        real = torch.randn(tuple(shape), dtype=torch.float64, device="cuda", generator=gen)
        spec = torch.fft.rfftn(real, dim=[a + 1 for a in axes])
        x[..., 0].copy_(spec.real)
        x[..., 1].copy_(spec.imag)
    in_copy = in_buf.clone()
    out_buf, y = buffer_view(oshape, out_strides, ocomps, out_dtype, "nan", None, offset[1])
    kw = dict(inverse=inverse, axis_mask=axis_mask, real_mode=b200fft.REAL_HALF if half else b200fft.REAL_FULL, bases=bases,
              in_strides=in_strides, out_strides=out_strides)
    plan = b200fft.plan_fft(in_dtype, out_dtype, tuple(ishape) + (icomps,), tuple(oshape) + (ocomps,), **kw)
    desc = plan.describe()
    assert plan.launches == len(axes), desc
    lines = desc.strip().split("\n")
    assert len(lines) == len(axes) and all("_str" in ln and "NVRTC" in ln for ln in lines), lines
    b200fft.fft(y, x, plan=plan)
    torch.cuda.synchronize()
    assert torch.equal(in_buf, in_copy), "the input was modified"
    mask = torch.ones(out_buf.shape, dtype=torch.bool, device="cuda")
    mask.as_strided(y.shape, y.stride(), y.storage_offset()).fill_(False)
    assert out_buf[mask].isnan().all(), "an element outside the output view was written"
    assert not y.isnan().any(), "an output element was not written"
    check(result(y, half, inverse), reference(x, shape, axes, icomps, half, inverse), out_dtype)
    # a second plan of the same problem: the same bits
    out2_buf, y2 = buffer_view(oshape, out_strides, ocomps, out_dtype, "nan", None, offset[1])
    plan2 = b200fft.plan_fft(in_dtype, out_dtype, tuple(ishape) + (icomps,), tuple(oshape) + (ocomps,), **kw)
    b200fft.fft(y2, x, plan=plan2)
    torch.cuda.synchronize()
    assert torch.equal(y, y2)
    if tags is not None:
        assert names_in(desc) == list(tags), (names_in(desc), tags)
    return desc, x, y

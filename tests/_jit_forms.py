"""One table of problems that reach every kernel form the plan-time specialisation tier (csrc/jit.cu) builds.

Each row is a problem (logical shape, dtypes, input components, half spectrum, direction, bases, axis mask, flags and
environment) and the names of the NVRTC kernels its plan must launch, in launch order: `tags[0]` is the kernel that
reads the user's array. A tag is the jit_name of the kernel (`jitrows600_25x24_c4_t160`, ...) or, where it depends on
a choice this table does not pin, its leading part up to a "_" or "(" (`jitcols37_`, `jitplane40x48(`).

`probe` names the host-only entry point that compiles the same axis without a GPU ("jit": b200fft.jit_probe, "split":
jit_split_probe, "split3": jit_split3_probe) and its arguments. The probes plan with rows_hint = 0, which the planner
treats as many rows, so a probed row kind has at least 297 rows (2 x 148 SMs) in `shape`: tests/test_host_jit_forms.py
asserts that the probe reports the row's full tags, and tests/test_gpu_jit_forms.py that the plan names them, so the
probe and the planner agree. `pair` joins a few-rows row with a many-rows row of the same axis where the planner's rules
pick a different kernel for each.

Shapes are logical: (batch, dims...) of the real-side array. A batch of None is filled in from the tile of tags[0] as
k * tile + 1 with k * tile >= 297: a ragged last tile at many rows.

tests/test_host_jit_forms.py checks that the table is complete: every one of the 21 kinds, every kind in both working
precisions (plane kinds: fp32 only), every kind that reads the user's array with every (input dtype, components) the
planner accepts for it."""

F32, F64, U8 = "float32", "float64", "uint8"
FEW, MANY = 2 * 148, 2 * 148 + 1  # rows_hint bounds of jit_plan_axis's few-rows rules

# the 21 kernel kinds (jit.cu: jit_name)
KINDS = ["jitrows", "jitcols", "jitscatter", "jitr2c", "jitr2creg", "jitr2codd", "jitc2r", "jitc2rodd", "jitsplitA",
         "jitsplitBcols", "jitsplitBrows", "jitplane", "jitr2cplane", "jitrowsIP", "jitsplitBr2c", "jitsplitAc2r",
         "jitsplitAc2rodd", "jitsplitBhalf", "jitsplitBreal", "jitsplit3A", "jitsplit3C"]
FP32_ONLY = {"jitplane", "jitr2cplane"}  # make_jit_plane_pass serves fp32 planes only

# (input dtype, input components) the planner accepts for the kinds that read the user's array; the others read the
# plan's temporary or workspace
_ANY = {(d, c) for d in (U8, F32, F64) for c in (1, 2)}
_REAL = {(F32, 1), (F64, 1)}        # half-spectrum forward: real rows in fp32 or fp64, no uint8
_WORK = {(F32, 2), (F64, 2)}        # the staged half spectrum / scatter source: complex in the working dtype only
ACCEPTED = {
    "jitrows": _ANY, "jitrowsIP": _ANY, "jitcols": _ANY, "jitsplitA": _ANY | _REAL, "jitsplit3A": _ANY,
    "jitscatter": _WORK, "jitr2c": _REAL, "jitr2creg": _REAL, "jitr2codd": _REAL,
    "jitc2r": _WORK, "jitc2rodd": _WORK, "jitsplitAc2r": _WORK, "jitsplitAc2rodd": _WORK,
    "jitplane": {(F32, 1), (F32, 2)}, "jitr2cplane": {(F32, 1)},
}

FLAG_NO_FUSED = 4  # b200fft.FLAG_NO_FUSED: per-axis passes, no plane or fused kernel in front


def kind_of(tag):
    """The kind a tag names: the longest kind it starts with that is followed by the transform length."""
    best = None
    for k in KINDS:
        if tag.startswith(k) and len(tag) > len(k) and tag[len(k)].isdigit() and (best is None or len(k) > len(best)):
            best = k
    assert best, tag
    return best


class Form:
    def __init__(self, id, shape, tags, *, in_dtype=F32, out_dtype=F32, comps=2, half=False, inverse=False, bases=None,
                 axis_mask=0, flags=0, env=None, probe=None, pair=None, permuted=None, scatter=False, exec_host=False,
                 note=""):
        self.id, self.shape, self.tags = id, tuple(shape), list(tags)
        self.in_dtype, self.out_dtype, self.comps, self.half, self.inverse = in_dtype, out_dtype, comps, half, inverse
        self.bases, self.axis_mask, self.flags, self.env = bases, axis_mask, flags, dict(env or {})
        self.probe, self.pair, self.permuted, self.scatter, self.exec_host, self.note = (
            probe, pair, permuted, scatter, exec_host, note)

    @property
    def kinds(self):
        return [kind_of(t) for t in self.tags]

    @property
    def f64(self):
        return self.out_dtype == F64

    def reads(self):
        """(input dtype, components) of the user's array as tags[0] reads it."""
        return (self.in_dtype, 1 if (self.half and not self.inverse) else self.comps)

    def rows(self):
        """Transforms per call of a row kind (rows_hint = batch x outer axes)."""
        n = 1
        for d in logical_shape(self)[:-1]:
            n *= d
        return n

    def __repr__(self):
        return self.id


def _p(fn, n, **kw):
    return (fn, dict(n=n, **kw))


def _rows(id, n, tags, *, batch=None, bases=None, probe=True, **kw):
    """A contiguous 1-D axis of n points; probed unless it is a few-rows row."""
    pr = None
    if probe:
        pr = _p("jit", n, bases=bases[0] if bases else None, inverse=kw.get("inverse", False),
                real_in=kw.get("comps", 2) == 1 and not kw.get("half"), half=(2 if kw.get("inverse") else 1) if kw.get("half") else 0,
                in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    return Form(id, (batch, n), tags, bases=bases, probe=pr, **kw)


def _cols(id, n, inner, tags, *, batch=2, bases=None, **kw):
    """The strided axis of (batch, n, inner), alone (axis_mask = 1): the first pass reads the user's array."""
    pr = _p("jit", n, inner=inner, bases=bases, inverse=kw.get("inverse", False), real_in=kw.get("comps", 2) == 1,
            in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    return Form(id, (batch, n, inner), tags, bases=[bases, [inner]] if bases else None, axis_mask=1, probe=pr, **kw)


def _split(id, n, tags, *, batch=2, inner=1, bases=None, **kw):
    half = kw.get("half", False)
    pr = _p("split", n, inner=inner, bases=bases, inverse=kw.get("inverse", False),
            real_in=kw.get("comps", 2) == 1 and not half, half=(2 if kw.get("inverse") else 1) if half else 0,
            in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    if inner == 1:
        return Form(id, (batch, n), tags, bases=[bases] if bases else None, probe=pr, **kw)
    return Form(id, (batch, n, inner), tags, bases=[bases, [inner]] if bases else None, axis_mask=1, probe=pr, **kw)


N3 = 3 * 2 ** 23  # the shortest lengths above 2^24 the three-pass split serves


def _split3(id, tags, *, bases=None, **kw):
    pr = _p("split3", N3, bases=bases, inverse=kw.get("inverse", False), real_in=kw.get("comps", 2) == 1,
            in_dtype=kw.get("in_dtype", F32), out_dtype=kw.get("out_dtype", F32))
    return Form(id, (1, N3), tags, bases=[bases] if bases else None, probe=pr, **kw)


FORMS = [
    # ---- jitrows: two exchange buffers, `tile` rows per CTA --------------------------------------------------------
    _rows("rows-pow2-unpacked", 256, ["jitrows256_32x8_c16_t128"], bases=[[32, 8]],
          note="no registered 256-point variant groups 32 x 8; power-of-two rows build without packed FADD2"),
    _rows("rows-mixed-packed", 600, ["jitrows600_30x20_c8_t160"]),
    _rows("rows-real", 600, ["jitrows600_30x20_c8_t160"], comps=1),
    _rows("rows-u8-real", 600, ["jitrows600_30x20_c8_t160_inu8"], in_dtype=U8, comps=1),
    _rows("rows-u8-complex", 600, ["jitrows600_30x20_c8_t160_inu8"], in_dtype=U8),
    _rows("rows-f64-in", 600, ["jitrows600_30x20_c8_t160_inf64"], in_dtype=F64),
    _rows("rows-f64-in-real", 600, ["jitrows600_30x20_c8_t160_inf64"], in_dtype=F64, comps=1),
    _rows("rows-f32-to-f64", 600, ["jitrows600_10x10x6_c3_t192_f64_inf32"], out_dtype=F64),
    _rows("rows-f32-to-f64-real", 600, ["jitrows600_10x10x6_c3_t192_f64_inf32"], out_dtype=F64, comps=1),
    _rows("rows-f64", 600, ["jitrows600_10x10x6_c3_t192_f64"], in_dtype=F64, out_dtype=F64, inverse=True),
    _rows("rows-u8-to-f64", 600, ["jitrows600_10x10x6_c3_t192_f64_inu8"], in_dtype=U8, out_dtype=F64, comps=1),
    # wide composite codelets (fp32): a stage list of three groups of <= 32 becomes two wide stages
    _rows("rows-wide36", 1296, ["jitrows1296_36x36_c6_t224"]),
    _rows("rows-wide45", 2025, ["jitrows2025_45x45_c2_t96"]),
    _rows("rows-wide48", 2304, ["jitrows2304_48x48_c2_t96"], inverse=True),
    _rows("rows-wide40", 1600, ["jitrows1600_40x40_c4_t160"], note="40 x 40 keeps its two wide stages at many rows"),
    # prime codelets: unrolled (<= 61) and looped (67..127) as the first and the last stage, fp32 and fp64
    _rows("rows-prime53-first", 424, ["jitrows424_53x8_c12_t96"], bases=[[53, 8]]),
    _rows("rows-prime97-first", 388, ["jitrows388_97x4_c16_t64"], bases=[[97, 4]], inverse=True),
    _rows("rows-prime41-last", 2624, ["jitrows2624_64x41_c3_t128"], bases=[[64, 41]]),
    _rows("rows-prime71-last", 9017, ["jitrows9017_127x71_c2_t160"], bases=[[127, 71]]),
    _rows("rows-prime53-first-f64", 424, ["jitrows424_53x8_c8_t64_f64"], bases=[[53, 8]], in_dtype=F64, out_dtype=F64),
    _rows("rows-prime97-first-f64", 388, ["jitrows388_97x4_c8_t32_f64"], bases=[[97, 4]], in_dtype=F64, out_dtype=F64, inverse=True),
    _rows("rows-prime41-last-f64", 2624, ["jitrows2624_64x41_c3_t128_f64"], bases=[[64, 41]], in_dtype=F64, out_dtype=F64),
    _rows("rows-prime71-last-f64", 9017, ["jitrows9017_127x71_c1_t96_f64"], bases=[[127, 71]], in_dtype=F64, out_dtype=F64),

    # ---- jitrowsIP: one row per CTA, 3-5 stages in one shared buffer ---------------------------------------------------
    _rows("rowsIP-given-order", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256"], permuted=False),
    _rows("rowsIP-permuted", 20000, ["jitrowsIP20000_20x40x25_c1_t512"], permuted=True,
          note="the descending stage order does not fit the register budget of the in-place middle stage"),
    _rows("rowsIP-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256"], comps=1),
    _rows("rowsIP-u8-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inu8"], in_dtype=U8, comps=1),
    _rows("rowsIP-u8-complex", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inu8"], in_dtype=U8, inverse=True),
    _rows("rowsIP-f64-in", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inf64"], in_dtype=F64),
    _rows("rowsIP-f64-in-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_inf64"], in_dtype=F64, comps=1),
    _rows("rowsIP-f64", 1024, ["jitrowsIP1024_16x8x8_c1_t128_f64"], in_dtype=F64, out_dtype=F64, pair="f64-1024"),
    _rows("rowsIP-f32-to-f64-real", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256_f64_inf32"], out_dtype=F64, comps=1),
    # an unrolled prime as the in-place middle stage; a looped prime (> 64 values per thread) never fits the middle, so
    # the planner moves it to an end
    _rows("rowsIP-prime37-middle", 18944, ["jitrowsIP18944_64x37x8_c1_t512"], bases=[[64, 37, 8]], permuted=False),
    _rows("rowsIP-prime37-middle-f64", 9472, ["jitrowsIP9472_64x37x4_c1_t256_f64"], bases=[[64, 37, 4]], in_dtype=F64, out_dtype=F64,
          permuted=False),
    _rows("rowsIP-prime67-moved", 17018, ["jitrowsIP17018_67x2x127_c1_t288"], bases=[[127, 67, 2]], permuted=True),
    _rows("rowsIP-prime67-moved-f64", 9514, ["jitrowsIP9514_67x2x71_c1_t160_f64"], bases=[[71, 67, 2]], in_dtype=F64, out_dtype=F64,
          permuted=True),

    # ---- few rows / many rows: the same axis, a different kernel ------------------------------------------------------
    # two wide stages with a radix-50 / 40 codelet become three narrow in-place stages at many rows only
    _rows("rows-2000-many", 2000, ["jitrowsIP2000_20x10x10_c1_t128"], pair="2000"),
    _rows("rows-2000-few", 2000, ["jitrows2000_50x40_"], batch=3, probe=False, pair="2000"),
    # 16-32 KB rows: the one-buffer kernel at many rows only
    _rows("rows-3000-many", 3000, ["jitrowsIP3000_20x15x10_c1_t160"], pair="3000"),
    _rows("rows-3000-few", 3000, ["jitrows3000_"], batch=FEW, probe=False, pair="3000"),
    # rows of 32 KB and more: the one-buffer kernel either way, 512 instead of 256 preferred threads at few rows
    _rows("rowsIP-10000-few", 10000, ["jitrowsIP10000_10x10x10x10_c1_t512"], batch=5, probe=False, pair="10000"),
    _rows("rowsIP-10000-many", 10000, ["jitrowsIP10000_10x10x10x10_c1_t256"], pair="10000"),
    _rows("rowsIP-f64-few", 9472, ["jitrowsIP9472_64x37x4_"], batch=3, probe=False, bases=[[64, 37, 4]], in_dtype=F64,
          out_dtype=F64),
    _rows("rows-f64-1024-few", 1024, ["jitrows1024_16x8x8_"], batch=7, probe=False, in_dtype=F64, out_dtype=F64, pair="f64-1024"),

    # ---- jitcols: strided axes -------------------------------------------------------------------------------------
    _cols("cols-inner5", 90, 5, ["jitcols90_10x9_w5_t64"], note="inner < 8: the tile is the inner extent"),
    _cols("cols-inner-tile-plus-odd", 100, 35, ["jitcols100_10x10_w32_t320"], batch=3),
    _cols("cols-w64", 36, 200, ["jitcols36_6x6_w64_t384"], note="64-wide tiles"),
    _cols("cols-real", 100, 35, ["jitcols100_10x10_w32_t320"], comps=1),
    _cols("cols-u8-real", 100, 35, ["jitcols100_10x10_w32_t320_inu8"], in_dtype=U8, comps=1),
    _cols("cols-u8-complex", 100, 35, ["jitcols100_10x10_w32_t320_inu8"], in_dtype=U8, inverse=True),
    _cols("cols-f64-in", 100, 35, ["jitcols100_10x10_w32_t320_inf64"], in_dtype=F64),
    _cols("cols-f64-in-real", 100, 35, ["jitcols100_10x10_w32_t320_inf64"], in_dtype=F64, comps=1, inverse=True),
    _cols("cols-f64", 100, 35, ["jitcols100_10x10_w16_t160_f64"], in_dtype=F64, out_dtype=F64),
    _cols("cols-u8-to-f64-real", 100, 35, ["jitcols100_10x10_w16_t160_f64_inu8"], in_dtype=U8, out_dtype=F64, comps=1),
    _cols("cols-f32-to-f64", 100, 35, ["jitcols100_10x10_w16_t160_f64_inf32"], out_dtype=F64, inverse=True),
    _cols("cols-prime43-first", 172, 20, ["jitcols172_43x4_w16_t64"], bases=[43, 4]),
    _cols("cols-prime89-first", 267, 20, ["jitcols267_89x3_w16_t64"], bases=[89, 3], inverse=True),
    _cols("cols-prime47-last", 3008, 3, ["jitcols3008_64x47_w3_t160"], bases=[64, 47]),
    _cols("cols-prime73-last", 9271, 2, ["jitcols9271_127x73_w2_t160"], bases=[127, 73]),
    _cols("cols-prime43-first-f64", 172, 20, ["jitcols172_43x4_w16_t64_f64"], bases=[43, 4], in_dtype=F64, out_dtype=F64),
    _cols("cols-prime89-first-f64", 267, 20, ["jitcols267_89x3_w8_t32_f64"], bases=[89, 3], in_dtype=F64, out_dtype=F64),
    _cols("cols-prime47-last-f64", 3008, 3, ["jitcols3008_64x47_w3_t160_f64"], bases=[64, 47], in_dtype=F64, out_dtype=F64, inverse=True),
    _cols("cols-prime67-last-f64", 5293, 2, ["jitcols5293_79x67_w2_t160_f64"], bases=[79, 67], in_dtype=F64, out_dtype=F64),

    # ---- jitscatter: the scattering store of a strided axis with no registered length (exec_scatter_at) ----------------
    Form("scatter", (4, 120, 36), ["jitcols120_", "jitscatter120_"], axis_mask=1, scatter=True),
    Form("scatter-f64", (4, 120, 36), ["jitcols120_", "jitscatter120_"], in_dtype=F64, out_dtype=F64, axis_mask=1,
         scatter=True),

    # ---- half spectrum, one tile per row ---------------------------------------------------------------------------
    _rows("r2c", 200, ["jitr2c100_10x10_c35_t352"], half=True, comps=1),
    _rows("r2c-f64", 200, ["jitr2c100_10x10_c16_t160_f64"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _rows("r2c-f64-in", 200, ["jitr2c100_10x10_c35_t352_inf64"], half=True, comps=1, in_dtype=F64),
    _rows("r2c-f32-to-f64", 200, ["jitr2c100_10x10_c16_t160_f64_inf32"], half=True, comps=1, out_dtype=F64),
    # H = 144 as 16 x 9: 16 points per row group, whole warps at any even tile (r2c_reg_ok). No length reaches the
    # R2C_REG -> R2C fallback of jit_plan_axis: P = H / r_last divides 32 and H <= 32 x 32, so the tile search always
    # finds a tile of whole warps within the shared-memory and thread limits
    _rows("r2creg", 288, ["jitr2creg144_16x9_c28_t256"], bases=[[32, 9]], half=True, comps=1),
    _rows("r2creg-f64", 288, ["jitr2creg144_16x9_c14_t128_f64"], bases=[[32, 9]], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _rows("r2creg-f64-in", 288, ["jitr2creg144_16x9_c28_t256_inf64"], bases=[[32, 9]], half=True, comps=1, in_dtype=F64),
    _rows("r2creg-f32-to-f64", 288, ["jitr2creg144_16x9_c14_t128_f64_inf32"], bases=[[32, 9]], half=True, comps=1, out_dtype=F64),
    Form("r2creg-smem", (300, 288), ["jitr2c144_16x9_"], bases=[[32, 9]], half=True, comps=1,
         env={"B200FFT_R2C_SMEM": "1"}, note="B200FFT_R2C_SMEM=1: the shared-memory unpack on a whole-warp length"),
    _rows("r2codd", 243, ["jitr2codd243_27x9_c21_t192"], half=True, comps=1),
    _rows("r2codd-f64", 243, ["jitr2codd243_9x9x3_c8_t224_f64"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _rows("r2codd-f64-in", 243, ["jitr2codd243_27x9_c21_t192_inf64"], half=True, comps=1, in_dtype=F64),
    _rows("c2r", 200, ["jitc2r100_10x10_c41_t416"], half=True, inverse=True),
    _rows("c2r-f64", 200, ["jitc2r100_10x10_c22_t224_f64"], half=True, inverse=True, in_dtype=F64, out_dtype=F64),
    _rows("c2rodd", 243, ["jitc2rodd243_27x9_c21_t192"], half=True, inverse=True),
    _rows("c2rodd-f64", 243, ["jitc2rodd243_9x9x3_c8_t224_f64"], half=True, inverse=True, in_dtype=F64, out_dtype=F64),
    # N-d: the strided passes after the R2C rows (before the C2R rows) see an odd n/2 + 1 = 101 inner extent
    Form("r2c-2d-odd-inner", (3, 37, 200), ["jitr2c100_", "jitcols37_"], half=True, comps=1, flags=FLAG_NO_FUSED),
    Form("c2r-2d-odd-inner", (3, 37, 200), ["jitcols37_", "jitc2r100_"], half=True, inverse=True, flags=FLAG_NO_FUSED),
    Form("r2c-2d-odd-inner-f64", (3, 37, 200), ["jitr2c100_", "jitcols37_"], half=True, comps=1, in_dtype=F64,
         out_dtype=F64),
    Form("c2r-2d-odd-inner-f64", (3, 37, 200), ["jitcols37_", "jitc2r100_"], half=True, inverse=True, in_dtype=F64,
         out_dtype=F64),

    # ---- long axes: two passes through a plan-owned temporary ----------------------------------------------------------
    _split("split-rows", 40000, ["jitsplitA200_20x10_w16_t160", "jitsplitBrows200_20x10_c25_t256"], exec_host=True),
    _split("split-rows-inv", 40000, ["jitsplitA200_20x10_w16_t160", "jitsplitBrows200_20x10_c25_t256"], inverse=True),
    _split("split-rows-real", 40000, ["jitsplitA200_20x10_w16_t160_realin", "jitsplitBrows200_20x10_c25_t256"], comps=1),
    _split("split-rows-u8-real", 40000, ["jitsplitA200_20x10_w16_t160_realin_inu8", "jitsplitBrows200_20x10_c25_t256"], in_dtype=U8, comps=1),
    _split("split-rows-u8-complex", 40000, ["jitsplitA200_20x10_w16_t160_inu8", "jitsplitBrows200_20x10_c25_t256"], in_dtype=U8, inverse=True),
    _split("split-rows-f64-in", 40000, ["jitsplitA200_20x10_w16_t160_inf64", "jitsplitBrows200_20x10_c25_t256"], in_dtype=F64, inverse=True),
    _split("split-rows-f64-in-real", 40000, ["jitsplitA200_20x10_w16_t160_realin_inf64", "jitsplitBrows200_20x10_c25_t256"], in_dtype=F64, comps=1),
    _split("split-rows-f64", 40000, ["jitsplitA100_10x10_w16_t160_f64", "jitsplitBrows400_10x8x5_c4_t160_f64"], in_dtype=F64, out_dtype=F64, exec_host=True),
    _split("split-rows-f64-inv", 40000, ["jitsplitA100_10x10_w16_t160_f64", "jitsplitBrows400_10x8x5_c4_t160_f64"], in_dtype=F64, out_dtype=F64, inverse=True),
    _split("split-rows-f64-real", 40000, ["jitsplitA100_10x10_w16_t160_f64_realin", "jitsplitBrows400_10x8x5_c4_t160_f64"], in_dtype=F64, out_dtype=F64, comps=1),
    _split("split-rows-u8-to-f64", 40000, ["jitsplitA100_10x10_w16_t160_f64_realin_inu8", "jitsplitBrows400_10x8x5_c4_t160_f64"], in_dtype=U8, out_dtype=F64, comps=1),
    _split("split-rows-f32-to-f64", 40000, ["jitsplitA100_10x10_w16_t160_f64_inf32", "jitsplitBrows400_10x8x5_c4_t160_f64"], out_dtype=F64),
    _split("split-cols", 20000, ["jitsplitA200_20x10_w16_t160", "jitsplitBcols100_10x10_w6_t64"], inner=6, exec_host=True),
    _split("split-cols-inv-ragged", 20000, ["jitsplitA200_20x10_w16_t160", "jitsplitBcols100_10x10_w16_t160"], inner=19, inverse=True),
    _split("split-cols-f64", 20000, ["jitsplitA100_10x10_w16_t160_f64", "jitsplitBcols200_8x5x5_w6_t160_f64"], inner=6, in_dtype=F64, out_dtype=F64, exec_host=True),
    _split("split-cols-f64-inv-ragged", 20000, ["jitsplitA100_10x10_w16_t160_f64", "jitsplitBcols200_8x5x5_w16_t416_f64"], inner=19, in_dtype=F64, out_dtype=F64,
           inverse=True),
    # long half-spectrum rows (fp32: tests/test_gpu_long_real.py)
    _split("split-r2c-f64", 40000, ["jitsplitA100_10x10_w16_t160_f64", "jitsplitBr2c200_8x5x5_c10_t256_f64"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _split("split-r2c-f32-to-f64", 40000, ["jitsplitA100_10x10_w16_t160_f64_inf32", "jitsplitBr2c200_8x5x5_c10_t256_f64"], half=True, comps=1, out_dtype=F64),
    _split("split-c2r-f64", 40000, ["jitsplitAc2r100_10x10_w16_t160_f64", "jitsplitBrows200_8x5x5_c10_t256_f64"], half=True, inverse=True, in_dtype=F64, out_dtype=F64,
           exec_host=True),
    _split("split-r2codd-f64", 59049, ["jitsplitA729_9x9x9_w8_t224_f64_realin", "jitsplitBhalf81_9x9_c27_t256_f64"], half=True, comps=1, in_dtype=F64, out_dtype=F64),
    _split("split-c2rodd-f64", 59049, ["jitsplitAc2rodd729_9x9x9_w8_t224_f64", "jitsplitBreal81_9x9_c27_t256_f64"], half=True, inverse=True, in_dtype=F64,
           out_dtype=F64),
    _split("split-r2c", 40000, ["jitsplitA200_20x10_w16_t160", "jitsplitBr2c100_10x10_c32_t320"], half=True, comps=1),
    _split("split-c2r", 40000, ["jitsplitAc2r200_20x10_w16_t160", "jitsplitBrows100_10x10_c40_t416"], half=True, inverse=True),
    _split("split-r2codd", 59049, ["jitsplitA243_27x9_w32_t288_realin", "jitsplitBhalf243_27x9_c27_t256"], half=True, comps=1),
    _split("split-c2rodd", 59049, ["jitsplitAc2rodd243_27x9_w32_t288", "jitsplitBreal243_27x9_c27_t256"], half=True, inverse=True),

    # ---- axes above 2^24 points: three passes ----------------------------------------------------------------------
    _split3("split3-f64-inv", ["jitsplit3A512_8x8x8_w8_t256_f64", "jitsplit3A192_16x12_w16_t192_f64", "jitsplit3C256_16x16_c8_t128_f64"], in_dtype=F64, out_dtype=F64, inverse=True),
    _split3("split3-real", ["jitsplit3A768_32x24_w8_t192_realin", "jitsplit3A1024_32x32_w8_t256", "jitsplit3C32_32_c128_t128"], comps=1),
    _split3("split3-u8-real-f64", ["jitsplit3A512_8x8x8_w8_t256_f64_realin_inu8", "jitsplit3A192_16x12_w16_t192_f64", "jitsplit3C256_16x16_c8_t128_f64"], in_dtype=U8, comps=1, out_dtype=F64),
    _split3("split3-u8-complex", ["jitsplit3A768_32x24_w8_t192_inu8", "jitsplit3A1024_32x32_w8_t256", "jitsplit3C32_32_c128_t128"], in_dtype=U8),
    _split3("split3-f64-in-real", ["jitsplit3A768_32x24_w8_t192_realin_inf64", "jitsplit3A1024_32x32_w8_t256", "jitsplit3C32_32_c128_t128"], in_dtype=F64, comps=1),
    _split3("split3-f32-complex", ["jitsplit3A768_32x24_w8_t192", "jitsplit3A1024_32x32_w8_t256", "jitsplit3C32_32_c128_t128"]),

    # ---- planes: the two innermost axes in one in-place tile (fp32) ---------------------------------------------------
    Form("plane", (3, 40, 48), ["jitplane40x48("]),
    Form("plane-inv", (3, 40, 48), ["jitplane40x48("], inverse=True),
    Form("plane-real", (3, 40, 48), ["jitplane40x48("], comps=1),
    Form("plane-r2c", (3, 40, 96), ["jitr2cplane40x96("], half=True, comps=1),
]


def by_id():
    return {f.id: f for f in FORMS}


def logical_shape(form):
    """form.shape with a batch of None filled in: k * tile + 1 rows, k * tile >= MANY (a ragged last tile)."""
    if form.shape[0] is not None:
        return form.shape
    import re
    tile = int(re.search(r"_c(\d+)_t", form.tags[0]).group(1))
    k = -(-MANY // tile)
    return (k * tile + 1,) + form.shape[1:]


def readers(form):
    """The kinds of `form` that read the user's array: the first pass, and the scattering store of a one-pass plan."""
    return [form.kinds[0]] + (["jitscatter"] if form.scatter else [])

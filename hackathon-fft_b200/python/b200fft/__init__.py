"""ctypes shim over libb200fft.so + a Python mirror of the reference's `fft` package API.

The reference's public surface is `plan_fft[...]()` and `fft(output, x, ctx, plan=plan)`
(fft/fft/fft.mojo:122-323). Host code for the product is the Mojo package in
hackathon-fft_b200/mojo/ (cannot be compiled in this image: no Mojo toolchain); this
module is the equivalent binding for the Python comparison harness, tests and bench.
It keeps the reference's names and argument meaning:

    plan = plan_fft(in_dtype, out_dtype, in_layout, out_layout, bases=..., inverse=...)
    fft(output, x, ctx, plan=plan)      # async on stream `ctx`; caller synchronises

There is NO CPU path here: importing works without a GPU (so the planner rules can be
unit-tested), but anything that computes raises B200FFTError unless libb200fft.so is
built and an sm_100 device is present.
"""
import ctypes
import os

__all__ = ["plan_fft", "fft", "Plan", "SlabPlan", "B200FFTError", "ordered_bases", "default_bases", "dry_run",
           "launch_count", "variant_info", "lib_path", "REAL_FULL", "REAL_HALF", "FLAG_FORCE_GENERIC", "FLAG_NO_FUSED", "FLAG_PREFER_FUSED",
           "FLAG_FORCE_RT", "GPUTest", "stream_synchronize", "host_register", "host_unregister", "MgpuPlan", "mgpu_split",
           "MGPU_BATCH_SHARD", "MGPU_SLAB"]

MAX_RANK = 8
U8, F32, F64 = 0, 1, 2
REAL_FULL, REAL_HALF = 0, 1
FLAG_FORCE_GENERIC, FLAG_NO_FUSED, FLAG_PREFER_FUSED, FLAG_FORCE_RT = 1, 4, 8, 16
MGPU_BATCH_SHARD, MGPU_SLAB = 0, 1


class GPUTest:
    """The reference's `_GPUTest` path forcer (_ndim_fft_gpu.mojo:453-459) mapped onto this library's kernel tiers,
    so the same small vectors exercise each of them (fft/tests.mojo:398-417):
        BLOCK       -> one compile-time tile kernel per axis (no fused N-d kernel)
        WARP        -> the runtime-length tier (rt.cu)
        DEVICE_WIDE -> the fused N-d persistent kernel wherever a variant matches (device-wide dependency counters)
        CLUSTER     -> the generic per-output-point kernel (the reference's own formulation)"""
    BLOCK, WARP, DEVICE_WIDE, CLUSTER = 0, 1, 2, 3
    FLAGS = {0: FLAG_NO_FUSED, 1: FLAG_FORCE_RT, 2: FLAG_PREFER_FUSED, 3: FLAG_FORCE_GENERIC}

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.normpath(os.path.join(_HERE, "..", "..", "lib", "libb200fft.so"))
_lib = None


class B200FFTError(RuntimeError):
    def __init__(self, status, detail):
        self.status = status
        super().__init__("b200fft status %d: %s" % (status, detail))


class _Desc(ctypes.Structure):
    _fields_ = [
        ("rank", ctypes.c_int32),
        ("dims", ctypes.c_int64 * MAX_RANK),
        ("batch", ctypes.c_int64),
        ("in_components", ctypes.c_int32),
        ("in_dtype", ctypes.c_int32),
        ("out_dtype", ctypes.c_int32),
        ("inverse", ctypes.c_int32),
        ("real_mode", ctypes.c_int32),
        ("axis_mask", ctypes.c_uint32),
        ("bases", ctypes.POINTER(ctypes.c_uint32)),
        ("bases_count", ctypes.POINTER(ctypes.c_int32)),
        ("device", ctypes.c_int32),
        ("flags", ctypes.c_uint32),
    ]


# every symbol include/b200fft.h declares: (name, restype, argtypes)
_u32p = ctypes.POINTER(ctypes.c_uint32)
_vp = ctypes.c_void_p
SYMBOLS = [
    ("b200fft_plan_create", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_Desc)]),
    ("b200fft_plan_create_strided", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_Desc), ctypes.POINTER(ctypes.c_int64),
                                                    ctypes.POINTER(ctypes.c_int64)]),
    ("b200fft_exec", ctypes.c_int, [_vp, _vp, _vp, _vp]),
    ("b200fft_exec_host", ctypes.c_int, [_vp, _vp, _vp]),
    ("b200fft_stream_synchronize", ctypes.c_int, [_vp]),
    ("b200fft_host_register", ctypes.c_int, [_vp, ctypes.c_size_t]),
    ("b200fft_host_unregister", ctypes.c_int, [_vp]),
    ("b200fft_exec_scatter", ctypes.c_int, [_vp, ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, _vp, _vp, _vp]),
    ("b200fft_exec_scatter_at", ctypes.c_int, [_vp, ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int64, _vp, _vp, _vp]),
    ("b200fft_malloc", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_size_t]),
    ("b200fft_free", ctypes.c_int, [_vp]),
    ("b200fft_ipc_export", ctypes.c_int, [_vp, ctypes.c_char_p]),
    ("b200fft_ipc_open", ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(_vp)]),
    ("b200fft_ipc_close", ctypes.c_int, [_vp]),
    ("b200fft_slab_create", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int]),
    ("b200fft_slab_recv_bytes", ctypes.c_size_t, [_vp]),
    ("b200fft_slab_timeout_offset", ctypes.c_size_t, [_vp]),
    ("b200fft_slab_exec", ctypes.c_int, [_vp, _vp, _vp, ctypes.POINTER(_vp), ctypes.c_int, _vp]),
    ("b200fft_slab_describe", ctypes.c_size_t, [_vp, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_slab_destroy", ctypes.c_int, [_vp]),
    ("b200fft_plan_destroy", ctypes.c_int, [_vp]),
    ("b200fft_mgpu_plan_create", ctypes.c_int, [ctypes.POINTER(_vp), ctypes.POINTER(_Desc), ctypes.c_int,
                                                 ctypes.POINTER(ctypes.c_int), ctypes.c_int]),
    ("b200fft_mgpu_plan_destroy", ctypes.c_int, [_vp]),
    ("b200fft_mgpu_ngpu", ctypes.c_int, [_vp]),
    ("b200fft_mgpu_shard", ctypes.c_int, [_vp, ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    ("b200fft_mgpu_in_bytes", ctypes.c_size_t, [_vp, ctypes.c_int]),
    ("b200fft_mgpu_out_bytes", ctypes.c_size_t, [_vp, ctypes.c_int]),
    ("b200fft_mgpu_exec", ctypes.c_int, [_vp, ctypes.POINTER(_vp), ctypes.POINTER(_vp)]),
    ("b200fft_mgpu_synchronize", ctypes.c_int, [_vp]),
    ("b200fft_mgpu_stream", _vp, [_vp, ctypes.c_int]),
    ("b200fft_mgpu_exec_host", ctypes.c_int, [_vp, _vp, _vp]),
    ("b200fft_mgpu_describe", ctypes.c_size_t, [_vp, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_mgpu_split", ctypes.c_int, [ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_int64),
                                           ctypes.POINTER(ctypes.c_int64)]),
    ("b200fft_plan_workspace_bytes", ctypes.c_size_t, [_vp]),
    ("b200fft_plan_get_bases", ctypes.c_int, [_vp, ctypes.c_int, _u32p, ctypes.c_int]),
    ("b200fft_plan_describe", ctypes.c_size_t, [_vp, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_plan_launches", ctypes.c_int, [_vp]),
    ("b200fft_plan_in_bytes", ctypes.c_size_t, [_vp]),
    ("b200fft_plan_out_bytes", ctypes.c_size_t, [_vp]),
    ("b200fft_ordered_bases", ctypes.c_int, [ctypes.c_uint64, _u32p, ctypes.c_int, _u32p, ctypes.c_int]),
    ("b200fft_default_bases", ctypes.c_int, [ctypes.c_uint64, ctypes.c_int, _u32p, ctypes.c_int]),
    ("b200fft_plan_dry_run", ctypes.c_int, [ctypes.POINTER(_Desc), ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_jit_probe", ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, _u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_jit_probe_strided", ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, _u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                  ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_jit_split_probe", ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, _u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_jit_split3_probe", ctypes.c_int, [ctypes.c_int64, ctypes.c_int64, _u32p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                 ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]),
    ("b200fft_schedule_dry_run", ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64,
                                                 ctypes.POINTER(ctypes.c_int64), ctypes.c_int]),
    ("b200fft_strerror", ctypes.c_char_p, [ctypes.c_int]),
    ("b200fft_last_error", ctypes.c_char_p, []),
    ("b200fft_version", ctypes.c_int, []),
    ("b200fft_launch_count", ctypes.c_uint64, []),
    ("b200fft_variant_count", ctypes.c_int, [ctypes.c_int]),
    ("b200fft_variant_info", ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]),
]


def lib_path():
    return _LIB_PATH


def lib():
    """Load libb200fft.so. Fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise B200FFTError(-1, "%s is missing: run __graft_entry__.build() (make -C hackathon-fft_b200/csrc); "
                                   "there is no CPU or PyTorch fallback" % _LIB_PATH)
        L = ctypes.CDLL(_LIB_PATH)
        for name, restype, argtypes in SYMBOLS:
            fn = getattr(L, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise B200FFTError(rc, lib().b200fft_last_error().decode() or lib().b200fft_strerror(rc).decode())


def _dtype_code(dt):
    """Accept 'float32'/'f32', numpy dtypes, torch dtypes."""
    name = str(dt).replace("torch.", "").replace("numpy.", "").replace("<class '", "").replace("'>", "")
    name = {"f32": "float32", "f64": "float64", "u8": "uint8"}.get(name, name)
    try:
        return {"uint8": U8, "float32": F32, "float64": F64}[name]
    except KeyError:
        raise B200FFTError(1, "unsupported dtype %r (uint8, float32, float64)" % (dt,))


def device_malloc(nbytes):
    """cudaMalloc through the library: a buffer whose base can be exported over CUDA IPC."""
    p = ctypes.c_void_p()
    _check(lib().b200fft_malloc(ctypes.byref(p), nbytes))
    return p.value


def device_free(ptr):
    _check(lib().b200fft_free(ptr))


def ipc_export(ptr):
    buf = ctypes.create_string_buffer(64)
    _check(lib().b200fft_ipc_export(ptr, buf))
    return buf.raw


def ipc_open(handle):
    p = ctypes.c_void_p()
    _check(lib().b200fft_ipc_open(handle, ctypes.byref(p)))
    return p.value


def ipc_close(ptr):
    _check(lib().b200fft_ipc_close(ptr))


def stream_synchronize(stream=None):
    """Block until `stream` (None = the legacy default stream) is idle: b200fft_stream_synchronize."""
    _check(lib().b200fft_stream_synchronize(_ptr(stream)))


def host_register(arr):
    """Page-lock a caller-owned host array so exec_host's copies overlap the kernels (cudaHostRegister)."""
    _check(lib().b200fft_host_register(_ptr(arr), arr.nbytes))


def host_unregister(arr):
    _check(lib().b200fft_host_unregister(_ptr(arr)))


def ordered_bases(length, bases):
    """`_build_ordered_bases` + validity (_utils.mojo:163-221). None if the reference rejects them."""
    arr = (ctypes.c_uint32 * len(bases))(*bases)
    out = (ctypes.c_uint32 * 64)()
    n = lib().b200fft_ordered_bases(length, arr, len(bases), out, 64)
    return None if n < 0 else [int(out[i]) for i in range(n)]


def default_bases(length, target="gpu"):
    """`_estimate_best_bases` (fft.mojo:49-104)."""
    out = (ctypes.c_uint32 * 64)()
    n = lib().b200fft_default_bases(length, 1 if target == "gpu" else 0, out, 64)
    return [int(out[i]) for i in range(n)]


def schedule(phases, batch):
    """Tile schedule of the fused N-d kernel for phases = [(tiles_per_transform, tiles_per_group, dep_div, quota)...]:
    list of (phase, first_item, first_tile, count) segments (host logic only)."""
    flat = [int(v) for ph in phases for v in ph]
    arr = (ctypes.c_int64 * len(flat))(*flat)
    n = lib().b200fft_schedule_dry_run(len(phases), arr, batch, None, 0)
    if n < 0:
        raise B200FFTError(1, "inconsistent phase description")
    out = (ctypes.c_int64 * (4 * max(1, n)))()
    lib().b200fft_schedule_dry_run(len(phases), arr, batch, out, n)
    return [tuple(int(out[4 * i + k]) for k in range(4)) for i in range(n)]


def jit_probe(n, inner=1, bases=None, inverse=False, real_in=False, half=0, in_dtype="float32", out_dtype="float32",
              strided=False):
    """Compile (NVRTC, no GPU needed) the specialised kernel the planner would pick for one axis; returns its report.
    strided=True: the form a strided plan runs (b200fft_plan_create_strided), column tiles over `inner` columns when
    inner > 1."""
    arr = (ctypes.c_uint32 * len(bases))(*bases) if bases else None
    buf = ctypes.create_string_buffer(1024)
    probe = lib().b200fft_jit_probe_strided if strided else lib().b200fft_jit_probe
    _check(probe(n, inner, arr, len(bases) if bases else 0, 1 if inverse else 0, 1 if real_in else 0, half,
                 _dtype_code(in_dtype), _dtype_code(out_dtype), buf, len(buf)))
    return buf.value.decode()


def jit_split_probe(n, inner=1, bases=None, inverse=False, real_in=False, half=0, in_dtype="float32", out_dtype="float32"):
    """Compile (NVRTC, no GPU needed) the two passes the planner builds for an axis too long for one tile; returns
    "<pass A report>; <pass B report>"."""
    arr = (ctypes.c_uint32 * len(bases))(*bases) if bases else None
    buf = ctypes.create_string_buffer(2048)
    _check(lib().b200fft_jit_split_probe(n, inner, arr, len(bases) if bases else 0, 1 if inverse else 0, 1 if real_in else 0,
                                         half, _dtype_code(in_dtype), _dtype_code(out_dtype), buf, len(buf)))
    return buf.value.decode()


def jit_split3_probe(n, inner=1, bases=None, inverse=False, real_in=False, half=0, in_dtype="float32", out_dtype="float32"):
    """Compile (NVRTC, no GPU needed) the three passes the planner builds for a contiguous axis longer than 2^24 points;
    returns "<pass 1 report>; <pass 2 report>; <pass 3 report>"."""
    arr = (ctypes.c_uint32 * len(bases))(*bases) if bases else None
    buf = ctypes.create_string_buffer(4096)
    _check(lib().b200fft_jit_split3_probe(n, inner, arr, len(bases) if bases else 0, 1 if inverse else 0, 1 if real_in else 0,
                                          half, _dtype_code(in_dtype), _dtype_code(out_dtype), buf, len(buf)))
    return buf.value.decode()


def launch_count():
    return int(lib().b200fft_launch_count())


def variant_info(tier):
    """The compiled-in kernel variants of `tier` (0 row / column, 1 fused N-d, 2 two-pass split), in registration
    order, as dicts of the fields b200fft_variant_info writes. `forms` is a list; `n` and `radices` are ints / a list
    of ints except for fused variants, whose `n` is the dims text ("64x64x64") and `radices` the phases' stage lists
    ("8x8;8x8|8x8"). Host-only."""
    out = []
    for i in range(lib().b200fft_variant_count(tier)):
        need = lib().b200fft_variant_info(tier, i, None, 0)
        if need < 0:
            raise B200FFTError(1, "variant %d of tier %d" % (i, tier))
        buf = ctypes.create_string_buffer(need)
        lib().b200fft_variant_info(tier, i, buf, len(buf))
        d = dict(tok.split("=", 1) for tok in buf.value.decode().split())
        d["forms"] = d["forms"].split(",")
        for k in ("tile", "threads", "smem", "smem_r2c", "smem_c2r", "full", "async"):
            if k in d:
                d[k] = int(d[k])
        if d["kind"] != "fused":
            d["n"] = int(d["n"])
            d["radices"] = [int(r) for r in d["radices"].split("x")]
        out.append(d)
    return out


def _make_desc(in_dtype, out_dtype, in_layout, out_layout, bases, inverse, real_mode, axis_mask, device, flags):
    in_layout, out_layout = tuple(int(v) for v in in_layout), tuple(int(v) for v in out_layout)
    # _check_layout_conditions_nd (fft.mojo:20-46): the parts that need both layouts
    if len(out_layout) <= 2:
        raise B200FFTError(2, "The rank should be bigger than 2. The first dimension represents the amount of "
                              "batches, and the last the complex dimension.")
    if len(in_layout) != len(out_layout):
        raise B200FFTError(2, "in_layout and out_layout must have equal rank")
    half = real_mode == REAL_HALF
    if not half:
        if out_layout[-1] != 2:
            raise B200FFTError(2, "out_layout must have the last dimension equal to 2")
        if out_layout[:-1] != in_layout[:-1]:
            raise B200FFTError(2, "out_layout and in_layout should have the same shape before the last dimension")
        dims = out_layout[1:-1]
    else:
        # logical (real-side) dims: forward = input dims, inverse = output dims
        dims = (out_layout if inverse else in_layout)[1:-1]
        cplx = (in_layout if inverse else out_layout)
        want = tuple(dims[:-1]) + (dims[-1] // 2 + 1, 2)
        if tuple(cplx[1:]) != want or (in_layout if not inverse else out_layout)[-1] != 1:
            raise B200FFTError(2, "REAL_HALF layouts must be real (B, dims..., 1) and complex (B, dims[:-1]..., n/2+1, 2)")
    if len(dims) > MAX_RANK:
        raise B200FFTError(2, "at most %d transformed axes" % MAX_RANK)
    d = _Desc()
    d.rank = len(dims)
    for i, v in enumerate(dims):
        d.dims[i] = v
    d.batch = out_layout[0]
    d.in_components = in_layout[-1]
    d.in_dtype = _dtype_code(in_dtype)
    d.out_dtype = _dtype_code(out_dtype)
    d.inverse = 1 if inverse else 0
    d.real_mode = real_mode
    d.axis_mask = axis_mask
    d.device = -1 if device is None else int(device)
    d.flags = flags
    keep = []
    if bases is not None:
        if len(bases) != len(dims):
            raise B200FFTError(3, "The bases list should have the same outer size as the amount of internal "
                                  "dimensions. e.g. (batches, dim_0, dim_1, dim_2, 2) -> len(bases) == 3")
        flat = [int(b) for bl in bases for b in bl]
        cnt = [len(bl) for bl in bases]
        flat_arr = (ctypes.c_uint32 * max(1, len(flat)))(*flat)
        cnt_arr = (ctypes.c_int32 * len(cnt))(*cnt)
        d.bases = ctypes.cast(flat_arr, _u32p)
        d.bases_count = ctypes.cast(cnt_arr, ctypes.POINTER(ctypes.c_int32))
        keep = [flat_arr, cnt_arr]
    return d, keep


def dry_run(in_dtype, out_dtype, in_layout, out_layout, *, bases=None, inverse=False, real_mode=REAL_FULL,
            axis_mask=0, flags=0):
    """Validate a plan request and return its stage list text, without touching CUDA."""
    d, keep = _make_desc(in_dtype, out_dtype, in_layout, out_layout, bases, inverse, real_mode, axis_mask, None, flags)
    buf = ctypes.create_string_buffer(4096)
    _check(lib().b200fft_plan_dry_run(ctypes.byref(d), buf, len(buf)))
    return buf.value.decode()


def _ptr(obj):
    if obj is None:
        return None
    if isinstance(obj, int):
        return obj
    if hasattr(obj, "data_ptr"):       # torch.Tensor
        return obj.data_ptr()
    if hasattr(obj, "ctypes"):         # numpy.ndarray (host buffers for exec_host)
        return obj.ctypes.data
    if hasattr(obj, "cuda_stream"):    # torch.cuda.Stream
        return obj.cuda_stream
    raise TypeError("cannot take a device pointer from %r" % type(obj))


class Plan:
    """Handle on a b200fft_plan: the runtime analogue of the reference's `_GPUPlan`
    (_ndim_fft_gpu.mojo:153-207): owns the device twiddle tables, built once, reused."""

    def __init__(self, handle, in_layout, out_layout, in_dtype, out_dtype, inverse, in_strides=None, out_strides=None):
        self._h = handle
        self.in_layout, self.out_layout = tuple(in_layout), tuple(out_layout)
        self.in_dtype, self.out_dtype, self.inverse = in_dtype, out_dtype, inverse
        # element strides over (batch, dims...) of each buffer; None = dense (both None: a dense plan)
        self.in_strides, self.out_strides = in_strides, out_strides

    @property
    def strided(self):
        return self.in_strides is not None or self.out_strides is not None

    def exec(self, output, x, stream=None):
        _check(lib().b200fft_exec(self._h, _ptr(output), _ptr(x), _ptr(stream)))

    def exec_host(self, h_out, h_in):
        _check(lib().b200fft_exec_host(self._h, _ptr(h_out), _ptr(h_in)))

    def exec_scatter(self, peer_ptrs, my_rank, x, work, stream=None):
        """Local slab transform with the exchange fused into the last pass's store (see b200fft.h)."""
        arr = (ctypes.c_void_p * len(peer_ptrs))(*[_ptr(p) for p in peer_ptrs])
        _check(lib().b200fft_exec_scatter(self._h, arr, len(peer_ptrs), my_rank, _ptr(x), _ptr(work), _ptr(stream)))

    def bases(self, axis):
        out = (ctypes.c_uint32 * 64)()
        n = lib().b200fft_plan_get_bases(self._h, axis, out, 64)
        return None if n < 0 else [int(out[i]) for i in range(n)]

    def describe(self):
        n = lib().b200fft_plan_describe(self._h, None, 0)
        buf = ctypes.create_string_buffer(int(n) + 1)
        lib().b200fft_plan_describe(self._h, buf, len(buf))
        return buf.value.decode()

    @property
    def launches(self):
        return int(lib().b200fft_plan_launches(self._h))

    @property
    def in_bytes(self):
        return int(lib().b200fft_plan_in_bytes(self._h))

    @property
    def out_bytes(self):
        return int(lib().b200fft_plan_out_bytes(self._h))

    @property
    def workspace_bytes(self):
        return int(lib().b200fft_plan_workspace_bytes(self._h))

    def destroy(self):
        if self._h:
            lib().b200fft_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class SlabPlan:
    """One rank's share of a slab-decomposed n^3 transform as a single fused kernel (b200fft_slab_*)."""

    def __init__(self, n, ranks, rank, inverse=False, device=None):
        h = ctypes.c_void_p()
        _check(lib().b200fft_slab_create(ctypes.byref(h), n, ranks, rank, 1 if inverse else 0,
                                         -1 if device is None else int(device)))
        self._h = h
        self.n, self.ranks, self.rank = n, ranks, rank

    @property
    def recv_bytes(self):
        return int(lib().b200fft_slab_recv_bytes(self._h))

    @property
    def timeout_offset(self):
        return int(lib().b200fft_slab_timeout_offset(self._h))

    def exec(self, x, work, peer_recv, buffer, stream=None):
        arr = (ctypes.c_void_p * len(peer_recv))(*[_ptr(p) for p in peer_recv])
        _check(lib().b200fft_slab_exec(self._h, _ptr(x), _ptr(work), arr, buffer, _ptr(stream)))

    def describe(self):
        buf = ctypes.create_string_buffer(512)
        lib().b200fft_slab_describe(self._h, buf, len(buf))
        return buf.value.decode()

    def destroy(self):
        if self._h:
            lib().b200fft_slab_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def mgpu_split(batch, ngpu, g):
    """(first, count) of the batch items device slot g owns under MGPU_BATCH_SHARD (host-only rule)."""
    first, count = ctypes.c_int64(), ctypes.c_int64()
    if lib().b200fft_mgpu_split(batch, ngpu, g, ctypes.byref(first), ctypes.byref(count)) != 0:
        raise B200FFTError(1, "mgpu_split(%r, %r, %r)" % (batch, ngpu, g))
    return int(first.value), int(count.value)


class MgpuPlan:
    """One host process driving several GPUs (b200fft_mgpu_*): batch sharding without communication, or the slab
    decomposition of ONE 3-D transform with the exchange fused into the Y pass's peer-to-peer stores.

    MGPU_SLAB over G devices, layouts (1, Z, Y, X, 2) complex (fp32 or fp64), or with real_mode=REAL_HALF the real
    (1, Z, Y, X, 1) and the half spectrum (1, Z, Y, X//2+1, 2); W = X//2+1. Per slot g:
      complex:               ins[g] (Z/G, Y, X, 2)  -> outs[g] (Z, Y/G, X, 2)
      REAL_HALF forward:     ins[g] (Z/G, Y, X) real (fp32 or fp64) -> outs[g] (Z, Y/G, W, 2)
      REAL_HALF inverse:     ins[g] (Z, Y/G, W, 2) -> outs[g] (Z/G, Y, X) real, scaled by 1/(Z*Y*X)
    Forward outputs are Y-slabs (rows y of slot h: h*Y/G + y_local). The half-spectrum inverse takes exactly those
    Y-slabs and returns z planes, so forward then inverse round-trips on the device buffers (the complex inverse keeps
    z planes in and Y-slabs out). shard(g) reports z planes, or y rows for the half-spectrum inverse."""

    def __init__(self, in_dtype, out_dtype, in_layout, out_layout, *, devices, mode=MGPU_BATCH_SHARD, bases=None,
                 inverse=False, real_mode=REAL_FULL, flags=0):
        d, keep = _make_desc(in_dtype, out_dtype, in_layout, out_layout, bases, inverse, real_mode, 0, None, flags)
        devs = [int(v) for v in devices]
        arr = (ctypes.c_int * len(devs))(*devs)
        h = ctypes.c_void_p()
        _check(lib().b200fft_mgpu_plan_create(ctypes.byref(h), ctypes.byref(d), len(devs), arr, mode))
        self._h = h
        self.devices, self.mode = devs, mode

    @property
    def ngpu(self):
        return int(lib().b200fft_mgpu_ngpu(self._h))

    def shard(self, g):
        first, count = ctypes.c_int64(), ctypes.c_int64()
        _check(lib().b200fft_mgpu_shard(self._h, g, ctypes.byref(first), ctypes.byref(count)))
        return int(first.value), int(count.value)

    def in_bytes(self, g):
        return int(lib().b200fft_mgpu_in_bytes(self._h, g))

    def out_bytes(self, g):
        return int(lib().b200fft_mgpu_out_bytes(self._h, g))

    def stream(self, g):
        return lib().b200fft_mgpu_stream(self._h, g)

    def exec(self, outs, ins):
        """Enqueue on every slot's stream; outs[g] / ins[g] live on device slot g. Call synchronize() before reading."""
        o = (ctypes.c_void_p * len(outs))(*[_ptr(t) for t in outs])
        i = (ctypes.c_void_p * len(ins))(*[_ptr(t) for t in ins])
        _check(lib().b200fft_mgpu_exec(self._h, o, i))

    def synchronize(self):
        _check(lib().b200fft_mgpu_synchronize(self._h))

    def exec_host(self, h_out, h_in):
        """The whole job from / to host memory in natural order, spread over the devices; blocks until h_out is complete."""
        _check(lib().b200fft_mgpu_exec_host(self._h, _ptr(h_out), _ptr(h_in)))

    def describe(self):
        n = lib().b200fft_mgpu_describe(self._h, None, 0)
        buf = ctypes.create_string_buffer(int(n) + 1)
        lib().b200fft_mgpu_describe(self._h, buf, len(buf))
        return buf.value.decode()

    def destroy(self):
        if self._h:
            lib().b200fft_mgpu_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def _dense_strides(layout):
    """Element strides over (batch, dims...) of a dense buffer of shape `layout` (last entry: 1 real / 2 complex)."""
    out, s = [], 1
    for v in reversed(tuple(layout)[:-1]):
        out.append(s)
        s *= int(v)
    return tuple(reversed(out))


def plan_fft(in_dtype, out_dtype, in_layout, out_layout, *, bases=None, inverse=False, runtime_twfs=True,
             max_cluster_size=8, _test=None, real_mode=REAL_FULL, axis_mask=0, device=None, flags=0, in_strides=None,
             out_strides=None):
    """Plan the FFT on GPU — the reference's `plan_fft[...](ctx=ctx)` (fft.mojo:160-210).

    in_layout / out_layout are the reference's layouts as shape tuples:
    (batches, dim_0[, dim_1...], 1|2) -> (batches, dim_0[, dim_1...], 2).
    `bases`: one list of radix bases per axis (any primes / composites whose powers multiply
    to the axis length); None = the reference's default rule. `runtime_twfs` and
    `max_cluster_size` are accepted for signature compatibility and ignored (twiddles always
    come from device tables here). `_test`: a GPUTest value forces a kernel tier (the role of the
    reference's `Optional[_GPUTest]`); any other non-None value forces the generic kernel.
    `in_strides` / `out_strides`: strided buffers (b200fft_plan_create_strided), one stride per dimension of the layout
    but the last, in ELEMENTS (complex pairs or real scalars) of that buffer; None = dense. A torch view `v` of complex
    pairs has element strides `[s // 2 for s in v.stride()[:-1]]`.
    """
    if _test is not None:
        flags |= GPUTest.FLAGS.get(_test, FLAG_FORCE_GENERIC) if isinstance(_test, int) else FLAG_FORCE_GENERIC
    d, keep = _make_desc(in_dtype, out_dtype, in_layout, out_layout, bases, inverse, real_mode, axis_mask, device, flags)
    h = ctypes.c_void_p()
    if in_strides is None and out_strides is None:
        _check(lib().b200fft_plan_create(ctypes.byref(h), ctypes.byref(d)))
        return Plan(h, in_layout, out_layout, in_dtype, out_dtype, inverse)
    strides = []
    for name, st, layout in (("in_strides", in_strides, in_layout), ("out_strides", out_strides, out_layout)):
        st = _dense_strides(layout) if st is None else tuple(int(v) for v in st)
        if len(st) != len(layout) - 1:
            raise B200FFTError(2, "%s needs %d strides (batch and each axis), got %d" % (name, len(layout) - 1, len(st)))
        strides.append(st)
    arrs = [(ctypes.c_int64 * len(st))(*st) for st in strides]
    _check(lib().b200fft_plan_create_strided(ctypes.byref(h), ctypes.byref(d), arrs[0], arrs[1]))
    return Plan(h, in_layout, out_layout, in_dtype, out_dtype, inverse, strides[0], strides[1])


def fft(output, x, ctx=None, *, plan):
    """Calculate the FFT on GPU — the reference's `fft(output, x, ctx, plan=plan)` (fft.mojo:262-323).

    `output` / `x` are device buffers (torch CUDA tensors or raw device pointers) with the
    plan's layouts; `ctx` is the CUDA stream (torch.cuda.Stream, raw handle, or None for the
    current torch stream). Asynchronous; the caller synchronises (bench.mojo:51-52).
    """
    for name, t, layout, st in (("output", output, plan.out_layout, plan.out_strides), ("x", x, plan.in_layout, plan.in_strides)):
        if hasattr(t, "shape") and tuple(t.shape) != tuple(layout):
            raise B200FFTError(2, "%s has shape %s, the plan was built for %s" % (name, tuple(t.shape), layout))
        if plan.strided and hasattr(t, "stride"):
            want = tuple(v * layout[-1] for v in (st or _dense_strides(layout))) + (1,)
            got = tuple(t.stride())
            # a dimension of extent 1 may carry any stride; the components of an element must be adjacent
            if any(g != w for g, w, n in zip(got, want, t.shape) if n > 1) or (layout[-1] == 2 and got[-1] != 1):
                raise B200FFTError(2, "%s has strides %s, the plan was built for %s" % (name, got, want))
        elif hasattr(t, "is_contiguous") and not t.is_contiguous():
            raise B200FFTError(2, "%s must be dense row-major" % name)
        if hasattr(t, "is_cuda") and not t.is_cuda:
            raise B200FFTError(5, "%s is not a CUDA tensor: there is no CPU path (use Plan.exec_host for host buffers)" % name)
    if ctx is None:
        try:
            import torch
            ctx = torch.cuda.current_stream().cuda_stream
        except Exception:
            ctx = None
    plan.exec(output, x, ctx)

"""ctypes binding of libsdfk.so (include/sdfk.h).  The product path: fails loudly when the CUDA
library is missing or a call fails -- there is no CPU fallback."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SDFK_LIB: another build of the same library (kernel A/B experiments: `python -m sdfkit_b200.build --variant name -DX=..`)
LIB_PATH = os.environ.get("SDFK_LIB") or os.path.join(_HERE, "libsdfk.so")

PROGRESS_FN = C.CFUNCTYPE(None, C.c_float, C.c_void_p)
WRITE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.c_void_p)
_fp = C.POINTER(C.c_float)
_vp = C.c_void_p
_i64p = C.POINTER(C.c_int64)

# name -> (restype, argtypes).  Every symbol include/sdfk.h declares is listed here.
SIGNATURES = {
    "sdfk_last_error": (C.c_char_p, []),
    "sdfk_version": (C.c_int, []),
    "sdfk_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "sdfk_ctx_create_on_stream": (C.c_int, [C.c_int, _vp, C.POINTER(_vp)]),
    "sdfk_ctx_create_multi": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(_vp)]),
    "sdfk_ctx_device_count": (C.c_int, [_vp, C.POINTER(C.c_int)]),
    "sdfk_ctx_last_wall_ms": (C.c_int, [_vp, C.POINTER(C.c_double)]),
    "sdfk_plan_layers": (C.c_int, [_vp, _vp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int)]),
    "sdfk_ctx_destroy": (C.c_int, [_vp]),
    "sdfk_ctx_synchronize": (C.c_int, [_vp]),
    "sdfk_ctx_stream": (C.c_int, [_vp, C.POINTER(_vp)]),
    "sdfk_ctx_timer_start": (C.c_int, [_vp]),
    "sdfk_ctx_timer_stop": (C.c_int, [_vp, _fp]),
    "sdfk_ctx_mark": (C.c_int, [_vp, C.c_int]),
    "sdfk_ctx_elapsed": (C.c_int, [_vp, C.c_int, C.c_int, _fp]),
    "sdfk_ctx_launch_count": (C.c_int, [_vp, _i64p]),
    "sdfk_ctx_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "sdfk_ctx_store_bandwidth": (C.c_int, [_vp, C.c_size_t, C.c_int, C.POINTER(C.c_double)]),
    "sdfk_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp)]),
    "sdfk_host_free": (C.c_int, [_vp]),
    "sdfk_sdf_compile": (C.c_int, [_vp, C.c_char_p, C.c_size_t, C.POINTER(_vp)]),
    "sdfk_sdf_destroy": (C.c_int, [_vp]),
    "sdfk_sdf_check": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "sdfk_sdf_eval": (C.c_int, [_vp, _fp, _fp, C.c_int64]),
    "sdfk_constdiv_verify": (C.c_int, [_vp, C.c_float, _i64p]),
    "sdfk_selftest_sqrt": (C.c_int, [_vp, _i64p]),
    "sdfk_voxels_sample": (C.c_int, [_vp, _vp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "sdfk_voxels_sample_slab": (C.c_int, [_vp, _vp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(_vp)]),
    "sdfk_voxels_sample_distances": (C.c_int, [_vp, _vp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(_vp)]),
    "sdfk_voxels_resample": (C.c_int, [_vp, _vp, C.c_int]),
    "sdfk_voxels_import": (C.c_int, [_vp, _fp, _fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "sdfk_voxels_export": (C.c_int, [_vp, _fp, _fp]),
    "sdfk_voxels_clip": (C.c_int, [_vp]),
    "sdfk_voxels_info": (C.c_int, [_vp, C.POINTER(C.c_int), C.POINTER(_vp), C.POINTER(_vp)]),
    "sdfk_voxels_layers": (C.c_int, [_vp, C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_int)]),
    "sdfk_voxels_part": (C.c_int, [_vp, C.c_int, C.POINTER(_vp)]),
    "sdfk_voxels_destroy": (C.c_int, [_vp]),
    "sdfk_mesh_create": (C.c_int, [_vp, _vp, C.c_float, C.c_int, _fp, _fp, PROGRESS_FN, _vp, C.POINTER(_vp)]),
    "sdfk_mesh_classify": (C.c_int, [_vp, _vp, C.c_float, C.c_int, C.c_int, C.c_int, C.POINTER(_vp), _i64p, _i64p]),
    "sdfk_mesh_emit": (C.c_int, [_vp, C.c_int64, C.c_int64, _fp, _fp]),
    "sdfk_mesh_emit_host": (C.c_int, [_vp, C.c_int64, C.c_int64, _fp, _fp, C.c_int]),
    "sdfk_mesh_counts": (C.c_int, [_vp, _i64p, _i64p]),
    "sdfk_sdf_to_mesh_host": (C.c_int, [_vp, _vp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, _fp, _fp, C.c_int,
                                        PROGRESS_FN, _vp, C.POINTER(_vp)]),
    "sdfk_mesh_host_ptrs": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "sdfk_mesh_export": (C.c_int, [_vp, _fp, _fp, _fp, C.POINTER(C.c_int32), _fp]),
    "sdfk_mesh_device_ptrs": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "sdfk_mesh_part": (C.c_int, [_vp, C.c_int, C.POINTER(_vp), _i64p, _i64p]),
    "sdfk_mesh_stats": (C.c_int, [_vp, C.POINTER(C.c_double)]),
    "sdfk_mesh_destroy": (C.c_int, [_vp]),
    "sdfk_obj_write": (C.c_int, [_vp, _fp, C.c_int64, _fp, C.c_int64, C.POINTER(C.c_int32), C.c_int64, WRITE_FN, _vp, _i64p]),
    "sdfk_selftest_float_text": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64)]),
    "sdfk_render": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, _fp]),
    "sdfk_render_depth": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_int, C.c_int, C.c_int, _fp]),
    "sdfk_render_bgr8": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int,
                                   C.POINTER(C.c_ubyte)]),
    "sdfk_render_depth_gray8": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int,
                                          C.POINTER(C.c_ubyte)]),
    "sdfk_render_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _fp, _fp, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, _vp]),
}


class SdfkError(RuntimeError):
    """A libsdfk call failed (status < 0); the message is sdfk_last_error()."""

    def __init__(self, code, message):
        super().__init__("libsdfk error %d: %s" % (code, message))
        self.code = code


class NotSupportedError(NotImplementedError):
    """The reference would run this on the CPU (e.g. an opaque lambda Sdf); the GPU path rejects it."""


_lib = None


def lib():
    """Load libsdfk.so (built in-tree by sdfkit_b200/build.py).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libsdfk.so is missing (%s): build it with `python -m sdfkit_b200.build` -- the SdfKit GPU path "
                "has no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)     # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code != 0:
        raise SdfkError(code, (lib().sdfk_last_error() or b"").decode("utf-8", "replace"))


def fptr(a):
    return None if a is None else a.ctypes.data_as(_fp)


def f32c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a if shape is None else a.reshape(shape)


class PinnedPool:
    """Page-locked host buffers for exports (sdfk_host_alloc), recycled when every numpy view of a buffer has been
    garbage collected -- pinning 100s of MB costs far more than copying them, so buffers are never freed eagerly."""
    _free = {}      # size class -> [pointer, ...]
    _seen = set()   # size classes that have been allocated before

    class _Block:
        def __init__(self, ptr, size):
            self.ptr, self.size = ptr, size

        def __del__(self):
            try:
                PinnedPool._free.setdefault(self.size, []).append(self.ptr)
            except Exception:
                pass

    @classmethod
    def empty(cls, shape, dtype):
        """A numpy array of `shape`/`dtype` living in pinned memory."""
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        size = 1 << max(12, (max(nbytes, 1) - 1).bit_length())
        lst = cls._free.setdefault(size, [])
        if lst:
            ptr = lst.pop()
        else:
            # `img = sdf.ToImage(...)` in a loop holds the previous result while the next one is made: the first miss of a
            # size class pins two buffers (pinning costs ~0.5 ms/MB), so the second call already finds a recycled one
            for _ in range(2 if (size <= (256 << 20) and size not in cls._seen) else 1):
                p = _vp()
                check(lib().sdfk_host_alloc(size, C.byref(p)))
                lst.append(p.value)
            cls._seen.add(size)
            ptr = lst.pop()
        block = cls._Block(ptr, size)
        buf = (C.c_ubyte * size).from_address(ptr)
        buf._block = block                       # the ctypes buffer keeps the block alive; numpy keeps the buffer alive
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


OPT_SIGN_PLANES = 1


class Context:
    """sdfk_ctx: one GPU + one stream, or -- Context(devices=[0, 1, ...]) -- N GPUs of one box behind one handle
    (sdfk_ctx_create_multi: z-slab / row-band sharding inside the library).  `default()` gives the per-process context
    (LOCAL_RANK aware)."""
    _default = None

    def __init__(self, device=None, stream=None, devices=None):
        h = _vp()
        if devices is not None:
            devices = [int(d) for d in devices]
            arr = (C.c_int * len(devices))(*devices)
            check(lib().sdfk_ctx_create_multi(len(devices), arr, C.byref(h)))
            device = devices[0]
        else:
            if device is None:
                device = int(os.environ.get("LOCAL_RANK", "0"))
            if stream is None:
                check(lib().sdfk_ctx_create(int(device), C.byref(h)))
            else:
                check(lib().sdfk_ctx_create_on_stream(int(device), _vp(int(stream)), C.byref(h)))
        self.handle = h
        self.device = int(device)
        self.devices = devices or [int(device)]

    def device_count(self):
        n = C.c_int()
        check(lib().sdfk_ctx_device_count(self.handle, C.byref(n)))
        return n.value

    def last_wall_ms(self):
        """Host wall clock of the last multi-GPU library call on this context (entry until every device had finished)."""
        ms = C.c_double()
        check(lib().sdfk_ctx_last_wall_ms(self.handle, C.byref(ms)))
        return ms.value

    @classmethod
    def default(cls):
        if cls._default is None:
            cls._default = cls()
        return cls._default

    def synchronize(self):
        check(lib().sdfk_ctx_synchronize(self.handle))

    def stream(self):
        s = _vp()
        check(lib().sdfk_ctx_stream(self.handle, C.byref(s)))
        return s.value or 0

    def timer_start(self):
        check(lib().sdfk_ctx_timer_start(self.handle))

    def timer_stop(self):
        ms = C.c_float()
        check(lib().sdfk_ctx_timer_stop(self.handle, C.byref(ms)))
        return ms.value

    def mark(self, slot):
        check(lib().sdfk_ctx_mark(self.handle, int(slot)))

    def elapsed(self, slot_a, slot_b):
        ms = C.c_float()
        check(lib().sdfk_ctx_elapsed(self.handle, int(slot_a), int(slot_b), C.byref(ms)))
        return ms.value

    def launch_count(self):
        n = C.c_int64()
        check(lib().sdfk_ctx_launch_count(self.handle, C.byref(n)))
        return n.value

    def constdiv_ok(self, divisor):
        """May the packed SDF body divide by this float32 constant with the 3-instruction sequence (sk2_divc)?  Decided by an
        exhaustive comparison with IEEE division on this context's GPU (all 2^32 dividends), once per constant."""
        d = np.float32(divisor)
        if not np.isfinite(d) or d == 0 or not (2.0 ** -30 <= abs(float(d)) <= 2.0 ** 30):
            return False
        cache = self.__dict__.setdefault("_constdiv", {})
        key = d.tobytes()
        if key not in cache:
            bad = C.c_int64()
            check(lib().sdfk_constdiv_verify(self.handle, C.c_float(float(d)), C.byref(bad)))
            cache[key] = bad.value == 0
        return cache[key]

    def selftest_sqrt(self):
        bad = C.c_int64()
        check(lib().sdfk_selftest_sqrt(self.handle, C.byref(bad)))
        return bad.value

    def set_option(self, option, value):
        check(lib().sdfk_ctx_set_option(self.handle, int(option), int(value)))

    def store_bandwidth(self, nbytes=4 << 30, reps=5):
        """GB/s of a store-only kernel in memory order (sdfk_ctx_store_bandwidth): the ceiling of the sampling kernels."""
        g = C.c_double()
        check(lib().sdfk_ctx_store_bandwidth(self.handle, int(nbytes), int(reps), C.byref(g)))
        return g.value

    def close(self):
        if self.handle:
            lib().sdfk_ctx_destroy(self.handle)
            self.handle = None
            if Context._default is self:
                Context._default = None

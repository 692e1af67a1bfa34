"""
ctypes binding of libshepseg_b200.so (C ABI declared in include/shepseg_b200.h).

There is no CPU fallback: importing this module without the built library raises, and
creating a Context without a CUDA device raises.  The library is built in-tree by
`__graft_entry__.build()` (or `make -C pyshepseg_b200/csrc`).
"""
import atexit
import ctypes
import os
import threading

import numpy

_HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(_HERE, 'libshepseg_b200.so')

SSG_U8, SSG_U16, SSG_I16, SSG_U32, SSG_I32 = 0, 1, 2, 3, 4
DTYPE_CODES = {
    numpy.dtype(numpy.uint8): SSG_U8,
    numpy.dtype(numpy.uint16): SSG_U16,
    numpy.dtype(numpy.int16): SSG_I16,
    numpy.dtype(numpy.uint32): SSG_U32,
    numpy.dtype(numpy.int32): SSG_I32,
}
SSG_MAX_BANDS = 64
SSG_MAX_CLUSTERS = 1024
SSG_EXTENT_TABLES = 10
ABI_VERSION = 2

SEG_PRESENT, SEG_NUMBERED, SEG_KEYTOP, SEG_KEYLEFT, SEG_INTRIM = 1, 2, 4, 8, 16
PAIR_LEFT = 1 << 63


class ShepsegB200Error(RuntimeError):
    pass


class TileParams(ctypes.Structure):
    _fields_ = [('dtype', ctypes.c_int), ('nBands', ctypes.c_int),
        ('nRows', ctypes.c_int64), ('nCols', ctypes.c_int64),
        ('centres', ctypes.c_void_p), ('k', ctypes.c_int), ('hasNull', ctypes.c_int),
        ('nullVal', ctypes.c_double), ('fourConnected', ctypes.c_int),
        ('minSegSize', ctypes.c_int), ('spectralThreshold', ctypes.c_double),
        ('trimTop', ctypes.c_int64), ('trimBottom', ctypes.c_int64), ('trimLeft', ctypes.c_int64),
        ('trimRight', ctypes.c_int64), ('stripRows', ctypes.c_int64), ('stripCols', ctypes.c_int64),
        ('extentsDev', ctypes.c_void_p), ('extentsCap', ctypes.c_int64)]


class TileResult(ctypes.Structure):
    _fields_ = [('numClumps', ctypes.c_uint32), ('numSegments', ctypes.c_uint32),
        ('singlePixelsEliminated', ctypes.c_uint32),
        ('smallSegmentsEliminated', ctypes.c_int64), ('numOversized', ctypes.c_uint32),
        ('numSinglePixelRounds', ctypes.c_uint32), ('numSmallPasses', ctypes.c_uint32),
        ('msAssign', ctypes.c_float), ('msClump', ctypes.c_float), ('msSingle', ctypes.c_float),
        ('msSmall', ctypes.c_float), ('msTotal', ctypes.c_float),
        ('extentsDone', ctypes.c_uint32), ('extentsStride', ctypes.c_uint32)]


class TileTables(ctypes.Structure):
    _fields_ = [('maxId', ctypes.c_uint32), ('countNew', ctypes.c_uint32),
        ('numPairs', ctypes.c_uint32), ('maxRankInTrim', ctypes.c_uint32)]


_c = ctypes
_vp, _i, _i64, _u32, _dbl, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_uint32, _c.c_double, _c.c_size_t

# name -> (restype, argtypes); exactly the functions include/shepseg_b200.h declares
SIGNATURES = {
    'ssg_abi_version': (_i, []),
    'ssg_device_count': (_i, []),
    'ssg_ctx_create': (_i, [_i, _c.POINTER(_vp)]),
    'ssg_ctx_create_priority': (_i, [_i, _c.POINTER(_vp)]),
    'ssg_ctx_destroy': (None, [_vp]),
    'ssg_last_error': (_c.c_char_p, [_vp]),
    'ssg_ctx_stream': (_vp, [_vp]),
    'ssg_ctx_synchronize': (_i, [_vp]),
    'ssg_ctx_reserve': (_i, [_vp, _i64, _i, _i, _i64]),
    'ssg_host_alloc': (_i, [_sz, _c.POINTER(_vp)]),
    'ssg_host_free': (_i, [_vp]),
    'ssg_assign': (_i, [_vp, _vp, _i, _i, _i64, _i64, _vp, _i, _i, _dbl, _vp]),
    'ssg_clump': (_i, [_vp, _vp, _i64, _i64, _c.c_int32, _i, _u32, _vp, _c.POINTER(_u32)]),
    'ssg_make_seg_size': (_i, [_vp, _vp, _i64, _vp, _i64]),
    'ssg_eliminate_single_pixels': (_i, [_vp, _vp, _i, _i, _i64, _i64, _vp, _vp, _i64, _u32, _i,
        _c.POINTER(_i64)]),
    'ssg_relabel_segments': (_i, [_vp, _vp, _i64, _vp, _i64, _u32]),
    'ssg_eliminate_small_segments': (_i, [_vp, _vp, _vp, _i, _i, _i64, _i64, _u32, _i, _dbl, _i, _u32,
        _c.POINTER(_i64)]),
    'ssg_segment_tile': (_i, [_vp, _vp, _c.POINTER(TileParams), _vp, _c.POINTER(TileResult)]),
    'ssg_segment_tile_device': (_i, [_vp, _vp, _c.POINTER(TileParams), _vp, _c.POINTER(TileResult)]),
    'ssg_upload_image': (_i, [_vp, _vp, _i, _i, _i64, _i64]),
    'ssg_staged_image': (_vp, [_vp]),
    'ssg_download_labels': (_i, [_vp, _vp]),
    'ssg_resident_labels': (_vp, [_vp]),
    'ssg_tile_tables_device': (_i, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64,
        _i64, _u32, _vp, _i64, _c.POINTER(TileTables)]),
    'ssg_tile_tables_fetch': (_i, [_vp, _vp, _vp, _vp, _vp]),
    'ssg_apply_lut_device': (_i, [_vp, _vp, _i64, _i64, _vp, _u32, _i64, _i64, _i64, _i64, _vp, _i64,
        _vp, _i64]),
    'ssg_apply_rel_lut_device': (_i, [_vp, _vp, _i64, _i64, _vp, _vp, _u32, _u32, _i64, _vp, _vp, _i64, _i64, _i64, _i64,
        _vp, _i64, _vp, _i64]),
    'ssg_window_overviews': (_i, [_vp, _vp, _i64, _i64, _i64, _i, _vp, _vp, _i64, _vp]),
    'ssg_dev_alloc': (_i, [_vp, _sz, _c.POINTER(_vp)]),
    'ssg_dev_free': (_i, [_vp, _vp]),
    'ssg_memcpy_h2d': (_i, [_vp, _vp, _vp, _sz]),
    'ssg_memcpy_d2h': (_i, [_vp, _vp, _vp, _sz]),
    'ssg_memcpy_d2d': (_i, [_vp, _vp, _vp, _sz]),
    'ssg_memcpy2d_d2d': (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    'ssg_memcpy2d_d2h': (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    'ssg_memcpy2d_h2d': (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    'ssg_memset_d': (_i, [_vp, _vp, _i, _sz]),
    'ssg_memcpy_d2h_async': (_i, [_vp, _vp, _vp, _sz]),
    'ssg_memcpy2d_d2h_async': (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    'ssg_mark': (_i, [_vp, _i]),
    'ssg_wait_mark': (_i, [_vp, _i]),
    'ssg_kmeans_begin': (_i, [_vp, _vp, _i64, _i, _vp, _i]),
    'ssg_kmeans_step': (_i, [_vp, _vp, _c.POINTER(_dbl), _c.POINTER(_c.c_uint64)]),
    'ssg_kmeans_labels': (_i, [_vp, _vp]),
    'ssg_kmeans_relocate': (_i, [_vp, _i, _vp, _vp]),
    'ssg_kmeans_update': (_i, [_vp, _c.POINTER(_dbl), _vp]),
    'ssg_kmeans_centres': (_i, [_vp, _vp]),
    'ssg_segment_stats': (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i64, _u32, _i, _vp, _vp, _i64, _vp, _vp, _vp]),
    'ssg_launch_count': (_c.c_uint64, [_vp]),
    'ssg_profile_enable': (_i, [_vp, _i]),
    'ssg_profile_fetch': (_i, [_vp, _c.c_char_p, _sz]),
}

_lib = None
_libLock = threading.Lock()


def load():
    """Load the shared library and declare every signature.  Raises if it is missing."""
    global _lib
    with _libLock:
        if _lib is None:
            if not os.path.exists(LIBPATH):
                raise ShepsegB200Error(
                    'libshepseg_b200.so is not built (%s); run `python -c "import '
                    '__graft_entry__ as g; g.build()"` or `make -C pyshepseg_b200/csrc`. '
                    'There is no CPU fallback.' % LIBPATH)
            lib = ctypes.CDLL(LIBPATH)
            for (name, (res, args)) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            if lib.ssg_abi_version() != ABI_VERSION:
                raise ShepsegB200Error('libshepseg_b200.so has ABI version %d, this binding needs %d: '
                    'rebuild it (make -C pyshepseg_b200/csrc)' % (lib.ssg_abi_version(), ABI_VERSION))
            _lib = lib
    return _lib


def ptr(a):
    """Pointer of a numpy array (must be C-contiguous) or pass through ints / None."""
    if a is None:
        return None
    if isinstance(a, numpy.ndarray):
        if not a.flags.c_contiguous:
            raise ValueError('array must be C-contiguous')
        return a.ctypes.data
    return a


class PinnedArray(object):
    """A numpy array over pinned host memory (ssg_host_alloc)."""
    def __init__(self, shape, dtype):
        lib = load()
        self.shape = tuple(int(s) for s in numpy.atleast_1d(shape))
        self.dtype = numpy.dtype(dtype)
        nbytes = int(numpy.prod(self.shape)) * self.dtype.itemsize
        p = ctypes.c_void_p()
        rc = lib.ssg_host_alloc(max(nbytes, 1), ctypes.byref(p))
        if rc != 0:
            raise ShepsegB200Error('pinned allocation of %d bytes failed' % nbytes)
        self._p = p
        buf = (ctypes.c_ubyte * max(nbytes, 1)).from_address(p.value)
        self.array = numpy.frombuffer(buf, dtype=self.dtype, count=int(numpy.prod(self.shape))
            ).reshape(self.shape)

    def free(self):
        if self._p is not None:
            self.array = None
            load().ssg_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context(object):
    """One ssg_ctx: a CUDA stream plus scratch memory on one device, used by one thread."""
    def __init__(self, device=0, highPriority=False):
        self.lib = load()
        self.device = int(device)
        h = ctypes.c_void_p()
        create = self.lib.ssg_ctx_create_priority if highPriority else self.lib.ssg_ctx_create
        rc = create(self.device, ctypes.byref(h))
        if rc != 0 or not h:
            raise ShepsegB200Error('cannot create a CUDA context on device %d (code %d): a B200 '
                'is required, there is no CPU fallback' % (self.device, rc))
        self.h = h

    def close(self):
        if getattr(self, 'h', None):
            self.lib.ssg_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def check(self, rc, what):
        if rc != 0:
            msg = self.lib.ssg_last_error(self.h)
            raise ShepsegB200Error('%s failed (code %d): %s' % (what, rc,
                msg.decode('utf-8', 'replace') if msg else ''))

    def call(self, name, *args):
        self.check(getattr(self.lib, name)(self.h, *args), name)

    @property
    def stream(self):
        return self.lib.ssg_ctx_stream(self.h)

    def synchronize(self):
        self.call('ssg_ctx_synchronize')

    def launch_count(self):
        return int(self.lib.ssg_launch_count(self.h))

    # ---- device memory -------------------------------------------------------------------
    def dev_alloc(self, nbytes):
        if os.environ.get('SSG_DEBUG_ALLOC'):
            import sys
            print('[ssg py] dev_alloc %d bytes' % nbytes, file=sys.stderr)
        p = ctypes.c_void_p()
        self.check(self.lib.ssg_dev_alloc(self.h, int(nbytes), ctypes.byref(p)), 'ssg_dev_alloc')
        return p.value

    def dev_free(self, p):
        if p:
            self.call('ssg_dev_free', p)

    def h2d(self, dst, src):
        src = numpy.ascontiguousarray(src)
        self.call('ssg_memcpy_h2d', dst, ptr(src), src.nbytes)
        self.synchronize()

    def d2h(self, dst, src, nbytes=None):
        self.call('ssg_memcpy_d2h', ptr(dst), src, dst.nbytes if nbytes is None else nbytes)


# Default contexts: one per (thread, device), held in thread-local storage so that a context
# (its stream, pinned words and multi-gigabyte scratch slab) dies with the thread that made it
# instead of piling up under reused thread idents.  Callers that run their own threads for long
# should pass context= explicitly and close it themselves.
_defaultLocal = threading.local()
_defaultAll = set()
_defaultLock = threading.Lock()


class _ThreadContexts(object):
    """The contexts of one thread; closing them when the thread-local storage is collected."""
    def __init__(self):
        self.byDevice = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def close(self):
        for ctx in self.byDevice.values():
            with _defaultLock:
                _defaultAll.discard(ctx)
            ctx.close()
        self.byDevice = {}


def _closeDefaultContexts():
    with _defaultLock:
        ctxs = list(_defaultAll)
        _defaultAll.clear()
    for ctx in ctxs:
        ctx.close()


atexit.register(_closeDefaultContexts)


def default_context(device=0):
    """A per-thread, per-device context for the simple (single call) entry points."""
    holder = getattr(_defaultLocal, 'holder', None)
    if holder is None:
        holder = _defaultLocal.holder = _ThreadContexts()
    ctx = holder.byDevice.get(int(device))
    if ctx is None or ctx.h is None:
        ctx = Context(device)
        holder.byDevice[int(device)] = ctx
        with _defaultLock:
            _defaultAll.add(ctx)
    return ctx

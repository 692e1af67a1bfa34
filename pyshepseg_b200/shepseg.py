"""
Drop-in for the hot path of pyshepseg.shepseg, computed on a B200.

Same function names, argument meaning, result object and in-place conventions as the
reference module (pyshepseg/shepseg.py); the numba loops and the scikit-learn predict are
replaced by CUDA kernels reached through the C ABI in include/shepseg_b200.h.  What stays
on the host, as in the reference: the k-means fit on the pixel subsample
(fitSpectralClusters, shepseg.py:252-314) and the resolution of maxSpectralDiff
(autoMaxSpectralDiff, shepseg.py:400-449).

There is no CPU fallback.  Without the built library or without a CUDA device every
compute function raises ShepsegB200Error.
"""
import ctypes
import time

import numpy

from . import _lib
from ._lib import ShepsegB200Error  # noqa: F401  (re-exported)

# shepseg.py:97-101
SegIdType = numpy.uint32
SEGNULLVAL = 0
MINSEGID = SEGNULLVAL + 1


class SegmentationResult(object):
    """
    Results of the segmentation process (shepseg.py:104-127).

    Attributes
    ----------
      segimg : numpy array (nRows, nCols) of uint32 segment ID numbers (starting from 1)
      kmeans : the fitted KMeans object (or whatever was passed as kmeansObj)
      maxSpectralDiff : the value used to limit segment merging
      singlePixelsEliminated : number of single pixels merged to adjacent segments
      smallSegmentsEliminated : number of small segments merged into adjacent segments
      timings : dict of device milliseconds per stage (extension; not in the reference)
    """
    def __init__(self):
        self.segimg = None
        self.kmeans = None
        self.maxSpectralDiff = None
        self.singlePixelsEliminated = None
        self.smallSegmentsEliminated = None
        self.timings = None


def _deviceImage(img):
    """The image as a C-contiguous array of a dtype the kernels take."""
    img = numpy.asarray(img)
    if img.ndim != 3:
        raise ValueError('img must have shape (nBands, nRows, nCols)')
    if not numpy.issubdtype(img.dtype, numpy.integer):
        raise TypeError('img must be an integer array (got %s)' % img.dtype)
    if img.dtype.itemsize > 2 or img.dtype not in _lib.DTYPE_CODES:
        # Values that fit 16 bits take the (faster) 16-bit kernels, and values that fit 32 bits
        # the 32-bit ones.  The reference widens every value to int64 or float64 before any
        # arithmetic, so the narrower type gives the same results.
        (lo, hi) = (int(img.min()), int(img.max())) if img.size else (0, 0)
        for t in (numpy.uint16, numpy.int16, numpy.uint32, numpy.int32):
            info = numpy.iinfo(t)
            if lo >= info.min and hi <= info.max:
                img = img.astype(t, copy=False)
                break
        else:
            raise NotImplementedError('image dtype %s with values outside 32 bits is not '
                'supported by the B200 path' % img.dtype)
    if img.shape[0] > _lib.SSG_MAX_BANDS:
        raise NotImplementedError('at most %d bands are supported' % _lib.SSG_MAX_BANDS)
    return numpy.ascontiguousarray(img)


def _centres(kmeansObj):
    c = getattr(kmeansObj, 'cluster_centers_', kmeansObj)
    return numpy.ascontiguousarray(c, dtype=numpy.float64)


def spectralThreshold(maxSpectralDiff):
    """
    maxSpectralDiff**2 as the reference's numba code evaluates it (shepseg.py:1060): the
    power is taken in maxSpectralDiff's own type (float32 for the numpy.float32 that 'auto'
    and None produce, float64 for a Python float, integer for a Python int) and the
    comparison with the float32 distance happens in float64.
    """
    if isinstance(maxSpectralDiff, numpy.float32):
        return float(numpy.float32(maxSpectralDiff) * numpy.float32(maxSpectralDiff))
    if isinstance(maxSpectralDiff, (int, numpy.integer)) and not isinstance(maxSpectralDiff, bool):
        return float(int(maxSpectralDiff) ** 2)
    return float(maxSpectralDiff) ** 2


def doShepherdSegmentation(img, numClusters=60, clusterSubsamplePcnt=1,
        minSegmentSize=50, maxSpectralDiff='auto', imgNullVal=None,
        fourConnected=True, verbose=False, fixedKMeansInit=False,
        kmeansObj=None, spectDistPcntile=50, context=None):
    """
    Perform Shepherd segmentation in memory, on the given multi-band img array
    (shepseg.py:130-249).  Parameters and the returned SegmentationResult are the
    reference's; `context` (extension) selects the _lib.Context / GPU to run on.
    """
    t0 = time.time()
    if kmeansObj is not None:
        km = kmeansObj
    else:
        km = fitSpectralClusters(img, numClusters, clusterSubsamplePcnt, imgNullVal,
            fixedKMeansInit)
    if verbose:
        print("Kmeans, in", round(time.time() - t0, 1), "seconds")

    maxSpectralDiff = autoMaxSpectralDiff(km, maxSpectralDiff, spectDistPcntile)
    t0 = time.time()
    ctx = context if context is not None else _lib.default_context()
    dimg = _deviceImage(img)
    (nBands, nRows, nCols) = dimg.shape
    seg = numpy.empty((nRows, nCols), dtype=SegIdType)
    res = segmentTile(ctx, dimg, _centres(km), imgNullVal, fourConnected, minSegmentSize,
        spectralThreshold(maxSpectralDiff), seg)
    if verbose:
        print("Found", res.numClumps, "clumps")
        print("Eliminated", res.singlePixelsEliminated, "single pixels")
        print("Eliminated", res.smallSegmentsEliminated, "segments, in",
            round(time.time() - t0, 1), "seconds")
        print("Final result has", res.numSegments, "segments")

    segResult = SegmentationResult()
    segResult.segimg = seg
    segResult.kmeans = km
    segResult.maxSpectralDiff = maxSpectralDiff
    segResult.singlePixelsEliminated = SegIdType(res.singlePixelsEliminated)
    segResult.smallSegmentsEliminated = int(res.smallSegmentsEliminated)
    segResult.timings = {'assign': res.msAssign, 'clump': res.msClump, 'single': res.msSingle,
        'small': res.msSmall, 'total': res.msTotal, 'numSmallPasses': res.numSmallPasses,
        'numSinglePixelRounds': res.numSinglePixelRounds, 'numOversized': res.numOversized,
        'numClumps': res.numClumps}
    return segResult


def makeTileParams(dtype, nBands, nRows, nCols, centres, imgNullVal, fourConnected,
        minSegmentSize, thr):
    """Fill the ssg_tile_params struct; `centres` must stay alive while it is used."""
    prm = _lib.TileParams()
    prm.dtype = _lib.DTYPE_CODES[numpy.dtype(dtype)]
    prm.nBands = int(nBands)
    prm.nRows = int(nRows)
    prm.nCols = int(nCols)
    prm.centres = centres.ctypes.data
    prm.k = int(centres.shape[0])
    prm.hasNull = int(imgNullVal is not None)
    prm.nullVal = 0.0 if imgNullVal is None else float(imgNullVal)
    prm.fourConnected = int(bool(fourConnected))
    prm.minSegSize = int(minSegmentSize)
    prm.spectralThreshold = float(thr)
    return prm


def segmentTile(ctx, img, centres, imgNullVal, fourConnected, minSegmentSize, thr, segOut):
    """
    One call of ssg_segment_tile: host image in, host labels out (segOut None keeps the
    labels resident on the device for the stitch).  Returns the ssg_tile_result struct.
    """
    (nBands, nRows, nCols) = img.shape
    if centres.shape[1] != nBands:
        raise ValueError('cluster centres have %d bands, image has %d' % (centres.shape[1], nBands))
    prm = makeTileParams(img.dtype, nBands, nRows, nCols, centres, imgNullVal, fourConnected,
        minSegmentSize, thr)
    res = _lib.TileResult()
    ctx.call('ssg_segment_tile', _lib.ptr(img), ctypes.byref(prm),
        None if segOut is None else _lib.ptr(segOut), ctypes.byref(res))
    return res


# Where the k-means fit runs: 'sklearn' (scikit-learn on the host, exactly the reference's call)
# or 'gpu' (Lloyd iterations on the device, ssg_kmeans_lloyd: same algorithm, centres equal to
# scikit-learn's within a tolerance, orders of magnitude faster on a million samples).  The
# environment variable SSG_KMEANS overrides the module default.
KMEANS_BACKEND = 'sklearn'


def fitSpectralClusters(img, numClusters, subsamplePcnt, imgNullVal, fixedKMeansInit, backend=None,
        context=None):
    """
    First step of Shepherd segmentation (shepseg.py:252-314): k-means on a subsample of the
    non-null pixels.  Returns a fitted sklearn.cluster.KMeans object either way; `backend`
    ('sklearn' / 'gpu', default KMEANS_BACKEND or $SSG_KMEANS) says who runs the iterations.
    """
    import os
    from sklearn.cluster import KMeans
    img = numpy.asarray(img)
    nBands = img.shape[0]
    pixels = numpy.moveaxis(img, 0, -1).reshape(-1, nBands)
    if imgNullVal is not None:
        pixels = pixels[(pixels != imgNullVal).all(axis=1)]
    sample = pixels[::int(round(100. / subsamplePcnt))]
    if backend is None:
        backend = os.environ.get('SSG_KMEANS', KMEANS_BACKEND)
    if backend == 'gpu':
        return _fitOnDevice(sample, numClusters, fixedKMeansInit, context)
    if fixedKMeansInit:
        km = KMeans(n_clusters=numClusters, n_init=1,
            init=diagonalClusterCentres(sample, numClusters))
    else:
        km = KMeans(n_clusters=numClusters, n_init=5, init='k-means++')
    km.fit(sample)
    return km


def _lloydOnDevice(ctx, X, centres, maxIter, tol):
    """
    The loop of scikit-learn's _kmeans_single_lloyd around the two device steps: assignment
    (ssg_kmeans_step), relocation of empty clusters as scikit-learn does it (the n_empty samples
    farthest from their centres, picked with the same numpy.argpartition expression, each becomes
    the sole member of an empty cluster), update (ssg_kmeans_update); stop when the labels repeat
    or the summed squared centre shift is <= tol.  Returns (centres, inertia, iterations).
    """
    (n, k) = (X.shape[0], centres.shape[0])
    ctx.call('ssg_kmeans_begin', _lib.ptr(X), n, X.shape[1], _lib.ptr(centres), k)
    counts = numpy.zeros(k, dtype=numpy.uint64)
    inertia = ctypes.c_double(0.0)
    changed = ctypes.c_uint64(0)
    shift = ctypes.c_double(0.0)
    cur = numpy.array(centres)
    strict = False
    it = 0
    for it in range(1, maxIter + 1):
        ctx.call('ssg_kmeans_step', _lib.ptr(counts), ctypes.byref(inertia), ctypes.byref(changed))
        empty = numpy.flatnonzero(counts == 0)
        if len(empty) > 0:
            labels = numpy.empty(n, dtype=numpy.int32)
            ctx.call('ssg_kmeans_labels', _lib.ptr(labels))
            ctx.call('ssg_kmeans_centres', _lib.ptr(cur))       # the centres this step assigned to
            distances = ((X - cur[labels]) ** 2).sum(axis=1)
            far = numpy.argpartition(distances, -len(empty))[:-len(empty) - 1:-1].astype(numpy.int64)
            # (both arrays must outlive the call: a temporary would be freed before the copy reads it)
            emptyIds = numpy.ascontiguousarray(empty.astype(numpy.int32))
            ctx.call('ssg_kmeans_relocate', len(empty), _lib.ptr(numpy.ascontiguousarray(far)),
                _lib.ptr(emptyIds))
        ctx.call('ssg_kmeans_update', ctypes.byref(shift), None)
        if changed.value == 0:
            strict = True
            break
        if shift.value <= tol:
            break
    ctx.call('ssg_kmeans_centres', _lib.ptr(cur))
    if not strict:
        # (scikit-learn assigns once more so that the inertia belongs to the final centres)
        ctx.call('ssg_kmeans_step', None, ctypes.byref(inertia), ctypes.byref(changed))
    return (cur, float(inertia.value), it)


def _fitOnDevice(sample, numClusters, fixedKMeansInit, context=None, maxIter=300, tol=1e-4):
    """
    scikit-learn's KMeans.fit restated around ssg_kmeans_lloyd: the data are centred on their mean
    (as scikit-learn does, for the arithmetic), tol is scaled by the mean feature variance, the
    initial centres are the diagonal ones (fixedKMeansInit) or scikit-learn's own k-means++ draw,
    five of them, keeping the fit with the lowest inertia.  The result is a scikit-learn KMeans
    object carrying the fitted centres, so predict() and everything else work as usual.
    """
    from sklearn.cluster import KMeans, kmeans_plusplus
    ctx = context if context is not None else _lib.default_context()
    X = numpy.ascontiguousarray(sample, dtype=numpy.float64)
    if X.shape[0] < numClusters:
        raise ValueError('n_samples=%d should be >= n_clusters=%d' % (X.shape[0], numClusters))
    mean = X.mean(axis=0)
    Xc = X - mean
    absTol = float(numpy.mean(numpy.var(Xc, axis=0)) * tol)
    if fixedKMeansInit:
        inits = [numpy.asarray(diagonalClusterCentres(sample, numClusters), dtype=numpy.float64)]
    else:
        rs = numpy.random.RandomState()
        inits = [kmeans_plusplus(X, numClusters, random_state=rs)[0] for _ in range(5)]
    best = None
    for init in inits:
        centres = numpy.ascontiguousarray(init - mean, dtype=numpy.float64)
        (centres, inertia, nIter) = _lloydOnDevice(ctx, Xc, centres, int(maxIter), absTol)
        if best is None or inertia < best[1]:
            best = (centres + mean, inertia, nIter)
    (centres, inertia, nIter) = best
    # a fitted scikit-learn object around those centres (fit on the centres themselves: trivially
    # converged; then the attributes are set to what the device computed)
    km = KMeans(n_clusters=numClusters, n_init=1, init=centres, max_iter=1)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        km.fit(centres)
    km.cluster_centers_ = numpy.ascontiguousarray(centres, dtype=numpy.float64)
    km.inertia_ = float(inertia)
    km.n_iter_ = int(nIter)
    km.labels_ = None
    return km


def diagonalClusterCentres(xSample, numClusters):
    """
    Initial centres evenly spaced along the diagonal of the data's bounding box, end points
    one step in from the corners, in the sample's dtype (shepseg.py:364-397).
    """
    lo = xSample.min(axis=0)
    hi = xSample.max(axis=0)
    step = (hi - lo) / (numClusters + 1)
    centres = numpy.empty((numClusters, xSample.shape[1]), dtype=xSample.dtype)
    for i in range(numClusters):
        centres[i] = lo + (i + 1) * step
    return centres


_msdCache = {}


def autoMaxSpectralDiff(km, maxSpectralDiff, distPcntile):
    """
    Work out what to use as the maxSpectralDiff (shepseg.py:400-449): 'auto' is the
    distPcntile-th percentile of the distances between cluster centres, None is ten times
    the largest distance, anything else is passed through.  The distances are formed with
    the reference's own numpy expressions (float64 math stored as float32), so the value and
    its dtype are the reference's.  Cached per centre set: the tiled driver calls this once
    per tile.
    """
    isAuto = isinstance(maxSpectralDiff, str) and maxSpectralDiff == 'auto'
    if not isAuto and maxSpectralDiff is not None:
        return maxSpectralDiff
    centres = numpy.asarray(getattr(km, 'cluster_centers_', km))
    key = (centres.shape, centres.tobytes(), isAuto, distPcntile)
    if key in _msdCache:
        return _msdCache[key]
    numClusters = centres.shape[0]
    dists = numpy.full(numClusters * (numClusters - 1) // 2, -1, dtype=numpy.float32)
    n = 0
    for i in range(numClusters - 1):
        for j in range(i + 1, numClusters):
            dists[n] = numpy.sqrt(((centres[i] - centres[j])**2).sum())
            n += 1
    if isAuto:
        value = numpy.percentile(dists, distPcntile)
    else:
        value = 10 * dists.max()
    if len(_msdCache) > 64:
        _msdCache.clear()
    _msdCache[key] = value
    return value


# ---------------------------------------------------------------------------------------
# Stage functions, with the reference's signatures and in-place behaviour
# ---------------------------------------------------------------------------------------
def applySpectralClusters(kmeansObj, img, imgNullVal, context=None):
    """
    Nearest-centre cluster number (1-based) for every pixel, SEGNULLVAL where any band is
    imgNullVal (shepseg.py:317-361).  Returns an int32 (nRows, nCols) array.
    """
    ctx = context if context is not None else _lib.default_context()
    dimg = _deviceImage(img)
    (nBands, nRows, nCols) = dimg.shape
    centres = _centres(kmeansObj)
    if centres.shape[1] != nBands:
        raise ValueError('cluster centres have %d bands, image has %d' % (centres.shape[1], nBands))
    out = numpy.empty((nRows, nCols), dtype=numpy.int32)
    ctx.call('ssg_assign', _lib.ptr(dimg), _lib.DTYPE_CODES[dimg.dtype], nBands, nRows, nCols,
        _lib.ptr(centres), centres.shape[0], int(imgNullVal is not None),
        0.0 if imgNullVal is None else float(imgNullVal), _lib.ptr(out))
    return out


def clump(img, ignoreVal, fourConnected=True, clumpId=1, context=None):
    """
    Clump equal-valued connected pixels (shepseg.py:452-541).  Returns (clumpimg, nextId)
    with the reference's raster-scan numbering and MAX_CLUMP_SIZE splitting.
    """
    ctx = context if context is not None else _lib.default_context()
    img = numpy.ascontiguousarray(img, dtype=numpy.int32)
    (nRows, nCols) = img.shape
    out = numpy.empty((nRows, nCols), dtype=SegIdType)
    nextId = ctypes.c_uint32(0)
    ctx.call('ssg_clump', _lib.ptr(img), nRows, nCols, int(ignoreVal), int(bool(fourConnected)),
        int(clumpId), _lib.ptr(out), ctypes.byref(nextId))
    return (out, int(nextId.value))


def makeSegSize(seg, context=None):
    """Histogram of segment ids, max(seg)+1 entries of uint32 (shepseg.py:544-569)."""
    ctx = context if context is not None else _lib.default_context()
    seg = numpy.ascontiguousarray(seg, dtype=SegIdType)
    n = (int(seg.max()) + 1) if seg.size else 1
    segSize = numpy.zeros(n, dtype=numpy.uint32)
    ctx.call('ssg_make_seg_size', _lib.ptr(seg), seg.size, _lib.ptr(segSize), n)
    return segSize


def _inplaceSeg(seg):
    if not (isinstance(seg, numpy.ndarray) and seg.dtype == SegIdType and seg.flags.c_contiguous
            and seg.flags.writeable):
        raise ValueError('seg must be a writeable C-contiguous uint32 array (it is modified in place)')


def eliminateSinglePixels(img, seg, segSize, minSegId, maxSegId, fourConnected, context=None):
    """
    Merge single-pixel segments into their spectrally nearest neighbouring pixel's segment,
    repeatedly, then relabel (shepseg.py:572-615).  seg and segSize are modified in place.
    """
    ctx = context if context is not None else _lib.default_context()
    dimg = _deviceImage(img)
    (nBands, nRows, nCols) = dimg.shape
    _inplaceSeg(seg)
    if not (segSize.dtype == numpy.uint32 and segSize.flags.c_contiguous):
        raise ValueError('segSize must be a C-contiguous uint32 array')
    # the kernels index segSize by segment id without a bound check of their own
    if seg.size and int(seg.max()) >= len(segSize):
        raise ValueError('segSize has %d entries but seg holds id %d' % (len(segSize), int(seg.max())))
    moved = ctypes.c_int64(0)
    ctx.call('ssg_eliminate_single_pixels', _lib.ptr(dimg), _lib.DTYPE_CODES[dimg.dtype], nBands,
        nRows, nCols, _lib.ptr(seg), _lib.ptr(segSize), len(segSize), int(minSegId),
        int(bool(fourConnected)), ctypes.byref(moved))


def relabelSegments(seg, segSize, minSegId, context=None):
    """
    Recode seg in place so that segment ids are contiguous: ids from minSegId up that own no
    pixel (segSize == 0) are squeezed out, the order of the others is kept (shepseg.py:739-777).
    segSize is not updated, as in the reference.
    """
    ctx = context if context is not None else _lib.default_context()
    _inplaceSeg(seg)
    segSize = numpy.ascontiguousarray(segSize, dtype=numpy.uint32)
    if seg.size and int(seg.max()) >= len(segSize):
        raise ValueError('segSize has %d entries but seg holds id %d' % (len(segSize), int(seg.max())))
    ctx.call('ssg_relabel_segments', _lib.ptr(seg), seg.size, _lib.ptr(segSize), len(segSize), int(minSegId))


def eliminateSmallSegments(seg, img, maxSegId, minSegSize, maxSpectralDiff, fourConnected,
        minSegId, context=None):
    """
    Merge segments smaller than minSegSize into their spectrally most similar larger
    neighbour, smallest first (shepseg.py:918-1000).  seg is modified in place; returns the
    number of segments eliminated.
    """
    ctx = context if context is not None else _lib.default_context()
    dimg = _deviceImage(img)
    (nBands, nRows, nCols) = dimg.shape
    _inplaceSeg(seg)
    # the per-segment tables have maxSegId + 1 entries and are indexed by segment id
    if seg.size and int(seg.max()) > int(maxSegId):
        raise ValueError('seg holds id %d, above maxSegId=%d' % (int(seg.max()), int(maxSegId)))
    numElim = ctypes.c_int64(0)
    ctx.call('ssg_eliminate_small_segments', _lib.ptr(seg), _lib.ptr(dimg),
        _lib.DTYPE_CODES[dimg.dtype], nBands, nRows, nCols, int(maxSegId), int(minSegSize),
        spectralThreshold(maxSpectralDiff), int(bool(fourConnected)), int(minSegId),
        ctypes.byref(numElim))
    return int(numElim.value)

"""
Drop-in for pyshepseg.tilingstats.calcPerSegmentStatsTiled on a B200.

The reference walks the label raster and one image band tile by tile, keeps a dictionary of
value histograms per segment (accumulateSegDict, tilingstats.py:467-517), evaluates a
segment's statistics as soon as its histogram holds as many pixels as the Histogram column
says it has (checkSegComplete / calcStatsForCompletedSegs, 519-617; SegmentStats, 923-1008)
and writes the raster attribute table page by page (writeCompletePages, 723-767).  None of the
results depend on that order, so here the whole band and the whole label raster go to the
device once, the per-segment histograms come out of one sort of (segment, value) keys, and one
thread per segment evaluates the statistics with the reference's arithmetic
(ssg_segment_stats, csrc/stats.cu).  The columns are bit identical to the reference's.

Kept from the reference's surface: calcPerSegmentStatsTiled (same arguments, same errors, the
RAT columns it creates through GDAL when GDAL is there), TiledStatsResult, PyShepSegStatsError,
the statistic names and STATID_* numbers.  calcPerSegmentStats is the same computation on
arrays (host numpy arrays, or device pointers for labels that are still resident).  Without
GDAL the columns of a built-in format go to a `<segfile>.rat.npz` side file.

Not rebuilt (SURVEY.md section 8 f4): the RIOS variants and the spatial statistics.
"""
import json
import os

import numpy

from . import _lib
from . import rasterfile
from . import timinghooks

STATID_MIN = 0
STATID_MAX = 1
STATID_MEAN = 2
STATID_STDDEV = 3
STATID_MEDIAN = 4
STATID_MODE = 5
STATID_PERCENTILE = 6
STATID_PIXCOUNT = 7
statIDdict = {
    'min': STATID_MIN,
    'max': STATID_MAX,
    'mean': STATID_MEAN,
    'stddev': STATID_STDDEV,
    'median': STATID_MEDIAN,
    'mode': STATID_MODE,
    'percentile': STATID_PERCENTILE,
    'pixcount': STATID_PIXCOUNT
}
MAX_STATS = 32

_STATS_DTYPES = dict(_lib.DTYPE_CODES)


class PyShepSegStatsError(Exception):
    pass


class TiledStatsResult(object):
    """Result of the per-segment statistics (tilingstats.py:71-82).  `columns` (not in the
    reference) holds what was written: column name -> array over segment ids."""
    def __init__(self):
        self.timings = None
        self.columns = None


def _gdal():
    try:
        from osgeo import gdal
        return gdal
    except ImportError:
        return None


def checkStatsSelection(statsSelection):
    """(statIds, params) of a statsSelection list (makeFastStatsSelection, tilingstats.py:798-864)."""
    if len(statsSelection) < 1:
        raise PyShepSegStatsError('no statistics selected')
    ids = numpy.zeros(len(statsSelection), dtype=numpy.int32)
    params = numpy.zeros(len(statsSelection), dtype=numpy.int32)
    for (i, sel) in enumerate(statsSelection):
        statName = sel[1]
        if statName not in statIDdict:
            raise KeyError(statName)           # (the reference's statIDdict[statName])
        ids[i] = statIDdict[statName]
        if statName == 'percentile':
            params[i] = sel[2]                 # (IndexError for a 2-tuple, as in the reference)
    return (ids, params)


def calcPerSegmentStats(img, seg, statsSelection, missingStatsValue=-9999, imgNullVal=None,
        maxSegId=None, segSize=None, context=None, shape=None, dtype=None):
    """
    The statistics of one image band per segment, as columns over segment ids 0..maxSegId:
    {columnName: int64 array, or float32 array for 'mean' and 'stddev'}.

    img and seg are 2-d numpy arrays of the same shape (seg uint32), or device pointers
    (ints, with `shape` and the image `dtype` given) on the device of `context`.  maxSegId
    defaults to the largest label (host arrays) and must be given for device pointers.
    With segSize (the Histogram column) given, the reference's completeness rule is applied:
    PyShepSegStatsError unless every segment 1..maxSegId has exactly that many pixels.
    """
    (ids, params) = checkStatsSelection(statsSelection)
    if len(ids) > MAX_STATS:
        groups = [statsSelection[i:i + MAX_STATS] for i in range(0, len(ids), MAX_STATS)]
        out = {}
        for g in groups:
            out.update(calcPerSegmentStats(img, seg, g, missingStatsValue, imgNullVal, maxSegId,
                segSize, context, shape, dtype))
        return out
    onDevice = not isinstance(seg, numpy.ndarray)
    if onDevice:
        if isinstance(img, numpy.ndarray) or shape is None or dtype is None or maxSegId is None:
            raise ValueError('device pointers need shape, dtype and maxSegId (and both rasters on the device)')
        dtype = numpy.dtype(dtype)
        nPixels = int(shape[0]) * int(shape[1])
        (segPtr, imgPtr) = (int(seg), int(img))
    else:
        img = numpy.asarray(img)
        if img.shape != seg.shape or seg.ndim != 2:
            raise PyShepSegStatsError("Images must be same size")
        dtype = img.dtype
        if dtype.kind == 'f':
            raise PyShepSegStatsError("Float image types not supported")
        seg = numpy.ascontiguousarray(seg, dtype=numpy.uint32)
        img = numpy.ascontiguousarray(img)
        nPixels = seg.size
        if maxSegId is None:
            maxSegId = int(seg.max()) if seg.size else 0
        (segPtr, imgPtr) = (_lib.ptr(seg), _lib.ptr(img))
    if dtype not in _STATS_DTYPES:
        raise PyShepSegStatsError('image type %s not supported (8, 16 and 32 bit integers are)' % dtype)
    if segSize is not None:
        maxSegId = len(segSize) - 1
    maxSegId = int(maxSegId)
    ctx = context if context is not None else _lib.default_context(0)
    nInt = int(numpy.count_nonzero((ids != STATID_MEAN) & (ids != STATID_STDDEV)))
    nFloat = len(ids) - nInt
    intOut = numpy.zeros((max(nInt, 1), maxSegId + 1), dtype=numpy.int64)
    floatOut = numpy.zeros((max(nFloat, 1), maxSegId + 1), dtype=numpy.float32)
    total = numpy.zeros(maxSegId + 1, dtype=numpy.uint32)
    hasNull = imgNullVal is not None
    ctx.call('ssg_segment_stats', segPtr, imgPtr, _STATS_DTYPES[dtype], nPixels, int(onDevice),
        int(hasNull), int(imgNullVal) if hasNull else 0, maxSegId, len(ids), _lib.ptr(ids),
        _lib.ptr(params), int(missingStatsValue), _lib.ptr(intOut), _lib.ptr(floatOut), _lib.ptr(total))
    if segSize is not None:
        # a segment is evaluated when its pixels found == its Histogram entry, a page written
        # when all its segments are; anything left over is the reference's error (207-209)
        want = numpy.asarray(segSize).astype(numpy.uint32)
        if (total[1:] != want[1:]).any() or (total[1:] == 0).any():
            raise PyShepSegStatsError('Not all pixels found during processing')
    out = {}
    (i, f) = (0, 0)
    for (sel, statId) in zip(statsSelection, ids):
        if statId in (STATID_MEAN, STATID_STDDEV):
            out[sel[0]] = floatOut[f]
            f += 1
        else:
            out[sel[0]] = intOut[i]
            i += 1
    return out


# ---------------------------------------------------------------------------------------
# File level
# ---------------------------------------------------------------------------------------
def equalProjection(proj1, proj2):
    """Same projection? (tilingstats.py:1011-1035; osr decides when the strings differ)"""
    if proj1 == proj2:
        return True
    try:
        from osgeo import osr
    except ImportError:
        return False
    (sr1, sr2) = (osr.SpatialReference(), osr.SpatialReference())
    (ok1, ok2) = (sr1.ImportFromWkt(proj1) == 0, sr2.ImportFromWkt(proj2) == 0) if hasattr(
        sr1, 'ImportFromWkt') else (True, True)
    if not (ok1 and ok2):
        return proj1 == proj2
    return bool(sr1.IsSame(sr2))


def doImageAlignmentChecks(segfile, imgfile, imgbandnum, update=True):
    """Open both files through GDAL and refuse misaligned or float rasters
    (tilingstats.py:409-463).  Returns (segds, segband, imgds, imgband)."""
    gdal = _gdal()
    segds = segfile
    if not isinstance(segds, gdal.Dataset):
        segds = gdal.Open(segfile, gdal.GA_Update if update else gdal.GA_ReadOnly)
    segband = segds.GetRasterBand(1)
    imgds = imgfile
    if not isinstance(imgds, gdal.Dataset):
        imgds = gdal.Open(imgfile, gdal.GA_ReadOnly)
    imgband = imgds.GetRasterBand(imgbandnum)
    if imgband.DataType in (gdal.GDT_Float32, gdal.GDT_Float64):
        raise PyShepSegStatsError("Float image types not supported")
    if segband.XSize != imgband.XSize or segband.YSize != imgband.YSize:
        raise PyShepSegStatsError("Images must be same size")
    if segds.GetGeoTransform() != imgds.GetGeoTransform():
        raise PyShepSegStatsError("Images must have same spatial extent and pixel size")
    if not equalProjection(segds.GetProjection(), imgds.GetProjection()):
        raise PyShepSegStatsError("Images must be in the same projection")
    return (segds, segband, imgds, imgband)


def checkHistColumn(existingColNames):
    """Index of the Histogram column, which must exist (tilingstats.py:656-679)."""
    histColNdx = -1
    for (i, name) in enumerate(existingColNames):
        if name == 'Histogram':
            histColNdx = i
    if histColNdx < 0:
        raise PyShepSegStatsError("Histogram column must exist before calculating per-segment stats")
    return histColNdx


def createStatColumns(statsSelection, attrTbl, existingColNames):
    """Create the requested RAT columns: Real for mean and stddev, Integer otherwise
    (tilingstats.py:682-720).  Returns their column indexes in the order of statsSelection."""
    gdal = _gdal()
    colIndexList = []
    for selection in statsSelection:
        (colName, statName) = selection[:2]
        if colName not in existingColNames:
            colType = gdal.GFT_Real if statName in ('mean', 'stddev') else gdal.GFT_Integer
            attrTbl.CreateColumn(colName, colType, gdal.GFU_Generic)
            colNdx = attrTbl.GetColumnCount() - 1
        else:
            print('Column {} already exists'.format(colName))
            colNdx = existingColNames.index(colName)
        colIndexList.append(colNdx)
    return colIndexList


def _readBand(band, dtype, timings):
    """The whole band into one host array, read in row strips."""
    (ysize, xsize) = (band.YSize, band.XSize)
    out = numpy.empty((ysize, xsize), dtype=dtype)
    strip = max(1, (64 << 20) // max(1, xsize * out.itemsize))
    with timings.interval('reading'):
        for y in range(0, ysize, strip):
            n = min(strip, ysize - y)
            out[y:y + n] = band.ReadAsArray(0, y, xsize, n)
    return out


def _statsThroughGdal(imgfile, imgbandnum, segfile, statsSelection, missingStatsValue, context):
    timings = timinghooks.Timers()
    (segds, segband, imgds, imgband) = doImageAlignmentChecks(segfile, imgfile, imgbandnum)
    attrTbl = segband.GetDefaultRAT()
    existingColNames = [attrTbl.GetNameOfCol(i) for i in range(attrTbl.GetColumnCount())]
    imgNullVal = imgband.GetNoDataValue()
    if imgNullVal is not None:
        imgNullVal = int(imgNullVal)           # (the reference casts to int64, tilingstats.py:160)
    histColNdx = checkHistColumn(existingColNames)
    segSize = numpy.asarray(attrTbl.ReadAsArray(histColNdx)).astype(numpy.uint32)
    checkStatsSelection(statsSelection)
    colIndexList = createStatColumns(statsSelection, attrTbl, existingColNames)
    seg = _readBand(segband, numpy.uint32, timings)
    first = imgband.ReadAsArray(0, 0, 1, 1)
    img = _readBand(imgband, first.dtype, timings)
    with timings.interval('accumulation'):
        cols = calcPerSegmentStats(img, seg, statsSelection, missingStatsValue, imgNullVal,
            segSize=segSize, context=context)
    with timings.interval('writing'):
        for (sel, colNdx) in zip(statsSelection, colIndexList):
            attrTbl.WriteArray(cols[sel[0]], colNdx)
        segds.FlushCache()
    del segds
    rtn = TiledStatsResult()
    rtn.timings = timings
    rtn.columns = cols
    return rtn


def ratPath(segfile):
    return segfile + '.rat.npz'


def readRat(segfile):
    """The columns written so far for a built-in format label raster."""
    if not os.path.exists(ratPath(segfile)):
        return {}
    with numpy.load(ratPath(segfile)) as z:
        return dict((k, z[k]) for k in z.files)


def _statsBuiltin(imgfile, imgbandnum, segfile, statsSelection, missingStatsValue, context):
    """Label rasters written by the built-in sinks (rasterfile.NpySink / TiffSink): the
    Histogram column is the `.hist.npy` side file, the new columns go to `.rat.npz`."""
    timings = timinghooks.Timers()
    segsrc = rasterfile.openRaster(segfile)
    imgsrc = rasterfile.openRaster(imgfile)
    if imgsrc.dtype.kind == 'f':
        raise PyShepSegStatsError("Float image types not supported")
    if (segsrc.xsize, segsrc.ysize) != (imgsrc.xsize, imgsrc.ysize):
        raise PyShepSegStatsError("Images must be same size")
    if tuple(segsrc.geotransform) != tuple(imgsrc.geotransform):
        raise PyShepSegStatsError("Images must have same spatial extent and pixel size")
    histfile = segfile + '.hist.npy'
    if not os.path.exists(histfile):
        raise PyShepSegStatsError("Histogram column must exist before calculating per-segment stats")
    segSize = numpy.load(histfile).astype(numpy.uint32)
    checkStatsSelection(statsSelection)
    with timings.interval('reading'):
        seg = numpy.ascontiguousarray(segsrc.readWindow([1], 0, 0, segsrc.xsize, segsrc.ysize)[0],
            dtype=numpy.uint32)
        img = numpy.ascontiguousarray(imgsrc.readWindow([imgbandnum], 0, 0, imgsrc.xsize, imgsrc.ysize)[0])
    imgNullVal = imgsrc.nodata[imgbandnum - 1]
    if imgNullVal is not None:
        imgNullVal = int(imgNullVal)
    with timings.interval('accumulation'):
        cols = calcPerSegmentStats(img, seg, statsSelection, missingStatsValue, imgNullVal,
            segSize=segSize, context=context)
    with timings.interval('writing'):
        rat = readRat(segfile)
        for sel in statsSelection:
            if sel[0] in rat:
                print('Column {} already exists'.format(sel[0]))
            rat[sel[0]] = cols[sel[0]]
        numpy.savez(ratPath(segfile), **rat)
        meta = {}
        if os.path.exists(segfile + '.json'):
            meta = json.load(open(segfile + '.json'))
        meta['rat'] = os.path.basename(ratPath(segfile))
        json.dump(meta, open(segfile + '.json', 'w'), indent=1)
    rtn = TiledStatsResult()
    rtn.timings = timings
    rtn.columns = cols
    return rtn


def calcPerSegmentStatsTiled(imgfile, imgbandnum, segfile, statsSelection, missingStatsValue=-9999,
        context=None):
    """
    Calculate the selected per-segment statistics of band imgbandnum (1-based) of imgfile
    over the segments of segfile and write them as columns of segfile's raster attribute
    table (tilingstats.py:85-215).  statsSelection is a list of (columnName, statName) or
    (columnName, 'percentile', p) with statName one of 'min', 'max', 'mean', 'stddev',
    'median', 'mode', 'percentile', 'pixcount'.  Pixels equal to imgfile's nodata value are
    ignored; a segment with no other pixels gets missingStatsValue.
    """
    gdal = _gdal()
    if gdal is not None:
        builtin = isinstance(segfile, str) and segfile.endswith('.npy')
        if not builtin:
            return _statsThroughGdal(imgfile, imgbandnum, segfile, statsSelection, missingStatsValue, context)
    if not isinstance(segfile, str):
        raise PyShepSegStatsError('an open dataset needs GDAL')
    return _statsBuiltin(imgfile, imgbandnum, segfile, statsSelection, missingStatsValue, context)

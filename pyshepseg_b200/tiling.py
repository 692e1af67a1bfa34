"""
Drop-in for pyshepseg.tiling.doTiledShepherdSegmentation on B200 GPUs.

The raster is cut into the same overlapping tiles as the reference (getTilesForFile,
tiling.py:376-443), every tile is segmented on a GPU with the same cluster centres
(shepseg.doShepherdSegmentation, called at tiling.py:1446/1586) and the tiles are stitched
with the reference's rules (stitchTiles / recodeTile / recodeSharedSegments /
relabelSegments / crossesMidline, tiling.py:950-1306).  Segment labels never leave the
device between segmentation and stitching: per-segment tables and the overlap votes are
computed by kernels (ssg_tile_tables_device), the few thousand numbers per tile that the
reference's sequential id bookkeeping needs come to the host (resolveTile below), and the
final ids are applied on the device straight into the trimmed output window
(ssg_apply_lut_device).

What is kept from the reference's surface: the function signature, TiledSegmentationResult,
SegmentationConcurrencyConfig (CONC_NONE and CONC_THREADS; a worker is a CUDA context on one
of `devices`), TileInfo / getTilesForFile, PyShepSegTilingError, the timer names.  What is
not rebuilt: the Fargate / subprocess managers and the TCP data channel (cloud
orchestration, SURVEY.md section 2 rows 3 and 12).
"""
import atexit
import copy
import ctypes
import os
import queue
import sys
import threading
import time

import numpy

from . import _lib
from . import rasterfile
from . import shepseg
from . import timinghooks

DFLT_TILESIZE = 4096
DFLT_OVERLAPSIZE = 1024
DFLT_TEMPFILES_DRIVER = 'KEA'
DFLT_TEMPFILES_EXT = 'kea'

# the reference reads the k-means subsample in blocks of this size (tiling.py:94, 288)
TILESIZE = 1024

CONC_NONE = "CONC_NONE"
CONC_THREADS = "CONC_THREADS"
CONC_FARGATE = "CONC_FARGATE"
CONC_SUBPROC = "CONC_SUBPROC"

HORIZONTAL = 0
VERTICAL = 1


class PyShepSegTilingError(Exception):
    pass


class TiledSegmentationResult(object):
    """Result of tiled segmentation (tiling.py:112-151)."""
    def __init__(self):
        self.maxSegId = None
        self.numTileRows = None
        self.numTileCols = None
        self.subsamplePcnt = None
        self.maxSpectralDiff = None
        self.kmeans = None
        self.hasEmptySegments = None
        self.outDs = None
        self.timings = None


class SegmentationConcurrencyConfig(object):
    """
    Concurrency configuration (tiling.py:590-634).  concurrencyType CONC_NONE runs the tiles
    one after the other on one GPU, devices[0]; CONC_THREADS runs `numWorkers` segmentation
    workers, each a CUDA context of its own, dealt round-robin over `devices` (extension; default:
    GPU 0).  With two or more distinct ids in `devices`, CONC_THREADS segments one mosaic on all
    of them from this process (MultiDeviceSegmenter): the tiles are shared out by
    distributed.partitionTiles, every device segments and stitches its own tiles, and the result
    goes to the one output raster, equal bit for bit to the same call on devices[0] alone.  A
    device that gets no worker segments its tiles in its stitch thread.  Repeated ids name one
    device ([0, 0] is GPU 0).  barrierTimeout bounds every wait of one device for the others.

    shardDevices (attribute, for tests and measurements only; None by default): the device of
    every shard of a MultiDeviceSegmenter, one shard per entry and repeats allowed, in place of
    the distinct ids of `devices`.  It lets the tests run several shards on one GPU.
    """
    def __init__(self, concurrencyType=CONC_NONE, numWorkers=0, maxConcurrentReads=20,
            tileCompletionTimeout=60, barrierTimeout=300, fargateCfg=None, devices=None):
        self.concurrencyType = concurrencyType
        self.numWorkers = numWorkers
        self.maxConcurrentReads = maxConcurrentReads
        self.tileCompletionTimeout = tileCompletionTimeout
        self.barrierTimeout = barrierTimeout
        self.fargateCfg = fargateCfg
        self.devices = [0] if devices is None else list(devices)
        self.shardDevices = None
        if concurrencyType == CONC_FARGATE and fargateCfg is None:
            raise PyShepSegTilingError("fargateCfg is required with CONC_FARGATE")
        if concurrencyType != CONC_FARGATE and fargateCfg is not None:
            raise PyShepSegTilingError("fargateCfg is only used with CONC_FARGATE")


class TileInfo(object):
    """Pixel coordinates of the tiles within an image (tiling.py:317-373)."""
    def __init__(self):
        self.tiles = {}
        self.ncols = None
        self.nrows = None

    def addTile(self, xpos, ypos, xsize, ysize, col, row):
        self.tiles[(col, row)] = (xpos, ypos, xsize, ysize)

    def getNumTiles(self):
        return len(self.tiles)

    def getTile(self, col, row):
        return self.tiles[(col, row)]


def _axisSpans(rasterSize, tileSize, overlapSize):
    """(pos, size) of the tiles along one axis: step tileSize-overlapSize, and the last tile
    grows to the edge as soon as a further whole tile would not fit (tiling.py:414-438)."""
    spans = []
    pos = 0
    while True:
        size = tileSize
        last = (pos + 2 * size) > rasterSize
        if last:
            size = rasterSize - pos
        if size > 0:
            spans.append((pos, size))
        if last:
            return spans
        pos += tileSize - overlapSize


def getTilesForFile(ds, tileSize, overlapSize):
    """
    TileInfo for a raster (tiling.py:376-443).  `ds` is anything with the raster size:
    a rasterfile.RasterSource, a GDAL dataset or an (xsize, ysize) tuple.
    """
    if isinstance(ds, tuple):
        (xs, ys) = ds
    elif hasattr(ds, 'RasterXSize'):
        (xs, ys) = (ds.RasterXSize, ds.RasterYSize)
    else:
        (xs, ys) = (ds.xsize, ds.ysize)
    tileInfo = TileInfo()
    cols = _axisSpans(int(xs), int(tileSize), int(overlapSize))
    rows = _axisSpans(int(ys), int(tileSize), int(overlapSize))
    for (r, (ypos, ysize)) in enumerate(rows):
        for (c, (xpos, xsize)) in enumerate(cols):
            tileInfo.addTile(xpos, ypos, xsize, ysize, c, r)
    tileInfo.ncols = len(cols)
    tileInfo.nrows = len(rows)
    return tileInfo


def getImgNullValue(src, bandNumbers):
    """The raster's null value; all bands must agree (tiling.py:229-256)."""
    vals = [src.nodata[b - 1] for b in bandNumbers]
    if any(v != vals[0] for v in vals):
        raise PyShepSegTilingError("Different null values in some bands")
    return vals[0]


def readSubsampledImage(src, bandNumbers, subsampleProp):
    """
    The pixel subsample used for the whole-file k-means fit: every skip-th row and column
    inside each 1024 x 1024 block, blocks restarting the stride (tiling.py:259-314).
    """
    skip = int(round(1. / subsampleProp))

    def picks(n):
        return numpy.concatenate([numpy.arange(p, min(p + TILESIZE, n), skip)
            for p in range(0, n, TILESIZE)])
    rows = picks(src.ysize)
    cols = picks(src.xsize)
    out = numpy.empty((len(bandNumbers), len(rows), len(cols)), dtype=src.dtype)
    for (i, r) in enumerate(rows):
        line = src.readWindow(bandNumbers, 0, int(r), src.xsize, 1)
        out[:, i, :] = line[:, 0, :][:, cols]
    return out


def fitSpectralClustersWholeFile(src, bandNumbers, numClusters=60, subsamplePcnt=None,
        imgNullVal=None, fixedKMeansInit=False):
    """
    Fit the spectral clusters on a subsample of the whole raster (tiling.py:154-226).
    Returns (kmeansObj, subsamplePcnt, imgNullVal).
    """
    if subsamplePcnt is None:
        prop = min(1, numpy.sqrt(1000000 / (src.xsize * src.ysize)))
        subsamplePcnt = 100 * prop**2
    else:
        prop = numpy.sqrt(subsamplePcnt / 100.0)
    if imgNullVal is None:
        imgNullVal = getImgNullValue(src, bandNumbers)
    img = readSubsampledImage(src, bandNumbers, prop)
    km = shepseg.fitSpectralClusters(img, numClusters, 100, imgNullVal, fixedKMeansInit)
    return (km, subsamplePcnt, imgNullVal)


# ---------------------------------------------------------------------------------------
# stitching: the sequential part (host) around the two device phases
# ---------------------------------------------------------------------------------------
def tileMargins(tileInfo, col, row, xsize, ysize, overlapSize):
    """Trimmed window [top,bottom) x [left,right) of a tile (tiling.py:997-1022)."""
    margin = int(overlapSize / 2)
    top = 0 if row == 0 else margin
    left = 0 if col == 0 else margin
    bottom = ysize if row == tileInfo.nrows - 1 else ysize - margin
    right = xsize if col == tileInfo.ncols - 1 else xsize - margin
    return (top, bottom, left, right)


def overviewBlockOwned(tileInfo, col, row, overlapSize, lvl, xoff=0, yoff=0):
    """
    (rows, cols) of the level-lvl overview block of tile (col, row)'s trimmed window that no later
    window writes again.  The reference writes every window's block, window[lvl//2::lvl,
    lvl//2::lvl] at (xOff // lvl, yOff // lvl), in row-major order (tiling.py:1360-1383); where a
    window edge is not a multiple of lvl the block overlaps the next window's and the later one
    wins.  A window that writes only this part gives the same overview whatever order the
    windows arrive in (the shards of a MultiDeviceSegmenter write theirs concurrently).  Column
    spans depend on the tile column only and row spans on the tile row only, so the later windows
    that overlap a block are the next one in the row and the ones of the next row.
    """
    def origin(c, r):
        (x, y, xs, ys) = tileInfo.tiles[(c, r)]
        (top, bottom, left, right) = tileMargins(tileInfo, c, r, xs, ys, overlapSize)
        return (x + left - xoff, y + top - yoff, bottom - top, right - left)
    (x0, y0, wr, wc) = origin(col, row)
    rows = len(range(lvl // 2, wr, lvl))
    cols = len(range(lvl // 2, wc, lvl))
    if row + 1 < tileInfo.nrows:
        rows = max(0, min(rows, origin(col, row + 1)[1] // lvl - y0 // lvl))
    if col + 1 < tileInfo.ncols:
        cols = max(0, min(cols, origin(col + 1, row)[0] // lvl - x0 // lvl))
    return (rows, cols)


def _modeByKey(keys, values, counts):
    """
    For every distinct key: the value with the largest summed count, smallest value on ties
    (scipy.stats.mode over the expanded list, tiling.py:1194).  Returns (keys, modes).
    keys < 2**31 and values < 2**32 (segment ids), so (key, value) packs into one sortable word.
    """
    packed = (keys.astype(numpy.uint64) << numpy.uint64(32)) | values.astype(numpy.uint64)
    order = numpy.argsort(packed, kind='stable')
    p = packed[order]
    c = counts[order].astype(numpy.int64)
    newGroup = numpy.ones(len(p), dtype=bool)
    newGroup[1:] = p[1:] != p[:-1]
    starts = numpy.flatnonzero(newGroup)
    gp = p[starts]                                  # one entry per (key, value), ascending
    gc = numpy.add.reduceat(c, starts)
    gk = (gp >> numpy.uint64(32)).astype(numpy.int64)
    newKey = numpy.ones(len(gk), dtype=bool)
    newKey[1:] = gk[1:] != gk[:-1]
    keyStarts = numpy.flatnonzero(newKey)
    best = numpy.maximum.reduceat(gc, keyStarts)    # the largest count of every key ...
    keyOfGroup = numpy.cumsum(newKey) - 1
    isBest = numpy.flatnonzero(gc == best[keyOfGroup])
    # ... and the first group that reaches it (groups of a key are in ascending value order)
    firstOfKey = numpy.ones(len(isBest), dtype=bool)
    firstOfKey[1:] = keyOfGroup[isBest][1:] != keyOfGroup[isBest][:-1]
    sel = isBest[firstOfKey]
    return (gk[sel], (gp[sel] & numpy.uint64(0xFFFFFFFF)).astype(numpy.int64))


def resolveTile(tables, rank, flags, pairKeys, pairCounts, offset, lutTop, lutLeft,
        simpleTileRecode=False):
    """
    The sequential step of the stitch for one tile (tiling.py:1024-1030, 1104-1126,
    1247-1267): given the tile's local tables, the running id offset (maxSegId so far) and
    the final-id tables of the upper / left neighbours, return (lut, trimmedMax).
    """
    n = int(tables.maxId) + 1
    if simpleTileRecode:
        lut = numpy.zeros(n, dtype=numpy.uint32)
        lut[1:] = numpy.arange(1, n, dtype=numpy.uint64) + offset
    else:
        # (whole-array arithmetic instead of boolean fancy indexing: this runs on the critical
        # path of the last tile, on a few hundred thousand segments)
        isNumbered = ((flags & _lib.SEG_NUMBERED) != 0).astype(numpy.uint32)
        lut = (rank.astype(numpy.uint32, copy=False) + numpy.uint32(offset)) * isNumbered
        if len(pairKeys) > 0:
            isLeft = (pairKeys >> numpy.uint64(63)) != 0
            segs = ((pairKeys >> numpy.uint64(32)) & numpy.uint64(0x7FFFFFFF)).astype(numpy.int64)
            nbr = (pairKeys & numpy.uint64(0xFFFFFFFF)).astype(numpy.int64)
            # top first, then left: the left vote overrides (tiling.py:1107-1121)
            for (sel, nbrLut) in ((~isLeft, lutTop), (isLeft, lutLeft)):
                if nbrLut is None or not sel.any():
                    continue
                (k, mode) = _modeByKey(segs[sel], nbrLut[nbr[sel]].astype(numpy.int64), pairCounts[sel])
                lut[k] = mode.astype(numpy.uint32)
    inTrim = ((flags & _lib.SEG_INTRIM) != 0).astype(numpy.uint32)
    trimmedMax = int((lut * inTrim).max()) if n > 0 else 0
    return (lut, trimmedMax)


class _DevicePool(object):
    """Reuses device buffers: cudaMalloc / cudaFree synchronise the whole device.  Shared by
    the worker threads of one device; every call goes through the caller's own context."""
    def __init__(self):
        self.free = []
        self.lock = threading.Lock()

    def get(self, ctx, nbytes):
        with self.lock:
            best = None
            for (i, (cap, p)) in enumerate(self.free):
                if cap >= nbytes and (best is None or cap < self.free[best][0]):
                    best = i
            if best is not None:
                return self.free.pop(best)
        return (nbytes, ctx.dev_alloc(nbytes))

    def put(self, buf):
        with self.lock:
            self.free.append(buf)

    def close(self, ctx):
        with self.lock:
            for (cap, p) in self.free:
                ctx.dev_free(p)
            self.free = []


class _Slot(object):
    """A context with its staging memory, kept alive between calls: creating contexts and
    pinned / device buffers costs far more than segmenting a tile."""
    def __init__(self, device, highPriority=False):
        self.ctx = _lib.Context(device, highPriority)
        self.pinned = None       # PinnedArray staging of one tile image
        self.devStage = None     # (cap, ptr): tile image gathered from a DeviceRaster
        self.window = None       # PinnedArray staging of one trimmed output window
        self.winDev = None       # (cap, ptr)
        self.ovBuf = None        # PinnedArray: the overview levels of one window, packed
        self.lock = threading.Lock()

    def overviewsFor(self, nItems):
        if self.ovBuf is None or self.ovBuf.array.size < nItems:
            if self.ovBuf is not None:
                self.ovBuf.free()
            self.ovBuf = _lib.PinnedArray((max(nItems, 1),), numpy.uint32)
        return self.ovBuf.array

    def pinnedFor(self, nItems, dtype):
        nbytes = nItems * numpy.dtype(dtype).itemsize
        if self.pinned is None or self.pinned.array.nbytes < nbytes:
            if self.pinned is not None:
                self.pinned.free()
            self.pinned = _lib.PinnedArray((nbytes,), numpy.uint8)
        return self.pinned.array[:nbytes].view(dtype)

    def devStageFor(self, nbytes):
        if self.devStage is None or self.devStage[0] < nbytes:
            if self.devStage is not None:
                self.ctx.dev_free(self.devStage[1])
            self.devStage = (nbytes, self.ctx.dev_alloc(nbytes))
        return self.devStage[1]

    def windowFor(self, nItems):
        if self.window is None or self.window.array.size < nItems:
            if self.window is not None:
                self.window.free()
            self.window = _lib.PinnedArray((nItems,), numpy.uint32)
        if self.winDev is None or self.winDev[0] < nItems * 4:
            if self.winDev is not None:
                self.ctx.dev_free(self.winDev[1])
            self.winDev = (nItems * 4, self.ctx.dev_alloc(nItems * 4))
        return (self.window.array, self.winDev[1])

    def close(self):
        if self.pinned is not None:
            self.pinned.free()
        if self.window is not None:
            self.window.free()
        if self.ovBuf is not None:
            self.ovBuf.free()
        if self.devStage is not None:
            self.ctx.dev_free(self.devStage[1])
        if self.winDev is not None:
            self.ctx.dev_free(self.winDev[1])
        self.ctx.close()


class _GpuState(object):
    """Everything kept per device between calls: slot 0 is the stitch / sequential context,
    slots 1.. are the segmentation workers; one pool of per-tile label buffers; the histogram."""
    def __init__(self, device):
        self.device = device
        self.slots = []
        self.pool = _DevicePool()
        self.lock = threading.Lock()
        self.hist = _DeviceHistogram()
        self.rasterBuf = None      # (cap, ptr): device copy of a host raster being segmented

    def slot(self, i):
        with self.lock:
            while len(self.slots) <= i:
                # slot 0 stitches: short kernels that must not queue behind the workers' long ones
                self.slots.append(_Slot(self.device, highPriority=(len(self.slots) == 0)))
            return self.slots[i]

    def close(self):
        if self.slots:
            if self.rasterBuf is not None:
                self.slots[0].ctx.dev_free(self.rasterBuf[1])
                self.rasterBuf = None
            self.hist.close(self.slots[0].ctx)
            self.pool.close(self.slots[0].ctx)
        for sl in self.slots:
            sl.close()
        self.slots = []


_gpuStates = {}
_gpuStatesLock = threading.Lock()


def gpuState(device, shard=0):
    """The state of one device; shard > 0: a further, separate state on the same device (several
    shards of a MultiDeviceSegmenter on one GPU each hold their stitch slot for a whole run)."""
    key = device if shard == 0 else (device, shard)
    with _gpuStatesLock:
        if key not in _gpuStates:
            _gpuStates[key] = _GpuState(device)
        return _gpuStates[key]


def releaseGpuState():
    """Free the contexts, pinned staging and device buffers kept between calls."""
    with _gpuStatesLock:
        for st in _gpuStates.values():
            st.close()
        _gpuStates.clear()


atexit.register(releaseGpuState)


class _RasterUploader(object):
    """
    A host raster that can be addressed in place goes to the GPU ONCE instead of tile by tile:
    overlapping tiles share 20-60 % of their pixels, and PCIe is the slowest link of the
    host-to-host path.  The raster is cut along every tile edge into cells; the cells go up in the
    order in which the tiles need them (a stream of its own), and a tile is gathered out of the
    device copy (device-to-device) as soon as its cells have landed.  The device copy holds the
    bounding box of the given tiles only (a shard of a MultiDeviceSegmenter copies its own).
    """
    def __init__(self, slot, hostBase, bandNumbers, ysize, xsize, item, devPtr, tiles, yoff, xoff=0):
        self.slot = slot
        self.hostBase = hostBase
        self.planes = [b - 1 for b in bandNumbers]      # planes of the host raster, in order
        (self.ysize, self.xsize, self.item) = (ysize, xsize, item)
        # tiles: [(key, xpos - xoff, ypos - yoff, xsize, ysize)] in the order they will be segmented
        self.tiles = [(k, x - xoff, y - yoff, xs, ys) for (k, x, y, xs, ys) in tiles]
        (self.boxX0, self.boxY0, self.boxH, self.boxW) = self.box(self.tiles)
        self.devPtr = devPtr                             # (len(bandNumbers), boxH, boxW)
        xs = sorted(set([0, xsize] + [t[1] for t in self.tiles] + [t[1] + t[3] for t in self.tiles]))
        ys = sorted(set([0, ysize] + [t[2] for t in self.tiles] + [t[2] + t[4] for t in self.tiles]))
        (self.xEdges, self.yEdges) = (xs, ys)
        self.ready = set()
        self.cond = threading.Condition()
        self.error = None
        self.bytes = 0
        self.thread = threading.Thread(target=self._run, daemon=True)

    @staticmethod
    def box(tiles):
        """(x0, y0, rows, cols) of the bounding box of [(key, x, y, xsize, ysize)]"""
        if not tiles:
            return (0, 0, 0, 0)
        (x0, y0) = (min(t[1] for t in tiles), min(t[2] for t in tiles))
        return (x0, y0, max(t[2] + t[4] for t in tiles) - y0, max(t[1] + t[3] for t in tiles) - x0)

    def devAddress(self, plane, y, x):
        """device address of pixel (y, x) of the host raster's window (plane: index in bandNumbers)"""
        return self.devPtr + ((plane * self.boxH + y - self.boxY0) * self.boxW + x - self.boxX0) * self.item

    def start(self):
        self.thread.start()

    def _cellsOf(self, t):
        (k, x, y, xs, ys) = t
        for (y0, y1) in zip(self.yEdges[:-1], self.yEdges[1:]):
            if y0 >= y + ys or y1 <= y:
                continue
            for (x0, x1) in zip(self.xEdges[:-1], self.xEdges[1:]):
                if x0 >= x + xs or x1 <= x:
                    continue
                yield (x0, y0, x1, y1)

    def _run(self):
        try:
            ctx = self.slot.ctx
            done = set()
            pitch = self.xsize * self.item
            with self.slot.lock:
                for t in self.tiles:
                    n = 0
                    for cell in self._cellsOf(t):
                        if cell in done:
                            continue
                        done.add(cell)
                        (x0, y0, x1, y1) = cell
                        for (i, pl) in enumerate(self.planes):
                            ctx.call('ssg_memcpy2d_h2d', self.devAddress(i, y0, x0), self.boxW * self.item,
                                self.hostBase + (pl * self.ysize + y0) * pitch + x0 * self.item, pitch,
                                (x1 - x0) * self.item, y1 - y0)
                        n += (x1 - x0) * (y1 - y0) * self.item * len(self.planes)
                    if n:
                        ctx.synchronize()
                    with self.cond:
                        self.ready.add(t[0])
                        self.bytes += n
                        self.cond.notify_all()
        except Exception as e:
            with self.cond:
                self.error = e
                self.cond.notify_all()

    def waitTile(self, key, timeout):
        with self.cond:
            ok = self.cond.wait_for(lambda: key in self.ready or self.error is not None, timeout)
            if self.error is not None:
                raise self.error
            if not ok:
                raise PyShepSegTilingError('timeout waiting for the raster upload')

    def join(self):
        self.thread.join()


class _Tile(object):
    def __init__(self, col, row, geom):
        (self.col, self.row) = (col, row)
        (self.xpos, self.ypos, self.xsize, self.ysize) = geom
        self.buf = None          # (capacity, device pointer) of the local labels
        self.numSegments = 0
        self.lut = None          # final id of every local id, once resolved
        self.uses = 0            # neighbours that still need the local labels
        self.done = threading.Event()
        self.error = None
        self.result = None


class TiledSegmenter(object):
    """
    Segments the tiles of one raster and stitches them.  One instance per call of
    doTiledShepherdSegmentation; bench.py drives it directly with the raster in pinned host
    memory or in HBM.
    """
    def __init__(self, src, bandNumbers, tileInfo, overlapSize, centres, imgNullVal, fourConnected,
            minSegmentSize, thr, simpleTileRecode, concurrencyCfg, timings, verbose=False,
            profile=False):
        self.src = src
        self.bandNumbers = list(bandNumbers)
        self.tileInfo = tileInfo
        self.overlapSize = int(overlapSize)
        self.centres = centres
        self.imgNullVal = imgNullVal
        self.fourConnected = fourConnected
        self.minSegmentSize = minSegmentSize
        self.thr = thr
        self.simple = simpleTileRecode
        self.cfg = concurrencyCfg
        self.timings = timings
        self.verbose = verbose
        self.profile = profile
        self.order = sorted(tileInfo.tiles.keys(), key=lambda cr: (cr[1], cr[0]))
        self.tiles = dict((cr, _Tile(cr[0], cr[1], tileInfo.tiles[cr])) for cr in self.order)
        for t in self.tiles.values():
            t.uses = int(t.col + 1 < tileInfo.ncols) + int(t.row + 1 < tileInfo.nrows)
            if (t.ysize < self.overlapSize or t.xsize < self.overlapSize) and len(self.tiles) > 1:
                raise PyShepSegTilingError("tiles must be at least overlapSize pixels on a side")
        if numpy.dtype(src.dtype).newbyteorder('=') not in _lib.DTYPE_CODES:
            raise PyShepSegTilingError("rasters of type {} are not supported (supported: {})".format(
                src.dtype, ', '.join(str(d) for d in _lib.DTYPE_CODES)))
        if len(self.bandNumbers) > _lib.SSG_MAX_BANDS:
            raise PyShepSegTilingError("at most {} bands are supported".format(_lib.SSG_MAX_BANDS))
        if len(set(self.cfg.devices)) > 1 and self.cfg.concurrencyType == CONC_THREADS:
            raise PyShepSegTilingError('a TiledSegmenter drives one GPU; MultiDeviceSegmenter runs '
                'one per device')
        self.device = self.cfg.devices[0]
        self.shard = 0           # which of the states of self.device this instance uses (gpuState)
        self.readSemaphore = threading.BoundedSemaphore(max(1, self.cfg.maxConcurrentReads))
        self.readLock = None     # serialises reads of a file source shared with other instances
        self.sinkLock = None     # serialises writes into a sink shared with other instances
        self.forceExit = threading.Event()
        self.workerError = None
        self.stopCause = None    # set by stop(): another part of the run failed
        self.stageMs = {'assign': 0.0, 'clump': 0.0, 'single': 0.0, 'small': 0.0, 'total': 0.0}
        self.launches = 0
        self.h2dBytes = 0
        self.d2hBytes = 0
        self.kernelMs = {}       # name -> [count, total ms] when profile=True
        self.statLock = threading.Lock()
        self.uploader = None     # _RasterUploader while a run streams the whole raster to the GPU
        self.timeline = [] if os.environ.get('SSG_TIMELINE') else None   # (ms, what) of one run
        self.t0 = time.perf_counter()

    def mark(self, what):
        if self.timeline is not None:
            self.timeline.append((round((time.perf_counter() - self.t0) * 1e3, 2), what))

    # ---- segmentation of one tile on a slot --------------------------------------------------
    def segmentOne(self, slot, pool, tile):
        ctx = slot.ctx
        self.mark('tile %d,%d read start' % (tile.col, tile.row))
        dtype = self.src.dtype.newbyteorder('=')
        item = dtype.itemsize
        nB = len(self.bandNumbers)
        nPix = tile.ysize * tile.xsize
        direct = self._directSource()
        ypos = tile.ypos - getattr(self.src, 'yoff', 0)   # a rank of a sharded run holds a window
        xpos = tile.xpos - getattr(self.src, 'xoff', 0)
        with self.timings.interval('reading'):
            if direct is not None:
                # the raster is addressable memory (HBM, or host memory that cudaMemcpy2D can
                # read in place): gather the tile's window band by band, no host staging copy
                (base, onDevice) = direct
                imgDev = slot.devStageFor(nB * nPix * item)
                copy = 'ssg_memcpy2d_d2d' if onDevice else 'ssg_memcpy2d_h2d'
                up = self.uploader
                if up is not None:      # the raster is on its way to the device in one piece
                    up.waitTile((tile.col, tile.row), self.cfg.tileCompletionTimeout)
                    copy = 'ssg_memcpy2d_d2d'
                for (i, b) in enumerate(self.bandNumbers):
                    if up is not None:
                        (srcPtr, pitch) = (up.devAddress(i, ypos, xpos), up.boxW * item)
                    else:
                        srcPtr = base + ((b - 1) * self.src.ysize * self.src.xsize + ypos * self.src.xsize + xpos) * item
                        pitch = self.src.xsize * item
                    ctx.call(copy, imgDev + i * nPix * item, tile.xsize * item, srcPtr, pitch,
                        tile.xsize * item, tile.ysize)
            else:
                with self.readSemaphore, self.readLock or _nullContext():
                    img = slot.pinnedFor(nB * nPix, dtype).reshape(nB, tile.ysize, tile.xsize)
                    self.src.readWindow(self.bandNumbers, xpos, ypos, tile.xsize, tile.ysize,
                        out=img)
        self.mark('tile %d,%d read issued' % (tile.col, tile.row))
        with self.timings.interval('segmentation'):
            if direct is None:
                ctx.call('ssg_upload_image', _lib.ptr(img), _lib.DTYPE_CODES[numpy.dtype(dtype)], nB,
                    tile.ysize, tile.xsize)
                imgDev = ctx.lib.ssg_staged_image(ctx.h)
            # the labels, followed by room for the per-segment existence tables of the stitch: the
            # final relabel of the segmentation fills them while it has the labels in its hands
            extCap = self._extentsCap(nPix)
            tile.buf = pool.get(ctx, nPix * 4 + extCap * _lib.SSG_EXTENT_TABLES)
            prm = shepseg.makeTileParams(dtype, nB, tile.ysize, tile.xsize, self.centres,
                self.imgNullVal, self.fourConnected, self.minSegmentSize, self.thr)
            (prm.trimTop, prm.trimBottom, prm.trimLeft, prm.trimRight) = tileMargins(self.tileInfo, tile.col,
                tile.row, tile.xsize, tile.ysize, self.overlapSize)
            ov = self.overlapSize
            prm.stripRows = 0 if (tile.row == 0 or self.simple) else min(ov, tile.ysize)
            prm.stripCols = 0 if (tile.col == 0 or self.simple) else min(ov, tile.xsize)
            prm.extentsDev = tile.buf[1] + nPix * 4
            prm.extentsCap = extCap
            res = _lib.TileResult()
            ctx.call('ssg_segment_tile_device', imgDev, ctypes.byref(prm), tile.buf[1], ctypes.byref(res))
        self.mark('tile %d,%d segmented (dev %.1f ms)' % (tile.col, tile.row, res.msTotal))
        tile.numSegments = int(res.numSegments)
        tile.result = res
        with self.statLock:
            if not isinstance(self.src, DeviceRaster) and self.uploader is None:
                self.h2dBytes += nB * nPix * item
            for k in self.stageMs:
                self.stageMs[k] += getattr(res, 'ms' + k.capitalize())

    @staticmethod
    def _extentsCap(nPix):
        """entries per existence table kept behind a tile's labels (a tile with more segments than
        this has its tables computed by the stitch instead)"""
        return ((nPix // 16 + 4096) + 15) // 16 * 16

    def _startUpload(self, state, slotIndex, order=None):
        """Stream the raster to the device in one piece (see _RasterUploader) when it is host
        memory addressable in place and several workers overlap the copy with the kernels."""
        direct = self._directSource()
        if direct is None or direct[1]:
            return
        dtype = self.src.dtype.newbyteorder('=')
        order = self.order if order is None else order
        tiles = [(cr, self.tiles[cr].xpos, self.tiles[cr].ypos, self.tiles[cr].xsize, self.tiles[cr].ysize)
            for cr in order]
        (bx, by, bh, bw) = _RasterUploader.box(tiles)     # (only the tiles' bounding box goes up)
        nbytes = len(self.bandNumbers) * bh * bw * dtype.itemsize
        slot = state.slot(slotIndex)
        if state.rasterBuf is None or state.rasterBuf[0] < nbytes:
            if state.rasterBuf is not None:
                slot.ctx.dev_free(state.rasterBuf[1])
            state.rasterBuf = (nbytes, slot.ctx.dev_alloc(max(nbytes, 1)))
        self.uploader = _RasterUploader(slot, direct[0], self.bandNumbers, self.src.ysize, self.src.xsize,
            dtype.itemsize, state.rasterBuf[1], tiles, getattr(self.src, 'yoff', 0), getattr(self.src, 'xoff', 0))
        self.uploader.start()

    def _finishUpload(self):
        if self.uploader is not None:
            self.uploader.join()
            self.h2dBytes += self.uploader.bytes
            self.uploader = None

    def _directSource(self):
        """(base pointer, on device?) when tile windows can be copied straight out of the
        raster's memory, else None (file sources go through a pinned staging read)."""
        if isinstance(self.src, DeviceRaster):
            return (self.src.devPtr, True)
        if isinstance(self.src, rasterfile.MemoryRaster) and not isinstance(self.src, rasterfile.NpySource):
            a = self.src.img
            if isinstance(a, numpy.ndarray) and a.flags.c_contiguous and a.dtype.isnative and \
                    a.dtype in _lib.DTYPE_CODES:
                return (a.ctypes.data, False)
        return None

    def _reserve(self, slot, segments):
        """Size a slot's device memory for the largest tile (or, for a slot that only stitches,
        for the largest overlap strips) before the first tile: growing later would put cudaMalloc
        and cudaFree, which synchronise the device, in the middle of the run."""
        maxPix = max(t.xsize * t.ysize for t in self.tiles.values())
        maxStrip = self.overlapSize * max(t.xsize + t.ysize for t in self.tiles.values())
        dtype = self.src.dtype.newbyteorder('=')
        direct = self._directSource() is not None
        if segments:
            # (with a directly addressable raster the tile image is gathered into the slot's own
            # staging buffer, so the context's image buffer is not needed)
            slot.ctx.call('ssg_ctx_reserve', maxPix, 0 if direct else len(self.bandNumbers),
                _lib.DTYPE_CODES[numpy.dtype(dtype)], 0)
        else:
            slot.ctx.call('ssg_ctx_reserve', 0, 0, 0, maxStrip * 24 + (64 << 20))

    def _worker(self, slot, pool, inQue):
        """A segmentation worker (tiling.py:1560-1613): pops tiles until the queue is empty.  Whatever
        goes wrong -- reserving memory included -- is recorded where the stitch loop looks
        (tile.error, like the reference's WorkerErrorRecord / checkWorkerExceptions) and every
        tile still waiting is released, so the main thread fails at once with the real cause."""
        tile = None
        try:
            with slot.lock:
                self._reserve(slot, True)
                before = slot.ctx.launch_count()
                self._profileStart(slot)
                while not self.forceExit.is_set():
                    try:
                        cr = inQue.get(block=False)
                    except queue.Empty:
                        break
                    tile = self.tiles[cr]
                    self.segmentOne(slot, pool, tile)
                    tile.done.set()
                    tile = None
                self._profileStop(slot)
                with self.statLock:
                    self.launches += slot.ctx.launch_count() - before
        except Exception as e:
            self.workerError = e
            self.forceExit.set()
            if tile is not None:
                tile.error = e
            for t in self.tiles.values():      # nobody will segment these now
                if not t.done.is_set():
                    if t.error is None:
                        t.error = e
                    t.done.set()

    def stop(self, cause):
        """End a run from another thread (another shard of a MultiDeviceSegmenter failed): the
        workers stop after their current tile and every tile not segmented yet reports `cause`."""
        self.stopCause = cause
        self.forceExit.set()
        for t in self.tiles.values():
            if not t.done.is_set():
                if t.error is None:
                    t.error = cause
                t.done.set()

    def _profileStart(self, slot):
        if self.profile:
            slot.ctx.call('ssg_profile_enable', 1)

    def _profileStop(self, slot):
        if not self.profile:
            return
        buf = ctypes.create_string_buffer(1 << 16)
        slot.ctx.call('ssg_profile_fetch', buf, len(buf))
        slot.ctx.call('ssg_profile_enable', 0)
        with self.statLock:
            for line in buf.value.decode().splitlines():
                (name, cnt, ms) = line.split()
                ent = self.kernelMs.setdefault(name, [0, 0.0])
                ent[0] += int(cnt)
                ent[1] += float(ms)

    # ---- the stitch of one tile (main thread) ------------------------------------------------
    def tileTables(self, slot, tile, topB, topStride, leftB, leftStride):
        """Device phase 1 of the stitch for one tile + the copy of its tables to the host.
        topB / leftB: device pointers of the neighbours' LOCAL labels under the overlaps."""
        ctx = slot.ctx
        (top, bottom, left, right) = tileMargins(self.tileInfo, tile.col, tile.row, tile.xsize,
            tile.ysize, self.overlapSize)
        tables = _lib.TileTables()
        with self.timings.interval('stitch_tables'):
            res = tile.result
            given = res is not None and res.extentsDone
            ctx.call('ssg_tile_tables_device', tile.buf[1], tile.ysize, tile.xsize, self.overlapSize,
                topB, topStride, leftB, leftStride, top, bottom, left, right, tile.numSegments,
                (tile.buf[1] + tile.ysize * tile.xsize * 4) if given else None,
                int(res.extentsStride) if given else 0, ctypes.byref(tables))
            n = int(tables.maxId) + 1
            rank = numpy.empty(n, dtype=numpy.uint32)
            flags = numpy.empty(n, dtype=numpy.uint8)
            pairKeys = numpy.empty(int(tables.numPairs), dtype=numpy.uint64)
            pairCounts = numpy.empty(int(tables.numPairs), dtype=numpy.uint32)
            ctx.call('ssg_tile_tables_fetch', _lib.ptr(rank), _lib.ptr(flags), _lib.ptr(pairKeys),
                _lib.ptr(pairCounts))
        self.d2hBytes += rank.nbytes + flags.nbytes + pairKeys.nbytes + pairCounts.nbytes
        from . import distributed
        return distributed.TileTable(tables.maxId, tables.countNew, rank, flags, pairKeys, pairCounts,
            maxRankInTrim=int(tables.maxRankInTrim))

    def applyLut(self, slot, tile, lut, maxId, sink, hist, histLen, deferred=None, fetchLen=0, rel=None):
        """Device phase 2: final ids over the trimmed window, on the device, then to the sink.
        deferred (a list, for the last tile of a run): if the window can travel on its own, the
        histogram copy is queued BEFORE it (mark 0), the window copy is left in flight (mark 1)
        and 'window' is appended to the list: the caller works on the histogram meanwhile.
        rel = (rank, flags, offset, crossLabels, crossIds) instead of lut: the lut is put together on
        the device (ssg_apply_rel_lut_device)."""
        ctx = slot.ctx

        def kernel(out, outStride):
            if rel is None:
                ctx.call('ssg_apply_lut_device', tile.buf[1], tile.ysize, tile.xsize, _lib.ptr(lut),
                    int(maxId), top, bottom, left, right, out, outStride, hist.dev, hist.cap)
                self.h2dBytes += lut.nbytes
            else:
                (rankArr, flagsArr, offset, crossLabels, crossIds) = rel
                ctx.call('ssg_apply_rel_lut_device', tile.buf[1], tile.ysize, tile.xsize,
                    None if rankArr is None else _lib.ptr(rankArr),
                    None if rankArr is None else _lib.ptr(flagsArr), int(maxId), int(offset), len(crossLabels),
                    _lib.ptr(crossLabels) if len(crossLabels) else None,
                    _lib.ptr(crossIds) if len(crossLabels) else None,
                    top, bottom, left, right, out, outStride, hist.dev, hist.cap)
                self.h2dBytes += (0 if rankArr is None else rankArr.nbytes + flagsArr.nbytes) + 8 * len(crossLabels)
        (top, bottom, left, right) = tileMargins(self.tileInfo, tile.col, tile.row, tile.xsize,
            tile.ysize, self.overlapSize)
        (wr, wc) = (bottom - top, right - left)
        hist.ensure(ctx, histLen)
        xout = tile.xpos + left - getattr(sink, 'xoff', 0)
        yout = tile.ypos + top - getattr(sink, 'yoff', 0)
        if isinstance(sink, DeviceMosaicSink):
            # the mosaic lives in HBM: write the window in place
            kernel(sink.devPtr + (yout * sink.xsize + xout) * 4, sink.xsize)
        else:
            (window, winDev) = slot.windowFor(wr * wc)
            kernel(winDev, wc)
            levels = [int(v) for v in (getattr(sink, 'levels', None) or [])]
            if levels:
                # the overview levels of the window, cut out on the device (tiling.py:1360-1383)
                shapes = [(len(range(lvl // 2, wr, lvl)), len(range(lvl // 2, wc, lvl))) for lvl in levels]
                total = sum(r * c for (r, c) in shapes)
                packed = slot.overviewsFor(total)
                starts = numpy.zeros(len(levels) + 1, dtype=numpy.int64)
                ctx.call('ssg_window_overviews', winDev, wr, wc, wc, len(levels),
                    _lib.ptr(numpy.array(levels, dtype=numpy.int32)), _lib.ptr(packed), packed.size, _lib.ptr(starts))
                with self.sinkLock or _nullContext():
                    for (j, (lvl, (r, c))) in enumerate(zip(levels, shapes)):
                        (ownRows, ownCols) = overviewBlockOwned(self.tileInfo, tile.col, tile.row, self.overlapSize,
                            lvl, getattr(sink, 'xoff', 0), getattr(sink, 'yoff', 0))
                        block = packed[starts[j]:starts[j] + r * c].reshape(r, c)[:ownRows, :ownCols]
                        sink.writeOverviewLevel(j, lvl, block, xout // lvl, yout // lvl)
                self.d2hBytes += total * 4
            arr = getattr(sink, 'array', None)
            if (type(sink) is rasterfile.MemorySink and isinstance(arr, numpy.ndarray) and
                    arr.flags.c_contiguous and arr.dtype == numpy.uint32):
                # the output raster is plain host memory: land the window in place (windows are
                # disjoint, so the shards of a MultiDeviceSegmenter need no sink lock for this)
                if deferred is not None:
                    hist.fetchAsync(ctx, fetchLen)
                    ctx.call('ssg_mark', 0)
                    ctx.call('ssg_memcpy2d_d2h_async', arr.ctypes.data + (yout * arr.shape[1] + xout) * 4,
                        arr.shape[1] * 4, winDev, wc * 4, wc * 4, wr)
                    ctx.call('ssg_mark', 1)
                    deferred.append('window')
                else:
                    ctx.call('ssg_memcpy2d_d2h', arr.ctypes.data + (yout * arr.shape[1] + xout) * 4,
                        arr.shape[1] * 4, winDev, wc * 4, wc * 4, wr)
            else:
                out = window[:wr * wc].reshape(wr, wc)
                ctx.call('ssg_memcpy_d2h', _lib.ptr(out), winDev, wr * wc * 4)
                with self.sinkLock or _nullContext():
                    sink.write(out, xout, yout)
                    if not levels:
                        sink.writeOverviews(out, xout, yout)
            self.d2hBytes += wr * wc * 4

    def stitchOne(self, slot, pool, tile, offset, sink, hist, deferred=None):
        self.mark('tile %d,%d stitch start' % (tile.col, tile.row))
        ov = self.overlapSize
        up = self.tiles.get((tile.col, tile.row - 1)) if tile.row > 0 else None
        lf = self.tiles.get((tile.col - 1, tile.row)) if tile.col > 0 else None
        topB = leftB = None
        (topStride, leftStride) = (0, 0)
        if not self.simple:
            if up is not None:      # the upper tile's bottom `ov` rows (its LOCAL labels)
                topB = up.buf[1] + (up.ysize - ov) * up.xsize * 4
                topStride = up.xsize
            if lf is not None:      # the left tile's right `ov` columns
                leftB = lf.buf[1] + (lf.xsize - ov) * 4
                leftStride = lf.xsize
        tb = self.tileTables(slot, tile, topB, topStride, leftB, leftStride)
        self.mark('tile %d,%d tables on host (%d segments, %d votes)' % (tile.col, tile.row, tb.maxId,
            len(tb.pairKeys)))
        tables = _lib.TileTables()
        (tables.maxId, tables.countNew, tables.numPairs) = (tb.maxId, tb.countNew, len(tb.pairKeys))
        with self.timings.interval('stitch_resolve'):
            (lut, trimmedMax) = resolveTile(tables, tb.rank, tb.flags, tb.pairKeys, tb.pairCounts, offset,
                None if up is None else up.lut, None if lf is None else lf.lut, self.simple)
        tile.lut = lut
        n = tb.maxId + 1
        self.mark('tile %d,%d resolved' % (tile.col, tile.row))
        self.applyLut(slot, tile, lut, tb.maxId, sink, hist,
            max(offset + tb.countNew, trimmedMax, int(lut.max()) if n else 0) + 1, deferred,
            max(offset, trimmedMax) + 1)
        self.mark('tile %d,%d window delivered' % (tile.col, tile.row))
        # the neighbours' labels are no longer needed once both users have run
        for nb in (up, lf):
            if nb is not None:
                nb.uses -= 1
                if nb.uses == 0 and nb.buf is not None:
                    pool.put(nb.buf)
                    nb.buf = None
        if tile.uses == 0:
            pool.put(tile.buf)
            tile.buf = None
        return max(offset, trimmedMax)

    # ---- driver ----------------------------------------------------------------------------
    def run(self, sink, comm=None, deferFinal=False):
        """Segment and stitch every tile; returns (maxSegId, histogram).  With a communicator of
        more than one rank (distributed.TorchComm) the tiles are shared out over the ranks and
        `sink` receives this rank's trimmed windows only.  deferFinal: return as soon as the
        histogram is on the host, possibly with the last window still on its way to the sink; the
        caller must then call finish() before it touches the output."""
        self.inFlight = None
        if comm is not None and comm.world > 1:
            return self.runSharded(sink, comm)
        cfg = self.cfg
        state = gpuState(self.device)
        pool = state.pool
        main = state.slot(0)
        hist = state.hist
        offset = 0
        workers = []
        numWorkers = cfg.numWorkers if cfg.concurrencyType == CONC_THREADS else 0
        main.lock.acquire()
        before = main.ctx.launch_count()
        try:
            self._reserve(main, numWorkers == 0)
            hist.reset(main.ctx)
            self._profileStart(main)
            if numWorkers > 0:
                # (row-major, the order of the stitch: starting the large corner tile first was
                # measured to be slower -- the GPU is the shared resource, and the small first
                # tiles then finish late and hold up the whole stitch chain)
                inQue = queue.Queue()
                for cr in self.order:
                    inQue.put(cr)
                with self.timings.interval('startworkers'):
                    self._startUpload(state, numWorkers + 1)
                    for w in range(numWorkers):
                        th = threading.Thread(target=self._worker, args=(state.slot(1 + w), pool, inQue),
                            daemon=True)
                        th.start()
                        workers.append(th)
            with self.timings.interval('stitchtiles') if numWorkers > 0 else _nullContext():
                deferred = []
                for cr in self.order:
                    tile = self.tiles[cr]
                    last = deferred if cr == self.order[-1] else None
                    if numWorkers > 0:
                        if not tile.done.wait(cfg.tileCompletionTimeout):
                            self.forceExit.set()
                            raise PyShepSegTilingError(("Timeout ({} seconds) waiting for completed "
                                "tile. Try increasing tileCompletionTimeout").format(cfg.tileCompletionTimeout))
                        if tile.error is not None:
                            raise PyShepSegTilingError("A segmentation worker failed on tile "
                                "col={} row={}: {}".format(tile.col, tile.row, tile.error))
                        offset = self.stitchOne(main, pool, tile, offset, sink, hist, last)
                    else:
                        if self.verbose:
                            print("Doing tile row={}, col={}".format(tile.row, tile.col))
                        self.segmentOne(main, pool, tile)
                        with self.timings.interval('stitchtiles'):
                            offset = self.stitchOne(main, pool, tile, offset, sink, hist, last)
            if deferred:
                # the histogram was queued ahead of the last window: it is here long before the window is
                main.ctx.call('ssg_wait_mark', 0)
                histogram = hist.collect()
                self.inFlight = main
                if not deferFinal:
                    self.finish()
            else:
                histogram = hist.fetch(main.ctx, offset + 1)
            self.d2hBytes += histogram.nbytes
        finally:
            self.forceExit.set()
            for th in workers:
                th.join()
            self._finishUpload()
            try:
                self._profileStop(main)
                for t in self.tiles.values():
                    if t.buf is not None:
                        pool.put(t.buf)
                        t.buf = None
                self.launches += main.ctx.launch_count() - before
            finally:
                main.lock.release()
        return (offset, histogram)


    def finish(self):
        """Wait for the last window of a run(deferFinal=True) to land in the sink."""
        if getattr(self, 'inFlight', None) is not None:
            self.inFlight.ctx.call('ssg_wait_mark', 1)
            self.inFlight = None

    def runSharded(self, sink, comm):
        """
        The tiles of the mosaic dealt over the ranks of `comm` (distributed.ShardedStitch): this
        rank segments its own tiles, keeps their labels in HBM, exchanges overlap strips with the
        ranks that own neighbouring tiles, and writes the trimmed windows of its tiles.
        Returns (maxSegId, histogram summed over the ranks; on rank 0 only when the ranks
        talk over NCCL).
        """
        from . import distributed
        import torch
        cfg = self.cfg
        state = gpuState(self.device, self.shard)
        pool = state.pool
        main = state.slot(0)
        hist = state.hist
        stitch = distributed.ShardedStitch(self.tileInfo, self.overlapSize, self.simple, comm, self.timings)
        mine = stitch.mine
        numWorkers = cfg.numWorkers if cfg.concurrencyType == CONC_THREADS else 0
        workers = []
        ov = self.overlapSize
        cudaDev = torch.device('cuda', self.device)
        # strips travel device to device (NCCL, or ThreadComm's copies) unless the communicator
        # is a host one (gloo)
        onDevice = getattr(comm, 'device', None) is not None and comm.device.type == 'cuda'
        stripDev = cudaDev if onDevice else torch.device('cpu')
        seg = self
        keep = []     # device copies of strips received through the host

        class Ops(object):
            def sendStrip(self, cr, which):
                t = seg.tiles[cr]
                if which == 'bottom':
                    out = torch.empty((ov, t.xsize), dtype=torch.int32, device=stripDev)
                    (src, spitch, rows) = (t.buf[1] + (t.ysize - ov) * t.xsize * 4, t.xsize * 4, ov)
                    width = t.xsize * 4
                else:
                    out = torch.empty((t.ysize, ov), dtype=torch.int32, device=stripDev)
                    (src, spitch, rows) = (t.buf[1] + (t.xsize - ov) * 4, t.xsize * 4, t.ysize)
                    width = ov * 4
                main.ctx.call('ssg_memcpy2d_d2d' if onDevice else 'ssg_memcpy2d_d2h', out.data_ptr(), width,
                    src, spitch, width, rows)
                main.ctx.synchronize()
                return out

            def recvStrip(self, cr, which, shape):
                return torch.empty(shape, dtype=torch.int32, device=stripDev)

            def _devStrip(self, t):
                if t.device.type == 'cuda':
                    return t
                d = t.to(cudaDev)
                torch.cuda.synchronize(cudaDev)
                keep.append(d)
                return d

            def tables(self, cr, top, left):
                t = seg.tiles[cr]
                (topB, topStride, leftB, leftStride) = (None, 0, None, 0)
                if top is not None:
                    if isinstance(top, str):
                        up = seg.tiles[(t.col, t.row - 1)]
                        (topB, topStride) = (up.buf[1] + (up.ysize - ov) * up.xsize * 4, up.xsize)
                    else:
                        top = self._devStrip(top)
                        (topB, topStride) = (top.data_ptr(), top.shape[1])
                if left is not None:
                    if isinstance(left, str):
                        lf = seg.tiles[(t.col - 1, t.row)]
                        (leftB, leftStride) = (lf.buf[1] + (lf.xsize - ov) * 4, lf.xsize)
                    else:
                        left = self._devStrip(left)
                        (leftB, leftStride) = (left.data_ptr(), left.shape[1])
                return seg.tileTables(main, t, topB, topStride, leftB, leftStride)

            def apply(self, cr, lut, tb):
                t = seg.tiles[cr]
                t.lut = lut
                seg.applyLut(main, t, lut, tb.maxId, sink, hist, int(lut.max()) + 1 if len(lut) else 1)

            def applyRel(self, cr, offset, crossLabels, crossIds, tb):
                t = seg.tiles[cr]
                top = offset + (tb.maxId if seg.simple else tb.countNew)
                if len(crossIds):
                    top = max(top, int(crossIds.max()))
                seg.applyLut(main, t, None, tb.maxId, sink, hist, top + 1, rel=(
                    None if seg.simple else tb.rank, tb.flags, offset,
                    numpy.ascontiguousarray(crossLabels, dtype=numpy.uint32),
                    numpy.ascontiguousarray(crossIds, dtype=numpy.uint32)))

        main.lock.acquire()
        before = main.ctx.launch_count()
        try:
            self._reserve(main, numWorkers == 0)
            hist.reset(main.ctx)
            self._profileStart(main)
            ops = Ops()
            # Tiles that feed another rank (their bottom / right strip lies under a remote tile's
            # overlap) are segmented first and their strips handed over while the rest is still
            # in work; a tile gets its stitch tables as soon as it and what lies under its
            # overlaps (own neighbours, received strips) exist.
            (feed, exchangeAfter) = stitch.feedPlan()
            order = feed + [cr for cr in mine if cr not in feed]
            exchangeAfter = min(exchangeAfter, len(order))
            tabled = set()

            def tryTables():
                for cr in mine:
                    if cr in tabled or not self.tiles[cr].done.is_set() or self.tiles[cr].error is not None:
                        continue
                    args = []
                    for (nb, which) in zip(stitch.neighbours(cr), ('bottom', 'right')):
                        if nb is None or self.simple:
                            args.append(None)
                        elif stitch.owner[nb] == comm.rank:
                            if not self.tiles[nb].done.is_set():
                                break
                            args.append('local')
                        else:
                            if stitch.received is None:
                                break
                            args.append(stitch.received[(nb, which)])
                    else:
                        tabled.add(cr)
                        stitch.early(cr, ops.tables(cr, args[0], args[1]))

            with self.timings.interval('segmentation_all'):
                if numWorkers > 0:
                    inQue = queue.Queue()
                    for cr in order:
                        inQue.put(cr)
                    self._startUpload(state, numWorkers + 1, order)
                    for w in range(numWorkers):
                        th = threading.Thread(target=self._worker, args=(state.slot(1 + w), pool, inQue),
                            daemon=True)
                        th.start()
                        workers.append(th)
                if exchangeAfter == 0:
                    stitch.exchangeStrips(ops)
                for (i, cr) in enumerate(order):
                    tile = self.tiles[cr]
                    if self.stopCause is not None:
                        raise PyShepSegTilingError('stopped: {}'.format(self.stopCause))
                    if numWorkers > 0:
                        if not tile.done.wait(cfg.tileCompletionTimeout):
                            self.forceExit.set()
                            raise PyShepSegTilingError(("Timeout ({} seconds) waiting for completed "
                                "tile. Try increasing tileCompletionTimeout").format(cfg.tileCompletionTimeout))
                        if tile.error is not None:
                            raise PyShepSegTilingError("A segmentation worker failed on tile col={} row={}: {}".format(
                                cr[0], cr[1], tile.error))
                    else:
                        self.segmentOne(main, pool, tile)
                        tile.done.set()
                    if i + 1 == exchangeAfter:
                        stitch.exchangeStrips(ops)
                    tryTables()
                for th in workers:
                    th.join()
            with self.timings.interval('stitchtiles'):
                (maxSegId, offsets, luts) = stitch.run(ops)
                with self.timings.interval('stitch_applywait'):
                    main.ctx.synchronize()
                with self.timings.interval('stitch_histogram'):
                    # Every rank takes the SAME branch and reduces the SAME number of entries:
                    # which collective runs must not hang on anything rank-local (a rank whose
                    # tiles carry small ids has a smaller histogram buffer than the others).
                    n = maxSegId + 1
                    hist.ensure(main.ctx, n)
                    if onDevice:
                        # summed over the ranks on the devices into rank 0, which alone holds the
                        # output's histogram (the other ranks return an empty one)
                        t = torch.empty(n, dtype=torch.int64, device=cudaDev)
                        main.ctx.call('ssg_memcpy_d2d', t.data_ptr(), hist.dev, n * 8)
                        main.ctx.synchronize()
                        t = comm.reduceSum(t)
                        if comm.rank == 0:
                            # converted on the device, copied into pinned memory (the caching
                            # host allocator hands the same block out again run after run)
                            f = t.to(torch.float64)
                            f[0] = 0
                            h = torch.empty(n, dtype=torch.float64, pin_memory=True)
                            h.copy_(f, non_blocking=True)
                            torch.cuda.current_stream(cudaDev).synchronize()
                            histogram = h.numpy()
                        else:
                            histogram = numpy.zeros(0)
                    else:
                        histogram = comm.allreduceSum(hist.fetch(main.ctx, n))
            self.d2hBytes += histogram.nbytes
            self.usedFallback = stitch.usedFallback
        finally:
            self.forceExit.set()
            for th in workers:
                th.join()
            self._finishUpload()
            try:
                self._profileStop(main)
                for t in self.tiles.values():
                    if t.buf is not None:
                        pool.put(t.buf)
                        t.buf = None
                self.launches += main.ctx.launch_count() - before
            finally:
                main.lock.release()
        return (maxSegId, histogram)


class MultiDeviceSegmenter(object):
    """
    One mosaic segmented on several GPUs from one process: one TiledSegmenter per shard, each
    running runSharded on a thread of its own over a distributed.ThreadComm, all writing into one
    sink.  shardDevices lists the device of every shard; doTiledShepherdSegmentation passes the
    distinct ids of concurrencyCfg.devices.  Shards on the same device (the tests run several on
    one GPU) each use a state of their own (gpuState).  The numWorkers workers are dealt
    round-robin over the shards; a shard without one segments its tiles in its stitch thread.

    Source: a host MemoryRaster is read in place by every shard, each streaming the cells of its
    own tiles to its device.  Reads of any other source are serialised through one lock, under
    one maxConcurrentReads semaphore for all shards.  Sink: window and overview writes of all
    shards go through one lock (windows landing in place in a plain MemorySink are disjoint and
    need none); every shard has synchronised its last window before run() returns.  Histogram:
    summed on the devices into shard 0's device (ThreadComm.reduceSum).  A failure anywhere stops
    every shard and run() raises it.
    """
    def __init__(self, shardDevices, src, bandNumbers, tileInfo, overlapSize, centres, imgNullVal,
            fourConnected, minSegmentSize, thr, simpleTileRecode, concurrencyCfg, timings, verbose=False):
        if isinstance(src, DeviceRaster):
            raise PyShepSegTilingError('a DeviceRaster lives on one GPU; segment it on that device alone')
        self.cfg = concurrencyCfg
        self.timings = timings
        self.timeline = [] if os.environ.get('SSG_TIMELINE') else None
        self.t0 = time.perf_counter()
        readSemaphore = threading.BoundedSemaphore(max(1, concurrencyCfg.maxConcurrentReads))
        (readLock, sinkLock) = (threading.Lock(), threading.Lock())
        n = len(shardDevices)
        self.shards = []
        self.labels = []
        perDevice = {}
        for (i, dev) in enumerate(shardDevices):
            cfg = copy.copy(concurrencyCfg)
            cfg.devices = [dev]
            cfg.numWorkers = len(range(i, concurrencyCfg.numWorkers, n))
            seg = TiledSegmenter(src, bandNumbers, tileInfo, overlapSize, centres, imgNullVal, fourConnected,
                minSegmentSize, thr, simpleTileRecode, cfg, timinghooks.Timers(), verbose)
            seg.shard = perDevice.get(dev, 0)
            perDevice[dev] = seg.shard + 1
            (seg.readSemaphore, seg.readLock, seg.sinkLock, seg.t0) = (readSemaphore, readLock, sinkLock, self.t0)
            self.shards.append(seg)
            self.labels.append('gpu%d' % dev if seg.shard == 0 else 'gpu%d.%d' % (dev, seg.shard))
        self.stageMs = None
        self.launches = self.h2dBytes = self.d2hBytes = 0
        self.usedFallback = False

    def mark(self, what):
        if self.timeline is not None:
            self.timeline.append((round((time.perf_counter() - self.t0) * 1e3, 2), what))

    def run(self, sink, comm=None, deferFinal=False):
        """Segment and stitch every tile into `sink`; returns (maxSegId, histogram)."""
        import torch
        from . import distributed
        if comm is not None:
            raise PyShepSegTilingError('a MultiDeviceSegmenter is its own communicator')
        n = len(self.shards)
        hub = distributed.ThreadHub(n, self.cfg.barrierTimeout)
        results = [None] * n

        def shardMain(i):
            seg = self.shards[i]
            try:
                results[i] = seg.runSharded(sink, distributed.ThreadComm(hub, i, torch.device('cuda', seg.device)))
            except BaseException as e:
                hub.abort(i, e)
                for other in self.shards:
                    if other is not seg:
                        other.stop('{} failed: {}'.format(self.labels[i], e))
        threads = [threading.Thread(target=shardMain, args=(i,), daemon=True) for i in range(n)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        if hub.failed is not None:
            (i, e) = hub.failed
            raise PyShepSegTilingError('segmentation on {} failed: {}'.format(self.labels[i], e)) from e
        self.stageMs = dict((k, sum(seg.stageMs[k] for seg in self.shards)) for k in self.shards[0].stageMs)
        for (seg, label) in zip(self.shards, self.labels):
            self.launches += seg.launches
            self.h2dBytes += seg.h2dBytes
            self.d2hBytes += seg.d2hBytes
            # every shard's intervals under the reference's names and under the shard's own
            self.timings.merge(seg.timings)
            self.timings.merge(timinghooks.Timers(dict((label + ':' + k, v) for (k, v) in seg.timings.pairs.items())))
            if self.timeline is not None and seg.timeline is not None:
                self.timeline += [(ms, label + ': ' + what) for (ms, what) in seg.timeline]
        if self.timeline is not None:
            self.timeline.sort(key=lambda e: e[0])
        self.usedFallback = self.shards[0].usedFallback
        return results[0]

    def finish(self):
        """(run() returns with every window in the sink)"""


class DeviceRaster(rasterfile.RasterSource):
    """A band-sequential (count, ysize, xsize) raster that already lives in GPU memory
    (devPtr is a device pointer on the segmenting GPU).  Used to measure the path with its
    input resident in HBM; tiles are gathered with device-to-device copies."""
    def __init__(self, devPtr, count, ysize, xsize, dtype, nodata=None, yoff=0, xoff=0):
        self.devPtr = int(devPtr)
        self.yoff = int(yoff)        # mosaic row / column of the buffer's first pixel (a rank's window)
        self.xoff = int(xoff)
        (self.count, self.ysize, self.xsize) = (int(count), int(ysize), int(xsize))
        self.dtype = numpy.dtype(dtype)
        self.nodata = [nodata] * self.count


class DeviceMosaicSink(rasterfile.RasterSink):
    """A uint32 (ysize, xsize) output mosaic in GPU memory: the stitch writes the trimmed
    windows in place and nothing but the small per-tile tables crosses PCIe."""
    def __init__(self, devPtr, xsize, ysize, yoff=0, xoff=0):
        self.devPtr = int(devPtr)
        (self.xsize, self.ysize) = (int(xsize), int(ysize))
        self.yoff = int(yoff)        # mosaic row / column of the buffer's first pixel (a rank's window)
        self.xoff = int(xoff)
        self.metadata = {}
        self.hist = None

    def setMetadataItem(self, key, value):
        self.metadata[key] = value

    def writeHistogram(self, hist):
        self.hist = hist


class _nullContext(object):
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


class _DeviceHistogram(object):
    """Growing uint64 histogram on the device (HistogramAccumulator, tiling.py:1915-1963)."""
    def __init__(self):
        self.dev = None
        self.cap = 0
        self.pinned = None
        (self.pending, self.pendingLen) = (0, 0)

    def ensure(self, ctx, n):
        if n <= self.cap:
            return
        newCap = max(n, 4 * self.cap, 1 << 20)
        p = ctx.dev_alloc(newCap * 8)
        ctx.call('ssg_memset_d', p, 0, newCap * 8)
        if self.dev is not None:
            ctx.call('ssg_memcpy_d2d', p, self.dev, self.cap * 8)
            ctx.synchronize()
            ctx.dev_free(self.dev)
        (self.dev, self.cap) = (p, newCap)

    def reset(self, ctx):
        """Empty the histogram for a new run (the buffer is kept between runs)."""
        if self.dev is not None:
            ctx.call('ssg_memset_d', self.dev, 0, self.cap * 8)

    def fetch(self, ctx, n):
        h = numpy.zeros(n, dtype=numpy.uint64)
        if self.dev is not None and n > 0:
            m = min(n, self.cap)
            ctx.call('ssg_memcpy_d2h', _lib.ptr(h), self.dev, m * 8)
        if n > 0:
            h[0] = 0     # the null count is always removed (tiling.py:1930-1931)
        return h.astype(numpy.float64)

    def fetchAsync(self, ctx, n):
        """Queue the copy of the first n bins into pinned memory (no wait); collect() converts"""
        if self.pinned is None or self.pinned.array.size < n:
            if self.pinned is not None:
                self.pinned.free()
            self.pinned = _lib.PinnedArray((max(n, 1 << 20),), numpy.uint64)
        self.pending = min(n, self.cap) if self.dev is not None else 0
        self.pendingLen = n
        if self.pending > 0:
            ctx.call('ssg_memcpy_d2h_async', _lib.ptr(self.pinned.array), self.dev, self.pending * 8)

    def collect(self):
        h = numpy.zeros(self.pendingLen, dtype=numpy.float64)
        h[:self.pending] = self.pinned.array[:self.pending]
        if self.pendingLen > 0:
            h[0] = 0
        return h

    def close(self, ctx):
        if self.dev is not None:
            ctx.dev_free(self.dev)
            self.dev = None
        if self.pinned is not None:
            self.pinned.free()
            self.pinned = None


def estimateStatsFromHisto(sink, hist):
    """STATISTICS_* metadata from the histogram (utils.estimateStatsFromHisto, utils.py:47-95).
    Same numbers as the reference's expressions (same products, same numpy sums), with fewer
    passes over the histogram: it is on the critical path of every tiled call."""
    nVals = hist.sum()
    if nVals <= 0:
        return
    nz = hist > 0
    first = int(numpy.argmax(nz))
    last = len(hist) - 1 - int(numpy.argmax(nz[::-1]))
    values = numpy.arange(len(hist))
    meanVal = (values * hist).sum() / nVals
    dev = values - meanVal
    stdDevVal = numpy.sqrt((hist * (dev * dev)).sum() / nVals)
    medianVal = int(numpy.searchsorted(hist.cumsum(), nVals / 2, side='left'))
    sink.setMetadataItem("STATISTICS_MINIMUM", repr(first))
    sink.setMetadataItem("STATISTICS_MAXIMUM", repr(last))
    sink.setMetadataItem("STATISTICS_MEAN", repr(float(meanVal)))
    sink.setMetadataItem("STATISTICS_STDDEV", repr(float(stdDevVal)))
    sink.setMetadataItem("STATISTICS_MODE", repr(int(numpy.argmax(hist))))
    sink.setMetadataItem("STATISTICS_MEDIAN", repr(medianVal))
    sink.setMetadataItem("STATISTICS_SKIPFACTORX", "1")
    sink.setMetadataItem("STATISTICS_SKIPFACTORY", "1")
    sink.setMetadataItem("STATISTICS_HISTOBINFUNCTION", "direct")


def checkForEmptySegments(hist, overlapSize):
    """Warn about segment ids with no pixels (tiling.py:1308-1341).  Unlike the reference,
    whose function forgets to return it, the flag is returned."""
    empty = numpy.where(hist[1:] == 0)[0] + 1
    if len(empty) > 0:
        print("\nWARNING: Found {} segments with zero pixels\n    Segment IDs: {}\n"
            "    This is caused by inconsistent joining of segmentation\n"
            "    tiles, and will probably cause trouble later on.\n"
            "    It is highly recommended to re-run with a larger overlap\n"
            "    size (currently {}), and if necessary a larger tile size\n".format(
                len(empty), empty, overlapSize), file=sys.stderr)
    return len(empty) > 0


def doTiledShepherdSegmentation(infile, outfile, tileSize=DFLT_TILESIZE,
        overlapSize=DFLT_OVERLAPSIZE, minSegmentSize=50, numClusters=60,
        bandNumbers=None, subsamplePcnt=None, maxSpectralDiff='auto',
        imgNullVal=None, fixedKMeansInit=False, fourConnected=True,
        verbose=False, simpleTileRecode=False, outputDriver='KEA',
        creationOptions=[], spectDistPcntile=50, kmeansObj=None,
        tempfilesDriver=DFLT_TEMPFILES_DRIVER, tempfilesExt=DFLT_TEMPFILES_EXT,
        tempfilesCreationOptions=[], writeHistogram=True, returnGDALDS=False,
        concurrencyCfg=None):
    """
    Run the Shepherd segmentation on a raster file tile by tile and stitch the tiles into
    one output raster (tiling.py:446-571).  Parameters as in the reference.  The temp-file
    arguments are accepted and ignored: tiles never go to disk, they stay in GPU memory until
    they are stitched.  outputDriver must be one GDAL offers, or 'GTiff' / 'NPY' / 'MEM' of the
    built-in writer when GDAL is absent.  With returnGDALDS the result's outDs is the open
    output object (a GDAL dataset with GDAL, else the rasterfile sink).

    Several GPUs: CONC_THREADS with two or more distinct ids in concurrencyCfg.devices segments
    the raster on all of them from this process and writes the one output raster (labels,
    histogram, overviews, statistics), equal bit for bit to the call with devices[0] alone.  The
    tiles are shared out by distributed.partitionTiles; the numWorkers workers are dealt
    round-robin over the devices, and a device that gets none segments its tiles in its stitch
    thread.  A failure on any device makes the call raise.  The result's maxSegId is the
    mosaic's; stageMs, gpuLaunches, h2dBytes and d2hBytes are summed over the devices; timings
    and timeline carry every device's entries, also under names prefixed by the device ('gpu1:').
    Not with concurrencyCfg.comm (one process per GPU) or a DeviceRaster input.
    """
    if concurrencyCfg is None:
        concurrencyCfg = SegmentationConcurrencyConfig()
    comm = getattr(concurrencyCfg, 'comm', None)
    shardDevices = getattr(concurrencyCfg, 'shardDevices', None) or list(dict.fromkeys(concurrencyCfg.devices))
    multiDevice = concurrencyCfg.concurrencyType == CONC_THREADS and len(shardDevices) > 1
    if (len(set(concurrencyCfg.devices)) > 1 or multiDevice) and comm is not None:
        raise PyShepSegTilingError('concurrencyCfg.comm (one process per GPU) and several devices '
            'in one process do not mix: give every process one device')
    if concurrencyCfg.concurrencyType not in (CONC_NONE, CONC_THREADS):
        if concurrencyCfg.concurrencyType in (CONC_FARGATE, CONC_SUBPROC):
            raise PyShepSegTilingError("concurrencyType {} is not part of the B200 build; use "
                "CONC_NONE or CONC_THREADS".format(concurrencyCfg.concurrencyType))
        raise ValueError("Unknown concurrencyType '{}'".format(concurrencyCfg.concurrencyType))
    if (overlapSize % 2) != 0:
        raise PyShepSegTilingError("Overlap size must be an even number")
    if not isinstance(outfile, rasterfile.RasterSink) and not rasterfile.driverAvailable(outputDriver):
        raise PyShepSegTilingError("This build does not support driver '{}'".format(outputDriver))

    timings = timinghooks.Timers()
    result = TiledSegmentationResult()
    with timings.interval('walltime'):
        try:
            src = rasterfile.openRaster(infile)
        except rasterfile.RasterError as e:
            raise PyShepSegTilingError(str(e))
        if bandNumbers is None:
            bandNumbers = range(1, src.count + 1)
        if multiDevice and isinstance(src, DeviceRaster):
            raise PyShepSegTilingError('a DeviceRaster lives on one GPU; segment it with one device')
        # one process per GPU (torchrun): concurrencyCfg.comm is a distributed.TorchComm, `src` is
        # this rank's row band of the raster and `outfile` the sink of this rank's windows
        sharded = comm is not None and comm.world > 1
        fullYsize = getattr(src, 'fullYsize', src.ysize)
        fullXsize = getattr(src, 'fullXsize', src.xsize)
        if kmeansObj is None:
            if sharded:
                raise PyShepSegTilingError("a sharded run needs kmeansObj (fit on one rank, "
                    "broadcast the centres)")
            with timings.interval('spectralclusters'):
                (kmeansObj, subsamplePcnt, imgNullVal) = fitSpectralClustersWholeFile(src,
                    bandNumbers, numClusters, subsamplePcnt, imgNullVal, fixedKMeansInit)
        elif imgNullVal is None:
            imgNullVal = getImgNullValue(src, bandNumbers)
        tileInfo = getTilesForFile((fullXsize, fullYsize), tileSize, overlapSize)
        if verbose:
            print("Found {} tiles, with {} rows and {} cols".format(tileInfo.getNumTiles(),
                tileInfo.nrows, tileInfo.ncols))
        msd = shepseg.autoMaxSpectralDiff(kmeansObj, maxSpectralDiff, spectDistPcntile)
        try:
            sink = rasterfile.createRaster(outfile, fullXsize, fullYsize, outputDriver,
                creationOptions, source=src)
        except rasterfile.RasterError as e:
            raise PyShepSegTilingError(str(e))
        sink.setMetadataItem('LAYER_TYPE', 'thematic')
        sink.setNoData(shepseg.SEGNULLVAL)
        args = (src, bandNumbers, tileInfo, overlapSize, shepseg._centres(kmeansObj), imgNullVal,
            fourConnected, minSegmentSize, shepseg.spectralThreshold(msd), simpleTileRecode, concurrencyCfg,
            timings, verbose)
        seg = MultiDeviceSegmenter(shardDevices, *args) if multiDevice else TiledSegmenter(*args)
        seg.mark('run start')
        (maxSegId, hist) = seg.run(sink, comm, deferFinal=True)
        seg.mark('run done')
        if len(hist) > 0:          # (ranks other than 0 of a sharded run hold no histogram)
            if writeHistogram:
                sink.writeHistogram(hist)
            result.hasEmptySegments = checkForEmptySegments(hist, overlapSize)
            estimateStatsFromHisto(sink, hist)
        seg.finish()          # (the last window travelled while the statistics were worked out)
        seg.mark('histogram and statistics written')
        if returnGDALDS:
            result.outDs = getattr(sink, 'ds', sink)
        else:
            sink.close()
        if not isinstance(infile, rasterfile.RasterSource):
            src.close()

    result.maxSegId = maxSegId
    result.numTileRows = tileInfo.nrows
    result.numTileCols = tileInfo.ncols
    result.subsamplePcnt = subsamplePcnt
    result.maxSpectralDiff = msd
    result.kmeans = kmeansObj
    result.timings = timings
    result.stageMs = seg.stageMs
    result.gpuLaunches = seg.launches
    result.h2dBytes = seg.h2dBytes
    result.d2hBytes = seg.d2hBytes
    result.timeline = seg.timeline
    return result

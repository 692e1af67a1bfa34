"""
GPU parity of uint32 and int32 images whose values do not fit in 16 bits.

The reference takes any integer image (shepseg.py:130-249).  On 32-bit values its arithmetic
differs from the 16-bit case in three places, which the CPU oracle restates: the assignment
converts x exactly to float64, the single-pixel distance squares int64 differences that can wrap
past 2**63, and the per-segment sums add exact doubles into float32 in raster order.  Every test
here compares labels and counts bit for bit (numpy.array_equal).
"""
import numpy
import pytest

import goldenutil
from oracle import oracle
from pyshepseg_b200 import synth, rasterfile

pytestmark = pytest.mark.gpu

U32_NULL = 4294967295
I32_NULL = -2147483648


@pytest.fixture(scope='module')
def shepseg():
    from pyshepseg_b200 import shepseg as mod
    return mod


@pytest.fixture(scope='module')
def tiling():
    from pyshepseg_b200 import tiling as mod
    return mod


def same(got, want, what):
    got = numpy.asarray(got)
    want = numpy.asarray(want)
    assert got.shape == want.shape, '%s: shape %s != %s' % (what, got.shape, want.shape)
    if not numpy.array_equal(got, want):
        bad = numpy.argwhere(got != want)
        first = tuple(bad[0])
        raise AssertionError('%s: %d of %d differ; first at %s: got %s want %s' % (
            what, len(bad), got.size, first, got[first], want[first]))


def wide_image(dtype, rows, cols, bands, seed, nullFrac=0.0, nullVal=None, cell=32):
    """uint32: synth_v1 * 65537, up to 4294901758; int32: (synth_v1 - 2000) * 500000, about
    -7.5e8 .. 1e9.  With nullFrac > 0 an upper left wedge is set to nullVal in all bands."""
    if dtype == numpy.uint32:
        base = synth.synth_v1(rows, cols, bands, seed=seed, cell=cell, lo=2000.0, hi=65000.0, noise=300.0)
        img = base.astype(numpy.uint32) * numpy.uint32(65537)
    else:
        base = synth.synth_v1(rows, cols, bands, seed=seed, cell=cell)
        img = ((base.astype(numpy.int64) - 2000) * 500000).astype(numpy.int32)
    if nullFrac > 0:
        rr = numpy.arange(rows)[:, None]
        cc = numpy.arange(cols)[None, :]
        img[:, (rr + cc) < numpy.sqrt(2.0 * nullFrac * rows * cols)] = nullVal
    return img


def against_oracle(shepseg, img, km, minSeg, nullVal, four, msd, what):
    # the values do not fit 16 bits: _deviceImage keeps the 32-bit array as it is
    assert shepseg._deviceImage(img).dtype == img.dtype, what
    want = oracle.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    got = shepseg.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    same(got.segimg, want.segimg, what + ' segimg')
    assert int(got.singlePixelsEliminated) == int(want.singlePixelsEliminated), what
    assert got.smallSegmentsEliminated == want.smallSegmentsEliminated, what
    assert got.timings['numClumps'] == want.numClumps, what
    return got


# ---- the reference's own outputs, through the 32-bit kernels ------------------------------------
def golden_wide_cases():
    cases = []
    for name in goldenutil.single_tile_names():
        cases.append((name, numpy.int32))
        cases.append((name, numpy.uint32))
    return cases


@pytest.mark.parametrize('name,dtype', golden_wide_cases(),
    ids=['%s-%s' % (n, numpy.dtype(d).name) for (n, d) in golden_wide_cases()])
def test_golden_fixtures_through_32bit_kernels(shepseg, monkeypatch, name, dtype):
    """The fixtures hold 16-bit values.  Numba computes the same on a 32-bit array holding them
    (int64 differences, one float32 rounding per add), so the reference's own outputs pin the
    32-bit kernels.  _deviceImage would narrow such an array back to 16 bits: it is bypassed."""
    c = goldenutil.load(name)
    m = c['meta']
    if dtype == numpy.uint32 and int(c['img'].min()) < 0:
        pytest.skip('negative values have no uint32 form')
    img = numpy.ascontiguousarray(c['img'].astype(dtype))
    monkeypatch.setattr(shepseg, '_deviceImage', numpy.ascontiguousarray)
    km = goldenutil.Centres(c['centres'])
    four = m['fourConnected']

    same(shepseg.applySpectralClusters(km, img, m['imgNullVal']), c['clusters'], 'applySpectralClusters')

    seg = c['clumps'].copy()
    segSize = shepseg.makeSegSize(seg)
    nextId = int(c['numClumps']) + 1
    shepseg.eliminateSinglePixels(img, seg, segSize, shepseg.MINSEGID, nextId - 1, four)
    same(seg, c['seg_singles'], 'eliminateSinglePixels')

    msd = shepseg.autoMaxSpectralDiff(km, goldenutil.msd_of(c), m['spectDistPcntile'])
    seg = c['seg_singles'].copy()
    numElim = shepseg.eliminateSmallSegments(seg, img, seg.max(), m['minSegmentSize'], msd, four,
        shepseg.MINSEGID)
    assert numElim == int(c['smallSegmentsEliminated'])
    same(seg, c['seg_final'], 'eliminateSmallSegments')

    segOut = numpy.empty(img.shape[1:], dtype=numpy.uint32)
    from pyshepseg_b200 import _lib
    res = shepseg.segmentTile(_lib.default_context(), img, km.cluster_centers_, m['imgNullVal'], four,
        m['minSegmentSize'], shepseg.spectralThreshold(msd), segOut)
    same(segOut, c['seg_final'], 'segmentTile')
    assert res.numClumps == int(c['numClumps'])
    assert res.singlePixelsEliminated == int(c['singlePixelsEliminated'])
    assert res.smallSegmentsEliminated == int(c['smallSegmentsEliminated'])


# ---- wide values against the oracle ---------------------------------------------------------------
WIDE_CASES = [
    # name, dtype, (rows, cols, bands), k, minSeg, nullFrac, nullVal, four, msd
    ('u32_3b', numpy.uint32, (1000, 1000, 3), 60, 50, 0.0, None, True, 'auto'),
    ('u32_1b_8conn', numpy.uint32, (800, 900, 1), 30, 40, 0.0, None, False, 'auto'),
    ('u32_odd_4b_null0', numpy.uint32, (997, 1003, 4), 40, 30, 0.05, 0, True, 'auto'),
    ('u32_6b_nullmax_msdnone', numpy.uint32, (900, 1000, 6), 30, 100, 0.1, U32_NULL, True, None),
    ('u32_10b_msdfloat', numpy.uint32, (700, 750, 10), 60, 50, 0.0, None, False, 3.0e8),
    ('i32_3b', numpy.int32, (1000, 1000, 3), 60, 50, 0.0, None, True, 'auto'),
    ('i32_1b_nullmin', numpy.int32, (800, 900, 1), 30, 40, 0.08, I32_NULL, True, 'auto'),
    ('i32_odd_4b_8conn', numpy.int32, (997, 1003, 4), 40, 30, 0.0, None, False, 'auto'),
    ('i32_6b_null0_msdfloat', numpy.int32, (900, 1000, 6), 30, 100, 0.1, 0, True, 1.0e9),
    ('i32_10b_msdnone', numpy.int32, (700, 750, 10), 60, 50, 0.0, None, True, None),
]


@pytest.mark.parametrize('case', WIDE_CASES, ids=[c[0] for c in WIDE_CASES])
def test_wide_values_against_oracle(shepseg, case):
    (name, dtype, (r, c, b), k, minSeg, nullFrac, nullVal, four, msd) = case
    img = wide_image(dtype, r, c, b, seed=len(name), nullFrac=nullFrac, nullVal=nullVal)
    km = goldenutil.Centres(synth.diagonal_centres(img, k, nullVal))
    against_oracle(shepseg, img, km, minSeg, nullVal, four, msd, name)


# ---- the int64 wrap of the single-pixel distance ------------------------------------------------
def wrap_image(bands):
    """Single pixels on the last row of an upper region, where the squared distance to the
    neighbour below passes 2**63 and wraps negative.  1 band: 0 above 4.2e9 and beside 1e9;
    3 bands of int32: -9e8 above 9e8 and beside -6e8 (differences of 1.8e9 per band)."""
    (rows, cols, row) = (48, 64, 20)
    rng = numpy.random.default_rng(bands)
    if bands == 1:
        (dtype, near, far, single) = (numpy.uint32, 1000000000, 4200000000, 0)
    else:
        (dtype, near, far, single) = (numpy.int32, -600000000, 900000000, -900000000)
    img = numpy.empty((bands, rows, cols), dtype=dtype)
    img[:, :row, :] = near
    img[:, row:, :] = far
    img += rng.integers(0, 1000, img.shape).astype(dtype)
    singles = [(row - 1, j) for j in range(3, cols - 3, 6)]
    for (i, j) in singles:
        img[:, i, j] = single
    centres = numpy.array([[near] * bands, [far] * bands, [single] * bands], dtype=numpy.float64)
    return (img, goldenutil.Centres(centres), singles)


def nearest_in_scan_order(img, i, j, wrap):
    """findNearestNeighbourPixel's choice (shepseg.py:677-736), 4-connected, among neighbours
    that all belong to large segments; Python integers, wrapped to int64 or not.  As in the
    reference, a negative best distance counts as none yet, so the wrapped distance wins only
    as the last neighbour in scan order (the one below)."""
    (minD, best) = (-1, None)
    for ii in (i - 1, i, i + 1):
        for jj in (j - 1, j, j + 1):
            if (ii, jj) == (i, j) or (ii != i and jj != j):
                continue
            d = sum((int(img[b, i, j]) - int(img[b, ii, jj])) ** 2 for b in range(img.shape[0]))
            if wrap:
                d = (d + 2 ** 63) % 2 ** 64 - 2 ** 63
            if minD < 0 or d < minD:
                (minD, best) = (d, (ii, jj))
    return best


@pytest.mark.parametrize('bands', [1, 3])
def test_single_pixel_distance_wraps_like_int64(shepseg, bands):
    (img, km, singles) = wrap_image(bands)
    for (i, j) in singles:
        assert nearest_in_scan_order(img, i, j, True) == (i + 1, j)
        assert nearest_in_scan_order(img, i, j, False) != (i + 1, j), 'the case does not test the wrap'
    clusters = oracle.applySpectralClusters(km, img, None)
    (seg, nextId) = oracle.clump(clusters, 0, True, 1)
    segSize = oracle.makeSegSize(seg)
    assert all(segSize[seg[i, j]] == 1 for (i, j) in singles)
    (refSeg, refSize) = (seg.copy(), segSize.copy())
    oracle.eliminateSinglePixels(img, refSeg, refSize, 1, nextId - 1, True)
    shepseg.eliminateSinglePixels(img, seg, segSize, shepseg.MINSEGID, nextId - 1, True)
    same(seg, refSeg, 'eliminateSinglePixels')
    same(segSize, refSize, 'eliminateSinglePixels segSize')
    for (i, j) in singles:
        assert seg[i, j] == seg[i + 1, j]
    against_oracle(shepseg, img, km, 10, None, True, 'auto', 'wrap %d bands' % bands)


# ---- assignment ties at large magnitude ------------------------------------------------------------
@pytest.mark.parametrize('dtype', [numpy.uint32, numpy.int32])
@pytest.mark.parametrize('k', [2, 17, 64])
def test_assignment_ties_at_large_magnitude(shepseg, dtype, k):
    """Integer centres and pixels exactly half way between two of them (and two identical
    centres): the float64 first-minimum argmin decides, as in the reference."""
    rng = numpy.random.default_rng(k)
    info = numpy.iinfo(dtype)
    nB = 3
    (rows, cols) = (128, 256)
    lo = int(info.min + (int(info.max) - int(info.min)) * 0.02)
    hi = int(info.max - (int(info.max) - int(info.min)) * 0.02)
    centres = rng.integers(lo, hi, (k, nB)).astype(numpy.float64)
    if k > 2:
        centres[1] = centres[0]
    img = rng.integers(lo, hi, (nB, rows, cols)).astype(dtype)
    for r in range(rows // 2):
        (a, b) = (rng.integers(0, k), rng.integers(0, k))
        mid = (centres[a].astype(numpy.int64) + centres[b].astype(numpy.int64)) // 2
        img[:, r, :] = (mid[:, None] + rng.integers(-1, 2, (nB, cols))).astype(dtype)
    img[:, rows - 1, :8] = info.min
    img[:, rows - 1, 8:16] = info.max
    km = goldenutil.Centres(centres)
    for nullVal in (None, int(img[0, 5, 5]), int(info.max)):
        want = oracle.applySpectralClusters(km, img, nullVal)
        got = shepseg.applySpectralClusters(km, img, nullVal)
        same(got, want, 'assignment (null %s)' % nullVal)


def test_null_value_near_the_top_of_uint32(shepseg):
    """4294967295 and 4294967200 are the same float32: only the first is null"""
    img = numpy.full((2, 16, 16), 4294967200, dtype=numpy.uint32)
    img[:, ::2, :] = U32_NULL
    img[1, 1, 1] = U32_NULL          # one band null is enough
    km = goldenutil.Centres(numpy.array([[1.0e9, 1.0e9], [4.0e9, 4.0e9]]))
    got = shepseg.applySpectralClusters(km, img, U32_NULL)
    same(got, oracle.applySpectralClusters(km, img, U32_NULL), 'nodata 4294967295')
    assert (got[::2] == 0).all() and got[1, 1] == 0 and (got[1, 2:] == 2).all()


# ---- stage functions --------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype,nullVal', [(numpy.uint32, U32_NULL), (numpy.int32, I32_NULL)])
def test_stage_functions(shepseg, dtype, nullVal):
    img = wide_image(dtype, 600, 700, 4, seed=21, nullFrac=0.05, nullVal=nullVal)
    km = goldenutil.Centres(synth.diagonal_centres(img, 40, nullVal))
    four = dtype == numpy.uint32

    clusters = shepseg.applySpectralClusters(km, img, nullVal)
    same(clusters, oracle.applySpectralClusters(km, img, nullVal), 'applySpectralClusters')

    (seg, nextId) = oracle.clump(clusters, 0, four, 1)
    segSize = oracle.makeSegSize(seg)
    (refSeg, refSize) = (seg.copy(), segSize.copy())
    oracle.eliminateSinglePixels(img, refSeg, refSize, 1, nextId - 1, four)
    shepseg.eliminateSinglePixels(img, seg, segSize, shepseg.MINSEGID, nextId - 1, four)
    same(seg, refSeg, 'eliminateSinglePixels seg')
    same(segSize, refSize, 'eliminateSinglePixels segSize')

    msd = shepseg.autoMaxSpectralDiff(km, 'auto', 50)
    ref = refSeg.copy()
    want = oracle.eliminateSmallSegments(ref, img, ref.max(), 40, msd, four, 1)
    got = shepseg.eliminateSmallSegments(seg, img, seg.max(), 40, msd, four, shepseg.MINSEGID)
    assert got == want
    same(seg, ref, 'eliminateSmallSegments')


# ---- which kernels an array goes to ---------------------------------------------------------------
def test_dtype_routing(shepseg):
    base = synth.synth_v1(300, 400, 3, seed=31)
    km = goldenutil.Centres(synth.diagonal_centres(base, 20))
    today = shepseg.doShepherdSegmentation(base, minSegmentSize=20, kmeansObj=km)
    # 16-bit values in wider arrays go to the 16-bit kernels, as before
    for dtype in (numpy.int32, numpy.uint32, numpy.int64):
        a = base.astype(dtype)
        assert shepseg._deviceImage(a).dtype == numpy.uint16
        res = shepseg.doShepherdSegmentation(a, minSegmentSize=20, kmeansObj=km)
        same(res.segimg, today.segimg, numpy.dtype(dtype).name)
    neg = (base.astype(numpy.int64) - 2000)
    assert shepseg._deviceImage(neg).dtype == numpy.int16
    # int64 and uint64 arrays with values in 32-bit range go to the 32-bit kernels
    for (dtype, img, want) in (
            (numpy.int64, wide_image(numpy.uint32, 300, 400, 3, seed=32), numpy.uint32),
            (numpy.uint64, wide_image(numpy.uint32, 300, 400, 3, seed=33), numpy.uint32),
            (numpy.int64, wide_image(numpy.int32, 300, 400, 3, seed=34), numpy.int32)):
        wide = img.astype(dtype)
        assert shepseg._deviceImage(wide).dtype == want
        km = goldenutil.Centres(synth.diagonal_centres(img, 20))
        res = shepseg.doShepherdSegmentation(wide, minSegmentSize=20, kmeansObj=km)
        ref = oracle.doShepherdSegmentation(img, minSegmentSize=20, kmeansObj=km)
        same(res.segimg, ref.segimg, '%s holding %s values' % (numpy.dtype(dtype).name, numpy.dtype(want).name))
    # beyond 32 bits: still refused
    for a in (numpy.array([[[0, 2 ** 32]]], dtype=numpy.int64),
              numpy.array([[[-2 ** 31 - 1, 5]]], dtype=numpy.int64),
              numpy.array([[[1, 2 ** 32 + 7]]], dtype=numpy.uint64)):
        with pytest.raises(NotImplementedError):
            shepseg._deviceImage(a)
        with pytest.raises(NotImplementedError):
            shepseg.applySpectralClusters(goldenutil.Centres(numpy.zeros((2, 1))), a, None)


# ---- tiled ------------------------------------------------------------------------------------------
def oracle_tiled(img, km, tileSize, overlap, minSeg, nullVal, four, simple=False):
    (nB, nR, nC) = img.shape
    ti = oracle.getTilesForFile(nC, nR, tileSize, overlap)
    segs = {}
    for ((col, row), (x, y, xs, ys)) in ti.tiles.items():
        sub = numpy.ascontiguousarray(img[:, y:y + ys, x:x + xs])
        segs[(col, row)] = oracle.doShepherdSegmentation(sub, minSegmentSize=minSeg, imgNullVal=nullVal,
            fourConnected=four, kmeansObj=km).segimg
    return oracle.stitchTiles(segs, ti, nC, nR, overlap, simpleTileRecode=simple)


TILED_CASES = [
    # name, dtype, (rows, cols, bands), tileSize, overlap, k, minSeg, nullFrac, nullVal, four, simple, workers
    ('u32_nullmax', numpy.uint32, (1500, 1700, 3), 400, 100, 30, 30, 0.1, U32_NULL, True, False, 0),
    ('u32_nullmax_2workers', numpy.uint32, (1500, 1700, 3), 400, 100, 30, 30, 0.1, U32_NULL, True, False, 2),
    ('i32_nullmin_8conn', numpy.int32, (1300, 1200, 4), 300, 60, 25, 25, 0.1, I32_NULL, False, False, 0),
    ('i32_null0_2workers', numpy.int32, (1300, 1200, 4), 300, 60, 25, 25, 0.1, 0, True, False, 2),
    ('u32_simple_recode', numpy.uint32, (1100, 1000, 3), 400, 100, 20, 30, 0.0, None, True, True, 0),
]


@pytest.mark.parametrize('case', TILED_CASES, ids=[c[0] for c in TILED_CASES])
def test_tiled_wide_values(tiling, case):
    (name, dtype, (r, c, b), tileSize, overlap, k, minSeg, nullFrac, nullVal, four, simple, workers) = case
    img = wide_image(dtype, r, c, b, seed=len(name) + 50, nullFrac=nullFrac, nullVal=nullVal)
    km = goldenutil.Centres(synth.diagonal_centres(img, k, nullVal))
    (mosaic, maxSegId, hist) = oracle_tiled(img, km, tileSize, overlap, minSeg, nullVal, four, simple)
    cfg = tiling.SegmentationConcurrencyConfig(concurrencyType=tiling.CONC_THREADS, numWorkers=workers) \
        if workers else None
    res = tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img, nodata=nullVal), None,
        tileSize=tileSize, overlapSize=overlap, minSegmentSize=minSeg, numClusters=k, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, simpleTileRecode=simple, outputDriver='MEM', returnGDALDS=True,
        concurrencyCfg=cfg)
    same(res.outDs.array, mosaic, name + ' mosaic')
    assert int(res.maxSegId) == maxSegId
    same(res.outDs.hist, hist, name + ' histogram')

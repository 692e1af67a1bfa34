"""
GPU parity of images of 17 to 64 bands.

Above 16 bands the assignment runs k_assign_many (centres in shared-memory tiles, band count known
at run time), the small-segment merge runs the 64-band record class of merge.cu (records
{size, list offset}, means in an array of their own) and the device k-means fit runs
k_lloyd_step<64>.  Every comparison of labels and counts is bit for bit (numpy.array_equal).
"""
import ctypes

import numpy
import pytest

import goldenutil
from oracle import oracle
from pyshepseg_b200 import synth, rasterfile

pytestmark = pytest.mark.gpu

U32_NULL = 4294967295


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


def image(dtype, rows, cols, bands, seed, nullFrac=0.0, nullVal=None, big=False):
    """synth_v1 in the value range of dtype: uint8 20..240; uint16 500..4000, or with big=True
    30000..65000 (float32 band sums of segments above 2^24 / 65000 pixels are inexact); int16 shifted
    by -2000; uint32 x 65537; int32 (x - 2000) x 500000.  With nullFrac > 0 an upper left wedge is
    nullVal in all bands."""
    if dtype == numpy.uint8:
        img = synth.synth_v1(rows, cols, bands, seed=seed, lo=20.0, hi=240.0, noise=6.0).astype(numpy.uint8)
    elif dtype == numpy.uint16 and big:
        img = synth.synth_v1(rows, cols, bands, seed=seed, lo=30000.0, hi=65000.0, noise=300.0)
    elif dtype == numpy.uint16:
        img = synth.synth_v1(rows, cols, bands, seed=seed)
    elif dtype == numpy.int16:
        img = (synth.synth_v1(rows, cols, bands, seed=seed).astype(numpy.int32) - 2000).astype(numpy.int16)
    elif dtype == numpy.uint32:
        base = synth.synth_v1(rows, cols, bands, seed=seed, lo=2000.0, hi=65000.0, noise=300.0)
        img = base.astype(numpy.uint32) * numpy.uint32(65537)
    else:
        base = synth.synth_v1(rows, cols, bands, seed=seed)
        img = ((base.astype(numpy.int64) - 2000) * 500000).astype(numpy.int32)
    if nullFrac > 0:
        rr = numpy.arange(rows)[:, None]
        cc = numpy.arange(cols)[None, :]
        img[:, (rr + cc) < numpy.sqrt(2.0 * nullFrac * rows * cols)] = nullVal
    return img


def against_oracle(shepseg, img, km, minSeg, nullVal, four, msd, what):
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


# ---- the reference's own outputs, padded with all-zero bands ----------------------------------------
def golden_padded_cases():
    cases = []
    for name in goldenutil.single_tile_names():
        for bands in (17, 32, 64):
            cases.append((name, bands, None))
        for dtype in (numpy.uint32, numpy.int32):
            cases.append((name, 64, dtype))
    return cases


@pytest.mark.parametrize('name,bands,dtype', golden_padded_cases(),
    ids=['%s-%d%s' % (n, b, '' if d is None else '-' + numpy.dtype(d).name) for (n, b, d) in golden_padded_cases()])
def test_golden_fixtures_padded_with_zero_bands(shepseg, monkeypatch, name, bands, dtype):
    """Zero bands (and zero centre coordinates) add exact zeros to every sum the reference forms:
    the distances of the assignment, the int64 distances of the single pixels and the float32
    distances of the merges.  So the reference's own stage outputs hold for the padded image.
    maxSpectralDiff is resolved from the unpadded centres (numpy's pairwise sum regroups when zeros
    are added).  With imgNullVal 0 every padded pixel would be null: there only the stages after
    the clump are compared."""
    c = goldenutil.load(name)
    m = c['meta']
    src = c['img']
    if dtype is not None:
        if dtype == numpy.uint32 and int(src.min()) < 0:
            pytest.skip('negative values have no uint32 form')
        src = src.astype(dtype)
        monkeypatch.setattr(shepseg, '_deviceImage', numpy.ascontiguousarray)
    img = numpy.zeros((bands,) + src.shape[1:], dtype=src.dtype)
    img[:src.shape[0]] = src
    centres = numpy.zeros((c['centres'].shape[0], bands))
    centres[:, :src.shape[0]] = c['centres']
    km = goldenutil.Centres(centres)
    nullVal = m['imgNullVal']
    four = m['fourConnected']

    if nullVal is None or nullVal != 0:
        same(shepseg.applySpectralClusters(km, img, nullVal), c['clusters'], 'applySpectralClusters')

    seg = c['clumps'].copy()
    segSize = shepseg.makeSegSize(seg)
    shepseg.eliminateSinglePixels(img, seg, segSize, shepseg.MINSEGID, int(c['numClumps']), four)
    same(seg, c['seg_singles'], 'eliminateSinglePixels')

    msd = shepseg.autoMaxSpectralDiff(goldenutil.Centres(c['centres']), goldenutil.msd_of(c),
        m['spectDistPcntile'])
    seg = c['seg_singles'].copy()
    numElim = shepseg.eliminateSmallSegments(seg, img, seg.max(), m['minSegmentSize'], msd, four,
        shepseg.MINSEGID)
    assert numElim == int(c['smallSegmentsEliminated'])
    same(seg, c['seg_final'], 'eliminateSmallSegments')

    if nullVal is None or nullVal != 0:
        from pyshepseg_b200 import _lib
        segOut = numpy.empty(img.shape[1:], dtype=numpy.uint32)
        res = shepseg.segmentTile(_lib.default_context(), numpy.ascontiguousarray(img), centres, nullVal,
            four, m['minSegmentSize'], shepseg.spectralThreshold(msd), segOut)
        same(segOut, c['seg_final'], 'segmentTile')
        assert res.numClumps == int(c['numClumps'])
        assert res.singlePixelsEliminated == int(c['singlePixelsEliminated'])
        assert res.smallSegmentsEliminated == int(c['smallSegmentsEliminated'])


# ---- the high bands are read -------------------------------------------------------------------------
def test_band_63_alone_equals_the_one_band_run(shepseg):
    one = synth.synth_v1(400, 500, 1, seed=63)
    img = numpy.zeros((64, 400, 500), dtype=numpy.uint16)
    img[63] = one[0]
    c1 = synth.diagonal_centres(one, 40)
    c64 = numpy.zeros((40, 64))
    c64[:, 63] = c1[:, 0]
    a = shepseg.doShepherdSegmentation(one, minSegmentSize=50, kmeansObj=goldenutil.Centres(c1))
    b = shepseg.doShepherdSegmentation(img, minSegmentSize=50, kmeansObj=goldenutil.Centres(c64))
    same(b.segimg, a.segimg, 'band 63 of 64 vs 1 band')
    assert int(b.singlePixelsEliminated) == int(a.singlePixelsEliminated)
    assert b.smallSegmentsEliminated == a.smallSegmentsEliminated
    assert b.timings['numClumps'] == a.timings['numClumps']
    assert int(a.segimg.max()) > 50


def test_only_band_40_varies(shepseg):
    img = numpy.full((48, 350, 420), 1000, dtype=numpy.uint16)
    img[40] = synth.synth_v1(350, 420, 1, seed=40)[0]
    km = goldenutil.Centres(synth.diagonal_centres(img, 30))
    got = against_oracle(shepseg, img, km, 30, None, True, 'auto', 'band 40')
    assert int(got.segimg.max()) > 50


# ---- varied data against the oracle ------------------------------------------------------------------
ORACLE_CASES = [
    # name, dtype, (rows, cols, bands), k, minSeg, nullFrac, nullVal, four, msd, big
    ('u16_17b', numpy.uint16, (400, 500, 17), 60, 50, 0.0, None, True, 'auto', False),
    ('u16_20b_8conn_null', numpy.uint16, (397, 503, 20), 40, 50, 0.1, 0, False, 'auto', False),
    ('u16_32b_msdnone', numpy.uint16, (300, 400, 32), 60, 400, 0.0, None, True, None, False),
    ('u16_48b_big', numpy.uint16, (350, 360, 48), 30, 400, 0.0, None, True, 'auto', True),
    ('u16_64b_minseg2', numpy.uint16, (301, 299, 64), 60, 2, 0.05, 0, True, 'auto', False),
    ('u16_64b_8conn_big', numpy.uint16, (300, 320, 64), 20, 400, 0.0, None, False, 'auto', True),
    ('u8_32b_msdfloat', numpy.uint8, (333, 444, 32), 50, 50, 0.0, None, True, 120.0, False),
    ('u8_64b_8conn_null', numpy.uint8, (300, 300, 64), 30, 50, 0.1, 0, False, 'auto', False),
    ('i16_17b_8conn', numpy.int16, (420, 380, 17), 40, 50, 0.0, None, False, 'auto', False),
    ('i16_48b_null', numpy.int16, (300, 350, 48), 60, 400, 0.1, -2000, True, None, False),
    ('u32_20b_nullmax', numpy.uint32, (350, 400, 20), 40, 50, 0.1, U32_NULL, True, 'auto', False),
    ('u32_64b_msdfloat', numpy.uint32, (250, 301, 64), 30, 50, 0.0, None, False, 3.0e9, False),
    ('i32_32b', numpy.int32, (320, 330, 32), 60, 2, 0.0, None, True, 'auto', False),
    ('i32_64b_null0_8conn', numpy.int32, (299, 250, 64), 30, 400, 0.1, 0, False, None, False),
]


def oracle_case(case):
    (name, dtype, (r, c, b), k, minSeg, nullFrac, nullVal, four, msd, big) = case
    img = image(dtype, r, c, b, seed=len(name) + b, nullFrac=nullFrac, nullVal=nullVal, big=big)
    km = goldenutil.Centres(synth.diagonal_centres(img, k, nullVal))
    return (img, km, minSeg, nullVal, four, msd)


@pytest.mark.parametrize('case', ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_many_bands_against_oracle(shepseg, case):
    (img, km, minSeg, nullVal, four, msd) = oracle_case(case)
    got = against_oracle(shepseg, img, km, minSeg, nullVal, four, msd, case[0])
    if minSeg > 2:
        assert got.smallSegmentsEliminated > 0


PACKED_ENVS = [
    {'SSG_SMALL_REGION_MB': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '7'},
]


@pytest.mark.parametrize('env', PACKED_ENVS, ids=['arena', 'no_arena', 'arena7'])
@pytest.mark.parametrize('case', ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_many_bands_packed_lists(shepseg, monkeypatch, case, env):
    for (key, value) in env.items():
        monkeypatch.setenv(key, value)
    (img, km, minSeg, nullVal, four, msd) = oracle_case(case)
    against_oracle(shepseg, img, km, minSeg, nullVal, four, msd, case[0] + ' packed')


# ---- assignment -----------------------------------------------------------------------------------------
@pytest.mark.parametrize('k', [2, 17, 64, 300, 1024])
def test_assignment_k_at_64_bands(shepseg, k):
    """k = 300 and 1024 take several centre tiles"""
    img = image(numpy.uint16, 150, 170, 64, seed=k, nullFrac=0.05, nullVal=0)
    rng = numpy.random.default_rng(k)
    centres = synth.diagonal_centres(img, k, 0) + rng.normal(0, 30, (k, 64))
    km = goldenutil.Centres(centres)
    for nullVal in (None, 0):
        same(shepseg.applySpectralClusters(km, img, nullVal), oracle.applySpectralClusters(km, img, nullVal),
            'k=%d (null %s)' % (k, nullVal))


@pytest.mark.parametrize('dtype', [numpy.uint32, numpy.int32, numpy.uint16])
@pytest.mark.parametrize('k', [2, 17, 64, 300])
def test_assignment_near_ties(shepseg, dtype, k):
    """Integer centres, pixels half way between two of them (and two identical centres), 40 bands:
    the float64 first-minimum argmin decides, as in the reference"""
    rng = numpy.random.default_rng(k)
    info = numpy.iinfo(dtype)
    nB = 40
    (rows, cols) = (64, 128)
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
        same(shepseg.applySpectralClusters(km, img, nullVal), oracle.applySpectralClusters(km, img, nullVal),
            'assignment (null %s)' % nullVal)


def test_null_value_near_the_top_of_uint32(shepseg):
    """4294967295 and 4294967200 are the same float32: only the first is null"""
    img = numpy.full((33, 16, 16), 4294967200, dtype=numpy.uint32)
    img[:, ::2, :] = U32_NULL
    img[32, 1, 1] = U32_NULL          # one band null is enough
    km = goldenutil.Centres(numpy.array([[1.0e9] * 33, [4.0e9] * 33]))
    got = shepseg.applySpectralClusters(km, img, U32_NULL)
    same(got, oracle.applySpectralClusters(km, img, U32_NULL), 'nodata 4294967295')
    assert (got[::2] == 0).all() and got[1, 1] == 0 and (got[1, 2:] == 2).all()


# ---- stage functions ------------------------------------------------------------------------------------
@pytest.mark.parametrize('dtype,nullVal', [(numpy.uint16, 0), (numpy.int32, 0)])
def test_stage_functions_32_bands(shepseg, dtype, nullVal):
    img = image(dtype, 400, 450, 32, seed=32, nullFrac=0.05, nullVal=nullVal)
    km = goldenutil.Centres(synth.diagonal_centres(img, 40, nullVal))
    four = dtype == numpy.uint16

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


# ---- tiled ------------------------------------------------------------------------------------------------
def oracle_tiled(img, km, tileSize, overlap, minSeg, nullVal, four):
    (nB, nR, nC) = img.shape
    ti = oracle.getTilesForFile(nC, nR, tileSize, overlap)
    segs = {}
    for ((col, row), (x, y, xs, ys)) in ti.tiles.items():
        sub = numpy.ascontiguousarray(img[:, y:y + ys, x:x + xs])
        segs[(col, row)] = oracle.doShepherdSegmentation(sub, minSegmentSize=minSeg, imgNullVal=nullVal,
            fourConnected=four, kmeansObj=km).segimg
    return oracle.stitchTiles(segs, ti, nC, nR, overlap)


@pytest.mark.parametrize('workers', [0, 2])
def test_tiled_24_bands(tiling, workers):
    img = image(numpy.uint16, 1100, 1000, 24, seed=24, nullFrac=0.1, nullVal=0)
    km = goldenutil.Centres(synth.diagonal_centres(img, 30, 0))
    (mosaic, maxSegId, hist) = oracle_tiled(img, km, 400, 100, 30, 0, True)
    cfg = tiling.SegmentationConcurrencyConfig(concurrencyType=tiling.CONC_THREADS, numWorkers=workers) \
        if workers else None
    res = tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img, nodata=0), None,
        tileSize=400, overlapSize=100, minSegmentSize=30, numClusters=30, imgNullVal=0,
        kmeansObj=km, outputDriver='MEM', returnGDALDS=True, concurrencyCfg=cfg)
    same(res.outDs.array, mosaic, 'mosaic')
    assert int(res.maxSegId) == maxSegId
    same(res.outDs.hist, hist, 'histogram')


# ---- the device k-means fit --------------------------------------------------------------------------------
@pytest.mark.parametrize('bands,k', [(32, 30), (64, 20)])
def test_lloyd_iterations_equal_sklearn(shepseg, bands, k):
    """As test_gpu_parity's check at up to 10 bands: from the same initial centres, after the same
    number of iterations, the centres agree with scikit-learn's to 1e-9 of the data range"""
    import warnings
    from sklearn.cluster import KMeans
    img = synth.synth_v1(300, 350, bands, seed=bands)
    sample = numpy.moveaxis(img, 0, -1).reshape(-1, bands)[::7]
    init = shepseg.diagonalClusterCentres(sample, k)
    span = float(img.max()) - float(img.min())
    for iters in (1, 5, 20):
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ref = KMeans(n_clusters=k, n_init=1, init=init, max_iter=iters, tol=0.0).fit(sample)
        got = shepseg._fitOnDevice(sample, k, True, maxIter=iters, tol=0.0)
        err = numpy.abs(got.cluster_centers_ - ref.cluster_centers_).max()
        assert err <= 1e-9 * span, '%d iterations: centres differ by %g (data range %g)' % (iters, err, span)
        assert abs(got.inertia_ - ref.inertia_) <= 1e-9 * ref.inertia_


def test_lloyd_fit_too_many_centres_for_shared_memory(shepseg):
    """64 bands: (k * 64 + k) float64 no longer fit 200 KB above 393 centres"""
    img = synth.synth_v1(100, 120, 64, seed=3)
    got = shepseg.fitSpectralClusters(img, 390, 100, None, True, backend='gpu')
    assert got.cluster_centers_.shape == (390, 64)
    with pytest.raises(shepseg.ShepsegB200Error, match='shared memory'):
        shepseg.fitSpectralClusters(img, 400, 100, None, True, backend='gpu')


# ---- the limit -----------------------------------------------------------------------------------------------
def test_65_bands_are_refused_at_every_layer(shepseg, tiling):
    from pyshepseg_b200 import _lib
    img = synth.synth_v1(20, 30, 65, seed=65)
    centres = numpy.ascontiguousarray(synth.diagonal_centres(img, 4))
    km = goldenutil.Centres(centres)
    with pytest.raises(NotImplementedError):
        shepseg.doShepherdSegmentation(img, minSegmentSize=5, kmeansObj=km)
    with pytest.raises(NotImplementedError):
        shepseg.applySpectralClusters(km, img, None)
    with pytest.raises(tiling.PyShepSegTilingError):
        tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img), None, tileSize=16, overlapSize=4,
            minSegmentSize=5, kmeansObj=km, outputDriver='MEM', returnGDALDS=True)

    ctx = _lib.Context(0)
    try:
        out = numpy.empty((20, 30), dtype=numpy.int32)
        with pytest.raises(_lib.ShepsegB200Error, match=r'\(code 1\)'):
            ctx.call('ssg_assign', _lib.ptr(img), _lib.SSG_U16, 65, 20, 30, _lib.ptr(centres), 4, 0, 0.0,
                _lib.ptr(out))
        prm = shepseg.makeTileParams(img.dtype, 65, 20, 30, centres, None, True, 5, 1.0e9)
        res = _lib.TileResult()
        seg = numpy.empty((20, 30), dtype=numpy.uint32)
        with pytest.raises(_lib.ShepsegB200Error, match=r'\(code 1\)'):
            ctx.call('ssg_segment_tile', _lib.ptr(img), ctypes.byref(prm), _lib.ptr(seg), ctypes.byref(res))
        with pytest.raises(_lib.ShepsegB200Error, match=r'\(code 1\)'):
            ctx.call('ssg_ctx_reserve', 600, 65, _lib.SSG_U16, 0)
        X = numpy.ascontiguousarray(numpy.moveaxis(img, 0, -1).reshape(-1, 65), dtype=numpy.float64)
        with pytest.raises(_lib.ShepsegB200Error, match=r'\(code 1\)'):
            ctx.call('ssg_kmeans_begin', _lib.ptr(X), X.shape[0], 65, _lib.ptr(centres), 4)
        # 64 is the limit itself
        ctx.call('ssg_ctx_reserve', 600, 64, _lib.SSG_U16, 0)
        got = shepseg.applySpectralClusters(goldenutil.Centres(centres[:, :64]), img[:64], None, context=ctx)
        same(got, oracle.applySpectralClusters(goldenutil.Centres(centres[:, :64]), img[:64], None), '64 bands')
    finally:
        ctx.close()

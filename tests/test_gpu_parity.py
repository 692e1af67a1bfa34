"""
GPU parity tests: the CUDA path (through the C ABI, via pyshepseg_b200.shepseg) against

  * the golden fixtures produced by the unmodified reference (tests/golden), stage by stage
    and end to end, bit for bit;
  * the CPU oracle on seeded inputs at sizes it finishes in seconds;
  * edge cases the reference's semantics define: empty / all-null / single-pixel rasters,
    a lone null pixel, odd sizes (unaligned rows), the clump-size cap.

Everything here is integer / index work: the bar is numpy.array_equal.
"""
import os

import numpy
import pytest

import goldenutil
from oracle import oracle
from pyshepseg_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def shepseg():
    from pyshepseg_b200 import shepseg as mod
    return mod


def same(got, want, what):
    """array_equal with a useful message"""
    got = numpy.asarray(got)
    want = numpy.asarray(want)
    assert got.shape == want.shape, '%s: shape %s != %s' % (what, got.shape, want.shape)
    if not numpy.array_equal(got, want):
        bad = numpy.argwhere(got != want)
        first = tuple(bad[0])
        raise AssertionError('%s: %d of %d differ; first at %s: got %s want %s; maxes %s / %s' % (
            what, len(bad), got.size, first, got[first], want[first], got.max(), want.max()))


@pytest.mark.parametrize('name', goldenutil.single_tile_names())
def test_golden_stages(shepseg, name):
    c = goldenutil.load(name)
    m = c['meta']
    img = c['img']
    km = goldenutil.Centres(c['centres'])
    four = m['fourConnected']

    clusters = shepseg.applySpectralClusters(km, img, m['imgNullVal'])
    assert clusters.dtype == numpy.int32
    same(clusters, c['clusters'], 'applySpectralClusters')

    (seg, nextId) = shepseg.clump(c['clusters'], shepseg.SEGNULLVAL, fourConnected=four,
        clumpId=shepseg.MINSEGID)
    assert seg.dtype == numpy.uint32
    assert nextId - 1 == int(c['numClumps'])
    same(seg, c['clumps'], 'clump')

    seg = c['clumps'].copy()
    segSize = shepseg.makeSegSize(seg)
    same(segSize, oracle.makeSegSize(seg), 'makeSegSize')
    refSize = segSize.copy()
    refSeg = seg.copy()
    oracle.eliminateSinglePixels(img, refSeg, refSize, 1, nextId - 1, four)
    shepseg.eliminateSinglePixels(img, seg, segSize, shepseg.MINSEGID, nextId - 1, four)
    same(seg, c['seg_singles'], 'eliminateSinglePixels seg')
    same(segSize, refSize, 'eliminateSinglePixels segSize')

    msd = shepseg.autoMaxSpectralDiff(km, goldenutil.msd_of(c), m['spectDistPcntile'])
    assert float(msd) == float(c['msd_value'])
    assert isinstance(msd, numpy.float32) == bool(c['msd_is_f32'])

    seg = c['seg_singles'].copy()
    numElim = shepseg.eliminateSmallSegments(seg, img, seg.max(), m['minSegmentSize'], msd,
        four, shepseg.MINSEGID)
    assert numElim == int(c['smallSegmentsEliminated'])
    same(seg, c['seg_final'], 'eliminateSmallSegments')


@pytest.mark.parametrize('name', goldenutil.single_tile_names())
def test_golden_end_to_end(shepseg, name):
    c = goldenutil.load(name)
    m = c['meta']
    res = shepseg.doShepherdSegmentation(c['img'], minSegmentSize=m['minSegmentSize'],
        maxSpectralDiff=goldenutil.msd_of(c), imgNullVal=m['imgNullVal'],
        fourConnected=m['fourConnected'], kmeansObj=goldenutil.Centres(c['centres']),
        spectDistPcntile=m['spectDistPcntile'])
    assert res.segimg.dtype == numpy.uint32 and res.segimg.flags.c_contiguous
    same(res.segimg, c['seg_final'], 'segimg')
    assert int(res.singlePixelsEliminated) == int(c['singlePixelsEliminated'])
    assert isinstance(res.singlePixelsEliminated, numpy.uint32)
    assert res.smallSegmentsEliminated == int(c['smallSegmentsEliminated'])
    assert res.timings['numClumps'] == int(c['numClumps'])
    assert float(res.maxSpectralDiff) == float(c['msd_value'])


def test_clump_cap_boundaries(shepseg):
    """shepseg.py:481,502 -- strips around the cap and flat blocks far above it"""
    g = numpy.load(os.path.join(goldenutil.GOLDEN_DIR, 'clump_only.npz'))
    for key in g.files:
        if key.startswith('strip_'):
            (_, n, four) = key.split('_')
            img = numpy.ones((1, int(n)), dtype=numpy.int32)
            (lab, nxt) = shepseg.clump(img, 0, bool(int(four)), 1)
            got = numpy.array([nxt] + list(numpy.bincount(lab.ravel())[1:]))
            same(got, g[key], key)
        elif key.startswith('flat_'):
            (_, shape, four) = key.split('_')
            (r, cc) = shape.split('x')
            img = numpy.full((int(r), int(cc)), 3, dtype=numpy.int32)
            (lab, nxt) = shepseg.clump(img, 0, bool(int(four)), 1)
            same(lab, g[key], key)
    for four in (0, 1):
        (lab, nxt) = shepseg.clump(g['mixed_img'], 0, bool(four), 7)
        same(lab, g['mixed_%d' % four], 'mixed_%d' % four)
        assert nxt == int(g['mixed_%d_next' % four])


def _against_oracle(shepseg, img, k, minSeg, nullVal, four, msd='auto', what=''):
    centres = synth.diagonal_centres(img, k, nullVal)
    km = goldenutil.Centres(centres)
    want = oracle.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    got = shepseg.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    same(got.segimg, want.segimg, what + ' segimg')
    assert int(got.singlePixelsEliminated) == int(want.singlePixelsEliminated), what
    assert got.smallSegmentsEliminated == want.smallSegmentsEliminated, what
    assert got.timings['numClumps'] == want.numClumps, what
    return got


ORACLE_CASES = [
    # name, (rows, cols, bands), k, minSeg, nullFrac, four, msd
    ('C1_1000x1000x3', (1000, 1000, 3), 60, 50, 0.0, True, 'auto'),
    ('C1_8conn', (1000, 1000, 3), 60, 50, 0.0, False, 'auto'),
    ('odd_997x1003x4', (997, 1003, 4), 40, 30, 0.05, True, 'auto'),
    ('six_band_null_k30', (1200, 1100, 6), 30, 100, 0.1, True, 'auto'),
    ('ten_band', (900, 950, 10), 60, 50, 0.0, True, 'auto'),
    ('msd_none_8conn', (800, 800, 4), 60, 50, 0.0, False, None),
    ('msd_small_float', (800, 800, 4), 60, 50, 0.0, True, 150.0),
    ('thin_3x5000', (3, 5000, 3), 20, 10, 0.0, True, 'auto'),
    ('tall_5000x2', (5000, 2, 3), 20, 10, 0.0, False, 'auto'),
]


@pytest.mark.parametrize('case', ORACLE_CASES, ids=[c[0] for c in ORACLE_CASES])
def test_against_oracle(shepseg, case):
    (name, (r, c, b), k, minSeg, nullFrac, four, msd) = case
    img = synth.synth_v1(r, c, b, seed=len(name), nullFrac=nullFrac, nullVal=0)
    _against_oracle(shepseg, img, k, minSeg, 0 if nullFrac > 0 else None, four, msd, name)


BASELINE_CASES = [
    # BASELINE.json configs at sizes the oracle does in ~10 s: C3 (Landsat-like, 6 bands, nodata
    # wedge, k=30, minSegmentSize=100, fixed centres) and C5 (10-band stack, 'auto', minSeg 50)
    ('C3_landsat_like_6band_null', (5000, 4400, 6), 30, 100, 0.10, True, 'auto'),
    ('C5_ten_band_auto', (3600, 3000, 10), 60, 50, 0.0, True, 'auto'),
]


@pytest.mark.parametrize('case', BASELINE_CASES, ids=[c[0] for c in BASELINE_CASES])
def test_baseline_configs_against_oracle(shepseg, case):
    (name, (r, c, b), k, minSeg, nullFrac, four, msd) = case
    img = synth.synth_tiled(r, c, b, seed=len(name))
    if nullFrac > 0:
        rr = numpy.arange(r)[:, None]
        cc = numpy.arange(c)[None, :]
        img[:, (rr + cc) < numpy.sqrt(2.0 * nullFrac * r * c)] = 0
    _against_oracle(shepseg, img, k, minSeg, 0 if nullFrac > 0 else None, four, msd, name)


def test_flat_cells_over_cap(shepseg):
    """Voronoi cells of constant colour, like the reference's own runtests image
    (cmdline/runtests.py:145-265): every region is far over MAX_CLUMP_SIZE."""
    img = synth.synth_flat(1100, 1300, 3, numCells=12, seed=3, border=7, nullVal=65535)
    for four in (True, False):
        got = _against_oracle(shepseg, img, 12, 50, 65535, four, 'auto', 'flat four=%s' % four)
        assert got.timings['numOversized'] > 0


def test_quantised_ties(shepseg):
    """exact float32 distance ties between different neighbours (SURVEY probe A19)"""
    img = (synth.synth_v1(900, 900, 3, seed=8) // 64 * 64).astype(numpy.uint16)
    _against_oracle(shepseg, img, 30, 50, None, True, 'auto', 'quantised')


def test_big_values_inexact_sums(shepseg):
    """band sums far above 2**24: float32 accumulation order matters (SURVEY probe A3)"""
    img = synth.synth_v1(700, 800, 3, seed=9, lo=30000, hi=62000, noise=300, cell=64)
    _against_oracle(shepseg, img, 8, 200, None, True, None, 'bigvalues')


@pytest.mark.parametrize('env', [
    {'SSG_SMALL_REGION_MB': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '7'},
], ids=['packed_lists_arena', 'packed_lists_all_chained', 'packed_lists_arena_runs_out'])
def test_small_segment_list_storage_and_grid(shepseg, env):
    """pixel lists normally live in per-segment regions; when that would take too much memory
    they are packed, merged lists rewritten into an arena while it lasts and chained after that.
    None of these ways of storing the lists may change a label."""
    img = synth.synth_v1(600, 700, 4, seed=10)
    km = goldenutil.Centres(synth.diagonal_centres(img, 40))
    want = oracle.doShepherdSegmentation(img, minSegmentSize=40, kmeansObj=km)
    os.environ.update(env)
    try:
        got = shepseg.doShepherdSegmentation(img, minSegmentSize=40, kmeansObj=km)
    finally:
        for k in env:
            del os.environ[k]
    same(got.segimg, want.segimg, str(env))
    assert got.smallSegmentsEliminated == want.smallSegmentsEliminated


def test_edge_rasters(shepseg):
    km = goldenutil.Centres(numpy.array([[100.0, 100, 100], [900, 900, 900], [2000, 2100, 2200]]))
    # all null
    img = numpy.zeros((3, 40, 50), dtype=numpy.uint16)
    res = shepseg.doShepherdSegmentation(img, minSegmentSize=10, imgNullVal=0, kmeansObj=km)
    assert res.segimg.shape == (40, 50) and not res.segimg.any()
    assert int(res.singlePixelsEliminated) == 0 and res.smallSegmentsEliminated == 0
    # 1 x 1
    img = numpy.full((3, 1, 1), 500, dtype=numpy.uint16)
    res = shepseg.doShepherdSegmentation(img, minSegmentSize=10, kmeansObj=km)
    want = oracle.doShepherdSegmentation(img, minSegmentSize=10, kmeansObj=km)
    same(res.segimg, want.segimg, '1x1')
    # one row, one column
    for shape in ((1, 300), (300, 1)):
        img = synth.synth_v1(shape[0], shape[1], 3, seed=4, cell=8)
        want = oracle.doShepherdSegmentation(img, minSegmentSize=5, kmeansObj=km)
        res = shepseg.doShepherdSegmentation(img, minSegmentSize=5, kmeansObj=km)
        same(res.segimg, want.segimg, str(shape))
    # repeated calls give the same answer (determinism of the atomics-based kernels)
    img = synth.synth_v1(333, 444, 3, seed=6)
    a = shepseg.doShepherdSegmentation(img, minSegmentSize=30, kmeansObj=km)
    b = shepseg.doShepherdSegmentation(img, minSegmentSize=30, kmeansObj=km)
    same(a.segimg, b.segimg, 'run twice')


def test_result_properties_large(shepseg):
    """size-independent properties at a benchmark-sized tile (4096 x 4096 x 4): ids are
    contiguous 1..n, no segment below minSegmentSize has a larger valid neighbour left
    unmerged ... checked cheaply as: contiguous ids, every id connected sizes >= 1, and
    idempotence of the label partition under the oracle's relabel."""
    img = synth.synth_tiled(4096, 4096, 4, seed=1)
    km = goldenutil.Centres(synth.diagonal_centres(img, 60))
    res = shepseg.doShepherdSegmentation(img, minSegmentSize=50, kmeansObj=km)
    seg = res.segimg
    n = int(seg.max())
    sizes = numpy.bincount(seg.ravel(), minlength=n + 1)
    assert sizes[0] == 0
    assert (sizes[1:] > 0).all()
    # ids increase with the raster position of each segment's first pixel is NOT a property
    # of the final raster (merges keep the target id), but the first pixel must be id 1's
    assert seg.flat[0] >= 1
    want = oracle.doShepherdSegmentation(img, minSegmentSize=50, kmeansObj=km)
    same(seg, want.segimg, '4096x4096x4 vs oracle')


ASSIGN_GRID_CASES = [
    # (dtype, bands, k, how the centres are drawn)
    (numpy.uint16, 4, 60, 'data'), (numpy.uint16, 3, 64, 'data'), (numpy.uint16, 2, 17, 'data'),
    (numpy.uint16, 1, 9, 'data'), (numpy.uint8, 4, 33, 'data'), (numpy.int16, 3, 40, 'data'),
    (numpy.uint16, 4, 60, 'integer'),        # integer centres: exact float64 ties, first minimum must win
    (numpy.uint16, 4, 12, 'outside'),        # centres outside the data type's range
    (numpy.int16, 4, 64, 'narrow'),          # all centres within a few units: one cell wide
]


@pytest.mark.parametrize('case', ASSIGN_GRID_CASES, ids=['%s_%db_k%d_%s' % (numpy.dtype(c[0]).name, c[1], c[2], c[3])
    for c in ASSIGN_GRID_CASES])
def test_assign_pruning_grid_equals_full_scan_and_oracle(shepseg, case):
    """The pruned assignment (a few candidate centres per box of band space, assign.cu) must give
    the float64 first-minimum argmin over ALL centres: compared with the oracle and with the
    full scan of the same library (SSG_ASSIGN_GRID=0), on values that sit on box boundaries, on
    the limits of the data type and on exact ties (shepseg.py:317-361)."""
    (dtype, nB, k, how) = case
    rng = numpy.random.default_rng(nB * 1000 + k)
    info = numpy.iinfo(dtype)
    (rows, cols) = (256, 512)
    lo = int(info.min + (info.max - info.min) * 0.05)
    hi = int(info.min + (info.max - info.min) * 0.4)
    img = rng.integers(lo, hi, (nB, rows, cols)).astype(dtype)
    img[:, :8, :] = rng.integers(info.min, info.max, (nB, 8, cols), endpoint=True).astype(dtype)   # anywhere
    img[:, 8, :64] = info.min
    img[:, 8, 64:128] = info.max
    if how == 'data':
        centres = rng.uniform(lo, hi, (k, nB))
    elif how == 'integer':
        centres = rng.integers(lo, hi, (k, nB)).astype(numpy.float64)
        centres[1] = centres[0]             # two identical centres: the first must win everywhere
        img[:, 9, :k] = ((centres[:k] + centres[(numpy.arange(k) + 1) % k]) // 2).T.astype(dtype)   # midpoints
    elif how == 'outside':
        centres = rng.uniform(-2.0 * info.max, 3.0 * info.max, (k, nB))
    else:
        centres = lo + rng.uniform(0.0, 3.0, (k, nB))
    # values on the boundaries of the grid boxes (powers of two around the centre range)
    for s in range(4, 14):
        img[:, 10 + (s - 4), :] = numpy.clip(numpy.floor(centres.min()) + rng.integers(-2, 3, (nB, cols)) +
            (rng.integers(-3, 40, (nB, cols)) << s), info.min, info.max).astype(dtype)
    km = goldenutil.Centres(centres)
    for nullVal in (None, int(img[0, 40, 40])):
        want = oracle.applySpectralClusters(km, img, nullVal)
        got = shepseg.applySpectralClusters(km, img, nullVal)
        same(got, want, 'pruned assignment vs oracle (null %s)' % nullVal)
        os.environ['SSG_ASSIGN_GRID'] = '0'
        try:
            full = shepseg.applySpectralClusters(km, img, nullVal)
        finally:
            del os.environ['SSG_ASSIGN_GRID']
        same(got, full, 'pruned assignment vs full scan (null %s)' % nullVal)


@pytest.mark.parametrize('bands,k', [(4, 60), (3, 12), (10, 30)])
def test_gpu_lloyd_iterations_equal_sklearn(shepseg, bands, k):
    """The Lloyd iterations on the device (ssg_kmeans_lloyd; shepseg.py:252-314, f3 of SURVEY.md
    section 8) are scikit-learn's: from the same initial centres, after the same number of
    iterations, the centres agree to 1e-9 of the data range (float64, another summation order)."""
    from sklearn.cluster import KMeans
    img = synth.synth_v1(400, 500, bands, seed=bands)
    sample = numpy.moveaxis(img, 0, -1).reshape(-1, bands)[::7]
    init = shepseg.diagonalClusterCentres(sample, k)
    span = float(img.max()) - float(img.min())
    for iters in (1, 5, 20):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            ref = KMeans(n_clusters=k, n_init=1, init=init, max_iter=iters, tol=0.0).fit(sample)
        got = shepseg._fitOnDevice(sample, k, True, maxIter=iters, tol=0.0)
        err = numpy.abs(got.cluster_centers_ - ref.cluster_centers_).max()
        assert err <= 1e-9 * span, '%d iterations: centres differ by %g (data range %g)' % (iters, err, span)
        assert abs(got.inertia_ - ref.inertia_) <= 1e-9 * ref.inertia_


def test_gpu_lloyd_fit_converges_to_sklearn_centres(shepseg):
    """On data with real clusters both fits converge, to the same centres: stated tolerance 1e-6
    of the data range (the north star's "centres within a stated tolerance"); the object that
    comes back is a fitted scikit-learn KMeans and assigns pixels like scikit-learn's own."""
    rng = numpy.random.default_rng(5)
    k = 12
    true = rng.uniform(500, 9000, (k, 4))
    lab = rng.integers(0, k, 300 * 320)
    img = numpy.clip(numpy.rint(true[lab] + rng.normal(0, 40, (len(lab), 4))), 1, 65534).astype(numpy.uint16)
    img = numpy.ascontiguousarray(img.T.reshape(4, 300, 320))
    ref = shepseg.fitSpectralClusters(img, k, 20, None, True, backend='sklearn')
    got = shepseg.fitSpectralClusters(img, k, 20, None, True, backend='gpu')
    span = float(img.max()) - float(img.min())
    err = numpy.abs(got.cluster_centers_ - ref.cluster_centers_).max()
    assert err <= 1e-6 * span, 'centres differ by %g (data range %g)' % (err, span)
    assert abs(got.inertia_ - ref.inertia_) <= 1e-9 * ref.inertia_
    pix = numpy.moveaxis(img[:, :50, :50], 0, -1).reshape(-1, 4)
    assert numpy.array_equal(got.predict(pix), ref.predict(pix))
    a = shepseg.doShepherdSegmentation(img, numClusters=k, minSegmentSize=20, kmeansObj=got)
    b = shepseg.doShepherdSegmentation(img, numClusters=k, minSegmentSize=20, kmeansObj=ref)
    assert numpy.array_equal(a.segimg, b.segimg)


def test_gpu_lloyd_fit_kmeanspp_and_nulls(shepseg):
    """k-means++ starts (five, the best kept) cannot be compared centre by centre with another
    random draw: the inertia must be in scikit-learn's range; null pixels stay out of the sample"""
    img = synth.synth_v1(500, 500, 3, seed=11, nullFrac=0.2)
    ref = shepseg.fitSpectralClusters(img, 20, 10, 0, False, backend='sklearn')
    got = shepseg.fitSpectralClusters(img, 20, 10, 0, False, backend='gpu')
    assert got.cluster_centers_.shape == (20, 3)
    assert got.inertia_ <= 1.05 * ref.inertia_
    assert (got.cluster_centers_.min(axis=0) > 0).all()      # no centre pulled to the null value

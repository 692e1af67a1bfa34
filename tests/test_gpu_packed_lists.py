"""
GPU parity of the packed pixel lists of the small-segment merge.

By default every small segment keeps its pixel list in a region of minSegmentSize-1 entries of its
own.  When the regions would take too much memory (a large minSegmentSize on a large tile) the
lists are packed instead: a merged list is copied into a fresh slice of an arena while the arena
lasts, and chained to the target's list after that.  SSG_SMALL_REGION_MB=0 forces the packed
lists, and SSG_SMALL_ARENA_PCT sizes the arena (0: every merge chains).  None of this may change
a label or a count: every case is compared with the CPU oracle bit for bit.
"""
import numpy
import pytest

import goldenutil
from oracle import oracle
from pyshepseg_b200 import synth, rasterfile

pytestmark = pytest.mark.gpu

PACKED_ENVS = [
    {'SSG_SMALL_REGION_MB': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '0'},
    {'SSG_SMALL_REGION_MB': '0', 'SSG_SMALL_ARENA_PCT': '7'},
]
ENV_IDS = ['arena', 'all_chained', 'arena_runs_out']


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


def image(kind, seed):
    if kind == 'uint8':
        return synth.synth_v1(400, 500, 4, seed=seed, lo=20.0, hi=230.0, noise=6.0, dtype=numpy.uint8)
    if kind == 'int16':       # about -2000 .. 1500
        base = synth.synth_v1(400, 500, 3, seed=seed)
        return (base.astype(numpy.int32) - 2500).astype(numpy.int16)
    if kind == 'uint32':      # up to about 4.3e9: the 32-bit kernels
        base = synth.synth_v1(400, 500, 3, seed=seed, lo=2000.0, hi=65000.0, noise=300.0)
        return base.astype(numpy.uint32) * numpy.uint32(65537)
    if kind == 'bigvalues':   # band sums far above 2**24: float32 sums depend on the order
        return synth.synth_v1(500, 600, 3, seed=seed, lo=30000, hi=62000, noise=300, cell=64)
    (bands, nullFrac) = {'b1': (1, 0.0), 'b6': (6, 0.0), 'b10': (10, 0.0), 'nulls': (4, 0.1)}[kind]
    return synth.synth_v1(400, 500, bands, seed=seed, nullFrac=nullFrac)


CASES = [
    # name, image, k, minSegmentSize, nodata, fourConnected, maxSpectralDiff
    ('one_band', 'b1', 20, 40, None, True, 'auto'),
    ('six_bands_8conn', 'b6', 40, 40, None, False, 'auto'),
    ('ten_bands', 'b10', 40, 40, None, True, 'auto'),
    ('uint8_8conn', 'uint8', 30, 30, None, False, 'auto'),
    ('int16_negative', 'int16', 30, 40, None, True, 'auto'),
    ('uint32_wide', 'uint32', 30, 40, None, True, 'auto'),
    ('big_values_inexact_sums', 'bigvalues', 8, 200, None, True, None),
    ('nulls', 'nulls', 40, 40, 0, True, 'auto'),
    ('min_seg_2', 'b6', 40, 2, None, True, 'auto'),
    ('min_seg_3_8conn', 'b6', 40, 3, None, False, 'auto'),
    # every small segment merges: lists grow through hundreds of sizes
    ('min_seg_400_long_chains', 'b1', 30, 400, None, True, None),
]


@pytest.mark.parametrize('env', PACKED_ENVS, ids=ENV_IDS)
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_packed_lists_against_oracle(shepseg, monkeypatch, case, env):
    (name, kind, k, minSeg, nullVal, four, msd) = case
    img = image(kind, len(name))
    km = goldenutil.Centres(synth.diagonal_centres(img, k, nullVal))
    want = oracle.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    for (key, value) in env.items():
        monkeypatch.setenv(key, value)
    got = shepseg.doShepherdSegmentation(img, minSegmentSize=minSeg, imgNullVal=nullVal,
        fourConnected=four, kmeansObj=km, maxSpectralDiff=msd)
    same(got.segimg, want.segimg, name)
    assert got.smallSegmentsEliminated == want.smallSegmentsEliminated, name
    # (at minSegmentSize 2 the single-pixel stage has already removed every small segment)
    assert minSeg == 2 or want.smallSegmentsEliminated > 0, name


@pytest.mark.parametrize('env', PACKED_ENVS, ids=ENV_IDS)
def test_packed_lists_tiled(tiling, monkeypatch, env):
    """a tiled run with packed lists gives the mosaic, histogram and maxSegId of the same run
    with per-segment regions"""
    img = synth.synth_v1(1100, 1300, 4, seed=21, nullFrac=0.05)
    km = goldenutil.Centres(synth.diagonal_centres(img, 40, 0))

    def run():
        res = tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img, nodata=0), None,
            tileSize=512, overlapSize=128, minSegmentSize=60, imgNullVal=0, kmeansObj=km,
            outputDriver='MEM', returnGDALDS=True)
        return (numpy.array(res.outDs.array), int(res.maxSegId), numpy.array(res.outDs.hist))

    (mosaic, maxSegId, hist) = run()
    for (key, value) in env.items():
        monkeypatch.setenv(key, value)
    (gotMosaic, gotMax, gotHist) = run()
    same(gotMosaic, mosaic, 'mosaic')
    assert gotMax == maxSegId
    same(gotHist, hist, 'histogram')

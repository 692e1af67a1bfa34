"""
One raster segmented on several GPUs from one process (tiling.MultiDeviceSegmenter, reached through
doTiledShepherdSegmentation with CONC_THREADS and two or more distinct devices).  On a box with one
GPU the shards all run on device 0 (concurrencyCfg.shardDevices, one shard per entry): the mosaic,
maxSegId, histogram, overviews and statistics must be the reference's (tests/golden/tiled_*.npz) or
the one-device call's.  The tests at the end need two or more visible devices and are skipped
otherwise.
"""
import os
import threading
import time

import numpy
import pytest

import goldenutil
from pyshepseg_b200 import rasterfile, synth, tiling

pytestmark = pytest.mark.gpu

GOLDEN = ['tiled_700x900', 'tiled_null_4x4', 'tiled_640_5x5_8conn', 'tiled_simple_recode']


def config(shards=None, workers=3, devices=None, conc=tiling.CONC_THREADS, barrierTimeout=120):
    cfg = tiling.SegmentationConcurrencyConfig(conc, numWorkers=workers, devices=devices,
        tileCompletionTimeout=120, barrierTimeout=barrierTimeout)
    if shards is not None:
        cfg.shardDevices = list(shards)
    return cfg


def run(case, cfg, src=None, outfile=None, driver='MEM', nullVal='meta'):
    m = case['meta']
    if nullVal == 'meta':
        nullVal = m['imgNullVal']
    if src is None:
        src = rasterfile.MemoryRaster(case['img'], nodata=nullVal)
    return tiling.doTiledShepherdSegmentation(src, outfile, tileSize=m['tileSize'], overlapSize=m['overlapSize'],
        minSegmentSize=m['minSegmentSize'], numClusters=m['numClusters'], imgNullVal=nullVal,
        fourConnected=m['fourConnected'], kmeansObj=goldenutil.Centres(case['centres']),
        simpleTileRecode=m['simpleTileRecode'], outputDriver=driver, returnGDALDS=True, concurrencyCfg=cfg)


def same(got, want, what):
    got = numpy.asarray(got)
    want = numpy.asarray(want)
    assert got.shape == want.shape, '%s: shape %s != %s' % (what, got.shape, want.shape)
    if not numpy.array_equal(got, want):
        bad = numpy.argwhere(got != want)
        raise AssertionError('%s: %d of %d differ; first at %s' % (what, len(bad), got.size, tuple(bad[0])))


def check_reference(res, c, what):
    m = c['meta']
    same(res.outDs.array, c['mosaic'], what + ' mosaic')
    assert int(res.maxSegId) == m['maxSegId'], what
    same(res.outDs.hist, c['hist'], what + ' histogram')
    assert res.outDs.metadata['STATISTICS_MAXIMUM'] == repr(m['maxSegId']), what


def check_same(res, one, what):
    same(res.outDs.array, one.outDs.array, what + ' mosaic')
    assert int(res.maxSegId) == int(one.maxSegId), what
    same(res.outDs.hist, one.outDs.hist, what + ' histogram')
    assert res.outDs.metadata == one.outDs.metadata, what
    for lvl in one.outDs.levels:
        same(res.outDs.overviews[lvl], one.outDs.overviews[lvl], '%s overview %d' % (what, lvl))


@pytest.mark.parametrize('shards', [2, 3, 4])
@pytest.mark.parametrize('name', GOLDEN)
def test_golden_on_shards(name, shards):
    c = goldenutil.load(name)
    res = run(c, config([0] * shards))
    check_reference(res, c, '%s on %d shards' % (name, shards))
    assert res.gpuLaunches > 0 and res.h2dBytes > 0 and res.d2hBytes > 0
    assert res.stageMs['total'] > 0
    # every shard's intervals under the reference's names and under its own prefix
    for label in ['gpu0'] + ['gpu0.%d' % i for i in range(1, shards)]:
        assert res.timings.getDurationsForName(label + ':stitchtiles') is not None
    assert res.timings.getDurationsForName('stitchtiles') is not None


@pytest.mark.parametrize('workers', [0, 1, 5])
def test_worker_counts(workers):
    c = goldenutil.load('tiled_640_5x5_8conn')
    check_reference(run(c, config([0, 0], workers=workers)), c, '%d workers over 2 shards' % workers)


def row_of_scenes(nulls):
    """a seeded raster of two tile rows and many tile columns, with a null wedge"""
    img = synth.synth_v1(686, 2900, 3, seed=77, cell=14)
    if nulls:
        (yy, xx) = numpy.mgrid[0:686, 0:2900]
        img[:, (xx - 3 * yy > 1500) | ((xx > 700) & (xx < 760))] = 0
    meta = {'tileSize': 256, 'overlapSize': 64, 'minSegmentSize': 20, 'numClusters': 16,
        'imgNullVal': 0 if nulls else None, 'fourConnected': True, 'simpleTileRecode': False}
    return {'img': img, 'centres': synth.diagonal_centres(img, 16), 'meta': meta}


@pytest.mark.parametrize('four', [True, False], ids=['4conn', '8conn'])
def test_row_of_scenes_equals_one_device(four):
    c = row_of_scenes(nulls=True)
    c['meta']['fourConnected'] = four
    (nB, nR, nC) = c['img'].shape
    sink = lambda: rasterfile.MemorySink(nC, nR, levels=[4, 8])      # noqa: E731  (overviews too)
    one = run(c, config(devices=[0]), outfile=sink())
    assert int(one.maxSegId) > 1000 and (one.outDs.array == 0).any()
    for shards in (2, 4):
        check_same(run(c, config([0] * shards, workers=2 * shards), outfile=sink()), one,
            'row of scenes on %d shards' % shards)


def written(directory):
    out = {}
    for name in sorted(os.listdir(directory)):
        if not name.startswith('in'):
            with open(os.path.join(directory, name), 'rb') as f:
                out[name] = f.read()
    return out


def tiff_sink_with_overviews(path, nC, nR, levels):
    """the built-in GTiff writer with overview levels kept beside the file (it writes none into it)"""
    sink = rasterfile.TiffSink(path, nC, nR)
    sink.levels = list(levels)
    sink.overviews = dict((lvl, numpy.zeros((-(-nR // lvl), -(-nC // lvl)), dtype=numpy.uint32)) for lvl in levels)
    return sink


def reference_overviews(mosaic, ti, overlap, lvl):
    """the reference's overview: whole blocks of every trimmed window, written in row-major order"""
    (nR, nC) = mosaic.shape
    out = numpy.zeros((-(-nR // lvl), -(-nC // lvl)), dtype=numpy.uint32)
    for (col, row) in sorted(ti.tiles, key=lambda cr: (cr[1], cr[0])):
        (x, y, xs, ys) = ti.tiles[(col, row)]
        (top, bottom, left, right) = tiling.tileMargins(ti, col, row, xs, ys, overlap)
        sub = mosaic[y + top:y + bottom, x + left:x + right][lvl // 2::lvl, lvl // 2::lvl]
        (xo, yo) = ((x + left) // lvl, (y + top) // lvl)
        sub = sub[:out.shape[0] - yo, :out.shape[1] - xo]
        out[yo:yo + sub.shape[0], xo:xo + sub.shape[1]] = sub
    return out


LEVELS = [8, 16]      # (tiled_null_4x4's window edges are not multiples of 8: neighbouring blocks overlap)


@pytest.mark.parametrize('shards', [2, 3, 4])
def test_overviews_where_windows_share_cells(shards):
    c = goldenutil.load('tiled_null_4x4')
    m = c['meta']
    (nB, nR, nC) = c['img'].shape
    ti = tiling.getTilesForFile((nC, nR), m['tileSize'], m['overlapSize'])
    one = run(c, config(devices=[0]), outfile=rasterfile.MemorySink(nC, nR, levels=LEVELS))
    for lvl in LEVELS:
        same(one.outDs.overviews[lvl], reference_overviews(c['mosaic'], ti, m['overlapSize'], lvl), 'one device')
    for _ in range(2):
        res = run(c, config([0] * shards, workers=shards), outfile=rasterfile.MemorySink(nC, nR, levels=LEVELS))
        check_reference(res, c, '%d shards' % shards)
        check_same(res, one, '%d shards' % shards)


def test_file_in_file_out(tmp_path):
    """a built-in GTiff source and a GTiff output with overview levels: every file written and the
    overviews equal the one-device call's"""
    c = goldenutil.load('tiled_null_4x4')
    (nB, nR, nC) = c['img'].shape
    outs = {}
    for (what, cfg) in (('one', config(devices=[0])), ('three', config([0, 0, 0], workers=4))):
        d = tmp_path / what
        d.mkdir()
        rasterfile.writeImage(str(d / 'in.tif'), c['img'], nodata=0)
        sink = tiff_sink_with_overviews(str(d / 'out.tif'), nC, nR, LEVELS)
        res = run(c, cfg, src=str(d / 'in.tif'), outfile=sink, nullVal=None)
        assert int(res.maxSegId) == c['meta']['maxSegId']
        overviews = dict((lvl, sink.overviews[lvl].copy()) for lvl in LEVELS)
        sink.close()
        outs[what] = (written(str(d)), overviews)
    assert sorted(outs['three'][0]) == sorted(outs['one'][0]) and len(outs['one'][0]) == 3
    for name in outs['one'][0]:
        assert outs['three'][0][name] == outs['one'][0][name], name
    for lvl in LEVELS:
        same(outs['three'][1][lvl], outs['one'][1][lvl], 'overview %d' % lvl)
    got = rasterfile.TiffSource(str(tmp_path / 'three' / 'out.tif'))
    same(got.readWindow([1], 0, 0, got.xsize, got.ysize)[0], c['mosaic'], 'mosaic read back')
    got.close()


def test_refusals():
    from pyshepseg_b200 import distributed
    c = goldenutil.load('tiled_700x900')
    cfg = config(devices=[0, 1])
    cfg.comm = distributed.LocalComm()
    with pytest.raises(tiling.PyShepSegTilingError, match='comm'):
        run(c, cfg)
    src = tiling.DeviceRaster(0, 3, 700, 900, numpy.uint16)
    with pytest.raises(tiling.PyShepSegTilingError, match='DeviceRaster'):
        run(c, config(devices=[0, 1]), src=src)
    with pytest.raises(tiling.PyShepSegTilingError, match='DeviceRaster'):
        run(c, config([0, 0]), src=src)


def test_one_device_meanings():
    """repeated ids are one device; CONC_NONE uses devices[0] alone"""
    c = goldenutil.load('tiled_700x900')
    check_reference(run(c, config(devices=[0, 0])), c, 'devices [0, 0]')
    check_reference(run(c, config(devices=[0, 1], conc=tiling.CONC_NONE, workers=0)), c, 'CONC_NONE')


class RaisingSink(rasterfile.MemorySink):
    """a sink that fails on one window (of the shard that owns the mosaic's last tile)"""
    def __init__(self, xsize, ysize, at):
        rasterfile.MemorySink.__init__(self, xsize, ysize)
        self.at = at

    def write(self, arr, xoff, yoff):
        if (xoff, yoff) == self.at:
            raise IOError('disk full at window (%d, %d)' % (xoff, yoff))
        rasterfile.MemorySink.write(self, arr, xoff, yoff)


def test_failing_sink_ends_the_call():
    c = goldenutil.load('tiled_640_5x5_8conn')
    m = c['meta']
    (nB, nR, nC) = c['img'].shape
    ti = tiling.getTilesForFile((nC, nR), m['tileSize'], m['overlapSize'])
    last = (ti.ncols - 1, ti.nrows - 1)
    (x, y, xs, ys) = ti.tiles[last]
    (top, bottom, left, right) = tiling.tileMargins(ti, last[0], last[1], xs, ys, m['overlapSize'])
    before = set(threading.enumerate())
    t0 = time.time()
    with pytest.raises(tiling.PyShepSegTilingError, match='disk full'):
        run(c, config([0, 0, 0], workers=3, barrierTimeout=100), outfile=RaisingSink(nC, nR, (x + left, y + top)))
    assert time.time() - t0 < 100
    for th in set(threading.enumerate()) - before:
        th.join(10)
        assert not th.is_alive(), 'thread %s left behind' % th.name
    # the cached GPU state serves the next call
    check_reference(run(c, config([0, 0, 0], workers=3)), c, 'the call after the failure')


def test_timeline_prefixed(monkeypatch):
    monkeypatch.setenv('SSG_TIMELINE', '1')
    c = goldenutil.load('tiled_700x900')
    res = run(c, config([0, 0]))
    whats = [w for (ms, w) in res.timeline]
    assert any(w.startswith('gpu0: tile') for w in whats) and any(w.startswith('gpu0.1: tile') for w in whats)
    assert [ms for (ms, w) in res.timeline] == sorted(ms for (ms, w) in res.timeline)


# ---- two or more GPUs ------------------------------------------------------------------------
def device_count():
    import torch
    return torch.cuda.device_count()


needs_two = pytest.mark.skipif(device_count() < 2, reason='needs two or more visible CUDA devices')


@needs_two
@pytest.mark.parametrize('source', ['memory', 'file'])
def test_several_devices_equal_one(source, tmp_path):
    c = goldenutil.load('tiled_null_4x4')
    assert (c['meta']['numTileRows'], c['meta']['numTileCols']) == (4, 4)

    def call(devices):
        if source == 'memory':
            return run(c, config(devices=devices, workers=2 * len(devices)))
        path = str(tmp_path / 'in.tif')
        if not os.path.exists(path):
            rasterfile.writeImage(path, c['img'], nodata=0)
        return run(c, config(devices=devices, workers=2 * len(devices)), src=path, nullVal=None)
    one = call([0])
    check_reference(one, c, 'devices [0]')
    for devices in ([0, 1], list(range(device_count()))):
        check_same(call(devices), one, 'devices %s' % devices)

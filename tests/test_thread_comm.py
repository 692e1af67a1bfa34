"""
The sharded stitch (pyshepseg_b200.distributed.ShardedStitch) over ThreadComm, the communicator
whose ranks are threads of one process (what tiling.MultiDeviceSegmenter runs on several GPUs).
The device work is the numpy stand-in of test_distributed_host; every rank's windows together
must be the mosaic of the oracle's sequential restatement of tiling.stitchTiles, with its
maxSegId.  A rank that fails must take every other rank out of its collective, and a rank that
never arrives must make the others give up after the barrier timeout.
"""
import threading
import time

import numpy
import pytest

from oracle import oracle
from pyshepseg_b200 import distributed
from test_distributed_host import NumpyOps, NumpyRelOps, make_tiles


def run_threads(world, case, forceSequential=False, opsFor=None, timeout=60, abortOnError=True):
    """ShardedStitch on `world` thread ranks; returns (maxSegIds, mosaic, usedFallback, errors, seconds)"""
    (kind, seed, nR, nC, tileSize, overlap, simple) = case
    (ti, allSegs) = make_tiles(kind, seed, nR, nC, tileSize, overlap)
    hub = distributed.ThreadHub(world, timeout)
    out = numpy.zeros((nR, nC), dtype=numpy.uint32)      # the ranks' windows are disjoint
    maxIds = [None] * world
    fallback = [None] * world
    errors = [None] * world

    def rank_main(rank):
        comm = distributed.ThreadComm(hub, rank)
        try:
            st = distributed.ShardedStitch(ti, overlap, simple, comm)
            st.forceSequential = forceSequential
            segs = dict((cr, allSegs[cr]) for cr in st.mine)
            cls = NumpyOps if seed % 2 else NumpyRelOps
            ops = (opsFor(rank, cls) if opsFor is not None else cls)(ti, segs, overlap, out)
            ops.simple = simple
            (maxIds[rank], offsets, luts) = st.run(ops)
            fallback[rank] = st.usedFallback
        except Exception as e:
            errors[rank] = e
            if abortOnError:
                hub.abort(rank, e)
    t0 = time.time()
    threads = [threading.Thread(target=rank_main, args=(r,), daemon=True) for r in range(world)]
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout + 30)
    assert not any(th.is_alive() for th in threads), 'a rank is still waiting'
    return (maxIds, out, fallback, errors, time.time() - t0)


CASES = [
    # name, world, (labels, seed, nR, nC, tileSize, overlap, simple), forced fall-back
    ('w2_4x3', 2, ('segmented', 11, 260, 300, 96, 32, False), False),
    ('w3_5x5', 3, ('segmented', 12, 330, 340, 96, 40, False), False),
    ('w4_6x6', 4, ('segmented', 16, 420, 430, 96, 32, False), False),
    ('w3_blobby', 3, ('blobby', 14, 260, 300, 96, 32, False), False),
    ('w4_row_of_scenes_blobby', 4, ('blobby', 19, 343, 1300, 128, 32, False), False),
    ('w2_forced_sequential', 2, ('blobby', 14, 260, 300, 96, 32, False), True),
    ('w4_forced_sequential', 4, ('segmented', 16, 420, 430, 96, 32, False), True),
    ('w2_simple', 2, ('segmented', 13, 260, 300, 96, 32, True), False),
    ('w3_blobby_simple', 3, ('blobby', 15, 260, 300, 96, 32, True), False),
    ('w4_simple', 4, ('segmented', 16, 420, 430, 96, 32, True), False),
    # more ranks than tiles: a rank without a tile still takes part in every collective
    ('w4_three_tiles', 4, ('segmented', 21, 120, 300, 96, 32, False), False),
    ('w3_three_tiles_simple', 3, ('segmented', 21, 120, 300, 96, 32, True), False),
]


@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_sharded_stitch_threads(case):
    (name, world, prm, forced) = case
    (kind, seed, nR, nC, tileSize, overlap, simple) = prm
    (maxIds, mosaic, fallback, errors, _) = run_threads(world, prm, forceSequential=forced)
    assert errors == [None] * world
    (ti, segs) = make_tiles(kind, seed, nR, nC, tileSize, overlap)
    (want, wantMax, _) = oracle.stitchTiles(segs, ti, nC, nR, overlap, simpleTileRecode=simple)
    assert maxIds == [wantMax] * world
    assert numpy.array_equal(mosaic, want)
    assert fallback == [forced] * world


class Failing(Exception):
    pass


def failing_ops(badRank):
    """rank badRank raises on the table of its second tile: after the strip exchange, while the
    other ranks are already in the first all-gather of the resolve"""
    def opsFor(rank, cls):
        if rank != badRank:
            return cls

        class Bad(cls):
            calls = 0

            def tables(self, cr, top, left):
                Bad.calls += 1
                if Bad.calls == 2:
                    raise Failing('table of tile %s' % (cr,))
                return cls.tables(self, cr, top, left)
        return Bad
    return opsFor


@pytest.mark.parametrize('world', [2, 3, 4])
def test_failing_rank_stops_every_rank(world):
    prm = ('segmented', 16, 420, 430, 96, 32, False)
    (maxIds, mosaic, fallback, errors, secs) = run_threads(world, prm, opsFor=failing_ops(1), timeout=120)
    assert isinstance(errors[1], Failing)
    for r in range(world):
        if r != 1:
            assert isinstance(errors[r], distributed.ThreadCommError)
            assert 'rank 1 failed' in str(errors[r]) and 'table of tile' in str(errors[r])
    assert secs < 60          # (the abort, not the 120 s barrier timeout, ended the wait)


def test_silent_rank_times_out():
    """a rank that leaves without aborting the hub: the others give up after the barrier timeout"""
    prm = ('segmented', 11, 260, 300, 96, 32, False)
    (maxIds, mosaic, fallback, errors, secs) = run_threads(2, prm, opsFor=failing_ops(1), timeout=3,
        abortOnError=False)
    assert isinstance(errors[1], Failing)
    assert isinstance(errors[0], distributed.ThreadCommError) and 'did not reach the barrier' in str(errors[0])
    assert secs < 30


def test_collectives():
    world = 3
    hub = distributed.ThreadHub(world, 30)
    got = [None] * world

    def rank_main(rank):
        comm = distributed.ThreadComm(hub, rank)
        ints = comm.allgatherInts(list(range(rank + 1)))
        arrs = comm.allgatherArray(numpy.arange(rank, dtype=numpy.int64))
        byts = comm.allgatherBytes(bytes([rank] * 3))
        total = comm.allreduceSum(numpy.full(4, rank + 1, dtype=numpy.int64))
        got[rank] = (ints, [a.tolist() for a in arrs], [b.tolist() for b in byts], total.tolist())
    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    for th in threads:
        th.start()
    for th in threads:
        th.join(60)
    want = ([[0], [0, 1], [0, 1, 2]], [[], [0], [0, 1]], [[0] * 3, [1] * 3, [2] * 3], [6] * 4)
    assert got == [want] * world

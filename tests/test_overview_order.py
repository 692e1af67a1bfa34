"""
tiling.overviewBlockOwned: every window writes only the part of its overview block that no later
window writes again, so the overviews do not depend on the order the windows arrive in (the shards
of a MultiDeviceSegmenter write theirs concurrently).  Written in any order, the clipped blocks must
give what the reference's row-major writes of whole blocks give (tiling.py:1360-1383), also on
geometries whose window edges are not multiples of the level.
"""
import numpy
import pytest

from pyshepseg_b200 import tiling


def overviews(mosaic, ti, overlap, lvl, order, clip):
    (nR, nC) = mosaic.shape
    out = numpy.zeros((-(-nR // lvl), -(-nC // lvl)), dtype=mosaic.dtype)
    for (col, row) in order:
        (x, y, xs, ys) = ti.tiles[(col, row)]
        (top, bottom, left, right) = tiling.tileMargins(ti, col, row, xs, ys, overlap)
        sub = mosaic[y + top:y + bottom, x + left:x + right][lvl // 2::lvl, lvl // 2::lvl]
        if clip:
            (r, c) = tiling.overviewBlockOwned(ti, col, row, overlap, lvl)
            sub = sub[:r, :c]
        (xo, yo) = ((x + left) // lvl, (y + top) // lvl)
        sub = sub[:out.shape[0] - yo, :out.shape[1] - xo]
        out[yo:yo + sub.shape[0], xo:xo + sub.shape[1]] = sub
    return out


GEOMETRIES = [
    # (nR, nC, tileSize, overlap)
    (620, 660, 180, 60),        # tests/golden/tiled_null_4x4
    (700, 900, 256, 64),
    (640, 640, 200, 120),
    (3000, 3000, 300, 30),
    (1234, 987, 250, 70),
    (500, 620, 256, 64),
]


@pytest.mark.parametrize('geom', GEOMETRIES, ids=['%dx%d_%d_%d' % g for g in GEOMETRIES])
@pytest.mark.parametrize('lvl', [2, 4, 5, 8, 16, 64])
def test_clipped_blocks_in_any_order_equal_row_major(geom, lvl):
    (nR, nC, tileSize, overlap) = geom
    ti = tiling.getTilesForFile((nC, nR), tileSize, overlap)
    rng = numpy.random.default_rng(nR + lvl)
    mosaic = rng.integers(1, 1 << 30, (nR, nC)).astype(numpy.uint32)
    rowMajor = sorted(ti.tiles, key=lambda cr: (cr[1], cr[0]))
    want = overviews(mosaic, ti, overlap, lvl, rowMajor, clip=False)
    assert numpy.array_equal(overviews(mosaic, ti, overlap, lvl, rowMajor, clip=True), want)
    for seed in range(3):
        order = list(rowMajor)
        numpy.random.default_rng(seed).shuffle(order)
        assert numpy.array_equal(overviews(mosaic, ti, overlap, lvl, order, clip=True), want)


def test_unclipped_blocks_depend_on_the_order():
    """(the test above is not vacuous: on this geometry whole blocks written in reverse order give
    other overviews than in row-major order)"""
    ti = tiling.getTilesForFile((660, 620), 180, 60)
    mosaic = numpy.random.default_rng(1).integers(1, 1 << 30, (620, 660)).astype(numpy.uint32)
    rowMajor = sorted(ti.tiles, key=lambda cr: (cr[1], cr[0]))
    assert not numpy.array_equal(overviews(mosaic, ti, 60, 8, rowMajor[::-1], clip=False),
        overviews(mosaic, ti, 60, 8, rowMajor, clip=False))

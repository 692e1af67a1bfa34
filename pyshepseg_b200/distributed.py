"""
One mosaic, its tiles sharded over the GPUs of one box: one process per GPU (torch.distributed,
TorchComm) or one thread per GPU in one process (ThreadComm, tiling.MultiDeviceSegmenter).

The path shards by tile: every tile is segmented independently given the shared cluster
centres (shepseg.doShepherdSegmentation per tile, tiling.py:1446/1586).  What the reference does
sequentially afterwards (stitchTiles, tiling.py:950-1064: tile after tile in row-major order,
carrying the running maxSegId and the recoded overlap strips of the finished neighbours) needs
three small exchanges when the tiles live on different ranks:

  strips   the LOCAL labels of an upper / left neighbour under a tile's overlap, when that
           neighbour lives on another rank (device-to-device send/recv, NCCL over NVLink).  A
           rank segments the tiles that feed other ranks first, so the exchange can run while
           the rest of its tiles are still in work (feedPlan / exchangeStrips);
  steps    one integer per tile, the highest rank among its self-numbered segments inside its
           trimmed window: the id offset of tile t is the sum over the tiles before it (one
           all-gather).  That is what the reference's "maxSegId = max(maxSegId, trimmed.max())"
           (tiling.py:1042-1043) amounts to unless a window holds an inherited id above the
           running maximum; the recurrence is checked on every tile after the resolve and the
           ranks fall back to the sequential order over all tables if it fails anywhere, so the
           result is the reference's in every case.  Until the offsets are known ids are handled
           SYMBOLICALLY, as (index of the tile that numbered the segment) << 32 | rank: such
           values order and compare like the final ids, so every vote can be taken before a
           single offset exists, and offset + rank is left to the device at the very end;
  look-ups the final ids of single labels of a tile on another rank: a crossing segment takes
           the final id of the neighbour segment it overlaps most (recodeSharedSegments,
           tiling.py:1128-1203), and that id may in turn be inherited from the neighbour's
           neighbour.  The owner of a tile answers what it has settled; requests travel with the
           steps' all-gather, so a mosaic costs two or three collectives.  No rank replays
           another rank's tiles and no tables are shipped (except in the fall-back).

Only the crossing segments of a tile (a few thousand) are ever handled here; nothing of a tile's
full length is computed on the host.  Everything in this module is host logic on numpy arrays;
the device work is behind the `ops` object the caller hands in (tiling.TiledSegmenter for the
GPU, plain numpy in the CPU tests).
"""
import io
import threading

import numpy

from . import _lib

KEY_FLAGS = _lib.SEG_KEYTOP | _lib.SEG_KEYLEFT


def rowMajor(tileInfo):
    return sorted(tileInfo.tiles.keys(), key=lambda cr: (cr[1], cr[0]))


# cost of segmenting a tile, in arbitrary units: a fixed part (the dependent phases of the merge
# kernels, whatever the tile's size) plus a part per pixel; measured on B200 (round 2 kernels) as
# 0.5 ms + 0.095 ms per megapixel
TILE_COST_FIXED = 0.5
TILE_COST_PER_MPIX = 0.095


def _tileCost(t):
    return TILE_COST_FIXED + TILE_COST_PER_MPIX * t[2] * t[3] / 1e6


def _splitBalanced(weights, k):
    """Cut the list into k contiguous non-empty groups with the smallest possible largest sum;
    returns the group index of every element."""
    n = len(weights)
    pre = numpy.concatenate([[0.0], numpy.cumsum(weights)])
    best = numpy.full((k + 1, n + 1), numpy.inf)
    cut = numpy.zeros((k + 1, n + 1), dtype=numpy.int64)
    best[0, 0] = 0.0
    for g in range(1, k + 1):
        for i in range(g, n - (k - g) + 1):
            v = numpy.maximum(best[g - 1, g - 1:i], pre[i] - pre[g - 1:i])     # last group = [j, i)
            j = int(numpy.argmin(v))
            (best[g, i], cut[g, i]) = (v[j], j + g - 1)
    groups = [0] * n
    i = n
    for g in range(k, 0, -1):
        j = int(cut[g, i])
        for e in range(j, i):
            groups[e] = g - 1
        i = j
    return groups


def partitionChunks(tileInfo, world):
    """owner rank of every tile: contiguous chunks of the row-major tile list (tiling.py:892-893)
    with as equal a share of the segmentation cost as the tile boundaries allow."""
    order = rowMajor(tileInfo)
    groups = _splitBalanced([_tileCost(tileInfo.tiles[cr]) for cr in order], min(world, len(order)))
    return dict((cr, g) for (cr, g) in zip(order, groups))


def partitionTiles(tileInfo, world):
    """
    owner rank of every tile.  The tile rows are cut into pr bands and every band, its tiles taken
    column by column, into pc contiguous pieces of as equal a segmentation cost as possible
    (pr * pc = world, ranks numbered band after band): a rank owns a block of whole tile columns
    plus at most a partial column at either end, so that it has remote upper or left neighbours
    only along the rim of its block, and only those tiles have to wait for another rank's
    strips before their stitch tables can be made.  Among the (pr, pc) that fit, the one with
    the smallest largest cost wins, fewer rim tiles on ties; contiguous chunks of the row-major
    list (pr = world bands cannot be formed, say) are the fall-back.  The reference deals tiles
    round-robin over its workers (tiling.py:892-893); which worker segments a tile does not
    change the result.
    """
    (nrows, ncols) = (tileInfo.nrows, tileInfo.ncols)
    if world <= 1:
        return dict((cr, 0) for cr in tileInfo.tiles)
    key = (world, tuple(sorted(tileInfo.tiles.items())))
    with _partitionLock:        # (the ranks of a ThreadComm ask from threads of one process)
        if key not in _partitionCache:
            _partitionCache.clear()
            _partitionCache[key] = _partitionTiles(tileInfo, world)
        return dict(_partitionCache[key])


_partitionCache = {}
_partitionLock = threading.Lock()


def _partitionTiles(tileInfo, world):
    (nrows, ncols) = (tileInfo.nrows, tileInfo.ncols)
    rowCost = [sum(_tileCost(tileInfo.tiles[(c, r)]) for c in range(ncols)) for r in range(nrows)]
    best = None
    for pr in range(1, world + 1):
        if world % pr:
            continue
        pc = world // pr
        if pr > nrows or pc > ncols:
            continue
        rg = _splitBalanced(rowCost, pr)
        owner = {}
        for band in range(pr):
            rows = [r for r in range(nrows) if rg[r] == band]
            cells = [(c, r) for c in range(ncols) for r in rows]          # column by column
            if len(cells) < pc:
                owner = None
                break
            groups = _splitBalanced([_tileCost(tileInfo.tiles[cr]) for cr in cells], pc)
            for (cr, g) in zip(cells, groups):
                owner[cr] = band * pc + g
        if owner is None:
            continue
        cost = numpy.zeros(world)
        rim = 0
        for ((c, r), t) in tileInfo.tiles.items():
            cost[owner[(c, r)]] += _tileCost(t)
            if (r > 0 and owner[(c, r - 1)] != owner[(c, r)]) or (c > 0 and owner[(c - 1, r)] != owner[(c, r)]):
                rim += 1
        key = (round(float(cost.max()), 6), rim)
        if best is None or key < best[0]:
            best = (key, owner)
    if best is None:
        return partitionChunks(tileInfo, world)
    return best[1]


class TileTable(object):
    """The host copy of what ssg_tile_tables_device computed for one tile."""
    def __init__(self, maxId, countNew, rank, flags, pairKeys, pairCounts, maxRankInTrim=None):
        self.givenMaxRankInTrim = maxRankInTrim      # (computed with the tables on the device)
        self.maxId = int(maxId)
        self.countNew = int(countNew)
        self.rank = numpy.ascontiguousarray(rank, dtype=numpy.uint32)
        self.flags = numpy.ascontiguousarray(flags, dtype=numpy.uint8)
        self.pairKeys = numpy.ascontiguousarray(pairKeys, dtype=numpy.uint64)
        self.pairCounts = numpy.ascontiguousarray(pairCounts, dtype=numpy.uint32)
        self._split = None

    @property
    def maxRankInTrim(self):
        if self.givenMaxRankInTrim is not None:
            return int(self.givenMaxRankInTrim)
        both = numpy.uint8(_lib.SEG_NUMBERED | _lib.SEG_INTRIM)
        return int(numpy.max(self.rank, where=(self.flags & both) == both, initial=0))

    @property
    def maxLabelInTrim(self):
        sel = numpy.flatnonzero(self.flags & _lib.SEG_INTRIM)
        return int(sel[-1]) if len(sel) else 0

    def prepare(self):
        """What the resolve needs of the tile besides look-ups of single labels, worked out once
        (as soon as the tables exist, while other tiles are still being segmented): the labels of
        the crossing segments, which of them lie in the trimmed window, the highest rank in the
        window, the decoded votes.  Nothing here is longer than a pass over the flag bytes."""
        if getattr(self, '_prepared', None) is None:
            crossing = numpy.flatnonzero((self.flags & numpy.uint8(KEY_FLAGS)) != 0)
            self._prepared = crossing
            self.crossInTrimMask = (self.flags[crossing] & _lib.SEG_INTRIM) != 0
            self.crossingInTrim = crossing[self.crossInTrimMask]
            self.cachedMaxRankInTrim = self.maxRankInTrim
            self.pairs()
        return self._prepared

    def rel(self):
        """rank where the tile numbered the segment itself, 0 elsewhere (a full-length array:
        only for building a whole lut on the host)"""
        return numpy.where((self.flags & _lib.SEG_NUMBERED) != 0, self.rank, numpy.uint32(0)).astype(numpy.uint32)

    def pairs(self):
        """(isLeft, segment, neighbour label, count) of the votes, decoded once."""
        if self._split is None:
            k = self.pairKeys
            self._split = ((k >> numpy.uint64(63)) != 0,
                ((k >> numpy.uint64(32)) & numpy.uint64(0x7FFFFFFF)).astype(numpy.int64),
                (k & numpy.uint64(0xFFFFFFFF)).astype(numpy.int64),
                self.pairCounts.astype(numpy.int64))
        return self._split


def packTables(tables):
    """{tile: TileTable} -> one uint8 array (for an all-gather of byte buffers)."""
    items = sorted(tables.items())
    total = 8
    for (cr, tb) in items:
        total += 24 + 32 + 8 * len(tb.pairKeys) + 4 * len(tb.rank) + 4 * len(tb.pairCounts) + len(tb.flags)
        total += (-total) % 8
    out = numpy.zeros(total, dtype=numpy.uint8)
    out[:8].view(numpy.int64)[0] = len(items)
    o = 8
    for (cr, tb) in items:
        body = 32 + 8 * len(tb.pairKeys) + 4 * len(tb.rank) + 4 * len(tb.pairCounts) + len(tb.flags)
        size = body + ((-(o + 24 + body)) % 8)
        out[o:o + 24].view(numpy.int64)[:] = (cr[0], cr[1], size)
        o += 24
        out[o:o + 32].view(numpy.int64)[:] = (tb.maxId, tb.countNew, len(tb.rank), len(tb.pairKeys))
        q = o + 32
        for a in (tb.pairKeys, tb.rank, tb.pairCounts, tb.flags):      # widest first: aligned
            nb = a.nbytes
            out[q:q + nb] = a.view(numpy.uint8)
            q += nb
        o += size
    return out


def unpackTables(b):
    b = numpy.frombuffer(b, dtype=numpy.uint8) if not isinstance(b, numpy.ndarray) else b
    n = int(b[:8].view(numpy.int64)[0])
    o = 8
    out = {}
    for _ in range(n):
        (c, r, size) = (int(v) for v in b[o:o + 24].view(numpy.int64))
        o += 24
        (maxId, countNew, nSeg, nPairs) = (int(v) for v in b[o:o + 32].view(numpy.int64))
        q = o + 32
        pairKeys = b[q:q + 8 * nPairs].view(numpy.uint64)
        q += 8 * nPairs
        rank = b[q:q + 4 * nSeg].view(numpy.uint32)
        q += 4 * nSeg
        pairCounts = b[q:q + 4 * nPairs].view(numpy.uint32)
        q += 4 * nPairs
        flags = b[q:q + nSeg]
        out[(c, r)] = TileTable(maxId, countNew, rank, flags, pairKeys, pairCounts)
        o += size
    return out


class MissingTable(Exception):
    """a look-up reached a tile whose table this rank does not hold"""


class LazyResolver(object):
    """
    Final ids from per-tile tables when the id offsets are known up front (offset of a tile = sum
    of countNew over the tiles before it), looked up per label:
      numbered segment           offset + rank                       (tiling.py:1264-1267)
      crossing segment           the mode of the final ids of the neighbour's labels under it,
                                 smallest id on ties, top overlap first, left overriding
                                 (tiling.py:1107-1121, 1194)
      anything else, and 0       0 (the segment belongs to a neighbour, tiling.py:1241)
    Only the crossing segments (a few thousand per tile) are stored; nothing of a tile's full
    length is computed here, so the work per tile is small enough for the thread that also
    feeds the GPU.  ids are uint32, or uint64 for the symbolic offsets of ShardedStitch.
    """
    def __init__(self, tables, offsets, simple=False, dtype=numpy.uint32):
        self.tables = tables
        self.offsets = offsets
        self.simple = simple
        self.dtype = numpy.dtype(dtype)
        self.UNKNOWN = self.dtype.type(numpy.iinfo(self.dtype).max)
        self.cross = {}         # tile -> (labels of its crossing segments ascending, their ids)
        self.scratch = {}       # tile -> bool array over its labels, all False between calls
        self.misses = 0         # look-ups that could not be answered yet
        self.remote = {}        # tile of another rank -> (labels ascending, their final ids)
        self.requests = {}      # tile of another rank -> [label arrays] still to be asked for

    def _crossOf(self, cr):
        if cr not in self.cross:
            if cr not in self.tables:
                raise MissingTable(cr)
            tb = self.tables[cr]
            if self.simple:
                crossing = numpy.zeros(0, dtype=numpy.int64)
            else:
                crossing = tb.prepare()
            self.cross[cr] = (crossing, numpy.full(len(crossing), self.UNKNOWN, dtype=self.dtype))
        return self.cross[cr]

    def _pos(self, crossing, labels):
        """(index into crossing, is a crossing label) per label"""
        if len(crossing) == 0:
            return (numpy.zeros(len(labels), dtype=numpy.int64), numpy.zeros(len(labels), dtype=bool))
        pos = numpy.searchsorted(crossing, labels)
        pos[pos >= len(crossing)] = 0
        return (pos, crossing[pos] == labels)

    def _lookup(self, cr, labels):
        """ids of the given labels of tile cr as far as known (UNKNOWN for open crossing ones)"""
        tb = self.tables[cr]
        off = self.dtype.type(self.offsets[cr])
        if self.simple:
            out = labels.astype(self.dtype) + off
            out[labels == 0] = 0
            return out
        (crossing, vals) = self._crossOf(cr)
        numbered = (tb.flags[labels] & _lib.SEG_NUMBERED) != 0
        out = numpy.where(numbered, tb.rank[labels].astype(self.dtype) + off, self.dtype.type(0))
        (pos, isCross) = self._pos(crossing, labels)
        out[isCross] = vals[pos[isCross]]
        return out

    def remoteIds(self, cr, labels):
        """final ids of labels of a tile owned by another rank, from the owner's answers so far;
        what is not known yet is queued in self.requests.  Returns (ids, complete)."""
        labels = numpy.asarray(labels, dtype=numpy.int64)
        out = numpy.zeros(len(labels), dtype=self.dtype)
        found = numpy.zeros(len(labels), dtype=bool)
        if cr in self.remote:
            (known, vals) = self.remote[cr]
            pos = numpy.searchsorted(known, labels)
            pos[pos >= len(known)] = 0
            found = known[pos] == labels
            out[found] = vals[pos[found]]
        if not found.all():
            self.requests.setdefault(cr, []).append(labels[~found])
            return (out, False)
        return (out, True)

    def addRemote(self, cr, labels, vals):
        if cr in self.remote:
            labels = numpy.concatenate([self.remote[cr][0], labels])
            vals = numpy.concatenate([self.remote[cr][1], vals])
        order = numpy.argsort(labels, kind='stable')
        self.remote[cr] = (labels[order].astype(numpy.int64), vals[order].astype(self.dtype))

    def answer(self, cr, labels):
        """what an owner can say about labels of its tile cr right now: (labels, final ids) of
        those that are settled"""
        labels = numpy.asarray(labels, dtype=numpy.int64)
        vals = self._finalIds(cr, labels)
        settled = vals != self.UNKNOWN
        return (labels[settled], vals[settled])

    def _finalIds(self, cr, labels):
        out = self._lookup(cr, labels)
        unknown = out == self.UNKNOWN
        if unknown.any():
            self._resolveCrossing(cr, numpy.unique(labels[unknown]))
            out = self._lookup(cr, labels)
        return out

    def finalIds(self, cr, labels):
        """final ids of the given local labels of tile cr (int64 array).  Entries whose value
        hangs on a table that is not here stay open (and come back as 0); self.misses counts
        them and self.requests says what to ask the owners for."""
        out = self._finalIds(cr, numpy.asarray(labels, dtype=numpy.int64))
        return numpy.where(out == self.UNKNOWN, 0, out).astype(self.dtype)

    def _resolveCrossing(self, cr, labels):
        """A crossing segment takes the vote of the left overlap if it crosses that one (the left
        recode is applied after the top one and overrides it, tiling.py:1107-1121), otherwise the
        vote of the top overlap."""
        from .tiling import _modeByKey
        tb = self.tables[cr]
        (crossing, vals) = self._crossOf(cr)
        (isLeft, segs, nbr, counts) = tb.pairs()
        if cr not in self.scratch:
            self.scratch[cr] = numpy.zeros(tb.maxId + 1, dtype=bool)
        mark = self.scratch[cr]
        keyLeft = (tb.flags[labels] & _lib.SEG_KEYLEFT) != 0
        for (sub, pairSide, nb) in ((labels[~keyLeft], ~isLeft, (cr[0], cr[1] - 1)),
                (labels[keyLeft], isLeft, (cr[0] - 1, cr[1]))):
            if len(sub) == 0:
                continue
            subPos = self._pos(crossing, sub)[0]
            mark[sub] = True
            sel = pairSide & mark[segs]
            mark[sub] = False
            if not sel.any():
                vals[subPos] = 0
                continue
            if nb not in self.tables:
                # a tile of another rank: its owner answers (entries stay open until then)
                (mapped, complete) = self.remoteIds(nb, nbr[sel])
                if not complete:
                    self.misses += 1
                    continue
            else:
                before = self.misses
                mapped = self.finalIds(nb, nbr[sel])
                if self.misses > before:
                    continue          # the neighbour's own answer is still open somewhere below
            vals[subPos] = 0
            if self.dtype.itemsize > 4:
                # symbolic ids do not fit the 32 bits _modeByKey packs: vote on their ranks in
                # ascending order (ties go to the smallest id either way)
                (uniq, inv) = numpy.unique(mapped, return_inverse=True)
                (k, mode) = _modeByKey(segs[sel], inv.astype(numpy.int64), counts[sel])
                vals[self._pos(crossing, k)[0]] = uniq[mode]
            else:
                (k, mode) = _modeByKey(segs[sel], mapped.astype(numpy.int64), counts[sel])
                vals[self._pos(crossing, k)[0]] = mode.astype(self.dtype)

    def settle(self, cr):
        """work on every open entry of own tile cr; True when none is left open"""
        if self.simple:
            return True
        (crossing, vals) = self._crossOf(cr)
        unknown = crossing[vals == self.UNKNOWN]
        if len(unknown) > 0:
            self._resolveCrossing(cr, unknown)
            return not (vals == self.UNKNOWN).any()
        return True

    def crossingIds(self, cr):
        """(labels of the crossing segments of tile cr, their ids; open ones as 0)"""
        (crossing, vals) = self._crossOf(cr)
        return (crossing, numpy.where(vals == self.UNKNOWN, 0, vals).astype(self.dtype))

    def fullLut(self, cr):
        """the whole lut of tile cr (an array over its labels)"""
        self.settle(cr)
        tb = self.tables[cr]
        off = self.dtype.type(self.offsets[cr])
        if self.simple:
            lut = numpy.arange(tb.maxId + 1, dtype=self.dtype) + off
            lut[0] = 0
            return lut
        rel = tb.rel().astype(self.dtype)
        lut = numpy.where(rel > 0, rel + off, self.dtype.type(0))
        (cl, cv) = self.crossingIds(cr)
        lut[cl] = cv
        return lut


def sequentialResolve(order, tables, simple=False):
    """The reference's order, tile after tile (tiling.resolveTile); returns (luts, offsets, maxSegId)."""
    from .tiling import resolveTile
    luts = {}
    offsets = {}
    offset = 0
    for cr in order:
        tb = tables[cr]
        offsets[cr] = offset
        t = _lib.TileTables()
        t.maxId = tb.maxId
        t.countNew = tb.countNew
        t.numPairs = len(tb.pairKeys)
        (lut, trimmedMax) = resolveTile(t, tb.rank, tb.flags, tb.pairKeys, tb.pairCounts, offset,
            luts.get((cr[0], cr[1] - 1)), luts.get((cr[0] - 1, cr[1])), simple)
        luts[cr] = lut
        offset = max(offset, trimmedMax)
    return (luts, offsets, offset)


class LocalComm(object):
    """world of one (and the interface the real communicators implement)"""
    rank = 0
    world = 1

    def allgatherInts(self, values):
        """list of ints from every rank -> list (per rank) of lists"""
        return [list(values)]

    def allgatherBytes(self, b):
        """uint8 array (or bytes) from every rank -> list of uint8 arrays"""
        return [numpy.frombuffer(b, dtype=numpy.uint8) if not isinstance(b, numpy.ndarray) else b]

    def allgatherArray(self, a):
        """int64 array from every rank -> list of int64 arrays"""
        return [numpy.asarray(a, dtype=numpy.int64)]

    def exchange(self, sends, recvs):
        """sends: [(dstRank, tensor)], recvs: [(srcRank, tensor)] in matching order per rank pair"""
        assert not sends and not recvs

    def allreduceSum(self, array):
        return array

    def reduceSum(self, t):
        """device tensor t of every rank -> their sum, on rank 0 (None on the other ranks)"""
        return t


class TorchComm(object):
    """torch.distributed process group (nccl on the GPUs, gloo in the CPU tests)"""
    def __init__(self, device=None):
        import torch
        import torch.distributed as dist
        self.torch = torch
        self.dist = dist
        self.rank = dist.get_rank()
        self.world = dist.get_world_size()
        self.device = device if device is not None else torch.device('cpu')

    def _t(self, a):
        return self.torch.from_numpy(numpy.ascontiguousarray(a)).to(self.device)

    def allgatherInts(self, values):
        n = self._t(numpy.array([len(values)], dtype=numpy.int64))
        sizes = [self.torch.zeros_like(n) for _ in range(self.world)]
        self.dist.all_gather(sizes, n)
        sizes = [int(s.item()) for s in sizes]
        m = max(sizes) if sizes else 0
        mine = numpy.zeros(max(m, 1), dtype=numpy.int64)
        mine[:len(values)] = values
        mine = self._t(mine)
        out = [self.torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(out, mine)
        return [o.cpu().numpy()[:sizes[i]].tolist() for (i, o) in enumerate(out)]

    def allgatherBytes(self, b):
        if not isinstance(b, numpy.ndarray):
            b = numpy.frombuffer(b, dtype=numpy.uint8)
        sizes = [s[0] for s in self.allgatherInts([len(b)])]
        m = max(max(sizes), 1)
        mine = numpy.zeros(m, dtype=numpy.uint8)
        mine[:len(b)] = b
        mine = self._t(mine)
        out = [self.torch.zeros_like(mine) for _ in range(self.world)]
        self.dist.all_gather(out, mine)
        return [o.cpu().numpy()[:sizes[i]] for (i, o) in enumerate(out)]

    def allgatherArray(self, a, quick=1 << 13):
        """int64 array from every rank -> list of int64 arrays.  One collective when every rank's
        array fits `quick` entries (slot 0 carries the length), otherwise the sizes first."""
        a = numpy.ascontiguousarray(a, dtype=numpy.int64)
        torch = self.torch
        if not hasattr(self, '_quickBufs') or self._quickBufs[0].numel() != quick + 1:
            self._quickBufs = (torch.zeros(quick + 1, dtype=torch.int64, device=self.device),
                torch.zeros(self.world * (quick + 1), dtype=torch.int64, device=self.device))
        (mine, everyone) = self._quickBufs
        host = numpy.zeros(quick + 1, dtype=numpy.int64)
        host[0] = len(a)
        if len(a) <= quick:
            host[1:1 + len(a)] = a
        mine.copy_(torch.from_numpy(host))
        self.dist.all_gather_into_tensor(everyone, mine)
        got = everyone.cpu().numpy().reshape(self.world, quick + 1)
        sizes = got[:, 0]
        if (sizes <= quick).all():
            return [got[r, 1:1 + int(sizes[r])].copy() for r in range(self.world)]
        return [b.view(numpy.int64) for b in self.allgatherBytes(a.view(numpy.uint8))]

    def exchange(self, sends, recvs):
        ops = []
        for (dst, t) in sends:
            ops.append(self.dist.P2POp(self.dist.isend, t, dst))
        for (src, t) in recvs:
            ops.append(self.dist.P2POp(self.dist.irecv, t, src))
        if ops:
            for w in self.dist.batch_isend_irecv(ops):
                w.wait()
        if self.device.type == 'cuda':
            self.torch.cuda.synchronize(self.device)

    def allreduceSum(self, array):
        t = self._t(array)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().numpy()

    def reduceSum(self, t):
        self.dist.reduce(t, 0)
        return t if self.rank == 0 else None


class ThreadCommError(RuntimeError):
    """a collective of ThreadComm could not complete: another rank failed or a barrier timed out"""


class ThreadHub(object):
    """What the ThreadComm ranks of one run share: a barrier and one slot per rank.  abort()
    breaks the barrier, so that a rank that fails takes every other rank out of its collective
    at once instead of leaving it waiting."""
    def __init__(self, world, timeout=None):
        self.world = int(world)
        self.barrier = threading.Barrier(self.world, timeout=timeout)
        self.timeout = timeout
        self.slots = [None] * self.world
        self.failed = None       # (rank, exception) of the first rank that failed
        self.lock = threading.Lock()

    def abort(self, rank, exc):
        with self.lock:
            if self.failed is None:
                self.failed = (rank, exc)
        self.barrier.abort()


class ThreadComm(object):
    """
    One rank of a world whose ranks are threads of one process (the LocalComm interface).  The
    collectives are exchanges of host data through the hub's slots between two barriers; the
    strips of exchange() and the histogram of reduceSum() are copied device to device (one plain
    torch copy per strip), so that nothing of a tile's size travels through the host.  `device`
    is the rank's CUDA device (torch.device), or None for host-only use.
    """
    def __init__(self, hub, rank, device=None):
        self.hub = hub
        self.rank = int(rank)
        self.world = hub.world
        self.device = device

    def _wait(self):
        try:
            self.hub.barrier.wait()
        except threading.BrokenBarrierError:
            failed = self.hub.failed
            if failed is not None:
                raise ThreadCommError('rank %d stopped: rank %d failed: %s' % (self.rank, failed[0], failed[1]))
            raise ThreadCommError('rank %d stopped: a rank did not reach the barrier within %s seconds' % (
                self.rank, self.hub.timeout))

    def _allgather(self, value):
        self.hub.slots[self.rank] = value
        self._wait()
        out = list(self.hub.slots)
        self._wait()          # (no rank refills its slot before every rank has read them all)
        return out

    def allgatherInts(self, values):
        return [list(v) for v in self._allgather(list(values))]

    def allgatherBytes(self, b):
        b = numpy.frombuffer(b, dtype=numpy.uint8) if not isinstance(b, numpy.ndarray) else b
        return self._allgather(b.copy())

    def allgatherArray(self, a):
        return self._allgather(numpy.array(a, dtype=numpy.int64))

    def exchange(self, sends, recvs):
        outbox = {}
        for (dst, t) in sends:
            outbox.setdefault(dst, []).append(t)
        boxes = self._allgather(outbox)
        taken = {}
        for (src, t) in recvs:
            i = taken.get(src, 0)
            taken[src] = i + 1
            t.copy_(boxes[src][self.rank][i])
        if recvs and self.device is not None and self.device.type == 'cuda':
            import torch
            torch.cuda.synchronize(self.device)
        self._wait()          # (a sender keeps its strips until every copy out of them has landed)

    def allreduceSum(self, array):
        return numpy.sum(self._allgather(numpy.asarray(array)), axis=0)

    def reduceSum(self, t):
        everyone = self._allgather(t)
        if self.rank == 0:
            import torch
            for other in everyone[1:]:
                t += other.to(t.device)     # (device to device; no copy when on the same device)
            if t.device.type == 'cuda':
                torch.cuda.synchronize(t.device)
        self._wait()          # (the other ranks keep their tensors until rank 0 has added them)
        return t if self.rank == 0 else None


class ShardedStitch(object):
    """
    The stitch of a mosaic whose tiles are spread over the ranks of `comm`.  The caller has
    segmented its own tiles and provides `ops`:

      ops.sendStrip(cr, which)            the LOCAL labels of tile cr's bottom ('bottom': last
                                          overlap rows) or right ('right': last overlap columns)
                                          strip as a contiguous tensor to send
      ops.recvStrip(cr, which, shape)     a tensor to receive such a strip of a remote tile into
      ops.tables(cr, top, left)           TileTable of own tile cr; top / left are None (no such
                                          neighbour), 'local' (the neighbour is an own tile) or
                                          the tensor received for it
      ops.apply(cr, lut, table)           write lut[tile] over the trimmed window of own tile cr
    """
    def __init__(self, tileInfo, overlapSize, simple, comm, timings=None):
        self.timings = timings
        self.tileInfo = tileInfo
        self.overlap = int(overlapSize)
        self.simple = simple
        self.comm = comm
        self.order = rowMajor(tileInfo)
        self.owner = partitionTiles(tileInfo, comm.world)
        self.mine = [cr for cr in self.order if self.owner[cr] == comm.rank]
        self.usedFallback = False
        self.forceSequential = False    # (tests) take the fall-back even if the check passes
        self.earlyTables = {}
        self.received = None
        symbolic = dict((cr, i << self.SHIFT) for (i, cr) in enumerate(self.order))
        self.resolver = LazyResolver({}, symbolic, simple, dtype=numpy.uint64)

    def neighbours(self, cr):
        (c, r) = cr
        up = (c, r - 1) if r > 0 else None
        left = (c - 1, r) if c > 0 else None
        return (up, left)

    def stripPlan(self):
        """(sends, recvs) of this rank as lists of (peerRank, tile, which, shape), in the
        row-major order of the receiving tile (both sides enumerate the same order)."""
        sends = []
        recvs = []
        ov = self.overlap
        if self.simple:
            return (sends, recvs)
        for cr in self.order:
            (xpos, ypos, xsize, ysize) = self.tileInfo.tiles[cr]
            (up, left) = self.neighbours(cr)
            for (nb, which) in ((up, 'bottom'), (left, 'right')):
                if nb is None or self.owner[nb] == self.owner[cr]:
                    continue
                (nx, ny, nxs, nys) = self.tileInfo.tiles[nb]
                shape = (ov, nxs) if which == 'bottom' else (nys, ov)
                if self.owner[nb] == self.comm.rank:
                    sends.append((self.owner[cr], nb, which, shape))
                if self.owner[cr] == self.comm.rank:
                    recvs.append((self.owner[nb], nb, which, shape))
        return (sends, recvs)

    def feedPlan(self):
        """(own tiles whose bottom or right strip a tile of another rank needs, in row-major
        order; after how many finished tiles every rank enters the strip exchange).  A rank that
        segments its feeding tiles FIRST can hand the strips over while it is still busy with
        the rest; the count is the largest number of feeding tiles any rank has, so that no rank
        sits in the exchange long before the strips it is waiting for exist."""
        feeds = dict((r, []) for r in range(self.comm.world))
        if not self.simple:
            for cr in self.order:
                for nb in self.neighbours(cr):
                    if nb is not None and self.owner[nb] != self.owner[cr] and nb not in feeds[self.owner[nb]]:
                        feeds[self.owner[nb]].append(nb)
        mine = sorted(feeds[self.comm.rank], key=lambda cr: (cr[1], cr[0]))
        return (mine, max(len(v) for v in feeds.values()))

    def exchangeStrips(self, ops):
        """The strip exchange, callable before run() (as soon as the feeding tiles are done)."""
        if self.received is None:
            with self._timed('stitch_strips'):
                self.received = self._exchangeStrips(ops)
        return self.received

    def _timed(self, name):
        import contextlib
        return self.timings.interval(name) if self.timings is not None else contextlib.nullcontext()

    def early(self, cr, table):
        """A table of an own tile that exists before run() (the caller computed it while other
        tiles were still being segmented): its lut is worked out as far as the tables at hand
        allow -- with symbolic offsets nothing has to wait for the other ranks' counts."""
        self.earlyTables[cr] = table
        self.resolver.tables[cr] = table
        table.prepare()
        if not self.simple:
            (up, left) = self.neighbours(cr)
            if all(nb is None or nb in self.resolver.tables for nb in (up, left)):
                self.resolver.requests = {}
                self.resolver.settle(cr)

    def run(self, ops):
        """returns (maxSegId, offsets of all tiles, luts of own tiles)"""
        received = self.exchangeStrips(ops)
        with self._timed('stitch_owntables'):
            tables = self._ownTables(ops, received)
        with self._timed('stitch_resolve'):
            (final, luts, offsets, maxSegId) = self._resolve(tables)
        with self._timed('stitch_apply'):
            for cr in self.mine:
                if cr in luts:
                    ops.apply(cr, luts[cr], tables[cr])
                elif hasattr(ops, 'applyRel'):
                    # offset + rank for the tile's own segments is left to the device; the host
                    # only hands over the ids of the crossing segments
                    ops.applyRel(cr, offsets[cr], final[cr][0], final[cr][1], tables[cr])
                else:
                    luts[cr] = self._fullLut(tables[cr], offsets[cr], final[cr])
                    ops.apply(cr, luts[cr], tables[cr])
        return (maxSegId, offsets, luts)

    def _fullLut(self, tb, offset, crossFinal):
        if self.simple:
            lut = numpy.arange(tb.maxId + 1, dtype=numpy.uint32) + numpy.uint32(offset)
            lut[0] = 0
            return lut
        rel = tb.rel()
        lut = numpy.where(rel > 0, rel + numpy.uint32(offset), numpy.uint32(0)).astype(numpy.uint32)
        lut[crossFinal[0]] = crossFinal[1]
        return lut

    def _exchangeStrips(self, ops):
        comm = self.comm
        # 1. strips of remote neighbours
        (sends, recvs) = self.stripPlan()
        received = {}
        sendList = [(peer, ops.sendStrip(cr, which)) for (peer, cr, which, shape) in sends]
        recvList = []
        for (peer, cr, which, shape) in recvs:
            t = ops.recvStrip(cr, which, shape)
            received[(cr, which)] = t
            recvList.append((peer, t))
        comm.exchange(sendList, recvList)
        return received

    def _ownTables(self, ops, received):
        comm = self.comm
        # 2. tables of own tiles
        tables = {}
        for cr in self.mine:
            if cr in self.earlyTables:
                tables[cr] = self.earlyTables[cr]
                continue
            (up, left) = self.neighbours(cr)
            top = lf = None
            if not self.simple:
                if up is not None:
                    top = 'local' if self.owner[up] == comm.rank else received[(up, 'bottom')]
                if left is not None:
                    lf = 'local' if self.owner[left] == comm.rank else received[(left, 'right')]
            tables[cr] = ops.tables(cr, top, lf)
            self.resolver.tables[cr] = tables[cr]
        return tables

    # The id offset of a tile is the sum of one integer per earlier tile, which the other ranks
    # only know when they are done.  Nothing else in the resolve needs the offsets' VALUES: ids
    # are handled as (index of the tile that numbered the segment) << 32 | rank, which sort like
    # the final ids (offsets grow with the tile index) and are equal exactly when those are, and
    # are turned into offset + rank at the very end.
    SHIFT = 32

    def _stepOf(self, tb):
        # The reference moves the running maximum on tile after tile:
        # maxSegId = max(maxSegId, trimmed.max()) (tiling.py:1042-1043).  Inside the trimmed
        # window a tile has its own numbered segments (offset + rank) and segments recoded to ids
        # of EARLIER tiles; unless one of those carries an id above the running maximum (a
        # neighbour's segment that was numbered without having a pixel in its own trimmed
        # window), the maximum moves on by the highest rank present in the window.  Take that as
        # the hypothesis -- offsets = running sum of one integer per tile -- and check the
        # recurrence on every tile afterwards.
        if self.simple:
            return tb.maxLabelInTrim
        tb.prepare()
        return tb.cachedMaxRankInTrim

    def _translate(self, lut, realOffsets):
        idx = (lut >> numpy.uint64(self.SHIFT)).astype(numpy.int64)
        return (realOffsets[idx] + (lut & numpy.uint64((1 << self.SHIFT) - 1))).astype(numpy.uint32)

    def _resolve(self, tables):
        comm = self.comm
        resolver = self.resolver
        index = dict((cr, i) for (i, cr) in enumerate(self.order))
        # Final ids of own tiles.  A crossing segment takes the final id of the neighbour
        # segment it overlaps most; when that neighbour tile lives on another rank its OWNER is
        # asked for the (symbolic) final ids of the labels in question (a few thousand per
        # boundary tile), and answers what it has settled.  An id inherited through several
        # tiles around a corner takes one more round per hop.  The first message of a rank also
        # carries the steps of its tiles, its last one the outcome of its check.
        steps = {}
        offsets = None
        realOffsets = None
        luts = {}       # whole luts: only after the fall-back
        final = {}      # own tile -> (labels of its crossing segments, their final ids)
        ok = None
        first = True
        for _round in range(len(self.order) + 4):
            resolver.requests = {}
            with self._timed('resolve_settle'):
                for cr in self.mine:          # (entries settled earlier are kept)
                    resolver.settle(cr)
            msg = []
            if first:
                head = [len(self.mine)]
                for cr in self.mine:
                    head += [cr[0], cr[1], self._stepOf(tables[cr])]
                msg.append(numpy.array(head, dtype=numpy.int64))
            nReq = len(resolver.requests)
            if nReq == 0 and not first and ok is None:
                # everything of this rank is settled and the offsets are known: translate and
                # check the hypothesis
                ok = 1
                for cr in self.mine:
                    tb = tables[cr]
                    (cl, cv) = resolver.crossingIds(cr)
                    final[cr] = (cl, self._translate(cv, realOffsets))
                    if self.simple:
                        trimmedMax = offsets[cr] + tb.maxLabelInTrim if tb.maxLabelInTrim else 0
                    else:
                        trimmedMax = offsets[cr] + tb.cachedMaxRankInTrim if tb.cachedMaxRankInTrim else 0
                        if tb.crossInTrimMask.any():
                            trimmedMax = max(trimmedMax, int(final[cr][1][tb.crossInTrimMask].max()))
                    if max(offsets[cr], trimmedMax) != offsets[cr] + steps[cr] or self.forceSequential:
                        ok = 0
            msg.append(numpy.array([nReq, -1 if ok is None else ok], dtype=numpy.int64))
            for (cr, parts) in sorted(resolver.requests.items()):
                labels = numpy.unique(numpy.concatenate(parts))
                msg += [numpy.array([cr[0], cr[1], len(labels)], dtype=numpy.int64), labels]
            with self._timed('resolve_gather%d' % min(_round, 2)):
                allReq = comm.allgatherArray(numpy.concatenate(msg))
            asked = []
            states = []
            for a in allReq:
                o = 0
                if first:
                    n = int(a[0])
                    for i in range(n):
                        steps[(int(a[1 + 3 * i]), int(a[2 + 3 * i]))] = int(a[3 + 3 * i])
                    o = 1 + 3 * n
                (n, state) = (int(a[o]), int(a[o + 1]))
                o += 2
                states.append(state)
                for _ in range(n):
                    (c, r, m) = (int(v) for v in a[o:o + 3])
                    asked.append(((c, r), a[o + 3:o + 3 + m]))
                    o += 3 + m
            if first:
                first = False
                offsets = {}
                realOffsets = numpy.zeros(len(self.order) + 1, dtype=numpy.uint64)
                offset = 0
                for (i, cr) in enumerate(self.order):
                    offsets[cr] = offset
                    realOffsets[i] = offset
                    offset += steps[cr]
                maxSegId = offset
            if not asked:
                if all(st >= 0 for st in states):
                    break
                continue          # (someone settled in this round and reports its check next)
            ans = []
            for (cr, labels) in asked:
                if self.owner[cr] == comm.rank:
                    (lab, vals) = resolver.answer(cr, labels)
                    ans += [numpy.array([cr[0], cr[1], len(lab)], dtype=numpy.int64), lab, vals.astype(numpy.int64)]
            with self._timed('resolve_answers'):
                allAns = comm.allgatherArray(numpy.concatenate(ans) if ans else numpy.zeros(0, numpy.int64))
            for a in allAns:
                o = 0
                while o < len(a):
                    (c, r, n) = (int(v) for v in a[o:o + 3])
                    if (c, r) in resolver.requests:
                        resolver.addRemote((c, r), a[o + 3:o + 3 + n], a[o + 3 + n:o + 3 + 2 * n].astype(numpy.uint64))
                    o += 3 + 2 * n
        else:
            raise RuntimeError('sharded stitch: look-ups across ranks did not settle')
        if min(states) == 0:
            # some window holds an inherited id above the running maximum: replay the
            # reference's sequential order over all tables, on every rank
            self.usedFallback = True
            known = {}
            for b in comm.allgatherBytes(packTables(tables)):
                known.update(unpackTables(b))
            (allLuts, offsets, maxSegId) = sequentialResolve(self.order, known, self.simple)
            luts = dict((cr, allLuts[cr]) for cr in self.mine)

        return (final, luts, offsets, maxSegId)

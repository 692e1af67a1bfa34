"""
Time the tiled segmentation of one 10980 x 10980 x 4 scene held as uint16, as uint32 and as int32.

    python tools/bench_wide_values.py --out DIR [--runs 3] [--size 10980]

The uint16 scene is bench.py's synthetic Sentinel-2-like raster (synth.synth_tiled, seed 1).  The
uint32 variant is the same scene times 65537 (up to about 4.3e9), the int32 one is
(scene - 2000) * 500000 (about -7.5e8 .. 1.2e9); their centres are the uint16 centres mapped the same
way.  Each run is doTiledShepherdSegmentation from host memory into a host mosaic, tile 4096,
overlap 1024, k = 60 fixed centres, minSegmentSize 50, three segmentation workers.  After one
warm-up run of each variant the variants alternate, `runs` rounds.

DIR/bench_wide_values.json gets, per variant: host ms per scene, Mpixel/s, the device ms of the
stages summed over the tiles, and the share of segments whose float32 band sums are not exact and
so take the ordered (raster-order) accumulation.  That share is worked out on tile (0, 0), from
the labels after the single-pixel stage, with the rule of eliminate.cu (k_finalize_sums2).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyshepseg_b200 import rasterfile, shepseg, synth, tiling  # noqa: E402


class KM(object):
    def __init__(self, centres):
        self.cluster_centers_ = numpy.ascontiguousarray(centres, dtype=numpy.float64)


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv'],
        capture_output=True, text=True, check=True).stdout
    return out.strip().splitlines()


def ordered_share(img, centres, tileSize, overlap):
    (nB, nR, nC) = img.shape
    ti = tiling.getTilesForFile((nC, nR), tileSize, overlap)
    (x, y, xs, ys) = ti.tiles[(0, 0)]
    sub = numpy.ascontiguousarray(img[:, y:y + ys, x:x + xs])
    km = KM(centres)
    clusters = shepseg.applySpectralClusters(km, sub, None)
    (seg, nextId) = shepseg.clump(clusters, shepseg.SEGNULLVAL, True, shepseg.MINSEGID)
    segSize = shepseg.makeSegSize(seg)
    shepseg.eliminateSinglePixels(sub, seg, segSize, shepseg.MINSEGID, nextId - 1, True)
    ids = seg.ravel()
    n = int(ids.max()) + 1
    size = numpy.bincount(ids, minlength=n)[1:].astype(numpy.float64)
    sums = numpy.array([numpy.bincount(ids, weights=sub[b].ravel().astype(numpy.float64), minlength=n)[1:]
        for b in range(nB)])
    alive = size > 0
    if img.dtype == numpy.uint16:
        big = (sums >= 2.0 ** 24).any(axis=0) | (size * 65535 >= 2.0 ** 32)
    elif img.dtype == numpy.uint32:
        big = (sums >= 2.0 ** 24).any(axis=0)
    else:
        big = size * 2.0 ** 31 >= 2.0 ** 24
    return {'segments': int(alive.sum()), 'ordered': int((big & alive).sum()),
        'share': float((big & alive).sum() / max(1, alive.sum()))}


def main():
    ap = argparse.ArgumentParser(description=__doc__.strip().splitlines()[0])
    ap.add_argument('--out', required=True)
    ap.add_argument('--runs', type=int, default=3)
    ap.add_argument('--size', type=int, default=10980)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    (tileSize, overlap, k, minSeg, workers) = (4096, 1024, 60, 50, 3)
    info = gpu_info()
    print('\n'.join(info), flush=True)

    t = time.time()
    u16 = synth.synth_tiled(args.size, args.size, 4, seed=1)
    c16 = synth.diagonal_centres(u16, k)
    u32 = u16.astype(numpy.uint32)
    u32 *= numpy.uint32(65537)
    i32 = u16.astype(numpy.int32)
    i32 -= 2000
    i32 *= 500000
    variants = {
        'uint16': (u16, c16),
        'uint32': (u32, c16 * 65537.0),
        'int32': (i32, (c16 - 2000.0) * 500000.0),
    }
    print('scene ready in %.1f s' % (time.time() - t), flush=True)

    nPix = args.size * args.size
    results = dict((name, {'ms': [], 'stage_ms': []}) for name in variants)
    sinks = dict((name, rasterfile.MemorySink(args.size, args.size)) for name in variants)

    def run(name):
        (img, centres) = variants[name]
        cfg = tiling.SegmentationConcurrencyConfig(concurrencyType=tiling.CONC_THREADS, numWorkers=workers,
            tileCompletionTimeout=600)
        t0 = time.perf_counter()
        res = tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img), sinks[name], tileSize=tileSize,
            overlapSize=overlap, minSegmentSize=minSeg, numClusters=k, kmeansObj=KM(centres),
            concurrencyCfg=cfg)
        ms = (time.perf_counter() - t0) * 1e3
        return (ms, dict(res.stageMs), int(res.maxSegId))

    for name in variants:
        (ms, _, maxSegId) = run(name)
        results[name]['maxSegId'] = maxSegId
        print('warm-up %s: %.0f ms, maxSegId %d' % (name, ms, maxSegId), flush=True)
    for r in range(args.runs):
        for name in variants:
            (ms, stages, _) = run(name)
            results[name]['ms'].append(round(ms, 2))
            results[name]['stage_ms'].append(dict((s, round(v, 2)) for (s, v) in stages.items()))
            print('run %d %s: %.0f ms  %s' % (r, name, ms, stages), flush=True)

    for (name, (img, centres)) in variants.items():
        d = results[name]
        med = float(numpy.median(d['ms']))
        d['ms_median'] = round(med, 2)
        d['mpix_per_s'] = round(nPix / med / 1e3, 1)
        d['stage_ms_median'] = dict((s, round(float(numpy.median([x[s] for x in d['stage_ms']])), 2))
            for s in d['stage_ms'][0])
        d['ordered_sums_tile00'] = ordered_share(img, centres, tileSize, overlap)
    out = {'gpu': info, 'scene': '%dx%dx4' % (args.size, args.size), 'tileSize': tileSize,
        'overlapSize': overlap, 'numClusters': k, 'minSegmentSize': minSeg, 'workers': workers,
        'runs': args.runs, 'variants': results}
    with open(os.path.join(args.out, 'bench_wide_values.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()

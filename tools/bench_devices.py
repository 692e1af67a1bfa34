"""
tools/bench_devices.py -- doTiledShepherdSegmentation on 1, 2, 4, ... GPUs of one box from ONE process
(CONC_THREADS, devices=[0 .. n-1]), host to host: the raster in pinned host memory (MemoryRaster),
the mosaic delivered into a pinned host MemorySink, every copy inside the timed call.

    python tools/bench_devices.py --out DIR [--workloads c4,c2] [--rounds 3] [--workers-per-device 3]
                                  [--c4-devices 1,2,4,8] [--c2-devices 1,2,4] [--shards-on-device0 2,4]
                                  [--timeline]

Workloads (bench.py's): c4 is the 40000 x 40000 x 4 uint16 mosaic (a seeded 10000 x 10000 patch laid
out 4 x 4, every other copy mirrored), c2 one 10980 x 10980 x 4 scene; tile 4096, overlap 1024,
k = 60 fixed centres (synth.diagonal_centres), minSegmentSize 50, maxSpectralDiff 'auto',
four-connected.  Device counts above the visible devices are skipped and listed as such; the
1-device configuration always runs first, whatever the lists say, as the parity reference.
--shards-on-device0 adds configurations 'Sx1' that run S shards all on GPU 0 (the
concurrencyCfg.shardDevices the tests use): not a scaling figure, but what the in-process
machinery (threads, ThreadComm, the shared sink) costs on one GPU.

Method: one warm-up call per configuration, then --rounds rounds in which the configurations of a
workload alternate.  Every call's mosaic (the whole array), maxSegId and histogram are compared
with the 1-device warm-up call's.  With --timeline the last call of every configuration runs again
with SSG_TIMELINE set and its per-device timeline (host ms since the call started) is kept.
Writes DIR/bench_devices.json: Mpixel/s (median and all calls) per device count, the device ms per
stage summed over the devices, the parity flags, the card name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pyshepseg_b200 import _lib, rasterfile, synth, tiling  # noqa: E402

PARAMS = {'tileSize': 4096, 'overlapSize': 1024, 'numClusters': 60, 'minSegmentSize': 50,
    'maxSpectralDiff': 'auto', 'fourConnected': True}


class KM(object):
    def __init__(self, centres):
        self.cluster_centers_ = numpy.ascontiguousarray(centres, dtype=numpy.float64)


def c4_raster():
    """bench.py's c4_40000 mosaic, built on the host"""
    (nB, N, P) = (4, 40000, 10000)
    patch = synth.synth_tiled(P, P, nB, seed=1)
    i = numpy.arange(N) % (2 * P)
    idx = numpy.where(i < P, i, 2 * P - 1 - i)
    img = _lib.PinnedArray((nB, N, N), numpy.uint16)
    for b in range(nB):
        rows = patch[b][idx]
        for r0 in range(0, N, 4000):
            img.array[b, r0:r0 + 4000] = rows[r0:r0 + 4000][:, idx]
    return (img, synth.diagonal_centres(patch, PARAMS['numClusters']))


def c2_raster():
    """bench.py's workload: one 10980 x 10980 x 4 scene"""
    img = _lib.PinnedArray((4, 10980, 10980), numpy.uint16)
    synth.synth_tiled(10980, 10980, 4, seed=1, out=img.array)
    return (img, synth.diagonal_centres(img.array, PARAMS['numClusters']))


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=index,name,power.limit,clocks.max.sm', '--format=csv,noheader'],
            capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except Exception as e:
        q = ['nvidia-smi unavailable: %s' % e]
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--workloads', default='c4,c2')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--workers-per-device', type=int, default=3)
    ap.add_argument('--c4-devices', default='1,2,4,8')
    ap.add_argument('--c2-devices', default='1,2,4')
    ap.add_argument('--shards-on-device0', default='')
    ap.add_argument('--timeline', action='store_true')
    args = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    if visible < 1:
        raise SystemExit('no CUDA device: this measures GPUs')
    report = {'cards_before': card(), 'visible_devices': visible, 'params': PARAMS,
        'workers_per_device': args.workers_per_device, 'workloads': {}}
    for wl in args.workloads.split(','):
        counts = [int(v) for v in getattr(args, wl + '_devices').split(',')]
        counts = [1] + [n for n in counts if n != 1]     # (the 1-device call is the parity reference)
        skipped = [n for n in counts if n > visible]
        counts = [n for n in counts if n <= visible]
        counts += ['%dx1' % int(v) for v in args.shards_on_device0.split(',') if v]
        t0 = time.time()
        (img, centres) = c4_raster() if wl == 'c4' else c2_raster()
        (nB, nR, nC) = img.array.shape
        print('%s: raster %s made in %.0f s' % (wl, img.array.shape, time.time() - t0), file=sys.stderr, flush=True)
        out = _lib.PinnedArray((nR, nC), numpy.uint32)
        src = rasterfile.MemoryRaster(img.array)
        km = KM(centres)

        def call(n):
            out.array.fill(0xFFFFFFFF)     # (a window that is not written shows)
            shards = [0] * int(n[:-2]) if isinstance(n, str) else list(range(n))
            cfg = tiling.SegmentationConcurrencyConfig(tiling.CONC_THREADS, numWorkers=args.workers_per_device * len(shards),
                devices=shards[:1] if isinstance(n, str) else shards, tileCompletionTimeout=600)
            if isinstance(n, str):
                cfg.shardDevices = shards
            sink = rasterfile.MemorySink(nC, nR, array=out.array)
            t = time.perf_counter()
            res = tiling.doTiledShepherdSegmentation(src, sink, tileSize=PARAMS['tileSize'],
                overlapSize=PARAMS['overlapSize'], minSegmentSize=PARAMS['minSegmentSize'],
                numClusters=PARAMS['numClusters'], maxSpectralDiff=PARAMS['maxSpectralDiff'],
                fourConnected=PARAMS['fourConnected'], kmeansObj=km, concurrencyCfg=cfg, returnGDALDS=True)
            return (time.perf_counter() - t, res)

        ref = None
        rec = dict((n, {'seconds': [], 'stage_ms': [], 'parity': []}) for n in counts)

        def record(n, secs, res):
            (mosaic, hist, maxSegId) = ref
            ok = {'mosaic': bool(numpy.array_equal(out.array, mosaic)), 'maxSegId': int(res.maxSegId) == maxSegId,
                'histogram': bool(numpy.array_equal(res.outDs.hist, hist))}
            rec[n]['parity'].append(ok)
            rec[n]['seconds'].append(secs)
            rec[n]['stage_ms'].append(dict(res.stageMs))
            print('  %s %s device(s): %.1f ms, %.0f Mpixel/s, parity %s' % (wl, n, secs * 1e3, nR * nC / secs / 1e6,
                all(ok.values())), file=sys.stderr, flush=True)
        for n in counts:      # warm-up, one call per configuration; the first, on 1 device, is the reference
            (secs, res) = call(n)
            if ref is None:
                ref = (out.array.copy(), numpy.array(res.outDs.hist), int(res.maxSegId))
            rec[n]['warmup_seconds'] = secs
            rec[n]['warmup_parity'] = {'mosaic': bool(numpy.array_equal(out.array, ref[0])),
                'maxSegId': int(res.maxSegId) == ref[2], 'histogram': bool(numpy.array_equal(res.outDs.hist, ref[1]))}
        for _ in range(args.rounds):
            for n in counts:
                record(n, *call(n))
        if args.timeline:
            os.environ['SSG_TIMELINE'] = '1'
            for n in counts:
                (secs, res) = call(n)
                rec[n]['timeline'] = {'seconds': secs, 'entries': res.timeline}
            del os.environ['SSG_TIMELINE']
        summary = {}
        for n in counts:
            s = rec[n]['seconds']
            med = float(numpy.median(s))
            summary[str(n)] = {'mpixel_per_s': nR * nC / med / 1e6, 'median_ms': med * 1e3,
                'all_ms': [round(v * 1e3, 1) for v in s],
                'stage_ms_median': dict((k, float(numpy.median([d[k] for d in rec[n]['stage_ms']])))
                    for k in rec[n]['stage_ms'][0]),
                'parity': all(all(p.values()) for p in rec[n]['parity']) and all(rec[n]['warmup_parity'].values()),
                'warmup_ms': rec[n]['warmup_seconds'] * 1e3}
            if 'timeline' in rec[n]:
                summary[str(n)]['timeline'] = rec[n]['timeline']
        report['workloads'][wl] = {'raster': [nB, nR, nC], 'segments': ref[2], 'devices': summary,
            'skipped_device_counts': skipped}
        del src, out, img
    report['cards_after'] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, 'bench_devices.json'), 'w') as f:
        json.dump(report, f, indent=1)
    brief = dict((wl, dict((n, (round(v['mpixel_per_s']), v['parity'])) for (n, v) in w['devices'].items()))
        for (wl, w) in report['workloads'].items())
    print(json.dumps(brief))


if __name__ == '__main__':
    main()

"""
Time the segmentation of one 10980 x 10980 scene of 16, 32 and 64 uint16 bands.

    python tools/bench_many_bands.py --out DIR [--runs 3] [--size 10980] [--bands 16,32,64]

The scene's first 16 bands are bench.py's synthetic raster generator (synth.synth_tiled, seed 1)
at 16 bands; band 16 j + b of the wider scenes is band (b + 5 j) % 16 rolled by 37 j rows and 53 j
columns, so that no two bands are equal.  k = 60 fixed diagonal centres, minSegmentSize 50,
maxSpectralDiff 'auto', four-connected.  Per band count:

  * resident: the scene is uploaded once (ssg_upload_image) and segmented as one tile from device
    memory (ssg_segment_tile_device), one warm-up and `runs` timed calls: the median of every ms*
    field of ssg_tile_result; then `runs` calls with per-launch events (ssg_profile_*) for the
    device time of the assignment kernel alone, against two lower bounds: FFMA (N k nB fused
    multiply-adds at 148 SMs x 128 lanes x the card's maximum SM clock) and bytes (N (2 nB + 4) at
    the 6.55 TB/s copy rate DESIGN.md records);
  * host to host: doTiledShepherdSegmentation from host memory into a host mosaic, tile 4096,
    overlap 1024, three segmentation workers, one warm-up and `runs` timed runs: Mpixel/s.

The card's name, power limit and maximum SM clock are read in the same run and written with the
numbers to DIR/bench_many_bands.json.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyshepseg_b200 import _lib, rasterfile, shepseg, synth, tiling  # noqa: E402

HBM_BYTES_PER_S = 6.55e12      # DESIGN.md: measured device-to-device copy rate of one B200
STAGES = ('msAssign', 'msClump', 'msSingle', 'msSmall', 'msTotal')


class KM(object):
    def __init__(self, centres):
        self.cluster_centers_ = numpy.ascontiguousarray(centres, dtype=numpy.float64)


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
        capture_output=True, text=True, check=True).stdout
    return out.strip().splitlines()


def scene(base, bands):
    if bands <= base.shape[0]:
        return numpy.ascontiguousarray(base[:bands])
    img = numpy.empty((bands,) + base.shape[1:], dtype=base.dtype)
    for i in range(bands):
        (j, b) = divmod(i, base.shape[0])
        img[i] = numpy.roll(base[(b + 5 * j) % base.shape[0]], (37 * j, 53 * j), axis=(0, 1))
    return img


def assign_ms(ctx):
    buf = ctypes.create_string_buffer(1 << 16)
    ctx.call('ssg_profile_fetch', buf, len(buf))
    for line in buf.value.decode().splitlines():
        (name, count, total) = line.split()
        if name in ('k_assign', 'k_assign_many', 'k_assign_grid'):
            return (name, float(total) / int(count))
    raise RuntimeError('no assignment kernel in the profile')


def resident(img, centres, runs, clockMHz):
    (nB, nR, nC) = img.shape
    N = nR * nC
    k = centres.shape[0]
    ctx = _lib.Context(0)
    try:
        ctx.call('ssg_upload_image', _lib.ptr(img), _lib.DTYPE_CODES[img.dtype], nB, nR, nC)
        dev = ctx.lib.ssg_staged_image(ctx.h)
        thr = shepseg.spectralThreshold(shepseg.autoMaxSpectralDiff(KM(centres), 'auto', 50))
        prm = shepseg.makeTileParams(img.dtype, nB, nR, nC, centres, None, True, 50, thr)
        fields = dict((s, []) for s in STAGES)
        for r in range(runs + 1):
            res = _lib.TileResult()
            ctx.call('ssg_segment_tile_device', dev, ctypes.byref(prm), None, ctypes.byref(res))
            if r > 0:
                for s in STAGES:
                    fields[s].append(round(float(getattr(res, s)), 3))
        # the kernel times in runs of their own: the profile brackets every launch with events
        kern = []
        ctx.call('ssg_profile_enable', 1)
        for r in range(runs):
            ctx.call('ssg_profile_fetch', ctypes.create_string_buffer(1 << 16), 1 << 16)      # (reset)
            ctx.call('ssg_segment_tile_device', dev, ctypes.byref(prm), None, ctypes.byref(_lib.TileResult()))
            ctx.synchronize()
            (name, ms) = assign_ms(ctx)
            kern.append(round(ms, 3))
        ctx.call('ssg_profile_enable', 0)
        ffmaMs = N * k * nB / (148 * 128 * clockMHz * 1e6) * 1e3
        bytesMs = N * (2 * nB + 4) / HBM_BYTES_PER_S * 1e3
        med = float(numpy.median(kern))
        return {'stage_ms_median': dict((s, float(numpy.median(v))) for (s, v) in fields.items()),
            'stage_ms': fields, 'segments': int(res.numSegments),
            'assign_kernel': name, 'assign_kernel_ms': kern, 'assign_kernel_ms_median': med,
            'ffma_bound_ms': round(ffmaMs, 3), 'bytes_bound_ms': round(bytesMs, 3),
            'assign_share_of_ffma_bound': round(ffmaMs / med, 3)}
    finally:
        ctx.close()


def host_to_host(img, centres, runs):
    (nB, nR, nC) = img.shape
    sink = rasterfile.MemorySink(nC, nR)
    ms = []
    for r in range(runs + 1):
        cfg = tiling.SegmentationConcurrencyConfig(concurrencyType=tiling.CONC_THREADS, numWorkers=3,
            tileCompletionTimeout=900)
        t0 = time.perf_counter()
        res = tiling.doTiledShepherdSegmentation(rasterfile.MemoryRaster(img), sink, tileSize=4096,
            overlapSize=1024, minSegmentSize=50, numClusters=centres.shape[0], kmeansObj=KM(centres),
            concurrencyCfg=cfg)
        if r > 0:
            ms.append(round((time.perf_counter() - t0) * 1e3, 1))
    med = float(numpy.median(ms))
    return {'ms': ms, 'ms_median': med, 'mpix_per_s': round(nR * nC / med / 1e3, 1), 'maxSegId': int(res.maxSegId)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.strip().splitlines()[0])
    ap.add_argument('--out', required=True)
    ap.add_argument('--runs', type=int, default=3)
    ap.add_argument('--size', type=int, default=10980)
    ap.add_argument('--bands', default='16,32,64')
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    info = gpu_info()
    print('\n'.join(info), flush=True)
    clockMHz = float(info[0].split(',')[2].split()[0])

    t = time.time()
    base = synth.synth_tiled(args.size, args.size, 16, seed=1)
    print('16-band scene ready in %.1f s' % (time.time() - t), flush=True)
    out = {'gpu': info, 'size': args.size, 'numClusters': 60, 'minSegmentSize': 50, 'runs': args.runs,
        'bands': {}}
    for bands in [int(b) for b in args.bands.split(',')]:
        img = scene(base, bands)
        centres = synth.diagonal_centres(img, 60)
        r = {'resident': resident(img, centres, args.runs, clockMHz)}
        print('%d bands resident: %s' % (bands, json.dumps(r['resident'])), flush=True)
        r['host_to_host'] = host_to_host(img, centres, args.runs)
        print('%d bands host to host: %s' % (bands, json.dumps(r['host_to_host'])), flush=True)
        out['bands'][str(bands)] = r
        del img
    with open(os.path.join(args.out, 'bench_many_bands.json'), 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()

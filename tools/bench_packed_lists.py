"""
Time the small-segment stage with packed pixel lists.

    python tools/bench_packed_lists.py [--out DIR] [--runs 5] [--size 4096]

Packed lists are what the merge uses when per-segment list regions would take too much memory (a
large minSegmentSize on a large tile); SSG_SMALL_REGION_MB=0 forces them at any size.  The tile is
bench.py's synthetic raster (synth.synth_tiled, seed 1, 4 bands, uint16) with k = 60 fixed
diagonal centres, maxSpectralDiff 'auto', four-connected.  Each configuration, minSegmentSize 50
and 1000, each with the default arena and with SSG_SMALL_ARENA_PCT=7 (the arena runs out and later
merges chain), runs once to warm up and then `runs` times through ssg_segment_tile.

Per configuration it prints, and writes to DIR/bench_packed_lists.json, the median and spread of
msSmall (the device time of the small-segment stage, ssg_tile_result), the pass count and the
SHA-256 of the label raster.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyshepseg_b200 import _lib, shepseg, synth  # noqa: E402

CONFIGS = [
    ('minseg50_arena', 50, {}),
    ('minseg50_arena_pct7', 50, {'SSG_SMALL_ARENA_PCT': '7'}),
    ('minseg1000_arena', 1000, {}),
    ('minseg1000_arena_pct7', 1000, {'SSG_SMALL_ARENA_PCT': '7'}),
]


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv'],
        capture_output=True, text=True, check=True).stdout
    return out.strip().splitlines()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument('--out', default=None)
    ap.add_argument('--runs', type=int, default=5)
    ap.add_argument('--size', type=int, default=4096)
    args = ap.parse_args()

    img = synth.synth_tiled(args.size, args.size, 4, seed=1)
    centres = numpy.ascontiguousarray(synth.diagonal_centres(img, 60), dtype=numpy.float64)
    thr = shepseg.spectralThreshold(shepseg.autoMaxSpectralDiff(centres, 'auto', 50))
    seg = numpy.empty(img.shape[1:], dtype=numpy.uint32)
    ctx = _lib.Context(0)
    report = {'gpu': gpu_info(), 'size': args.size, 'runs': args.runs, 'configs': {}}
    for (name, minSeg, env) in CONFIGS:
        env = dict(env, SSG_SMALL_REGION_MB='0')
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            ms = []
            for i in range(args.runs + 1):
                res = shepseg.segmentTile(ctx, img, centres, None, True, minSeg, thr, seg)
                if i > 0:
                    ms.append(float(res.msSmall))
        finally:
            for (k, v) in saved.items():
                if v is None:
                    del os.environ[k]
                else:
                    os.environ[k] = v
        r = {'msSmall_median': float(numpy.median(ms)), 'msSmall_min': min(ms), 'msSmall_max': max(ms),
            'numSmallPasses': int(res.numSmallPasses), 'smallSegmentsEliminated': int(res.smallSegmentsEliminated),
            'labels_sha256': hashlib.sha256(seg.tobytes()).hexdigest()}
        report['configs'][name] = r
        print('%-24s msSmall median %8.2f (%.2f .. %.2f)  passes %5d  eliminated %8d  labels %s' % (
            name, r['msSmall_median'], r['msSmall_min'], r['msSmall_max'], r['numSmallPasses'],
            r['smallSegmentsEliminated'], r['labels_sha256'][:16]))
    ctx.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'bench_packed_lists.json'), 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()

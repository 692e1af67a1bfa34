"""
The CPU oracle on uint32 and int32 images at full 32-bit range: its assignment against
scikit-learn's KMeans.predict, which the reference calls (shepseg.py:317-361), and, where the
reference is installed in oracle/_ref/, the whole segmentation against the unmodified reference.
"""
import json
import os
import subprocess
import sys
import warnings

import numpy
import pytest

from oracle import oracle
from pyshepseg_b200 import synth
import goldenutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.path.join(ROOT, 'oracle', '_ref')


def full_range_image(dtype, seed):
    """512 x 512 x 3: smooth fields spread over the whole range of dtype, a null wedge"""
    info = numpy.iinfo(dtype)
    base = synth.synth_v1(512, 512, 3, seed=seed, lo=1.0, hi=65534.0, noise=500.0).astype(numpy.float64)
    img = numpy.rint(info.min + (base - 1.0) / 65533.0 * (float(info.max) - float(info.min)))
    img = numpy.clip(img, info.min, info.max).astype(dtype)
    rr = numpy.arange(512)[:, None]
    cc = numpy.arange(512)[None, :]
    img[:, (rr + cc) < 80] = info.max
    return img


@pytest.mark.parametrize('dtype', [numpy.uint32, numpy.int32])
def test_oracle_assignment_equals_sklearn_predict(dtype):
    from sklearn.cluster import KMeans
    img = full_range_image(dtype, seed=7 if dtype == numpy.uint32 else 8)
    nullVal = int(numpy.iinfo(dtype).max)
    centres = synth.diagonal_centres(img, 30, nullVal)
    km = KMeans(n_clusters=len(centres), n_init=1, init=centres, max_iter=1)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        km.fit(centres)
    km.cluster_centers_ = centres
    pixels = numpy.moveaxis(img, 0, -1).reshape(-1, img.shape[0])
    want = km.predict(pixels).astype(numpy.int32) + 1
    want[(pixels == nullVal).any(axis=1)] = 0
    got = oracle.applySpectralClusters(goldenutil.Centres(centres), img, nullVal)
    assert numpy.array_equal(got.ravel(), want)
    assert len(numpy.unique(got)) > 20


RUNNER = r'''
import json, sys, warnings
import numpy
sys.path.insert(0, %(ref)r)
from sklearn.cluster import KMeans
from pyshepseg import shepseg
spec = json.load(open(sys.argv[1]))
for c in spec['cases']:
    d = numpy.load(c['npz'])
    centres = d['centres']
    km = KMeans(n_clusters=len(centres), n_init=1, init=centres, max_iter=1)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        km.fit(centres)
    km.cluster_centers_ = centres
    res = shepseg.doShepherdSegmentation(d['img'], numClusters=len(centres), minSegmentSize=c['minSeg'],
        maxSpectralDiff=c['msd'], imgNullVal=c['nullVal'], fourConnected=c['four'], kmeansObj=km)
    numpy.savez(c['out'], segimg=res.segimg, single=int(res.singlePixelsEliminated),
        small=int(res.smallSegmentsEliminated))
'''


def live_cases():
    """(img, centres, minSeg, msd, nullVal, four): wide uint32 and int32 fields, and single pixels
    whose squared distance to the neighbour below wraps past 2**63"""
    cases = []
    u = synth.synth_v1(140, 170, 3, seed=301, cell=12, lo=2000.0, hi=65000.0, noise=300.0)
    u = u.astype(numpy.uint32) * numpy.uint32(65537)
    u[:, :12, :12] = 4294967295
    cases.append((u, synth.diagonal_centres(u, 12, 4294967295), 10, 'auto', 4294967295, True))
    s = synth.synth_v1(150, 130, 4, seed=302, cell=12)
    s = ((s.astype(numpy.int64) - 2000) * 500000).astype(numpy.int32)
    cases.append((s, synth.diagonal_centres(s, 14), 12, None, None, False))
    w = numpy.full((1, 48, 64), 1000000000, dtype=numpy.uint32)
    w[:, 20:, :] = 4200000000
    w += numpy.random.default_rng(303).integers(0, 1000, w.shape).astype(numpy.uint32)
    w[:, 19, 3::6] = 0
    cases.append((w, numpy.array([[1.0e9], [4.2e9], [0.0]]), 10, 'auto', None, True))
    return cases


@pytest.mark.skipif(not os.path.isdir(os.path.join(REFERENCE, 'pyshepseg')),
    reason='the reference is not installed in oracle/_ref')
def test_oracle_equals_reference_on_32bit_images(tmp_path):
    try:
        import numba  # noqa: F401
        import sklearn  # noqa: F401
    except ImportError:
        pytest.skip('numba / scikit-learn missing: the reference cannot run here')
    spec = []
    cases = live_cases()
    for (i, (img, centres, minSeg, msd, nullVal, four)) in enumerate(cases):
        npz = str(tmp_path / ('in%d.npz' % i))
        numpy.savez(npz, img=img, centres=numpy.asarray(centres, dtype=numpy.float64))
        spec.append({'npz': npz, 'out': str(tmp_path / ('out%d.npz' % i)), 'minSeg': minSeg, 'msd': msd,
            'nullVal': nullVal, 'four': four})
    specFile = str(tmp_path / 'spec.json')
    json.dump({'cases': spec}, open(specFile, 'w'))
    script = str(tmp_path / 'run_reference.py')
    open(script, 'w').write(RUNNER % {'ref': REFERENCE})
    subprocess.run([sys.executable, script, specFile], check=True, timeout=900, cwd=str(tmp_path))
    for (c, (img, centres, minSeg, msd, nullVal, four)) in zip(spec, cases):
        ref = numpy.load(c['out'])
        got = oracle.doShepherdSegmentation(img, minSegmentSize=minSeg, maxSpectralDiff=msd,
            imgNullVal=nullVal, fourConnected=four, kmeansObj=goldenutil.Centres(centres))
        assert numpy.array_equal(got.segimg, ref['segimg'])
        assert int(got.singlePixelsEliminated) == int(ref['single'])
        assert int(got.smallSegmentsEliminated) == int(ref['small'])

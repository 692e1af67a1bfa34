"""
The CPU oracle on images of 17 to 64 bands: its assignment against scikit-learn's
KMeans.predict, which the reference calls (shepseg.py:317-361).  This pins the assignment contract
above 16 bands to the library the reference uses, without needing the reference itself.
"""
import warnings

import numpy
import pytest

from oracle import oracle
from pyshepseg_b200 import synth
import goldenutil


def many_band_image(bands, dtype):
    """256 x 256 synth_v1; int16 shifted to negatives, uint32 spread over the full range (x 65537);
    a 20 x 20 null corner"""
    img = synth.synth_v1(256, 256, bands, seed=bands, cell=16)
    if dtype == numpy.int16:
        img = (img.astype(numpy.int32) - 2000).astype(numpy.int16)
    elif dtype == numpy.uint32:
        img = img.astype(numpy.uint32) * numpy.uint32(65537)
    img[:, :20, :20] = -2000 if dtype == numpy.int16 else 0
    return img


@pytest.mark.parametrize('bands,dtype', [(17, numpy.uint16), (32, numpy.uint16), (64, numpy.uint16),
                                         (32, numpy.int16), (48, numpy.uint32)],
                         ids=['17-uint16', '32-uint16', '64-uint16', '32-int16', '48-uint32'])
def test_oracle_assignment_equals_sklearn_predict(bands, dtype):
    from sklearn.cluster import KMeans
    img = many_band_image(bands, dtype)
    nullVal = int(img[0, 0, 0])
    centres = synth.diagonal_centres(img, 60, nullVal)
    km = KMeans(n_clusters=len(centres), n_init=1, init=centres, max_iter=1)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        km.fit(centres)
    km.cluster_centers_ = centres
    pixels = numpy.moveaxis(img, 0, -1).reshape(-1, bands)
    want = km.predict(pixels).astype(numpy.int32) + 1
    want[(pixels == nullVal).any(axis=1)] = 0
    got = oracle.applySpectralClusters(goldenutil.Centres(centres), img, nullVal)
    assert numpy.array_equal(got.ravel(), want)
    assert len(numpy.unique(got)) > 10

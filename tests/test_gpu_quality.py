"""frtest-style round-trip quality harness (upstream other/frtest.cpp:30-250) on the GPU path,
beside the same harness driven through upstream compiled in-tree (oracle/_ref).

Upstream's test fills a 1-channel float image with a de-biased, power-normalised cosine of
circular frequency th, resizes it by k = 0.95^n > SizeCoeff (passed as NEGATIVE k: uniform, no
centring, frtest.cpp:109-111) and back, and accumulates per frequency
    FR = 10 log10 mean(rms(dst)^2),  DR = 10 log10 mean(rms(src*p1g - back*p2g)^2),
    PE = 20 log10 max |src*p1g - back*p2g|
over the k sweep (frtest.cpp:224-250).  Here: same statistics, IS_UPS = 1 (upsizing first, as
upstream's default build), fewer frequencies and a narrower image so the test runs in
seconds.  The product must reproduce the oracle's numbers (stored in tests/golden/upstream.json)
within 0.01 dB (it is bit-exact, so the difference is 0).
"""
import math

import numpy as np
import pytest

import avir_b200 as ab
import cases as cs
import oracle_ref as o

pytestmark = pytest.mark.gpu

BIAS, SIZE_COEFF, OFFS = 0.0, 0.3, 32
W, H = 2048, 12


def _source(th):
    row = np.cos(np.arange(W, dtype=np.float64) * th).astype(np.float32).astype(np.float64)
    row -= row.mean()
    row = (row.astype(np.float32)).astype(np.float64)
    s2 = 1.0 / math.sqrt(float((row ** 2).sum()) / W)
    row = (row * s2 + BIAS).astype(np.float32)
    return np.ascontiguousarray(np.broadcast_to(row[None, :, None], (H, W, 1))).astype(np.float32)


def _rms(a):
    return math.sqrt(float(((a.astype(np.float64) - BIAS) ** 2).sum()) / a.size)


def _stats(resize, th):
    src = _source(th)
    p1g = 1.0 / _rms(src[0, OFFS:W - OFFS, 0])
    avgd = avgd2 = peakd = 0.0
    n = 0
    k = 1.0
    while k > SIZE_COEFF:
        dw, dh = int(math.ceil(W / k)), int(math.ceil(H / k))
        dst = resize(src, dw, dh, -k)             # frtest.cpp:109-111
        back = resize(dst, W, H, -1.0 / k)        # frtest.cpp:116-118
        r = _rms(dst[0, OFFS:dw - OFFS, 0])
        p2g = 1.0 / _rms(back[0, OFFS:W - OFFS, 0])
        d = (src[0, OFFS:W - OFFS, 0].astype(np.float64) - BIAS) * p1g - \
            (back[0, OFFS:W - OFFS, 0].astype(np.float64) - BIAS) * p2g
        avgd += r * r
        avgd2 += float((d ** 2).sum()) / d.size
        peakd = max(peakd, float(np.abs(d).max()))
        n += 1
        k *= 0.95
    return (10.0 * math.log10(avgd / n), 10.0 * math.log10(avgd2 / n), 20.0 * math.log10(peakd), n)


@pytest.mark.parametrize("frac", [0.02, 0.2, 0.6, 0.95])
def test_frtest_round_trip_statistics_match_upstream(frac):
    th = math.pi * frac
    rs = ab.CImageResizer(16, 0, 0, ab.FP_DEF)

    def gpu(img, nw, nh, k):
        return rs.resizeImage(img, nw, nh, k, out_dtype=np.float32)

    def ref(img, nw, nh, k):
        return o.ref_resize(img, nw, nh, np.float32, fpclass=o.FP_DEF, k=k, resbits=16)

    g = _stats(gpu, th)
    r = cs.upstream("frtest:%r" % frac, lambda: list(_stats(ref, th)))
    assert g[3] == r[3] == 24  # 0.95^n > 0.3
    for a, b, name in zip(g[:3], r[:3], ("FR", "DR", "PE")):
        assert abs(a - b) <= 0.01, (name, a, b)
    # sanity of the harness itself: pass-band frequencies come back with > 60 dB dynamic range
    if frac <= 0.2:
        assert g[1] < -60.0, g

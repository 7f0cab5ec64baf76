"""CPU tests of the oracle itself: the restatement against independent float64 numpy/scipy
implementations of the same formulas, against the reference README's published feature
counts (the only known answers the reference holds for extraction, SURVEY.md 8c; checked on crops of its demo
photographs against the reference library's counts), and the
matcher's quirk register on crafted inputs.  Golden fixtures produced by the reference
library on the GPU box are checked in test_golden_cpu.py."""
import os

import numpy as np
import pytest
from scipy.ndimage import correlate1d

import oracle
from cudasift_b200.synth import synth_descriptors, synth_image

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _taps9(sigma):
    k = np.zeros(9, np.float32)
    oracle.lib().oracle_lowpass_taps(sigma, k.ctypes.data)
    return k


def test_taps_are_normalised_gaussians():
    k = _taps9(1.0)
    assert abs(k.sum() - 1.0) < 1e-6 and np.allclose(k, k[::-1])
    g = np.exp(-np.arange(-4, 5) ** 2 / 2.0); g /= g.sum()
    assert np.allclose(k, g, atol=1e-6)
    k5 = np.zeros(5, np.float32)
    oracle.lib().oracle_scaledown_taps(0.5, k5.ctypes.data)
    assert np.allclose(k5, [0.010334, 0.207561, 0.564210, 0.207561, 0.010334], atol=2e-6)   # SURVEY 8(a7)
    lap = oracle.laplace_taps(5).reshape(8, 12, 16)
    for octave in range(1, 6):
        for s in range(8):
            t = lap[octave, s, :5]
            assert abs(t[0] + 2 * t[1:].sum() - 1.0) < 1e-6
    # effective sigmas at the finest octave (SURVEY A.2): 2^((i-1)/5)
    t = lap[5, 1, :5].astype(np.float64)
    assert abs(np.log(t[0] / t[1]) * 2 - 1.0) < 1e-4          # sigma = 1.0 for scale 1


def test_lowpass_matches_float64_convolution():
    img = synth_image(200, 120, seed=3)
    out = oracle.lowpass(img, 1.0)
    k = _taps9(1.0).astype(np.float64)
    ref = correlate1d(correlate1d(img.astype(np.float64), k, axis=1, mode="nearest"), k, axis=0, mode="nearest")
    assert np.max(np.abs(out - ref)) < 2e-4


def test_scaledown_matches_float64_convolution():
    img = synth_image(203, 121, seed=4)
    out = oracle.scaledown(img)
    assert out.shape == (60, 101)
    k5 = np.zeros(5, np.float32)
    oracle.lib().oracle_scaledown_taps(0.5, k5.ctypes.data)
    k = k5.astype(np.float64)
    full = correlate1d(correlate1d(img.astype(np.float64), k, axis=1, mode="nearest"), k, axis=0, mode="nearest")
    assert np.max(np.abs(out - full[0:120:2, 0:202:2])) < 2e-4


def test_scaleup_is_bilinear():
    img = synth_image(40, 30, seed=5)
    up = oracle.scaleup(img)
    assert np.array_equal(up[0::2, 0::2], img)
    assert np.allclose(up[0, 1], 0.5 * (img[0, 0] + img[0, 1]))
    assert np.allclose(up[1, 1], 0.25 * (img[0, 0] + img[0, 1] + img[1, 0] + img[1, 1]))


def test_dog_matches_float64_convolution():
    img = synth_image(160, 96, seed=6)
    d = oracle.dog(img, 5, 5)
    lap = oracle.laplace_taps(5).reshape(8, 12, 16)
    blurs = []
    for s in range(8):
        h = lap[5, s, :5].astype(np.float64)
        k = np.concatenate([h[:0:-1], h])
        blurs.append(correlate1d(correlate1d(img.astype(np.float64), k, axis=0, mode="nearest"), k, axis=1, mode="nearest"))
    for s in range(7):
        assert np.max(np.abs(d[s] - (blurs[s + 1] - blurs[s]))) < 3e-4


def test_tex2d_matches_bilinear_with_8bit_weights():
    img = synth_image(64, 48, seed=7)
    rng = np.random.default_rng(0)
    xs, ys = rng.uniform(-2, 66, 500).astype(np.float32), rng.uniform(-2, 50, 500).astype(np.float32)
    got = oracle.tex2d(img, xs, ys)
    xb, yb = xs.astype(np.float64) - 0.5, ys.astype(np.float64) - 0.5
    i, j = np.floor(xb), np.floor(yb)
    a, b = xb - i, yb - j
    i0, i1 = np.clip(i, 0, 63).astype(int), np.clip(i + 1, 0, 63).astype(int)
    j0, j1 = np.clip(j, 0, 47).astype(int), np.clip(j + 1, 0, 47).astype(int)
    ref = (1 - a) * (1 - b) * img[j0, i0] + a * (1 - b) * img[j0, i1] + (1 - a) * b * img[j1, i0] + a * b * img[j1, i1]
    grad = np.abs(img[j0, i1] - img[j0, i0]) + np.abs(img[j1, i0] - img[j0, i0]) + np.abs(img[j1, i1] - img[j0, i0])
    assert np.all(np.abs(got - ref) <= grad / 256.0 + 1e-3)    # within the 1.8 fixed-point quantisation
    # measured B200 behaviour (scripts/tex_calib.py): weights are whole 1/256ths that sum to 1
    hot = np.zeros((16, 16), np.float32); hot[8, 8] = 65536.0
    wq = oracle.tex2d(hot, np.array([8.59521484375, 7.955078125], np.float32), np.array([8.8134765625, 8.00048828125], np.float32))
    assert list(wq) == [40960.0, 15104.0]
    # exact at texel centres
    assert np.allclose(oracle.tex2d(img, np.array([10.5], np.float32), np.array([7.5], np.float32)), img[7, 10])


def test_extract_invariants():
    img = synth_image(640, 480, seed=11)
    pts, total = oracle.extract(img, 5, 1.0, 3.0)
    assert 100 < len(pts) <= total
    assert np.all(pts["xpos"] >= 0) and np.all(pts["xpos"] < 640) and np.all(pts["ypos"] < 480)
    assert set(np.unique(pts["subsampling"])) <= {1.0, 2.0, 4.0, 8.0, 16.0}
    n = np.linalg.norm(pts["data"], axis=1)
    assert np.allclose(n, 1.0, atol=1e-4)
    assert pts["data"].max() <= 0.2 / np.sqrt(0.04 * 1) + 1e-3   # clamp 0.2 then renormalise (< 1)
    assert np.all((pts["orientation"] >= 0) & (pts["orientation"] < 360.0001))
    assert np.all(np.abs(pts["sharpness"]) > 3.0 - 1.0)          # refined value stays near |DoG| > thresh
    assert np.all(pts["edgeness"] < 10.0)                        # tra^2/det < edgeLimit
    # output grouped coarsest octave first (cudaSiftH.cu:153-161)
    assert np.all(np.diff(pts["subsampling"]) <= 0)
    # a higher threshold yields a subset of the extrema
    pts2, _ = oracle.extract(img, 5, 1.0, 5.0)
    assert len(pts2) < len(pts)


def test_extract_scaleup_and_lowest_scale():
    img = synth_image(160, 120, seed=12)
    up, _ = oracle.extract(img, 3, 1.0, 2.0, 0.0, True)
    assert len(up) > 0 and up["xpos"].max() < 160 and up["ypos"].max() < 120
    a, _ = oracle.extract(img, 3, 1.0, 2.0, 0.0)
    b, _ = oracle.extract(img, 3, 1.0, 2.0, 3.0)
    assert 0 < len(b) < len(a) and b["scale"].min() >= 3.0 - 1e-3


CROP = (390, 760, 300, 400)      # y0, x0, height, width: the centre of the reference's 1920x1080 demo photographs


@pytest.mark.parametrize("name", ["img1", "img2"])
def test_demo_photo_crop_feature_counts(name):
    """The reference's demo photographs data/img1.png, data/img2.png at the demo's parameters (mainSift.cpp:58-68):
    its README.md:33 publishes 'MatchSiftData 1911 x 2086 features' for the whole images.  What is stored is a
    400x300 grey centre crop of each (tests/golden/<name>_crop.png) with the reference library's own feature count
    on it (reference_checks.npz); the oracle must be within the same +-0.5 % of it."""
    import cv2
    g = np.load(os.path.join(GOLDEN, "reference_checks.npz"))
    img = cv2.imread(os.path.join(GOLDEN, name + "_crop.png"), 0)
    assert img.shape == CROP[2:]
    expected = int(g[name + "_crop_count"])
    pts, _ = oracle.extract(img.astype(np.float32), 5, 1.0, 3.0)
    assert abs(len(pts) - expected) <= 0.005 * expected, (len(pts), expected)


# ------------------------------------------------------------------ matcher
def _brute(s1, s2):
    n2 = (len(s2) // 32) * 32
    sc = s1["data"].astype(np.float64) @ s2["data"][:n2].astype(np.float64).T
    return sc


def test_match_against_float64_bruteforce():
    s1, s2 = synth_descriptors(257, 1), synth_descriptors(500, 2)
    m = oracle.match(s1, s2)
    sc = _brute(s1, s2)
    top = np.sort(sc, axis=1)[:, ::-1]
    clear = (top[:, 0] - top[:, 1]) > 1e-5
    assert clear.sum() > 200
    assert np.array_equal(m["match"][clear], np.argmax(sc, axis=1)[clear])
    assert np.allclose(m["score"], top[:, 0], atol=2e-6)
    assert np.all(m["match"] < 480)                              # Q7: tail 500 % 32 = 20 never visited
    idx = m["match"]
    assert np.array_equal(m["match_xpos"], s2["xpos"][idx]) and np.array_equal(m["match_ypos"], s2["ypos"][idx])
    assert np.all(m["ambiguity"] <= 1.0 + 1e-6) and np.all(m["ambiguity"] > 0)


def test_match_quirks():
    s2 = synth_descriptors(64, 5)
    s1 = synth_descriptors(4, 6)
    # Q10: exact duplicates in different partitions -> lowest partition wins, not lowest index
    s1["data"][0] = s2["data"][40]          # partition (40%32)//4 = 2
    s2["data"][7] = s2["data"][40]          # partition 1, lower index
    s2["data"][33] = s2["data"][40]         # partition 0 (33%32=1), higher index than 7
    m = oracle.match(s1, s2)
    assert m["match"][0] == 33
    # Q9: 'second' only sees partition 0's second and other partitions' maxima
    assert m["ambiguity"][0] == pytest.approx(1.0, abs=2e-6)
    # Q7: fewer than 32 candidates -> nothing visited
    m2 = oracle.match(s1, s2[:31])
    assert np.all(m2["match"] == -1) and np.all(m2["score"] == 0) and np.all(m2["ambiguity"] == 0)
    # Q11: only strictly positive scores can match
    neg = s1.copy(); neg["data"] *= -1
    m3 = oracle.match(neg, s2)
    assert np.all(m3["match"] == -1)
    # threads give identical results
    big1, big2 = synth_descriptors(100, 8), synth_descriptors(96, 9)
    a, b = oracle.match(big1, big2), oracle.match(big1, big2, threads=4)
    assert a.tobytes() == b.tobytes()

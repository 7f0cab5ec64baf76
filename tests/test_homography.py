"""FindHomography (matching.cu:1000-1087), the consumer of MatchSiftData's output (SURVEY 8f-1).
CPU: the oracle recovers a planted homography.  GPU: product == oracle under the same srand()
seed, and == the stored result of the reference library."""
import numpy as np
import pytest

import oracle
from cudasift_b200 import SIFT_DTYPE

H_TRUE = np.array([[0.98, -0.05, 30.0], [0.04, 1.01, -12.0], [1.0e-5, -2.0e-5, 1.0]])


def planted(n=600, outliers=0.4, seed=3, noise=0.3):
    rng = np.random.default_rng(seed)
    p = np.zeros(n, SIFT_DTYPE)
    x, y = rng.uniform(0, 1280, n), rng.uniform(0, 960, n)
    q = H_TRUE @ np.stack([x, y, np.ones(n)])
    mx, my = q[0] / q[2] + rng.normal(0, noise, n), q[1] / q[2] + rng.normal(0, noise, n)
    bad = rng.random(n) < outliers
    mx[bad], my[bad] = rng.uniform(0, 1280, bad.sum()), rng.uniform(0, 960, bad.sum())
    p["xpos"], p["ypos"], p["match_xpos"], p["match_ypos"] = x, y, mx, my
    p["score"] = np.where(bad, rng.uniform(0.5, 0.9, n), rng.uniform(0.86, 0.99, n))
    p["ambiguity"] = np.where(bad, rng.uniform(0.7, 1.0, n), rng.uniform(0.3, 0.94, n))
    return p, bad


def test_oracle_recovers_planted_homography():
    p, bad = planted()
    H, n = oracle.find_homography(p, numLoops=1000, minScore=0.85, maxAmbiguity=0.95, thresh=3.0, seed=1)
    assert n >= 0.9 * (~bad).sum()
    pts = np.array([[100.0, 200.0, 1.0], [1000.0, 800.0, 1.0], [640.0, 480.0, 1.0]]).T
    a, b = H.astype(np.float64) @ pts, H_TRUE @ pts
    assert np.max(np.abs(a[:2] / a[2] - b[:2] / b[2])) < 1.0
    # fewer than 8 points / fewer than 8 eligible points: identity, 0 matches (matching.cu:1016,1040)
    H0, n0 = oracle.find_homography(p[:7], seed=1)
    assert n0 == 0 and np.array_equal(H0, np.eye(3, dtype=np.float32))
    H1, n1 = oracle.find_homography(p, minScore=2.0, seed=1)
    assert n1 == 0 and np.array_equal(H1, np.eye(3, dtype=np.float32))


@pytest.mark.gpu
def test_find_homography_equals_oracle(cs):
    p, _ = planted(n=1500, seed=5)
    sd = cs.InitSiftData(cs.SiftData(), 2048, False, True)
    sd._buf.upload(p); sd.numPts = len(p)
    for loops, thresh in ((1000, 3.0), (10000, 5.0)):
        Hg, ng, ms = cs.FindHomography(sd, loops, 0.85, 0.95, thresh, seed=7)
        Ho, no = oracle.find_homography(p, loops, 0.85, 0.95, thresh, seed=7)
        assert ng == no, (ng, no)
        assert np.allclose(Hg, Ho, rtol=1e-4, atol=1e-6), (Hg, Ho)
    sd.numPts = 7
    H0, n0, _ = cs.FindHomography(sd, seed=1)
    assert n0 == 0 and np.array_equal(H0, np.eye(3, dtype=np.float32))


@pytest.mark.gpu
def test_find_homography_vs_reference(cs):
    """Against the reference's FindHomography after srand(11) on the same points (tests/golden/reference_checks.npz)."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))
    Hr, nr = g["homography_H"], int(g["homography_numfit"])
    p, _ = planted(n=1600, seed=9)            # multiple of 16: the reference reads no padding entries
    sd = cs.InitSiftData(cs.SiftData(), 2048, False, True)
    sd._buf.upload(p); sd.numPts = len(p)
    Hg, ng, _ = cs.FindHomography(sd, 2000, 0.85, 0.95, 4.0, seed=11)
    assert abs(ng - nr) <= max(2, 0.005 * nr), (ng, nr)
    assert np.allclose(Hg.ravel()[:8], Hr[:8], rtol=2e-3, atol=1e-5), (Hg, Hr)


def test_improve_homography_host():
    """ImproveHomography (geomFuncs.cpp:6-72) is host code in the reference and here: product (own 8x8
    Cholesky) against the numpy restatement, and against the planted geometry."""
    import cudasift_b200 as cs
    from oracle.geom import improve_homography
    p, bad = planted(n=900, seed=11, noise=0.25)
    # a deliberately rough start (what a short RANSAC would hand over)
    H0 = H_TRUE.copy(); H0[0, 2] += 1.5; H0[1, 2] -= 1.0; H0[0, 0] *= 1.001
    H0 = (H0 * 1.7).astype(np.float32)                       # not normalised: [8] != 1 on input
    for loops, mins, maxa, thr in ((5, 0.0, 0.80, 3.0), (1, 0.85, 0.95, 5.0), (8, 0.0, 1.0, 2.0)):
        q = p.copy()
        Hp, nfit = cs.ImproveHomography(q, H0, loops, mins, maxa, thr)
        Ho, nfo, erro = improve_homography(p, H0, loops, mins, maxa, thr)
        assert nfit == nfo, (nfit, nfo)
        assert np.allclose(Hp.reshape(9), Ho, rtol=1e-5, atol=1e-7), (Hp, Ho)
        assert np.allclose(q["match_error"], erro, rtol=1e-3, atol=1e-3)
        assert Hp[2, 2] == 1.0
        assert nfit >= 0.95 * (~bad).sum()
    pts = np.array([[100.0, 200.0, 1.0], [1000.0, 800.0, 1.0], [640.0, 480.0, 1.0]]).T
    a, b = Hp.astype(np.float64) @ pts, H_TRUE @ pts
    assert np.max(np.abs(a[:2] / a[2] - b[:2] / b[2])) < 0.15     # refinement beats the 1.5 px start
    # no eligible matches: singular normal equations -> zero solution, match_error still filled
    q = p.copy()
    Hz, nz = cs.ImproveHomography(q, H0, 2, 2.0, 0.0, 3.0)
    assert np.array_equal(Hz.reshape(9)[:8], np.zeros(8, np.float32)) and Hz[2, 2] == 1.0
    Hzo, nzo, _ = improve_homography(p, H0, 2, 2.0, 0.0, 3.0)
    assert nz == nzo and np.array_equal(Hz.reshape(9), Hzo)


def _golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "improve_homography.npz"))


def test_improve_homography_pinned_by_opencv():
    """SURVEY 8 f3: the vectorised restatement AND the product against golden vectors produced by the reference's
    own solver (cv::solve(DECOMP_CHOLESKY) through cv2 inside a statement-by-statement port of geomFuncs.cpp:6-72);
    the port is re-run live when cv2 imports."""
    import cudasift_b200 as cs
    from oracle.geom import improve_homography, improve_homography_cv2
    g = _golden()
    p, H0 = g["points"], g["H0"]
    p2, _ = planted(n=900, seed=11, noise=0.25)
    assert p.tobytes() == p2.tobytes()                       # the fixture's inputs are the seeded ones
    try:
        import cv2  # noqa: F401
        live = True
    except ImportError:
        live = False
    for k, (loops, mins, maxa, thr) in enumerate(g["cases"]):
        Hg, ng, eg = g["H_%d" % k], int(g["numfit_%d" % k]), g["err_%d" % k]
        Ho, no, eo = improve_homography(p, H0, int(loops), mins, maxa, thr)
        q = p.copy()
        Hp, npd = cs.ImproveHomography(q, H0, int(loops), mins, maxa, thr)
        for H, n, e, who in ((Ho, no, eo, "oracle"), (Hp.reshape(9), npd, q["match_error"], "product")):
            assert n == ng, (who, k, n, ng)
            # float32 outputs of an 8x8 double solve: different summation orders agree to a few ulp
            assert np.allclose(H, Hg, rtol=2e-6, atol=1e-9), (who, k, H, Hg)
            assert np.allclose(e, eg, rtol=1e-4, atol=2e-4), (who, k)
        if live:
            Hc, nc, ec = improve_homography_cv2(p, H0, int(loops), mins, maxa, thr)
            assert nc == ng and np.array_equal(Hc, Hg) and np.array_equal(ec, eg)

"""GPU parity of ExtractSift: against the oracle, against the stored results of the reference library,
determinism, API paths and edge cases."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from compare import compare_sets, reference_summary
from cudasift_b200.synth import synth_image

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def canon(pts):
    """Canonical order (the reference's own order is nondeterministic, quirk Q2)."""
    key = np.lexsort((pts["orientation"], pts["scale"], pts["xpos"], pts["ypos"], pts["subsampling"]))
    return pts[key]


def _extract(cs, arr, **kw):
    return cs.extract_host(arr, **kw)


def _assert_close(rep, min_frac=0.995, desc_tol=1e-3, bad_desc=0.01):
    n = max(rep["na"], rep["nb"])
    assert rep["pairs"] >= min_frac * n, rep
    assert rep["pos_err"] < 1e-2 and rep["scale_rel"] < 1e-3 and rep["ori_err"] < 0.5, rep
    assert rep["desc_bad"] <= bad_desc * rep["pairs"], rep


def test_extract_vs_oracle_synthetic(cs):
    arr = synth_image(640, 480, seed=1000)
    got = _extract(cs, arr, thresh=3.0)
    want, _ = oracle.extract(arr, 5, 1.0, 3.0)
    assert abs(len(got) - len(want)) <= 2
    rep = compare_sets(canon(got), canon(want))
    _assert_close(rep)


def test_extract_vs_oracle_1080p(cs):
    arr = synth_image(1920, 1080, seed=1001)
    got = _extract(cs, arr, thresh=3.0)
    want, _ = oracle.extract(arr, 5, 1.0, 3.0)
    assert abs(len(got) - len(want)) <= 0.002 * len(want) + 2
    _assert_close(compare_sets(canon(got), canon(want)))


def test_extract_deterministic(cs):
    arr = synth_image(800, 600, seed=5)
    a, b = canon(_extract(cs, arr)), canon(_extract(cs, arr))
    assert len(a) == len(b)
    for f in ("xpos", "ypos", "scale", "orientation", "sharpness", "edgeness", "subsampling", "data"):
        assert np.array_equal(a[f], b[f]), f


# (width, height, seed, ExtractSift keywords) of the synthetic inputs compared with the reference
REF_CASES = [(1280, 960, 1000, dict(thresh=3.0)), (1920, 1080, 1000, dict(thresh=3.0)),
             (640, 480, 7, dict(thresh=2.0, scaleUp=True)), (800, 600, 8, dict(thresh=3.0, numOctaves=1)),
             (800, 600, 8, dict(thresh=3.0, numOctaves=3))]


def ref_case_image(case):
    return synth_image(case[0], case[1], seed=case[2])


def _assert_matches_reference(mine, g, kw):
    """`mine` (canonical order) against a compare.reference_summary of two reference runs on the same input."""
    assert int(g["count1"]) == int(g["count2"]) == len(mine) > 100, (kw, int(g["count1"]), int(g["count2"]), len(mine))
    for f in ("xpos", "ypos", "scale", "sharpness", "edgeness", "subsampling"):
        assert sha(mine[f]) == str(g[f + "_sha"]), (kw, f)
    do = lambda a, b: np.minimum(np.abs(a - b) % 360.0, 360.0 - np.abs(a - b) % 360.0)
    ori_noise = float(g["ori_noise"])
    ori_err = float(do(mine["orientation"], g["orientation"]).max())
    fin_ref = np.ones(len(mine), bool)
    fin_ref[g["nonfinite"]] = False
    assert np.array_equal(np.isfinite(mine["data"]).all(axis=1), fin_ref)      # quirk Q21 rows
    rows = g["rows"]
    keep = fin_ref[rows]
    de = np.abs(mine["data"][rows[keep]] - g["data"][keep]).max(axis=1)
    d_noise, d_err = float(g["desc_noise"]), float(de.max())
    bad_noise, bad_err = int(g["desc_bad_noise"]), int((de > 2e-5).sum())
    print(kw, "points", len(mine), "ori noise/err", ori_noise, ori_err, "desc max noise/err", d_noise, d_err,
          "rows > 2e-5 noise/err", bad_noise, bad_err, "median err", float(np.median(de)))
    assert ori_err <= max(2.0 * ori_noise, 1e-3), (kw, ori_err, ori_noise)
    # a last-bit difference of the orientation moves sample positions across the texture unit's 1/256 coordinate
    # grid: a few descriptors differ by ~1e-4 (the reference does the same between two of its own runs)
    assert float(np.median(de)) <= 1e-6, (kw, float(np.median(de)))
    # measured on the B200 (6 cases): rows > 2e-5: reference vs itself 1..14, product vs reference 0..10; max 2.0e-4 both
    assert bad_err <= 2 * bad_noise + 5, (kw, bad_err, bad_noise)
    assert d_err <= max(2.0 * d_noise, 3e-4), (kw, d_err, d_noise)
    assert d_err <= 1e-3 and ori_err <= 0.36                    # BASELINE.json: 1e-3 (orientation: of 360 degrees)


def test_extract_vs_reference(cs):
    """The headline parity test: reference ExtractSift and the product on identical inputs.
    BASELINE.json asks for x/y/scale/orientation and descriptors within 1e-3 relative; what is asserted is what was
    measured: positions, scales, sharpness and edgeness BIT-IDENTICAL, orientation and descriptors within twice the
    reference's own run-to-run noise (its histograms are accumulated with shared-memory float atomics, quirk Q3).
    The reference's results are stored under tests/golden/: for the synthetic cases, digests of the bit-exact fields,
    every orientation and the descriptors of a seeded sample of rows (reference_checks.npz); for config #1, both
    reference runs in full on a 640x480 crop of the reference's data/left.pgm (extract_left_crop.npz)."""
    g = np.load(os.path.join(GOLDEN, "reference_checks.npz"))
    for k, case in enumerate(REF_CASES):
        summary = {key[len("extract%d_" % k):]: g[key] for key in g.files if key.startswith("extract%d_" % k)}
        _assert_matches_reference(canon(_extract(cs, ref_case_image(case), **case[3])), summary, case[3])
    left = np.load(os.path.join(GOLDEN, "extract_left_crop.npz"))     # config #1: data/left.pgm, mainSift.cpp:59
    kw = dict(thresh=float(left["thresh"]))
    summary = reference_summary(canon(left["run1"]), canon(left["run2"]), seed=0, sample=None)
    _assert_matches_reference(canon(_extract(cs, left["image"].astype(np.float32), **kw)), summary, kw)


def test_cxx_api_equals_c_abi(cs, selflib):
    arr = synth_image(640, 480, seed=31)
    a = canon(selflib.extract(arr, thresh=3.0))                       # InitSiftData/ExtractSift (mangled C++)
    b = canon(_extract(cs, arr, thresh=3.0))                          # cs_extract_host
    c = canon(selflib.extract(arr, thresh=3.0, use_temp=False))       # internal arena (tempMemory == NULL)
    assert a.tobytes() == c.tobytes()
    for f in ("xpos", "ypos", "scale", "orientation", "data"):
        assert np.array_equal(a[f], b[f]), f


def test_extract_python_mirror(cs):
    """mainSift.cpp:49-69 through the Python mirror of the API."""
    arr = synth_image(640, 480, seed=32)
    img = cs.CudaImage().Allocate(640, 480, cs.iAlignUp(640, 128), False, None, arr)
    img.Download()
    sd = cs.InitSiftData(cs.SiftData(), 4096, True, True)
    tmp = cs.AllocSiftTempMemory(640, 480, 5, False)
    n1 = cs.ExtractSift(sd, img, 5, 1.0, 3.0, 0.0, False, tmp)
    n2 = cs.ExtractSift(sd, img, 5, 1.0, 3.0, 0.0, False, tmp)
    cs.FreeSiftTempMemory(tmp)
    assert n1 == n2 == sd.numPts > 100
    want, _ = oracle.extract(arr, 5, 1.0, 3.0)
    assert abs(n1 - len(want)) <= 2
    cs.FreeSiftData(sd)


def test_edge_cases(cs):
    arr = synth_image(320, 240, seed=33)
    # numOctaves = 1, odd sizes, scaleUp, lowestScale, tiny image, maxPts overflow
    for kw in ({"numOctaves": 1}, {"numOctaves": 3, "scaleUp": True, "thresh": 2.0}, {"lowestScale": 3.0, "thresh": 2.0}):
        got = canon(_extract(cs, arr, **kw))
        o = dict(numOctaves=5, initBlur=1.0, thresh=3.0, lowestScale=0.0, scaleUp=False); o.update(kw)
        want, _ = oracle.extract(arr, o["numOctaves"], o["initBlur"], o["thresh"], o["lowestScale"], o["scaleUp"])
        assert abs(len(got) - len(want)) <= 2, kw
        _assert_close(compare_sets(got, canon(want)), min_frac=0.98)
    odd = synth_image(333, 201, seed=34)
    got, (want, _) = _extract(cs, odd), oracle.extract(odd, 5, 1.0, 3.0)
    assert abs(len(got) - len(want)) <= 2
    tiny = synth_image(20, 12, seed=35)
    assert len(_extract(cs, tiny, numOctaves=5)) == len(oracle.extract(tiny, 5, 1.0, 3.0)[0])
    few = _extract(cs, arr, thresh=1.0, maxPts=50)                     # quirk Q18: clamp, never overflow
    assert len(few) == 50
    flat = np.full((64, 64), 100.0, np.float32)
    assert len(_extract(cs, flat)) == 0


def test_extractor_pipeline_and_u8_upload(cs):
    """The pipelined extractor (CUDA-graph submit path after the second call) returns what the
    synchronous call returns; an 8-bit upload gives the same records as its float image."""
    import ctypes
    arr8 = np.clip(np.rint(synth_image(640, 480, seed=41)), 0, 255).astype(np.uint8)
    arrf = arr8.astype(np.float32)
    want = canon(_extract(cs, arrf, thresh=3.0))
    ex = cs.Extractor(640, 480, 5, 8192)
    ex.host_image()[:] = arrf
    got = []
    for rep in range(4):                      # reps >= 2 run through the captured graph
        ex.submit_host(ex.host_image().ctypes.data, 1.0, 3.0, 0.0)
        n = ex.wait()
        got.append(canon(ex.host_points(n).copy()))
    p8 = cs.lib().cs_host_alloc_pinned(640 * 480)
    ctypes.memmove(p8, arr8.ctypes.data, 640 * 480)
    ex.submit_host_u8(p8, 1.0, 3.0, 0.0)
    n = ex.wait()
    got.append(canon(ex.host_points(n).copy()))
    cs.lib().cs_host_free_pinned(p8)
    for g in got:
        assert len(g) == len(want)
        for f in ("xpos", "ypos", "scale", "orientation", "subsampling", "data"):
            assert np.array_equal(g[f], want[f]), f
    ex.close()


def test_detector_variants_identical(cs):
    """Every compiled detector configuration (CTA size, columns per horizontal task, row pairs per
    vertical task) produces the same keypoints, bit for bit: tiling must not influence the results."""
    arr = synth_image(1000, 700, seed=21)
    L = cs.lib()
    try:
        assert L.cs_set_tuning(b"detect_variant", 0) == 0
        base = canon(_extract(cs, arr, thresh=2.0))
        assert len(base) > 500
        for v in range(1, 8):
            assert L.cs_set_tuning(b"detect_variant", v) == 0
            got = canon(_extract(cs, arr, thresh=2.0))
            assert len(got) == len(base), v
            for f in ("xpos", "ypos", "scale", "sharpness", "edgeness", "orientation", "subsampling"):
                assert np.array_equal(got[f], base[f]), (v, f)
            assert np.array_equal(got["data"], base["data"]), v
    finally:
        L.cs_set_tuning(b"detect_variant", 0)
    assert L.cs_set_tuning(b"no_such_key", 1) < 0


def test_dense_candidates_low_threshold(cs):
    """thresh close to 0 flags almost every pixel: the thread-per-item extrema path, the keypoint queue
    overflow path and the maxPts clamp are all exercised; counts agree with the oracle."""
    arr = synth_image(320, 240, seed=9)
    got = _extract(cs, arr, thresh=0.05)
    want, _ = oracle.extract(arr, 5, 1.0, 0.05)
    assert len(want) > 2000
    assert abs(len(got) - len(want)) <= 0.003 * len(want) + 2
    _assert_close(compare_sets(canon(got), canon(want)), min_frac=0.99)

"""GPU tests of the batched TMA pipeline (round 2): identical to the round-1 per-image kernels (which are pinned to the
reference), batches equal single images, the reference's cap of 32 extrema per block."""
import ctypes
import hashlib
import os

import numpy as np
import pytest

import oracle
from compare import compare_sets
from cudasift_b200.synth import synth_image

pytestmark = pytest.mark.gpu

FIELDS = ("xpos", "ypos", "scale", "sharpness", "edgeness", "orientation", "subsampling", "data")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def canon(p):
    return p[np.lexsort((p["orientation"], p["scale"], p["xpos"], p["ypos"], p["subsampling"]))]


def dev_image(cs, img):
    h, w = img.shape
    pitch = cs.iAlignUp(w, 128)
    ci = cs.CudaImage().Allocate(w, h, pitch, False, None, img)
    ci.Download()
    return ci, pitch


def run_extractor(cs, img, legacy, octaves=5, thresh=3.0, scaleUp=False, levels=False):
    cs.set_tuning("legacy", 1 if legacy else 0)
    try:
        h, w = img.shape
        ex = cs.Extractor(w, h, octaves, 32768, scaleUp)
        ci, pitch = dev_image(cs, img)
        ex.submit_device(ci.d_data, pitch, 1.0, thresh, 0.0)
        n = ex.wait()
        pts = ex.device_points_at(0, n)
        lv = []
        if levels:
            for l in range(octaves):
                try:
                    lv.append(ex.read_level(0, l))
                except cs.CudaSiftError:
                    break
        ex.close()
    finally:
        cs.set_tuning("legacy", 0)
    return pts, lv


def assert_identical(a, b, what):
    a, b = canon(a), canon(b)
    assert len(a) == len(b), (what, len(a), len(b))
    for f in FIELDS:
        assert np.array_equal(a[f], b[f]), (what, f)


@pytest.mark.parametrize("w,h,octaves,thresh,up", [(1920, 1080, 5, 3.0, False), (1280, 960, 5, 3.0, False), (641, 479, 4, 2.0, False),
                                                   (150, 100, 3, 1.0, False), (640, 480, 5, 3.0, True), (300, 200, 1, 2.0, False),
                                                   (1000, 700, 7, 3.0, False), (257, 131, 2, 1.5, False), (20, 12, 5, 0.5, False)])
def test_batched_pipeline_equals_round1_kernels(cs, w, h, octaves, thresh, up):
    """Pyramid levels and keypoint records of the TMA pipeline are bit-identical to the round-1 kernels, which
    test_pyramid_gpu / test_extract_gpu pin to the reference library and the oracle."""
    img = synth_image(w, h, seed=7)
    pn, ln = run_extractor(cs, img, False, octaves, thresh, up, levels=True)
    po, lo = run_extractor(cs, img, True, octaves, thresh, up, levels=True)
    assert len(ln) == len(lo) > 0
    for l, (a, b) in enumerate(zip(ln, lo)):
        assert a.shape == b.shape and np.array_equal(a, b), ("level", l)
    assert_identical(pn, po, "records")


def test_dropin_call_equals_round1(cs):
    img = synth_image(1280, 960, seed=3)
    a = cs.extract_host(img)
    cs.set_tuning("legacy", 1)
    try:
        b = cs.extract_host(img)
    finally:
        cs.set_tuning("legacy", 0)
    assert len(a) > 500
    assert_identical(a, b, "cs_extract_host")


def test_batch_equals_single_images(cs):
    """A batch of six different images (device pointers, host buffers, a partial batch, the captured graph) gives every
    image exactly the records it gets alone."""
    w, h = 960, 540
    imgs = [synth_image(w, h, seed=100 + i) for i in range(6)]
    singles = [run_extractor(cs, im, False)[0] for im in imgs]
    ex = cs.Extractor(w, h, 5, 16384, False, batch=6)
    cis = [dev_image(cs, im) for im in imgs]
    for rep in range(4):                       # reps >= 2 run through the captured graph
        order = list(range(6)) if rep % 2 == 0 else [3, 1, 5, 0, 2, 4]
        ex.submit_device_batch([cis[i][0].d_data for i in order], cis[0][1], 1.0, 3.0, 0.0)
        counts = ex.wait_batch(6)
        for slot, i in enumerate(order):
            assert_identical(ex.device_points_at(slot, counts[slot]), singles[i], ("device", rep, slot))
    ptrs = []
    for i in range(6):
        hp = cs.lib().cs_extractor_host_image_at(ex.handle, i)
        ctypes.memmove(hp, imgs[i].ctypes.data, w * h * 4)
        ptrs.append(hp)
    ex.submit_host_batch(ptrs, 1.0, 3.0, 0.0)
    counts = ex.wait_batch(6)
    for i in range(6):
        assert_identical(ex.host_points_at(i, counts[i]), singles[i], ("host", i))
    ex.submit_device_batch([c[0].d_data for c in cis[:3]], cis[0][1], 1.0, 3.0, 0.0)
    counts = ex.wait_batch(3)
    for i in range(3):
        assert_identical(ex.device_points_at(i, counts[i]), singles[i], ("partial", i))
    with pytest.raises(cs.CudaSiftError):
        ex.submit_device_batch([c[0].d_data for c in cis] + [cis[0][0].d_data], cis[0][1], 1.0, 3.0, 0.0)   # 7 > batch
    ex.close()


def test_unaligned_image_takes_the_legacy_path(cs):
    """An image TMA cannot address (pitch not a multiple of 4 floats) still extracts through the drop-in call."""
    img = synth_image(333, 201, seed=34)
    L = cs.lib()
    pitch = 335                                                    # odd pitch
    buf = cs.DeviceBuffer(pitch * 201 * 4)
    padded = np.zeros((201, pitch), np.float32); padded[:, :333] = img
    buf.upload(padded)
    pts = cs.DeviceBuffer(8192 * 576)
    n = L.cs_extract(buf.ptr, 333, 201, pitch, 5, 1.0, 3.0, 0.0, 0, None, pts.ptr, None, 8192)
    assert n > 0, L.cs_last_error()
    want = cs.extract_host(img)
    assert_identical(pts.download(cs.SIFT_DTYPE, n), want, "odd pitch")


def test_extrema_cap_mechanism_vs_oracle(cs):
    """The reference keeps at most 32 extrema per (30x8 block, scale) (cudaSiftD.cu:1371,1379).  DoG planes that come
    out of the blur chain never hold 33, so the limit is lowered (product and oracle alike) to make the cap -- per-cell
    counters, overflow list, fix-up kernel, removal + compaction -- do work."""
    img = synth_image(320, 240, seed=9)
    try:
        for limit in (4, 5):
            cs.set_tuning("cap32_limit", limit)
            oracle.set_cap_limit(limit)
            got = cs.extract_host(img, thresh=0.05)
            want, _ = oracle.extract(img, 5, 1.0, 0.05)
            dropped = oracle.last_dropped()
            assert dropped > 20, dropped
            assert abs(len(got) - len(want)) <= 0.003 * len(want) + 2, (limit, len(got), len(want))
            rep = compare_sets(canon(got), canon(want))
            assert rep["pairs"] >= 0.99 * len(want), (limit, rep)
        cs.set_tuning("cap32_limit", 5)
        capped = cs.extract_host(img, thresh=0.05)
        cs.set_tuning("cap32", 0)
        free = cs.extract_host(img, thresh=0.05)
        assert len(free) > len(capped) + 20                        # the switch: CUDASIFT_NO_CAP32 / cs_set_tuning("cap32", 0)
        # every capped keypoint is one of the uncapped ones, untouched
        key = lambda p: set(zip(p["subsampling"].tolist(), p["xpos"].tolist(), p["ypos"].tolist(), p["scale"].tolist(), p["orientation"].tolist()))
        assert key(capped) <= key(free)
    finally:
        cs.set_tuning("cap32", 1)
        cs.set_tuning("cap32_limit", 32)
        oracle.set_cap_limit(32)
    # default limit: the product, the oracle (cap on) and the round-1 kernels (no cap) agree on a dense input
    a = cs.extract_host(img, thresh=0.05)
    want, _ = oracle.extract(img, 5, 1.0, 0.05)
    assert oracle.last_dropped() == 0
    assert abs(len(a) - len(want)) <= 0.003 * len(want) + 2


def dense_cases():
    """Dense, low-threshold inputs and their thresholds: clipped noise, and a synthetic image."""
    rng = np.random.default_rng(5)
    noise = np.clip(128 + 60 * rng.standard_normal((480, 640)), 1, 254).astype(np.float32)
    return ((noise, 0.5), (synth_image(640, 480, seed=12), 0.1))


def test_dense_input_vs_reference(cs):
    """Dense, low-threshold input against the reference itself (its results are stored in
    tests/golden/reference_checks.npz): equal counts and positions (the cap included)."""
    g = np.load(os.path.join(GOLDEN, "reference_checks.npz"))
    for k, (arr, th) in enumerate(dense_cases()):
        got = canon(cs.extract_host(arr, thresh=th))
        assert int(g["dense%d_count" % k]) == len(got) > 3000, (int(g["dense%d_count" % k]), len(got))
        for f in ("xpos", "ypos", "scale", "sharpness", "edgeness", "subsampling"):
            assert sha(got[f]) == str(g["dense%d_%s_sha" % (k, f)]), f

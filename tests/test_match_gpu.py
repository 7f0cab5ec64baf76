"""GPU parity of MatchSiftData: match indices (and here all five output fields) bit-exact
against the oracle and against the reference library on identical SiftData arrays."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from cudasift_b200.synth import synth_descriptors

pytestmark = pytest.mark.gpu
FIELDS = ("score", "ambiguity", "match", "match_xpos", "match_ypos")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _eq(a, b, what):
    for f in FIELDS:
        assert np.array_equal(a[f], b[f]), "%s: field %s differs in %d rows" % (what, f, int((a[f] != b[f]).sum()))


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("n1,n2", [(1, 32), (100, 64), (257, 500), (1000, 1031), (2000, 2000)])
def test_match_bit_exact_vs_oracle(cs, n1, n2, mode):
    s1, s2 = synth_descriptors(n1, 1), synth_descriptors(n2, 2)
    got, _ = cs.match_host(s1, s2, mode=mode)
    _eq(got, oracle.match(s1, s2, threads=8), "mode %d %dx%d" % (mode, n1, n2))


@pytest.mark.parametrize("mode", [1, 2])
def test_match_quirks(cs, mode):
    s2, s1 = synth_descriptors(640, 5), synth_descriptors(300, 6)
    s1["data"][0] = s2["data"][40]; s2["data"][7] = s2["data"][40]; s2["data"][33] = s2["data"][40]   # Q10 ties
    s1["data"][1] = s2["data"][639]                       # best candidate in the unvisited tail? (640 % 32 == 0: visited)
    s1["data"][2] *= -1                                   # Q11: no positive score
    s1["data"][3] = 0
    got, _ = cs.match_host(s1, s2, mode=mode)
    want = oracle.match(s1, s2)
    _eq(got, want, "quirks")
    assert got["match"][0] == 33 and got["match"][2] == -1 and got["match"][3] == -1
    got2, _ = cs.match_host(s1, s2[:630], mode=mode)      # Q7: tail of 22 ignored
    _eq(got2, oracle.match(s1, s2[:630]), "tail")
    got3, _ = cs.match_host(s1, s2[:31], mode=mode)       # nothing visited
    assert np.all(got3["match"] == -1) and np.all(got3["score"] == 0)
    # SIFT-like (clamped) descriptors and near-duplicate candidates
    a, b = synth_descriptors(500, 11, sift_like=True), synth_descriptors(800, 12, sift_like=True)
    b["data"][100:200] = b["data"][0:100] * np.float32(1.0) + np.float32(1e-7)
    got4, _ = cs.match_host(a, b, mode=mode)
    _eq(got4, oracle.match(a, b, threads=8), "near duplicates")


@pytest.mark.parametrize("n", [2000, 10000])
def test_match_bit_exact_vs_reference(cs, n):
    """BASELINE.json config #3: 2000x2000 then 10000x10000 synthetic descriptors, against the sha256 digests of the
    reference's five output fields (tests/golden/reference_checks.npz)."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))
    s1, s2 = synth_descriptors(n, 1), synth_descriptors(n, 2)

    def _eq_ref(a, what):
        for f in FIELDS:
            assert _sha(a[f]) == str(g["match%d_%s_sha" % (n, f)]), "%s: field %s differs" % (what, f)
    for mode in (1, 2):
        got, _ = cs.match_host(s1, s2, mode=mode)
        _eq_ref(got, "mode %d vs reference %d" % (mode, n))
    if n == 2000:
        _eq_ref(oracle.match(s1, s2, threads=8), "oracle vs reference")


def test_match_device_api(cs):
    """MatchSiftData through the SiftData mirror (host copy of the 5 fields, matching.cu:1195-1199)."""
    s1, s2 = synth_descriptors(300, 3), synth_descriptors(352, 4)
    d1 = cs.InitSiftData(cs.SiftData(), 512, True, True)
    d2 = cs.InitSiftData(cs.SiftData(), 512, False, True)
    d1._buf.upload(s1); d2._buf.upload(s2)
    d1.numPts, d2.numPts = 300, 352
    ms = cs.MatchSiftData(d1, d2)
    assert ms > 0
    want = oracle.match(s1, s2)
    _eq(d1.h_data[:300], want, "host copy")
    dev = d1._buf.download(cs.SIFT_DTYPE, 300)
    _eq(dev, want, "device records")
    assert np.array_equal(dev["data"], s1["data"])        # descriptors untouched
    d1.numPts = 0
    assert cs.MatchSiftData(d1, d2) == 0.0                # matching.cu:1095-1096


def test_match_large_tensor_equals_exact(cs):
    """Beyond the sizes the CPU oracle can check quickly: the tensor path against the exact
    SIMT path (itself bit-identical to the oracle/reference at smaller sizes)."""
    n1, n2 = 20000, 24000
    s1, s2 = synth_descriptors(n1, 21, sift_like=True), synth_descriptors(n2, 22, sift_like=True)
    a, _ = cs.match_host(s1, s2, mode=1)
    b, _ = cs.match_host(s1, s2, mode=2)
    _eq(b, a, "tensor vs exact %dx%d" % (n1, n2))
    st = cs.match_stats()
    assert st[3] == 2 and st[2] < 0.01 * n1, st            # tensor path taken, <1 % rows needed the fallback


def test_match_extracted_descriptors(cs):
    """End to end on real descriptors (many zeros, clamped at 0.2): ExtractSift on two views of a
    scene, MatchSiftData on both paths, identical output; unambiguous matches recover the shift."""
    from cudasift_b200.synth import synth_image
    img = synth_image(1280, 960, seed=77)
    shifted = np.roll(img, (7, 11), axis=(0, 1))
    p1, p2 = cs.extract_host(img, thresh=3.0), cs.extract_host(shifted, thresh=3.0)
    assert len(p1) > 500 and len(p2) > 500
    a, _ = cs.match_host(p1, p2, mode=1)
    b, _ = cs.match_host(p1, p2, mode=2)
    _eq(b, a, "extracted descriptors")
    _eq(a, oracle.match(p1, p2, threads=8), "exact path vs oracle")
    good = (a["score"] > 0.9) & (a["ambiguity"] < 0.9)
    dx, dy = a["match_xpos"][good] - a["xpos"][good], a["match_ypos"][good] - a["ypos"][good]
    assert good.sum() > 100            # the synthetic scene repeats shapes: many matches are ambiguous by design
    # chance level for a random pairing is ~0 (the scene repeats shapes and np.roll wraps, so many of the
    # 'good' matches are legitimately elsewhere): 15 % within half a pixel of the true shift shows that
    # positions and descriptors belong together
    hit = (np.abs(dx - 11) < 0.5) & (np.abs(dy - 7) < 0.5)
    assert hit.mean() > 0.15, (hit.mean(), good.sum())


def test_match_out_of_range_inputs_take_the_exact_path(cs):
    """|x| >= 8 (or NaN/Inf) cannot be bounded by the split-FP16 screening: the device-side gate sends
    every row through the exact kernel, no host round trip, same results as mode 1."""
    s1, s2 = synth_descriptors(600, 11), synth_descriptors(700, 12)
    s2["data"][5, 17] = 100.0
    a, _ = cs.match_host(s1, s2, mode=1)
    b, _ = cs.match_host(s1, s2, mode=2)
    _eq(b, a, "out of range")
    assert cs.match_stats()[2] > len(s1)            # flagged: everything went the exact way
    s2 = synth_descriptors(700, 12)
    s1["data"][3, 0] = np.nan
    a, _ = cs.match_host(s1, s2, mode=1)
    b, _ = cs.match_host(s1, s2, mode=2)
    for f in ("score", "ambiguity", "match", "match_xpos", "match_ypos"):
        assert a[f].tobytes() == b[f].tobytes(), f
    # and the next call with clean inputs is back on the tensor path (the flag areas alternate)
    s1 = synth_descriptors(600, 11)
    a, _ = cs.match_host(s1, s2, mode=1)
    b, _ = cs.match_host(s1, s2, mode=2)
    _eq(b, a, "clean again")
    assert cs.match_stats()[2] < 0.01 * len(s1)


def test_match_triplicates_fall_back_per_row(cs):
    """Three identical candidates in one partition (p2 = 0, 32, 64) tie the three largest group maxima of
    every row that likes them: such rows cannot be certified and are re-scanned exactly -- same output."""
    s1, s2 = synth_descriptors(512, 21), synth_descriptors(640, 22)
    s2["data"][32] = s2["data"][0]
    s2["data"][64] = s2["data"][0]
    s1["data"][:64] = s2["data"][0] * 0.999 + s1["data"][:64] * 0.001      # rows whose best match is the triplicate
    a, _ = cs.match_host(s1, s2, mode=1)
    b, _ = cs.match_host(s1, s2, mode=2)
    _eq(b, a, "triplicates")
    st = cs.match_stats()
    assert 0 < st[2] < len(s1)
    assert (a["match"][:64] == 0).all()             # lowest index wins the tie (matching.cu:354, strict '>')

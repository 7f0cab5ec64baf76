#!/usr/bin/env python
"""Record what the tests that compare with the UNMODIFIED reference library compared against.

Run on a GPU where the reference was built into oracle/_ref (cudasift_b200/build.py):

  python tests/golden/make_reference_checks.py OUTDIR

and commit OUTDIR/reference_checks.npz, OUTDIR/img1_crop.png and OUTDIR/img2_crop.png under tests/golden/.
Bit-exact results are kept as sha256 digests of the arrays; the rest as small arrays or a seeded sample of rows:
  stages77_*, dog78_*     LowPass / ScaleDown / ScaleUp / DoG planes     (tests/test_pyramid_gpu.py)
  match{n}_*              MatchSiftData n x n, the five output fields    (tests/test_match_gpu.py)
  homography_*            FindHomography after srand(11)                 (tests/test_homography.py)
  dense{k}_*              ExtractSift on dense, low-threshold inputs     (tests/test_batch_gpu.py)
  extract{k}_*            two ExtractSift runs per synthetic case        (tests/test_extract_gpu.py, compare.reference_summary)
  img{1,2}_crop_count     ExtractSift on 400x300 grey crops of the reference's demo photographs (tests/test_oracle_cpu.py)
"""
import ctypes
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cudasift_b200 as cs                      # noqa: E402
import reflib                                   # noqa: E402
from compare import reference_summary          # noqa: E402
from cudasift_b200 import build                 # noqa: E402
from cudasift_b200.synth import synth_descriptors, synth_image   # noqa: E402

MATCH_FIELDS = ("score", "ambiguity", "match", "match_xpos", "match_ypos")
POS_FIELDS = ("xpos", "ypos", "scale", "sharpness", "edgeness", "subsampling")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def canon(p):
    return p[np.lexsort((p["orientation"], p["scale"], p["xpos"], p["ypos"], p["subsampling"]))]


def main(out):
    import cv2
    from test_batch_gpu import dense_cases
    from test_extract_gpu import REF_CASES, ref_case_image
    from test_homography import planted
    from test_oracle_cpu import CROP
    os.makedirs(out, exist_ok=True)
    cs.InitCuda(0)
    ref = reflib.load_reference()
    assert ref is not None, "reference library missing: build it into oracle/_ref first"
    g = {}
    # ---- image stages ----
    arr = synth_image(640, 480, seed=77)
    g["stages77_lowpass_sha"] = sha(ref.lowpass(arr, 1.0))
    g["stages77_scaledown_sha"] = sha(ref.scaledown(arr))
    g["stages77_scaleup_sha"] = sha(ref.scaleup(np.ascontiguousarray(arr[:200, :256])))
    arr = synth_image(640, 480, seed=78)
    for octave in (5, 2):
        g["dog78_oct%d_sha" % octave] = sha(ref.dog(arr, 5, octave))
    # ---- matching ----
    for n in (2000, 10000):
        m, _ = ref.match(synth_descriptors(n, 1), synth_descriptors(n, 2))
        for f in MATCH_FIELDS:
            g["match%d_%s_sha" % (n, f)] = sha(m[f])
    # ---- FindHomography ----
    p, _ = planted(n=1600, seed=9)
    f = ref.L._Z14FindHomographyR8SiftDataPfPiifff
    f.restype = ctypes.c_double
    f.argtypes = [ctypes.POINTER(reflib.CSiftData), ctypes.c_void_p, ctypes.POINTER(ctypes.c_int), ctypes.c_int,
                  ctypes.c_float, ctypes.c_float, ctypes.c_float]
    sd = cs.InitSiftData(cs.SiftData(), 2048, False, True)
    sd._buf.upload(p); sd.numPts = len(p)
    rsd = reflib.CSiftData(len(p), 2048, None, sd.d_data)
    Hr = np.zeros(9, np.float32); nr = ctypes.c_int(0)
    ctypes.CDLL(None).srand(11)
    with reflib.quiet_stdout():
        f(ctypes.byref(rsd), Hr.ctypes.data, ctypes.byref(nr), 2000, 0.85, 0.95, 4.0)
    g["homography_H"], g["homography_numfit"] = Hr, np.int32(nr.value)
    cs.FreeSiftData(sd)
    # ---- extraction ----
    for k, (im, th) in enumerate(dense_cases()):
        r = canon(ref.extract(im, thresh=th))
        g["dense%d_count" % k] = np.int32(len(r))
        for fld in POS_FIELDS:
            g["dense%d_%s_sha" % (k, fld)] = sha(r[fld])
    for k, case in enumerate(REF_CASES):
        im, kw = ref_case_image(case), case[3]
        r1, r2 = canon(ref.extract(im, **kw)), canon(ref.extract(im, **kw))
        for key, v in reference_summary(r1, r2, seed=k).items():
            g["extract%d_%s" % (k, key)] = v
        print("extract case", k, kw, len(r1), len(r2))
    for name in ("img1", "img2"):
        grey = cv2.imread(os.path.join(build.REF_DIR, "data", name + ".png"), 0)
        y0, x0, h, w = CROP
        crop = np.ascontiguousarray(grey[y0:y0 + h, x0:x0 + w])
        assert cv2.imwrite(os.path.join(out, name + "_crop.png"), crop, [cv2.IMWRITE_PNG_COMPRESSION, 9])
        g[name + "_crop_count"] = np.int32(len(ref.extract(crop.astype(np.float32), 5, 1.0, 3.0)))
        print(name, "crop", int(g[name + "_crop_count"]))
    np.savez_compressed(os.path.join(out, "reference_checks.npz"), **g)
    print("written to", out)


if __name__ == "__main__":
    main(sys.argv[1])

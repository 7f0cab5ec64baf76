"""examples/sift_demo.cpp: a g++-compiled caller of include/cudaSift.h + cudaImage.h (the role of the
reference's mainSift.cpp:25-93, SURVEY 8f-4), run end to end and cross-checked with the ctypes API."""
import os
import re
import subprocess

import numpy as np
import pytest

from cudasift_b200 import build as _build
from cudasift_b200.synth import synth_image



def _write_pgm(path, img):
    a = np.clip(np.rint(img), 0, 255).astype(np.uint8)
    with open(path, "wb") as f:
        f.write(b"P5\n# synthetic\n%d %d\n255\n" % (a.shape[1], a.shape[0]))
        f.write(a.tobytes())
    return a.astype(np.float32)


@pytest.mark.gpu
def test_demo_program(cs, tmp_path):
    demo = _build.build_demo()
    assert demo and os.path.exists(demo)
    left = synth_image(1280, 960, seed=5)
    right = np.roll(left, (9, -13), axis=(0, 1))
    l8 = _write_pgm(str(tmp_path / "l.pgm"), left)
    r8 = _write_pgm(str(tmp_path / "r.pgm"), right)
    out = str(tmp_path / "marked.pgm")
    r = subprocess.run([demo, str(tmp_path / "l.pgm"), str(tmp_path / "r.pgm"), "--thresh", "3.0", "--repeat", "3", "--out", out,
                        "--print", "2"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0, r.stdout
    m = re.search(r"Number of original features: (\d+) (\d+)", r.stdout)
    n1, n2 = int(m.group(1)), int(m.group(2))
    assert n1 == len(cs.extract_host(l8, thresh=3.0)) and n2 == len(cs.extract_host(r8, thresh=3.0))
    m = re.search(r"Number of matching features: (\d+) (\d+)", r.stdout)
    numFit, numMatches = int(m.group(1)), int(m.group(2))
    assert numFit > 50 and numMatches > 50, r.stdout
    H = np.array([float(v) for v in re.search(r"Homography:\s+((?:\S+\s+){9})", r.stdout).group(1).split()]).reshape(3, 3)
    # the planted shift; RANSAC draws by record index and the record order is unspecified (atomic slot
    # allocation, as in the reference), so the fit moves by a fraction of a pixel from run to run
    assert abs(H[0, 2] + 13) < 1.5 and abs(H[1, 2] - 9) < 1.5 and abs(H[0, 0] - 1) < 0.01, H
    with open(out, "rb") as f:
        assert f.read(2) == b"P5"
    assert os.path.getsize(out) > 1280 * 960


def _run_demo(demo, args):
    r = subprocess.run([demo] + args, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=180)
    assert r.returncode == 0, r.stdout
    m = re.search(r"Number of original features: (\d+) (\d+)", r.stdout)
    f = re.search(r"Number of matching features: (\d+) (\d+)", r.stdout)
    return (int(m.group(1)), int(m.group(2))), (int(f.group(1)), int(f.group(2))), r.stdout


@pytest.mark.gpu
def test_demo_png_input_and_reference_drawing(cs, tmp_path):
    """SURVEY 8 f4: the reference demo's second input pair is PNG (mainSift.cpp:37-38) and its output is the drawing of
    PrintMatchData (mainSift.cpp:150-200).  The demo decodes PNG itself (zlib) and --style reference draws the same
    primitives; feature counts must equal the ctypes API on the identically converted grey image."""
    cv2 = pytest.importorskip("cv2")
    # a colour pair in the demo photographs' size (1920x1080 RGB), the second shifted: three different channels, so
    # that the colour-to-grey conversion matters
    base = [np.clip(synth_image(1920, 1080, seed=s), 0, 255).astype(np.uint8) for s in (61, 62)]
    bgr = np.stack([base[0], np.roll(base[0], 3, axis=1), base[1]], axis=2)
    p1, p2 = str(tmp_path / "img1.png"), str(tmp_path / "img2.png")
    assert cv2.imwrite(p1, bgr) and cv2.imwrite(p2, np.roll(bgr, (9, -13), axis=(0, 1)))
    demo = _build.build_demo()
    out = str(tmp_path / "drawn.pgm")
    (n1, n2), (fit, matches), log = _run_demo(demo, [p1, p2, "--thresh", "2.0", "--repeat", "1", "--out", out, "--style", "reference"])
    g1 = cv2.cvtColor(cv2.imread(p1, cv2.IMREAD_COLOR), cv2.COLOR_BGR2GRAY).astype(np.float32)
    g2 = cv2.cvtColor(cv2.imread(p2, cv2.IMREAD_COLOR), cv2.COLOR_BGR2GRAY).astype(np.float32)
    assert n1 == len(cs.extract_host(g1, thresh=2.0)) and n2 == len(cs.extract_host(g2, thresh=2.0)), log
    assert matches > 100 and fit > 100, log                      # the pair overlaps (README.md:33 reports ~1000+ matches)
    with open(out, "rb") as f:
        hdr = f.readline() + f.readline() + f.readline()
        drawn = np.frombuffer(f.read(), np.uint8).reshape(g1.shape)
    assert hdr.startswith(b"P5")
    changed = int((drawn != np.clip(g1, 0, 255).astype(np.uint8)).sum())
    assert changed > 20 * n1 // 4, changed                        # crosses and match lines were drawn


@pytest.mark.gpu
def test_demo_managed_memory_flavour(cs, tmp_path):
    """SURVEY 8 f4 / cudaSift.h:27-32: the MANAGEDMEM flavour (SiftData::m_data in unified memory) is built
    (libcudasift_b200_managed.so + the demo compiled with -DMANAGEDMEM) and gives the same counts as the default build."""
    demo, demo_m = _build.build_demo(), _build.build_demo(managed=True)
    assert demo_m and os.path.exists(demo_m)
    left = synth_image(960, 720, seed=8)
    right = np.roll(left, (5, 7), axis=(0, 1))
    _write_pgm(str(tmp_path / "l.pgm"), left)
    _write_pgm(str(tmp_path / "r.pgm"), right)
    args = [str(tmp_path / "l.pgm"), str(tmp_path / "r.pgm"), "--thresh", "3.0", "--repeat", "2", "--print", "1"]
    c0, f0, log0 = _run_demo(demo, args)
    c1, f1, log1 = _run_demo(demo_m, args)
    assert c0 == c1, (log0, log1)
    assert f1[0] > 50 and abs(f1[0] - f0[0]) <= max(3, f0[0] // 50), (f0, f1)     # RANSAC draws depend on record order

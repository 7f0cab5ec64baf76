"""GPU parity of the image stages (LowPass, ScaleDown, ScaleUp, Laplace/DoG): bit-exact
against the oracle and against the stored results of the reference library itself."""
import hashlib
import os

import numpy as np
import pytest

import oracle
from cudasift_b200.synth import synth_image

pytestmark = pytest.mark.gpu


def _upload(cs, arr, pitch=None):
    img = cs.CudaImage().Allocate(arr.shape[1], arr.shape[0], pitch, False, None, arr)
    img.Download()
    return img


def _blank(cs, w, h, pitch=None):
    img = cs.CudaImage().Allocate(w, h, pitch, True)
    img.Download()
    return img


SIZES = [(640, 480), (500, 333), (1920, 1080), (135, 67), (33, 20)]


@pytest.mark.parametrize("w,h", SIZES)
def test_lowpass_bit_exact_vs_oracle(cs, w, h):
    arr = synth_image(w, h, seed=w + h)
    src, dst = _upload(cs, arr), _blank(cs, w, h)
    for sigma in (1.0, 0.7):
        assert cs.lib().cs_lowpass(src.d_data, dst.d_data, w, h, src.pitch, sigma) == 0
        got = dst.Readback()
        assert np.array_equal(got, oracle.lowpass(arr, sigma)), "LowPass differs from the oracle"


@pytest.mark.parametrize("w,h", SIZES)
def test_scaledown_bit_exact_vs_oracle(cs, w, h):
    arr = synth_image(w, h, seed=2 * w + h)
    src, dst = _upload(cs, arr), _blank(cs, w // 2, h // 2)
    assert cs.lib().cs_scaledown(src.d_data, dst.d_data, w, h, src.pitch, dst.pitch) == 0
    assert np.array_equal(dst.Readback(), oracle.scaledown(arr))


def test_scaleup_bit_exact_vs_oracle(cs):
    arr = synth_image(321, 123, seed=9)
    src, dst = _upload(cs, arr), _blank(cs, 642, 246)
    assert cs.lib().cs_scaleup(src.d_data, dst.d_data, 321, 123, src.pitch, dst.pitch) == 0
    assert np.array_equal(dst.Readback(), oracle.scaleup(arr))


@pytest.mark.parametrize("w,h,octave", [(640, 480, 5), (500, 333, 3), (120, 67, 1), (1920, 1080, 5)])
def test_dog_planes_bit_exact_vs_oracle(cs, w, h, octave):
    arr = synth_image(w, h, seed=3 * w + h)
    src = _upload(cs, arr)
    buf = cs.DeviceBuffer(7 * h * src.pitch * 4)
    buf.zero()
    assert cs.lib().cs_dog_planes(src.d_data, buf.ptr, w, h, src.pitch, 5, octave) == 0
    got = buf.download(np.float32, 7 * h * src.pitch).reshape(7, h, src.pitch)[:, :, :w]
    want = oracle.dog(arr, 5, octave)
    assert np.array_equal(got, want), "DoG planes differ from the oracle (max %g)" % np.abs(got - want).max()


def test_laplace_taps_equal_oracle(cs):
    for n in (1, 3, 5, 7):
        k = np.zeros(8 * 12 * 16, np.float32)
        assert cs.lib().cs_laplace_taps(n, 0.0, k.ctypes.data) == 0
        o = oracle.laplace_taps(n)
        for octave in range(1, n + 1):
            assert np.array_equal(k.reshape(8, 12, 16)[octave, :8, :5], o.reshape(8, 12, 16)[octave, :8, :5])


# ---------------------------------------------------------------- against the reference itself
def _reference_checks():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_stages_bit_exact_vs_reference(cs, selflib):
    """Oracle and product against the sha256 digests of the reference's LowPass / ScaleDown / ScaleUp."""
    g = _reference_checks()
    arr = synth_image(640, 480, seed=77)
    for sigma in (1.0,):
        assert _sha(oracle.lowpass(arr, sigma)) == str(g["stages77_lowpass_sha"]), "oracle LowPass != reference"
        assert _sha(selflib.lowpass(arr, sigma)) == str(g["stages77_lowpass_sha"]), "product LowPass != reference"
    assert _sha(oracle.scaledown(arr)) == str(g["stages77_scaledown_sha"]), "oracle ScaleDown != reference"
    assert _sha(selflib.scaledown(arr)) == str(g["stages77_scaledown_sha"]), "product ScaleDown != reference"
    small = np.ascontiguousarray(arr[:200, :256])
    assert _sha(oracle.scaleup(small)) == _sha(selflib.scaleup(small)) == str(g["stages77_scaleup_sha"])


@pytest.mark.parametrize("octave", [5, 2])
def test_dog_bit_exact_vs_reference(cs, octave):
    o = oracle.dog(synth_image(640, 480, seed=78), 5, octave)
    assert _sha(o) == str(_reference_checks()["dog78_oct%d_sha" % octave]), "oracle DoG != reference"

"""CPU: numpy restatement vs the live OpenCV/NumPy wheels (oracle/cv2_port.py issues the very
calls the reference makes).  Skipped if cv2 is not importable."""
import numpy as np
import pytest

from oracle import corruption_oracle as orc
from oracle import cv2_port
from tests.helpers import synth

pytestmark = pytest.mark.skipif(not cv2_port.available(), reason="opencv not importable")


@pytest.mark.parametrize("shape", [(1, 1), (2, 3), (17, 9), (64, 64), (255, 333), (360, 480), (765, 1360), (541, 961)])
def test_restatement_matches_live_cv2(shape):
    h, w = shape
    for kind in ("uniform", "binary"):
        img = synth(h * 7 + w, h, w, kind)
        assert np.array_equal(orc.apply_motion_blur(img, 9, 0), cv2_port.blur(img, 9, 0))
        assert np.array_equal(orc.apply_lowres(img, 0.5), cv2_port.lowres(img, 0.5))
        np.random.seed(1)
        a = orc.apply_noise(img, 15)
        np.random.seed(1)
        assert np.array_equal(a, cv2_port.noise(img, 15))


def test_letterbox_resize_matches_cv2():
    import cv2
    for h, w in [(765, 1360), (720, 1280), (1050, 1400), (360, 480), (333, 517)]:
        img = synth(h + w, h, w)
        nh, nw, top, left = orc.letterbox_geometry(h, w, 640, 640)
        assert np.array_equal(orc.resize_linear(img, nh, nw), cv2.resize(img, (nw, nh), interpolation=cv2.INTER_LINEAR))

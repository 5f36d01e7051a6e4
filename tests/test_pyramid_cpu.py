"""The Gaussian pyramid on the CPU: the integer restatement (oracle/cv_pyramid_oracle.py) against the installed cv2 and
against frontend.gaussian_pyramid, and the C library's blur taps and level table against the restatement."""
import ctypes as C

import numpy as np
import pytest

cv2 = pytest.importorskip('cv2')

BLUR_SHAPES = [(600, 800, 3), (600, 800), (37, 53, 3), (120, 91), (5, 7, 3), (5, 7), (1, 9), (1, 9, 3), (2, 2), (9, 1)]
EXTRA_SIGMAS = [1.6, 0.7, 4.3]


def _sigmas():
    from oracle import cv_pyramid_oracle as cp
    return cp.pyramid_sigmas() + EXTRA_SIGMAS


@pytest.mark.parametrize('shape', BLUR_SHAPES)
def test_blur_restatement_equals_cv2(shape):
    from oracle import cv_pyramid_oracle as cp
    rng = np.random.default_rng(sum(shape))
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    for sigma in _sigmas():
        want = cv2.GaussianBlur(img, (0, 0), sigmaX=sigma, sigmaY=sigma)
        assert np.array_equal(cp.gaussian_blur_u8(img, sigma), want), sigma


@pytest.mark.parametrize('shape', [(37, 53, 3), (40, 56), (1, 1), (2, 3, 3), (300, 401, 3)])
def test_upsample_restatement_equals_cv2(shape):
    from oracle import cv_pyramid_oracle as cp
    img = np.random.default_rng(7).integers(0, 256, shape, dtype=np.uint8)
    want = cv2.resize(img, (0, 0), fx=2, fy=2, interpolation=cv2.INTER_LINEAR_EXACT)
    assert np.array_equal(cp.upsample2_u8(img), want)


@pytest.mark.parametrize('h,w,grey,seed', [(600, 800, False, 100), (600, 800, True, 100), (301, 417, False, 5),
                                           (240, 320, True, 3), (40, 56, False, 9)])
def test_pyramid_restatement_equals_frontend(h, w, grey, seed):
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image
    from oracle import cv_pyramid_oracle as cp
    img = make_textured_image(h, w, seed=seed)
    if grey:
        img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    want = fe.gaussian_pyramid(img)
    got = cp.gaussian_pyramid_u8(img)
    assert len(got) == len(want)
    for i, (g, x) in enumerate(zip(got, want)):
        assert g.shape == x.shape and np.array_equal(g, x), 'level %d' % i


def test_c_gaussian_taps_equal_restatement():
    from gims_b200 import _lib, build
    from oracle import cv_pyramid_oracle as cp
    build.build()
    taps = (C.c_int * 127)()
    n = C.c_int(0)
    for sigma in _sigmas():
        assert _lib.lib().gims_debug_gaussian_kernel(sigma, taps, C.byref(n)) == 0
        want = cp.gaussian_taps(sigma)
        assert n.value == len(want) and int(want.sum()) == 256
        assert np.array_equal(np.frombuffer(taps, dtype=np.int32)[:n.value], want), sigma


@pytest.mark.parametrize('h,w', [(600, 800), (800, 600), (301, 417), (417, 301), (240, 320), (40, 56), (75, 99),
                                 (1200, 1600), (123, 1001), (17, 23)])
def test_c_pyramid_layout_equals_frontend(h, w):
    from gims_b200 import _lib, build
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image
    from oracle import cv_pyramid_oracle as cp
    build.build()
    img = make_textured_image(h, w, seed=1)
    want = [lv.shape for lv in fe.gaussian_pyramid(img)]
    assert [s + (3,) for s in cp.level_shapes(h, w)] == want
    n = C.c_int(-1)
    assert _lib.lib().gims_pyramid_layout(h, w, 3, C.byref(n), None, None, None) == 0
    assert n.value == len(want)
    off = np.zeros(n.value, dtype=np.int64)
    hh = np.zeros(n.value, dtype=np.int32)
    ww = np.zeros(n.value, dtype=np.int32)
    assert _lib.lib().gims_pyramid_layout(h, w, 3, C.byref(n), off.ctypes.data, hh.ctypes.data, ww.ctypes.data) == 0
    assert [(int(a), int(b), 3) for a, b in zip(hh, ww)] == want
    # levels are disjoint, in order, 256-byte aligned
    assert off[0] == 0 and (off % 256 == 0).all()
    assert (off[1:] >= off[:-1] + hh[:-1].astype(np.int64) * ww[:-1] * 3).all()
    ws = _lib.lib().gims_pyramid_workspace_bytes(h, w, 3)
    assert ws >= 2 * int(hh[0]) * int(ww[0]) * 3


def test_halving_rounds_ties_to_even():
    from oracle import cv_pyramid_oracle as cp
    assert cp.seed_size(301) == 150 and cp.seed_size(75) == 38 and cp.seed_size(5) == 2
    assert cv2.resize(np.zeros((301, 75), np.uint8), (0, 0), fx=0.5, fy=0.5, interpolation=cv2.INTER_NEAREST).shape == (150, 38)


def test_c_pyramid_rejects_bad_arguments():
    from gims_b200 import _lib, build
    build.build()
    n = C.c_int(0)
    assert _lib.lib().gims_pyramid_layout(10, 10, 2, C.byref(n), None, None, None) != 0
    assert _lib.lib().gims_pyramid_layout(0, 10, 3, C.byref(n), None, None, None) != 0
    assert _lib.lib().gims_pyramid_layout(1, 1, 1, C.byref(n), None, None, None) == 0 and n.value == 0

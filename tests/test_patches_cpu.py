"""Row f-2 on the CPU: the restatement of OpenCV's fixed-point cubic warp (oracle/cv_warp_oracle.py) against the installed
cv2, the C library's weight table against the restatement, and the vectorised per-keypoint maps against the reference's
per-keypoint construction (utils/library.py:84-110 as mirrored by frontend.extract_patches)."""
import ctypes as C

import numpy as np
import pytest

cv2 = pytest.importorskip('cv2')


def _image(h, w, seed, channels=3):
    rng = np.random.default_rng(seed)
    shape = (h, w, channels) if channels > 1 else (h, w)
    return cv2.GaussianBlur(rng.integers(0, 256, shape, dtype=np.uint8), (0, 0), 1.2)


def test_warp_restatement_equals_cv2():
    from oracle import cv_warp_oracle as cw
    tab = cw.bicubic_table()
    assert (tab.reshape(32 * 32, 16).sum(1) == 1 << 15).all()
    rng = np.random.default_rng(1)
    for channels in (3, 1):
        img = _image(90, 120, 2 + channels, channels)
        for _ in range(4):
            ang, sc = rng.uniform(0, 2 * np.pi), rng.uniform(0.3, 3.0)
            rot = np.float32([[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]]) / sc
            shift = rot @ rng.uniform(-10, 130, 2)                 # some patches hang over the border
            m = np.hstack([rot, [[15.5 - shift[0]], [15.5 - shift[1]]]])
            ref = cv2.warpAffine(img, m, (32, 32), flags=cv2.INTER_CUBIC, borderMode=cv2.BORDER_CONSTANT)
            assert np.array_equal(ref, cw.warp_affine_cubic_u8(img, m, (32, 32), tab))


def test_c_weight_table_equals_restatement():
    from gims_b200 import _lib, build
    from oracle import cv_warp_oracle as cw
    build.build()
    buf = (C.c_short * (32 * 32 * 16))()
    assert _lib.lib().gims_debug_bicubic_table(buf) == 0
    assert np.array_equal(np.frombuffer(buf, dtype=np.int16).reshape(32, 32, 4, 4), cw.bicubic_table().astype(np.int16))


def test_patch_maps_equal_per_keypoint_construction():
    from gims_b200 import frontend as fe
    from gims_b200.synth import make_textured_image
    from oracle import cv_warp_oracle as cw
    img = make_textured_image(240, 320, seed=4)
    kps = fe.detect(img, 200)
    assert len(kps) > 50
    level, inv = fe.patch_maps(kps)
    r = (fe.PATCH_SUPPORT - 1) / 2
    for i, kp in enumerate(kps):
        octave, layer, scale = fe._unpack_octave(kp)
        step = kp.size * scale * 0.5
        centre = np.array(kp.pt) * scale
        angle = 360.0 - kp.angle
        if abs(angle - 360.0) < 1.19209e-07:
            angle = 0.0
        phi = np.deg2rad(angle)
        s, c = np.sin(phi), np.cos(phi)
        rot = np.float32([[c, -s], [s, c]]) / step
        shift = np.matmul(rot, centre)
        affine = np.hstack([rot, [[r - shift[0]], [r - shift[1]]]])
        assert level[i] == (octave - fe.FIRST_OCTAVE) * (fe.LAYERS + 3) + layer
        assert np.allclose(inv[i], cw.invert_affine(affine), rtol=1e-15, atol=0)


def test_level_check_rejects_keypoints_outside_the_pyramid():
    from gims_b200 import _lib
    from gims_b200 import frontend as fe
    n_levels = 8 * (fe.LAYERS + 3)
    inside = [cv2.KeyPoint(10, 10, 4, 0, 1, o) for o in (0xFF, 0x500 | 6)]     # level 0, the last level
    fe._check_levels(fe.patch_maps(inside)[0], n_levels)
    below = cv2.KeyPoint(10, 10, 4, 0, 1, 0xFE)                                  # octave -2: level -6
    past = cv2.KeyPoint(10, 10, 4, 0, 1, 7)                                      # octave 7: level 48
    for kp, level in ((below, -6), (past, n_levels)):
        assert fe.patch_maps([kp])[0][0] == level
        with pytest.raises(_lib.GimsError, match='level %d of a %d-level' % (level, n_levels)):
            fe._check_levels(fe.patch_maps(inside + [kp])[0], n_levels)

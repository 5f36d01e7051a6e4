"""SIFT detection on the CPU: the numpy restatement (oracle/cv_sift_oracle.py) that csrc/sift.cu follows, pinned
primitive by primitive to the installed cv2, and its keypoints against cv2.SIFT's within the tolerance cv2's own
optimised and unoptimised paths need to agree with each other."""
import numpy as np
import pytest

cv2 = pytest.importorskip('cv2')

IMAGES = [(600, 800, 3, 100), (600, 800, 3, 101), (301, 417, 3, 5), (240, 320, 1, 3), (40, 56, 3, 9)]
BAR = 0.99


def sift_image(h, w, channels, seed):
    from gims_b200.synth import make_textured_image
    img = make_textured_image(h, w, seed=seed)
    return cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if channels == 1 else img


def records(kps):
    """cv2.KeyPoint list -> the record dict the oracle returns."""
    return {'pt': np.array([k.pt for k in kps], dtype=np.float32).reshape(-1, 2),
            'size': np.array([k.size for k in kps], dtype=np.float32),
            'angle': np.array([k.angle for k in kps], dtype=np.float32),
            'response': np.array([k.response for k in kps], dtype=np.float32),
            'octave': np.array([k.octave for k in kps], dtype=np.int64).astype(np.int32)}


def agreement(a, b):
    """Share of the keypoints of `a` that `b` has too: same octave and layer (octave & 0xffff), |dpt| <= 0.01 px,
    |dsize| <= 1e-3 relative, circular |dangle| <= 0.5 degrees."""
    from scipy.spatial import cKDTree
    n = len(a['pt'])
    if n == 0:
        return 1.0
    if len(b['pt']) == 0:
        return 0.0
    tree = cKDTree(b['pt'].astype(np.float64))
    hits = 0
    for i, near in enumerate(tree.query_ball_point(a['pt'].astype(np.float64), 0.01)):
        for j in near:
            d = abs(float(a['angle'][i]) - float(b['angle'][j])) % 360.0
            if ((int(a['octave'][i]) & 0xffff) == (int(b['octave'][j]) & 0xffff)
                    and abs(float(a['size'][i]) - float(b['size'][j])) <= 1e-3 * float(b['size'][j])
                    and min(d, 360.0 - d) <= 0.5):
                hits += 1
                break
    return hits / n


def top(rec, k):
    """The k strongest records (the rule of frontend.detect, ties in order)."""
    if len(rec['response']) <= k:
        return rec
    o = np.argsort(-rec['response'], kind='stable')[:k]
    return {key: v[o] for key, v in rec.items()}


def _cv2_detect(img, optimized=True):
    from gims_b200 import frontend as fe
    was = cv2.useOptimized()
    cv2.setUseOptimized(optimized)
    try:
        return records(fe.detect(img))
    finally:
        cv2.setUseOptimized(was)


def test_grey_conversion_equals_cv2():
    from oracle import cv_sift_oracle as so
    c = np.stack(np.meshgrid(np.arange(256), np.arange(256), np.arange(0, 256, 3), indexing='ij'), -1)
    img = c.reshape(-1, 64, 3).astype(np.uint8)
    assert np.array_equal(so.grey(img), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    g = img[..., 1]
    assert np.array_equal(so.grey(g), g) and np.array_equal(so.grey(g[..., None]), g)


@pytest.mark.parametrize('shape', [(600, 800), (37, 53), (1, 1), (2, 3)])
def test_upsample_equals_cv2(shape):
    from oracle import cv_sift_oracle as so
    f = np.random.default_rng(3).integers(0, 256, shape).astype(np.float32)
    want = cv2.resize(f, (2 * shape[1], 2 * shape[0]), interpolation=cv2.INTER_LINEAR)
    assert np.array_equal(so.upsample2_f32(f), want)


@pytest.mark.parametrize('shape', [(1200, 1600), (75, 100), (9, 13), (3, 40)])
def test_float_blur_close_to_cv2(shape):
    from oracle import cv_sift_oracle as so
    f = np.random.default_rng(4).integers(0, 256, shape).astype(np.float32)
    for sigma in [so.init_sigma()] + so.octave_sigmas():
        want = cv2.GaussianBlur(f, (0, 0), sigmaX=sigma, sigmaY=sigma)
        assert len(so.gaussian_kernel_f32(sigma)) == (int(np.rint(sigma * 8 + 1)) | 1)
        assert np.abs(so.blur_f32(f, sigma) - want).max() <= 1e-4, sigma


def test_kernel_sizes():
    from oracle import cv_sift_oracle as so
    assert [len(so.gaussian_kernel_f32(s)) for s in [so.init_sigma()] + so.octave_sigmas()] == [11, 11, 13, 17, 21, 27]


def test_fast_atan2_equals_cv2():
    from oracle import cv_sift_oracle as so
    v = np.linspace(-300, 300, 601, dtype=np.float32)
    y, x = (a.ravel() for a in np.meshgrid(v, v))
    assert np.array_equal(so.fast_atan2(y, x), cv2.phase(x, y, angleInDegrees=True).ravel())
    assert so.fast_atan2(np.float32(1), np.float32(3)) == np.float32(cv2.fastAtan2(1, 3))


def test_exp_and_magnitude_equal_opencv_code():
    """With optimisations on, cv2 hands exp and magnitude to Intel IPP; OpenCV's own code is what runs without."""
    from oracle import cv_sift_oracle as so
    x = np.linspace(-120, 0, 400001, dtype=np.float32)
    v = np.linspace(-300, 300, 601, dtype=np.float32)
    gy, gx = (a.ravel() for a in np.meshgrid(v, v))
    was = cv2.useOptimized()
    cv2.setUseOptimized(False)
    try:
        want_exp = cv2.exp(x).ravel()
        want_mag = cv2.magnitude(gx, gy).ravel()
    finally:
        cv2.setUseOptimized(was)
    assert np.array_equal(so.exp32f(x), want_exp)
    assert np.array_equal(so.magnitude(gx, gy), want_mag)


@pytest.mark.parametrize('h,w,channels,seed', IMAGES)
def test_oracle_agrees_with_cv2(h, w, channels, seed):
    from oracle import cv_sift_oracle as so
    img = sift_image(h, w, channels, seed)
    got = so.detect(img)
    want = _cv2_detect(img)
    unopt = _cv2_detect(img, optimized=False)
    a, b = agreement(got, want), agreement(want, got)
    ta, tb = agreement(top(got, 2048), top(want, 2048)), agreement(top(want, 2048), top(got, 2048))
    print('%dx%dx%d: oracle %d / cv2 %d keypoints, agreement %.4f / %.4f, top-2048 %.4f / %.4f; cv2 optimised vs not '
          '%.4f / %.4f' % (h, w, channels, len(got['pt']), len(want['pt']), a, b, ta, tb, agreement(want, unopt),
                           agreement(unopt, want)))
    assert min(a, b, ta, tb) >= BAR
    # cv2's order: sorted by (x, y, -size, angle, -response, -octave), no duplicate (pt, size, angle)
    key = np.lexsort((-got['octave'], -got['response'], got['angle'], -got['size'], got['pt'][:, 1], got['pt'][:, 0]))
    assert np.array_equal(key, np.arange(len(key)))


def test_oracle_max_keypoints_takes_the_strongest():
    from oracle import cv_sift_oracle as so
    img = sift_image(240, 320, 1, 3)
    full = so.detect(img)
    got = so.detect(img, 300)
    assert len(got['pt']) == 300
    assert np.all(np.diff(got['response']) <= 0)
    assert got['response'][-1] >= np.sort(full['response'])[::-1][299]


def test_sift_abi_rejects_bad_arguments():
    from gims_b200 import _lib, build
    build.build()
    L = _lib.lib()
    assert L.gims_sift_workspace_bytes(600, 800, 3, 16384) > 4 * 1200 * 1600 * 11
    assert L.gims_sift_workspace_bytes(600, 800, 4, 16384) == 0
    assert L.gims_sift_workspace_bytes(600, 800, 3, 0) == 0
    assert L.gims_sift_detect(None, 600, 800, 3, -1, 16, None, 0, None, None, None, None, None, None, None, None) != 0

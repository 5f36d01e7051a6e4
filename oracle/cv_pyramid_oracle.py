"""TEST INFRASTRUCTURE (like everything under oracle/): a numpy integer restatement of the 8-bit Gaussian pyramid that
frontend.gaussian_pyramid builds with OpenCV (utils/library.py:234-293) — the algorithm csrc/pyramid.cu implements on the
GPU.  Every step is OpenCV's fixed-point arithmetic for CV_8U (imgproc/src/smooth.dispatch.cpp: getGaussianKernelBitExact,
getGaussianKernelFixedPoint_ED, the fixed-point separable filter; imgproc/src/resize.cpp: INTER_LINEAR_EXACT and
INTER_NEAREST), so the restatement equals OpenCV byte for byte.  tests/test_pyramid_cpu.py pins it to the installed cv2,
and the C library's taps and level table to it."""
import math

import numpy as np

FRAC_BITS = 8                 # fraction bits of the blur taps; the row pass is in 1/256, the column pass in 2^-16
PER_OCTAVE = 6                # nOctaveLayers + 3
SEED_LAYER = 3                # nOctaveLayers
FIRST_OCTAVE = -1


def gaussian_taps(sigma):
    """The integer taps (sum 256) cv2.GaussianBlur uses for an 8-bit image: n = cvRound(6 sigma + 1) | 1, exp(-x^2 /
    (2 sigma^2)) normalised in double, the left half quantised with the rounding error carried on, mirrored, centre =
    256 - 2 * (sum of the left half)."""
    n = int(np.rint(sigma * 3 * 2 + 1)) | 1
    n2 = n // 2
    vals = [math.exp((x * x) * (-0.125 / (sigma * sigma))) for x in range(1 - n, 0, 2)]
    mul = 1.0 / (2 * sum(vals) + 1.0)
    m = 1 << FRAC_BITS
    out = np.zeros(n, dtype=np.int64)
    err, tot = 0.0, 0
    for i in range(n2):
        a = vals[i] * mul * m + err
        v = int(np.rint(a))
        err = a - v
        out[i] = out[n - 1 - i] = v
        tot += v
    out[n2] = m - 2 * tot
    return out


def reflect101(n, r):
    """Source indices -r .. n + r - 1 under BORDER_REFLECT_101, reflected as often as needed (a 1-pixel side reads 0)."""
    idx = np.arange(-r, n + r)
    if n == 1:
        return np.zeros_like(idx)
    p = 2 * (n - 1)
    idx = np.mod(idx, p)
    return np.where(idx >= n, p - idx, idx)


def _hwc(img):
    x = img.astype(np.int64)
    return x if x.ndim == 3 else x[..., None]


def _u8(out, like):
    out = out.astype(np.uint8)
    return out if like.ndim == 3 else out[..., 0]


def gaussian_blur_u8(img, sigma):
    """cv2.GaussianBlur(img, (0, 0), sigma, sigma) for uint8 (H, W[, C])."""
    k = gaussian_taps(sigma)
    r = len(k) // 2
    x = _hwc(img)
    h, w = x.shape[:2]
    xi = x[:, reflect101(w, r)]
    row = sum(k[j] * xi[:, j:j + w] for j in range(len(k)))          # 1/256 units, < 2^16
    yi = row[reflect101(h, r)]
    col = sum(k[j] * yi[j:j + h] for j in range(len(k)))             # 2^-16 units
    return _u8((col + (1 << 15)) >> 16, img)


def upsample2_u8(img):
    """cv2.resize(img, (0, 0), fx=2, fy=2, interpolation=INTER_LINEAR_EXACT): destination i reads 64/256 of source a
    and 192/256 of source b = i // 2, a = b - 1 (i even) or b + 1 (i odd), clamped; rows first, then columns."""
    x = _hwc(img)
    h, w = x.shape[:2]

    def taps(n):
        i = np.arange(2 * n)
        a = np.where(i % 2 == 0, i // 2 - 1, i // 2 + 1)
        return np.clip(a, 0, n - 1), i // 2
    a, b = taps(w)
    row = 64 * x[:, a] + 192 * x[:, b]
    a, b = taps(h)
    col = 64 * row[a] + 192 * row[b]
    return _u8((col + (1 << 15)) >> 16, img)


def seed_size(n):
    """cvRound(n * 0.5): ties to even, so 301 gives 150."""
    return int(np.rint(n * 0.5))


def octave_seed_u8(img):
    """cv2.resize(img, (0, 0), fx=0.5, fy=0.5, interpolation=INTER_NEAREST)."""
    h, w = img.shape[:2]
    return np.ascontiguousarray(img[::2, ::2][:seed_size(h), :seed_size(w)])


def n_octaves(h, w):
    """frontend.gaussian_pyramid's octave count for an h x w image (the base level is 2h x 2w)."""
    return int(np.round(np.log(np.float32(min(2 * h, 2 * w))) / np.log(2.0) - 2) - FIRST_OCTAVE)


def pyramid_sigmas():
    """The incremental sigmas of level 1 .. 5 of an octave, computed as frontend.gaussian_pyramid computes them."""
    k = np.float32(2.0 ** (1.0 / 3))
    out = []
    for i in range(1, PER_OCTAVE):
        prev = (k ** np.float32(i - 1)) * 1.6
        total = prev * k
        out.append(math.sqrt(total * total - prev * prev))
    return out


def level_shapes(h, w):
    """(height, width) of every level."""
    shapes, ch, cw = [], 2 * h, 2 * w
    for o in range(n_octaves(h, w)):
        if o > 0:
            ch, cw = seed_size(ch), seed_size(cw)
        shapes += [(ch, cw)] * PER_OCTAVE
    return shapes


def gaussian_pyramid_u8(img):
    """Every level of frontend.gaussian_pyramid(img), as a list of uint8 arrays."""
    sig = pyramid_sigmas()
    levels = []
    for o in range(n_octaves(*img.shape[:2])):
        for i in range(PER_OCTAVE):
            if i == 0:
                lv = upsample2_u8(img) if o == 0 else octave_seed_u8(levels[(o - 1) * PER_OCTAVE + SEED_LAYER])
            else:
                lv = gaussian_blur_u8(levels[-1], sig[i - 1])
            levels.append(np.ascontiguousarray(lv))
    return levels

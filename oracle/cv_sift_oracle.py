"""TEST INFRASTRUCTURE (like everything under oracle/): a vectorised numpy restatement of OpenCV 4.x `SIFT::detect` with
the settings of frontend.SIFT_CONFIG (3 layers per octave, contrastThreshold 0.001, edgeThreshold 80, sigma 1.6, the
image doubled first) — the algorithm csrc/sift.cu implements on the GPU.

OpenCV does not reproduce its own detector bit for bit (its SIMD and scalar paths differ in the last bits of the float
blur), so this module fixes ONE float32 order of operations and the CUDA code follows it exactly: the device detector is
judged bit for bit against this module and with a tolerance against cv2 (tests/test_sift_cpu.py,
tests/test_gpu_sift.py).  Every float32 operation below is rounded on its own; `_fma` marks the fused multiply-adds of
OpenCV's SIMD code (fastAtan2, the histogram smoothing).  tests/test_sift_cpu.py pins fastAtan2 to cv2.phase, and exp32f
and magnitude32f to cv2.exp and cv2.magnitude with optimisations off: with them on, OpenCV hands those two to Intel IPP,
whose code is not public.

Keypoint records: pt float32 (N, 2), size, angle, response float32 (N,), octave int32 (N,) packed as cv2.KeyPoint.octave
(octave byte, layer << 8, cvRound((xi + 0.5) * 255) << 16)."""
import math

import numpy as np

from .cv_pyramid_oracle import n_octaves, reflect101

F = np.float32
LAYERS = 3
PER_OCTAVE = LAYERS + 3          # Gaussian levels per octave
DOG_PER_OCTAVE = LAYERS + 2
BORDER = 5                       # SIFT_IMG_BORDER
MAX_STEPS = 5                    # SIFT_MAX_INTERP_STEPS
SIGMA = 1.6
CONTRAST = F(0.001)
EDGE = F(80.0)
N_BINS = 36
FLT_EPSILON = F(np.finfo(np.float32).eps)
LU_EPS = F(FLT_EPSILON * F(10))
IMG_SCALE = F(F(1) / F(255))
DERIV_SCALE = F(IMG_SCALE * F(0.5))
CROSS_SCALE = F(IMG_SCALE * F(0.25))

# cv::hal::exp32f (core/src/mathfuncs_core.simd.hpp)
_EXP_A0 = .9670371139572337719125840413672004409288e-2
_EXP_A4 = F(1.000000000000002438532970795181890933776 / _EXP_A0)
_EXP_A3 = F(.6931471805521448196800669615864773144641 / _EXP_A0)
_EXP_A2 = F(.2402265109513301490103372422686535526573 / _EXP_A0)
_EXP_A1 = F(.5550339366753125211915322047004666939128e-1 / _EXP_A0)
_EXP_PRESCALE = F(1.4426950408889634073599246810019 * 64)
_EXP_POSTSCALE = F(1.0 / 64)
_EXP_MIN = F(-3000.0 * 64 / (1.4426950408889634073599246810019 * 64))
_EXP_MAX = F(3000.0 * 64 / (1.4426950408889634073599246810019 * 64))
EXP_TABLE = np.array([2.0 ** (j / 64.0) * _EXP_A0 for j in range(64)], dtype=np.float32)

# cv::fastAtan2 (core/src/mathfuncs_core.simd.hpp): degrees
_R2D = F(180 / math.pi)
ATAN_P1 = F(F(0.9997878412794807) * _R2D)
ATAN_P3 = F(F(-0.3258083974640975) * _R2D)
ATAN_P5 = F(F(0.1555786518463281) * _R2D)
ATAN_P7 = F(F(-0.04432655554792128) * _R2D)
ATAN_EPS = F(np.finfo(np.float64).eps)


def _fma(a, b, c):
    """float32 a * b + c with one rounding (the product is exact in float64)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(np.float32)


def exp32f(x):
    """cv::hal::exp32f of a float32 array as OpenCV's own (non-IPP) code computes it: the 64-entry 2^(j/64) table and a
    degree-4 polynomial, every operation rounded (the baseline SIMD path has no fused multiply-add)."""
    x = np.minimum(np.maximum(np.asarray(x, np.float32), _EXP_MIN), _EXP_MAX) * _EXP_PRESCALE
    xi = np.rint(x).astype(np.int32)
    xf = (x - xi.astype(np.float32)) * _EXP_POSTSCALE
    e = np.clip((xi >> 6) + 127, 0, 255).astype(np.int32)
    yf = EXP_TABLE[xi & 63] * (e << 23).view(np.float32)
    z = (((xf + _EXP_A1) * xf + _EXP_A2) * xf + _EXP_A3) * xf + _EXP_A4
    return z * yf


def fast_atan2(y, x):
    """cv::fastAtan2 in degrees [0, 360) of float32 arrays, as its SIMD loop computes it."""
    y = np.asarray(y, np.float32)
    x = np.asarray(x, np.float32)
    ax, ay = np.abs(x), np.abs(y)
    c = np.minimum(ax, ay) / (np.maximum(ax, ay) + ATAN_EPS)
    cc = c * c
    a = _fma(_fma(_fma(cc, ATAN_P7, ATAN_P5), cc, ATAN_P3), cc, ATAN_P1) * c
    a = np.where(ax >= ay, a, F(90) - a)
    a = np.where(x < 0, F(180) - a, a)
    return np.where(y < 0, F(360) - a, a)


def magnitude(x, y):
    """cv::hal::magnitude32f as OpenCV's own (non-IPP) code computes it: sqrt(x * x + y * y), every operation rounded."""
    x = np.asarray(x, np.float32)
    y = np.asarray(y, np.float32)
    return np.sqrt(x * x + y * y)


def grey(image):
    """The 8-bit grey image SIFT starts from: cvtColor(BGR2GRAY) for colour (fixed point, weights 3735 / 19235 / 9798,
    >> 15 with rounding), grey and (H, W, 1) as they are."""
    a = np.asarray(image)
    if a.dtype != np.uint8 or not (a.ndim == 2 or (a.ndim == 3 and a.shape[2] in (1, 3))):
        raise ValueError('need a uint8 (H, W), (H, W, 1) or (H, W, 3) image')
    if a.ndim == 3 and a.shape[2] == 3:
        b, g, r = (a[..., k].astype(np.int32) for k in range(3))
        return ((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15).astype(np.uint8)
    return a.reshape(a.shape[0], a.shape[1])


def upsample2_f32(img):
    """cv2.resize(float image, x2, INTER_LINEAR): destination 2k reads 0.25 s[k - 1] + 0.75 s[k], 2k + 1 reads
    0.75 s[k] + 0.25 s[k + 1], indices clamped.  Exact for 8-bit data (multiples of 1/16)."""
    x = np.asarray(img, np.float32)

    def axis(n):
        i = np.arange(2 * n)
        return np.clip(np.where(i % 2 == 0, i // 2 - 1, i // 2 + 1), 0, n - 1), i // 2
    a, b = axis(x.shape[1])
    row = F(0.25) * x[:, a] + F(0.75) * x[:, b]
    a, b = axis(x.shape[0])
    return F(0.25) * row[a] + F(0.75) * row[b]


def gaussian_kernel_f32(sigma):
    """getGaussianKernel(cvRound(8 sigma + 1) | 1, sigma, CV_32F): the bit-exact double kernel, rounded to float32."""
    n = int(np.rint(sigma * 8 + 1)) | 1
    n2 = n // 2
    vals = [math.exp((x * x) * (-0.125 / (sigma * sigma))) for x in range(1 - n, 0, 2)]
    mul = 1.0 / (2 * sum(vals) + 1.0)
    k = np.empty(n, dtype=np.float32)
    for i in range(n2):
        k[i] = k[n - 1 - i] = F(vals[i] * mul)
    k[n2] = F(mul)
    return k


def _blur_axis(x, k):
    """Symmetric 1-D filter along axis 1 under BORDER_REFLECT_101: k[r] x[0] + sum_j k[r + j] (x[-j] + x[j]), j = 1..r
    in order, every operation rounded to float32."""
    r = len(k) // 2
    w = x.shape[1]
    xi = x[:, reflect101(w, r)]
    acc = k[r] * xi[:, r:r + w]
    for j in range(1, r + 1):
        acc = acc + k[r + j] * (xi[:, r - j:r - j + w] + xi[:, r + j:r + j + w])
    return acc


def blur_f32(img, sigma):
    """cv2.GaussianBlur(float32 img, (0, 0), sigma): the row pass, then the column pass."""
    k = gaussian_kernel_f32(sigma)
    return np.ascontiguousarray(_blur_axis(_blur_axis(np.asarray(img, np.float32), k).T, k).T)


def init_sigma():
    """sqrtf(max(1.6f^2 - 4 * 0.5f^2, 0.01f)): the blur that takes the doubled image to sigma 1.6."""
    s = F(SIGMA)
    return float(np.sqrt(max(F(s * s) - F(F(0.5) * F(0.5)) * F(4), F(0.01))))


def octave_sigmas():
    """The incremental sigmas of level 1 .. 5 of an octave, in double as buildGaussianPyramid computes them."""
    k = 2.0 ** (1.0 / LAYERS)
    out = []
    for i in range(1, PER_OCTAVE):
        prev = k ** (i - 1) * SIGMA
        total = prev * k
        out.append(math.sqrt(total * total - prev * prev))
    return out


def level_shape(h, w, o):
    """(rows, cols) of octave o: the doubled image, halved (rounding down) once per octave."""
    return (2 * h) >> o, (2 * w) >> o


def scale_space(image):
    """(gauss, dog): per octave the 6 float32 Gaussian levels and the 5 differences of neighbouring levels.  The octave
    count is frontend.gaussian_pyramid's, since keypoints index that pyramid."""
    g = grey(image)
    h, w = g.shape
    base = blur_f32(upsample2_f32(g.astype(np.float32)), init_sigma())
    sig = octave_sigmas()
    gauss = []
    for o in range(n_octaves(h, w)):
        if o == 0:
            lv = [base]
        else:
            rows, cols = level_shape(h, w, o)
            lv = [np.ascontiguousarray(gauss[o - 1][LAYERS][::2, ::2][:rows, :cols])]
        for i in range(1, PER_OCTAVE):
            lv.append(blur_f32(lv[-1], sig[i - 1]))
        gauss.append(lv)
    dog = [[lv[i + 1] - lv[i] for i in range(DOG_PER_OCTAVE)] for lv in gauss]
    return gauss, dog


def _flat(levels):
    """All levels in one float32 vector, with per-level offsets."""
    offs = np.cumsum([0] + [l.size for l in levels[:-1]]).astype(np.int64)
    return np.concatenate([l.ravel() for l in levels]), offs


def candidates(dog):
    """(o, layer, r, c) int64 arrays of every scale-space extremum: a nonzero DoG value of layer 1..3 at least 5 px from
    the border that is >= all 26 neighbours (positive) or <= all of them (negative)."""
    out = []
    for o, d in enumerate(dog):
        rows, cols = d[0].shape
        if rows <= 2 * BORDER or cols <= 2 * BORDER:
            continue
        for i in range(1, LAYERS + 1):
            v = d[i][BORDER:rows - BORDER, BORDER:cols - BORDER]
            is_max = v > 0
            is_min = v < 0
            for dl in (-1, 0, 1):
                for dr in (-1, 0, 1):
                    for dc in (-1, 0, 1):
                        if dl == 0 and dr == 0 and dc == 0:
                            continue
                        n = d[i + dl][BORDER + dr:rows - BORDER + dr, BORDER + dc:cols - BORDER + dc]
                        is_max &= v >= n
                        is_min &= v <= n
            r, c = np.nonzero(is_max | is_min)
            k = len(r)
            out.append((np.full(k, o), np.full(k, i), r + BORDER, c + BORDER))
    if not out:
        e = np.zeros(0, dtype=np.int64)
        return e, e, e, e
    return tuple(np.concatenate([x[j] for x in out]).astype(np.int64) for j in range(4))


def lu_solve3(A, b):
    """hal::LU32f on a stack of 3 x 3 systems (partial pivoting, eps = 10 FLT_EPSILON): x with A x = b, or 0 where a
    pivot is below eps (Matx::solve returns zeros then)."""
    A = A.astype(np.float32).copy()
    b = b.astype(np.float32).copy()
    n = len(A)
    rows = np.arange(n)
    singular = np.zeros(n, dtype=bool)
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        for i in range(3):
            k = np.full(n, i)
            for j in range(i + 1, 3):
                k = np.where(np.abs(A[:, j, i]) > np.abs(A[rows, k, i]), j, k)
            singular |= np.abs(A[rows, k, i]) < LU_EPS
            ai, ak = A[rows, i].copy(), A[rows, k].copy()
            A[rows, i], A[rows, k] = ak, ai
            bi, bk = b[rows, i].copy(), b[rows, k].copy()
            b[rows, i], b[rows, k] = bk, bi
            d = F(-1) / A[:, i, i]
            for j in range(i + 1, 3):
                alpha = A[:, j, i] * d
                for kk in range(i + 1, 3):
                    A[:, j, kk] = A[:, j, kk] + alpha * A[:, i, kk]
                b[:, j] = b[:, j] + alpha * b[:, i]
        for i in (2, 1, 0):
            s = b[:, i].copy()
            for kk in range(i + 1, 3):
                s = s - A[:, i, kk] * b[:, kk]
            b[:, i] = s / A[:, i, i]
    b[singular] = 0
    return b


def refine(dog, o, layer, r, c):
    """adjustLocalExtrema for every candidate.  Returns (keep mask, o, layer, r, c, xc, xr, xi, contrast) — the
    position after the interpolation steps, the sub-pixel offsets and the interpolated DoG value."""
    flat, offs = _flat([l for d in dog for l in d])
    widths = np.array([d[0].shape[1] for d in dog], dtype=np.int64)
    heights = np.array([d[0].shape[0] for d in dog], dtype=np.int64)
    n = len(o)
    layer, r, c = layer.copy(), r.copy(), c.copy()
    xi = np.zeros(n, np.float32)
    xr = np.zeros(n, np.float32)
    xc = np.zeros(n, np.float32)
    live = np.ones(n, dtype=bool)        # still iterating
    done = np.zeros(n, dtype=bool)       # converged
    W = widths[o]

    def at(idx, dl, dr, dc):
        ii = idx
        return flat[offs[o[ii] * DOG_PER_OCTAVE + layer[ii] + dl] + (r[ii] + dr) * W[ii] + c[ii] + dc]

    def derivs(ii):
        v = at(ii, 0, 0, 0)
        g = np.stack([(at(ii, 0, 0, 1) - at(ii, 0, 0, -1)) * DERIV_SCALE,
                      (at(ii, 0, 1, 0) - at(ii, 0, -1, 0)) * DERIV_SCALE,
                      (at(ii, 1, 0, 0) - at(ii, -1, 0, 0)) * DERIV_SCALE], axis=1)
        v2 = v * F(2)
        dxx = (at(ii, 0, 0, 1) + at(ii, 0, 0, -1) - v2) * IMG_SCALE
        dyy = (at(ii, 0, 1, 0) + at(ii, 0, -1, 0) - v2) * IMG_SCALE
        dss = (at(ii, 1, 0, 0) + at(ii, -1, 0, 0) - v2) * IMG_SCALE
        dxy = (at(ii, 0, 1, 1) - at(ii, 0, 1, -1) - at(ii, 0, -1, 1) + at(ii, 0, -1, -1)) * CROSS_SCALE
        dxs = (at(ii, 1, 0, 1) - at(ii, 1, 0, -1) - at(ii, -1, 0, 1) + at(ii, -1, 0, -1)) * CROSS_SCALE
        dys = (at(ii, 1, 1, 0) - at(ii, 1, -1, 0) - at(ii, -1, 1, 0) + at(ii, -1, -1, 0)) * CROSS_SCALE
        return v, g, dxx, dyy, dss, dxy, dxs, dys

    big = F(2147483647 // 3)
    for _ in range(MAX_STEPS):
        ii = np.nonzero(live)[0]
        if len(ii) == 0:
            break
        _, g, dxx, dyy, dss, dxy, dxs, dys = derivs(ii)
        H = np.stack([np.stack([dxx, dxy, dxs], 1), np.stack([dxy, dyy, dys], 1), np.stack([dxs, dys, dss], 1)], 1)
        X = lu_solve3(H, g)
        xi[ii], xr[ii], xc[ii] = -X[:, 2], -X[:, 1], -X[:, 0]
        conv = (np.abs(xi[ii]) < F(0.5)) & (np.abs(xr[ii]) < F(0.5)) & (np.abs(xc[ii]) < F(0.5))
        done[ii[conv]] = True
        live[ii[conv]] = False
        mv = ii[~conv]
        with np.errstate(invalid='ignore'):
            huge = (np.abs(xi[mv]) > big) | (np.abs(xr[mv]) > big) | (np.abs(xc[mv]) > big) | \
                ~np.isfinite(xi[mv]) | ~np.isfinite(xr[mv]) | ~np.isfinite(xc[mv])
        live[mv[huge]] = False
        mv = mv[~huge]
        c[mv] += np.rint(xc[mv]).astype(np.int64)
        r[mv] += np.rint(xr[mv]).astype(np.int64)
        layer[mv] += np.rint(xi[mv]).astype(np.int64)
        out = (layer[mv] < 1) | (layer[mv] > LAYERS) | (c[mv] < BORDER) | (c[mv] >= W[mv] - BORDER) | \
            (r[mv] < BORDER) | (r[mv] >= heights[o[mv]] - BORDER)
        live[mv[out]] = False
    keep = done.copy()
    contr = np.zeros(n, np.float32)
    ii = np.nonzero(keep)[0]
    if len(ii):
        v, g, dxx, dyy, _, dxy, _, _ = derivs(ii)
        t = g[:, 0] * xc[ii]
        t = t + g[:, 1] * xr[ii]
        t = t + g[:, 2] * xi[ii]
        cv = v * IMG_SCALE + t * F(0.5)
        contr[ii] = cv
        ok = ~(np.abs(cv) * F(LAYERS) < CONTRAST)
        tr = dxx + dyy
        det = dxx * dyy - dxy * dxy
        ok &= ~((det <= 0) | (tr * tr * EDGE >= F((EDGE + F(1)) * (EDGE + F(1))) * det))
        keep[ii[~ok]] = False
    return keep, o, layer, r, c, xc, xr, xi, contr


def keypoint_fields(o, layer, r, c, xc, xr, xi, contr):
    """The cv2.KeyPoint fields at the doubled-image scale: x, y, size, response float32 and the packed octave."""
    s = (np.int64(1) << o).astype(np.float32)
    x = (c.astype(np.float32) + xc) * s
    y = (r.astype(np.float32) + xr) * s
    p = np.exp2(((layer.astype(np.float32) + xi) / F(LAYERS)).astype(np.float64)).astype(np.float32)
    size = F(SIGMA) * p * s * F(2)
    octv = o + (layer << 8) + (np.rint((xi.astype(np.float64) + 0.5) * 255).astype(np.int64) << 16)
    return x, y, size, np.abs(contr), octv.astype(np.int64)


def smooth_hist(t):
    """The [1 4 6 4 1] / 16 circular smoothing of calcOrientationHist: bins 0..31 as its SIMD loop (fused), 32..35 as its
    scalar tail.  `t`: (N, 36) float32."""
    n = t.shape[1]
    tn2, tn1 = np.roll(t, 2, axis=1), np.roll(t, 1, axis=1)
    tp1, tp2 = np.roll(t, -1, axis=1), np.roll(t, -2, axis=1)
    a, b = tn2 + tp2, tn1 + tp1
    fused = _fma(a, F(1 / 16), _fma(b, F(4 / 16), t * F(6 / 16)))
    plain = a * F(1 / 16) + b * F(4 / 16) + t * F(6 / 16)
    return np.where(np.arange(n) < 32, fused, plain)


def orientation_hists(gauss, o, layer, r, c, size):
    """calcOrientationHist at each refined keypoint: the 36-bin smoothed histogram of gradient orientations on Gaussian
    level (o, layer) around (r, c), radius cvRound(4.5 scl), Gaussian weight of sigma 1.5 scl, scl = size / 2 / 2^o.
    Each bin sums its pixels in row-major window order.  Returns (N, 36) float32."""
    flat, offs = _flat([l for lv in gauss for l in lv])
    widths = np.array([lv[0].shape[1] for lv in gauss], dtype=np.int64)
    heights = np.array([lv[0].shape[0] for lv in gauss], dtype=np.int64)
    n = len(o)
    scl = (size * F(0.5)) / (np.int64(1) << o).astype(np.float32)
    radius = np.rint(F(4.5) * scl).astype(np.int64)
    sw = F(1.5) * scl
    escale = F(-1) / (F(2) * sw * sw)
    hist = np.zeros((n, N_BINS), np.float32)
    base = offs[o * PER_OCTAVE + layer]
    W, Hh = widths[o], heights[o]
    for R in np.unique(radius):
        ii = np.nonzero(radius == R)[0]
        m = len(ii)
        rows = np.arange(m)
        h = np.zeros((m, N_BINS), np.float32)
        for di in range(-R, R + 1):
            y = r[ii] + di
            oky = (y > 0) & (y < Hh[ii] - 1)
            for dj in range(-R, R + 1):
                x = c[ii] + dj
                ok = oky & (x > 0) & (x < W[ii] - 1)
                yy, xx = np.where(ok, y, 1), np.where(ok, x, 1)
                p = base[ii] + yy * W[ii] + xx
                dx = flat[p + 1] - flat[p - 1]
                dy = flat[p - W[ii]] - flat[p + W[ii]]
                wt = exp32f(F(di * di + dj * dj) * escale[ii])
                ori = fast_atan2(dy, dx)
                mag = magnitude(dx, dy)
                b = np.rint(F(N_BINS / 360.0) * ori).astype(np.int64)
                b = np.where(b >= N_BINS, b - N_BINS, b)
                b = np.where(b < 0, b + N_BINS, b)
                h[rows[ok], b[ok]] = h[rows[ok], b[ok]] + wt[ok] * mag[ok]
        hist[ii] = h
    return smooth_hist(hist)


def peaks(hist):
    """Orientation peaks: every bin above both neighbours and >= 0.8 of the maximum, refined by a parabola.  Returns
    (keypoint index, angle) with angle = 360 - 10 bin (0 within FLT_EPSILON of 360), in keypoint then bin order."""
    omax = hist.max(axis=1)
    thr = omax * F(0.8)
    hl, hr = np.roll(hist, 1, axis=1), np.roll(hist, -1, axis=1)
    is_peak = (hist > hl) & (hist > hr) & (hist >= thr[:, None])
    k, j = np.nonzero(is_peak)
    a, b, m = hl[k, j], hr[k, j], hist[k, j]
    with np.errstate(divide='ignore', invalid='ignore'):
        bn = j.astype(np.float32) + F(0.5) * (a - b) / (a - F(2) * m + b)
    bn = np.where(bn < 0, F(N_BINS) + bn, np.where(bn >= F(N_BINS), bn - F(N_BINS), bn))
    ang = F(360) - F(360.0 / N_BINS) * bn
    ang = np.where(np.abs(ang - F(360)) < FLT_EPSILON, F(0), ang)
    return k, ang.astype(np.float32)


def detect(image, max_keypoints=-1):
    """SIFT keypoints of one uint8 image, as records (pt, size, angle, response, octave) in cv2's order: sorted by
    (x, y, -size, angle, -response, -octave) with duplicates of (pt, size, angle) removed; with 0 < max_keypoints < N
    the strongest `max_keypoints` by response, ties in the sorted order."""
    gauss, dog = scale_space(image)
    keep, o, layer, r, c, xc, xr, xi, contr = refine(dog, *candidates(dog))
    ii = np.nonzero(keep)[0]
    o, layer, r, c, xc, xr, xi, contr = (a[ii] for a in (o, layer, r, c, xc, xr, xi, contr))
    x, y, size, resp, octv = keypoint_fields(o, layer, r, c, xc, xr, xi, contr)
    k, ang = peaks(orientation_hists(gauss, o, layer, r, c, size))
    x, y, size, resp, octv = x[k], y[k], size[k], resp[k], octv[k]
    order = np.lexsort((-octv, -resp, ang, -size, y, x))
    x, y, size, ang, resp, octv = (a[order] for a in (x, y, size, ang, resp, octv))
    dup = np.zeros(len(x), dtype=bool)
    dup[1:] = (x[1:] == x[:-1]) & (y[1:] == y[:-1]) & (size[1:] == size[:-1]) & (ang[1:] == ang[:-1])
    x, y, size, ang, resp, octv = (a[~dup] for a in (x, y, size, ang, resp, octv))
    octv = (octv & ~255) | ((octv - 1) & 255)
    rec = {'pt': np.stack([x * F(0.5), y * F(0.5)], axis=1).astype(np.float32).reshape(-1, 2),
           'size': (size * F(0.5)).astype(np.float32), 'angle': ang.astype(np.float32),
           'response': resp.astype(np.float32), 'octave': octv.astype(np.int32)}
    if 0 < max_keypoints < len(x):
        top = np.argsort(-rec['response'], kind='stable')[:max_keypoints]
        rec = {k2: v[top] for k2, v in rec.items()}
    return rec

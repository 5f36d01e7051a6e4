"""numpy restatement of the RANSAC homography estimator of gims_b200/csrc/homography.cu.

It replaces the `cv2.findHomography(src, dst, cv2.RANSAC, thresh)` call of eval_homography.py and eval_matches.py.  cv2's
estimator cannot be restated bit for bit at a reasonable cost (its solvers go through a Jacobi eigen-decomposition), so
this module fixes one deterministic algorithm that follows cv2's classic RANSACPointSetRegistrator + findHomography step
for step.  The device equals it bit for bit; the tests hold it to cv2 by outcome.  It differs from cv2 in three places:
  - samples come from a counter-based RNG (splitmix64 of the seed, the hypothesis, the attempt, the slot and the retry),
    so that hypotheses can be drawn in parallel; a pair's result does not depend on its position in a batch;
  - the iteration bound N(g) is the least k >= 1 with q^k <= 1 - confidence, q^k by sequential multiplication, instead of
    cvRound(log(1 - c) / log(q)): at most one iteration more than cv2, and no `log`, whose last bit differs between libms;
  - the minimal solver, the refit and the Levenberg-Marquardt steps solve their 8x8 normal equations by Gaussian
    elimination with partial pivoting instead of an eigen-decomposition.
Every sum over points is 256 strided partials (partial p takes points p, p+256, ... in order, starting from +0.0),
combined by a halving tree (p += p+128, then +64, ..., +1).  Every product and sum is spelled out element-wise: no
np.dot / @ / np.sum on floating-point data, whose order of operations and use of FMA are unspecified.
"""
import numpy as np

MAX_ATTEMPTS = 1000       # sampling attempts per hypothesis
MAX_RETRIES = 64          # draws per sample slot until an index differs from the ones already drawn
WAVE = 256                # hypotheses evaluated together; the result does not depend on it
LM_ITERS = 10
REFIT_ROUNDS = 3
PIVOT_EPS = 1e-12
DBL_EPSILON = np.finfo(np.float64).eps
FLT_EPSILON = float(np.finfo(np.float32).eps)
_U64 = np.uint64


def splitmix64(x):
    """splitmix64 mix of (x + golden gamma), uint64 with wrap-around; x is a uint64 array or scalar."""
    x = np.asarray(x, dtype=_U64)
    with np.errstate(over='ignore'):
        z = x + _U64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> _U64(27))) * _U64(0x94D049BB133111EB)
    return z ^ (z >> _U64(31))


def fixed_sum(t):
    """Sum over the last axis in the fixed order: 256 strided partials from +0.0, then the halving tree."""
    t = np.asarray(t, dtype=np.float64)
    n = t.shape[-1]
    rows = max(1, -(-n // 256))
    pad = np.zeros(t.shape[:-1] + (rows * 256,), dtype=np.float64)
    pad[..., :n] = t
    pad = pad.reshape(t.shape[:-1] + (rows, 256))
    part = np.zeros(t.shape[:-1] + (256,), dtype=np.float64)
    for r in range(rows):
        part = part + pad[..., r, :]
    s = 128
    while s:
        part = part[..., :s] + part[..., s:2 * s]
        s >>= 1
    return part[..., 0]


def n_iters_bound(good, m, confidence, max_iters):
    """N(g): the least k >= 1 with q^k <= 1 - confidence, q = 1 - (g/m)^4, capped at max_iters."""
    w = float(good) / float(m)
    q = 1.0 - ((w * w) * w) * w
    lim = 1.0 - confidence
    k, prod = 1, q
    while not (prod <= lim) and k < max_iters:
        prod = prod * q
        k += 1
    return k


def _solve8(A, b):
    """Gaussian elimination with partial pivoting on (B, 8, 8) x = (B, 8), fp64.  The pivot is the first maximal |a|
    (ties to the lowest row); a pivot <= 1e-12 * max|diag A| is a failure.  Returns (x, ok)."""
    A = np.array(A, dtype=np.float64)
    b = np.array(b, dtype=np.float64)
    B = A.shape[0]
    ar = np.arange(B)
    dmax = np.zeros(B)
    for i in range(8):
        d = np.abs(A[:, i, i])
        dmax = np.where(d > dmax, d, dmax)
    thr = PIVOT_EPS * dmax
    ok = np.ones(B, dtype=bool)
    for k in range(8):
        r = np.full(B, k)
        best = np.abs(A[:, k, k])
        for i in range(k + 1, 8):
            v = np.abs(A[:, i, k])
            better = v > best
            r = np.where(better, i, r)
            best = np.where(better, v, best)
        ok &= best > thr
        rowk, rowr = A[ar, k].copy(), A[ar, r].copy()
        A[ar, r], A[ar, k] = rowk, rowr
        bk, br = b[ar, k].copy(), b[ar, r].copy()
        b[ar, r], b[ar, k] = bk, br
        with np.errstate(all='ignore'):
            for i in range(k + 1, 8):
                f = A[:, i, k] / A[:, k, k]
                for j in range(k + 1, 8):
                    A[:, i, j] = A[:, i, j] - f * A[:, k, j]
                b[:, i] = b[:, i] - f * b[:, k]
    x = np.zeros((B, 8))
    with np.errstate(all='ignore'):
        for i in range(7, -1, -1):
            s = b[:, i]
            for j in range(i + 1, 8):
                s = s - A[:, i, j] * x[:, j]
            x[:, i] = s / A[:, i, i]
    return x, ok


def _mat3(a, b):
    """(B, 9) x (B, 9) row-major 3x3 products, each entry (a0 b0 + a1 b1) + a2 b2."""
    c = np.empty_like(a)
    for i in range(3):
        for j in range(3):
            c[:, 3 * i + j] = (a[:, 3 * i] * b[:, j] + a[:, 3 * i + 1] * b[:, 3 + j]) + a[:, 3 * i + 2] * b[:, 6 + j]
    return c


def dlt(xs, ys, xd, yd):
    """Normalised DLT with h33 = 1 for B point sets: xs, ys, xd, yd are (B, n) float32.  Returns (H (B, 9) fp64 with
    H[8] = 1, ok (B,)).  Normalisation as cv2's HomographyEstimatorCallback::runKernel: centroid, then per axis
    n / sum|x - c|; a sum below DBL_EPSILON is a failure.  A non-finite H is a failure."""
    xs, ys, xd, yd = (np.asarray(v, dtype=np.float32).astype(np.float64) for v in (xs, ys, xd, yd))
    n = float(xs.shape[-1])
    with np.errstate(all='ignore'):
        cxs, cys, cxd, cyd = (fixed_sum(v) / n for v in (xs, ys, xd, yd))
        sums = [fixed_sum(np.abs(v - c[:, None])) for v, c in ((xs, cxs), (ys, cys), (xd, cxd), (yd, cyd))]
        ok = np.ones(xs.shape[0], dtype=bool)
        for s in sums:
            ok &= ~(np.abs(s) < DBL_EPSILON)
        sxs, sys_, sxd, syd = (n / s for s in sums)
        X = (xs - cxs[:, None]) * sxs[:, None]
        Y = (ys - cys[:, None]) * sys_[:, None]
        u = (xd - cxd[:, None]) * sxd[:, None]
        v = (yd - cyd[:, None]) * syd[:, None]
        zero, one = np.zeros_like(X), np.ones_like(X)
        r1 = [X, Y, one, zero, zero, zero, -(u * X), -(u * Y)]
        r2 = [zero, zero, zero, X, Y, one, -(v * X), -(v * Y)]
        A = np.zeros((xs.shape[0], 8, 8))
        b = np.zeros((xs.shape[0], 8))
        for a in range(8):
            for c in range(a, 8):
                A[:, a, c] = A[:, c, a] = fixed_sum(r1[a] * r1[c] + r2[a] * r2[c])
            b[:, a] = fixed_sum(r1[a] * u + r2[a] * v)
        h, ok2 = _solve8(A, b)
        ok &= ok2
        B = xs.shape[0]
        hn = np.concatenate([h, np.ones((B, 1))], axis=1)
        inv_dst = np.zeros((B, 9))
        inv_dst[:, 0], inv_dst[:, 2], inv_dst[:, 4], inv_dst[:, 5], inv_dst[:, 8] = 1.0 / sxd, cxd, 1.0 / syd, cyd, 1.0
        nrm_src = np.zeros((B, 9))
        nrm_src[:, 0], nrm_src[:, 2] = sxs, -(cxs * sxs)
        nrm_src[:, 4], nrm_src[:, 5], nrm_src[:, 8] = sys_, -(cys * sys_), 1.0
        T = _mat3(_mat3(inv_dst, hn), nrm_src)
        H = T / T[:, 8:9]
    ok &= np.isfinite(H).all(axis=1)
    return H, ok


def reproj_err(Hf, x, y, xd, yd):
    """cv2's HomographyEstimatorCallback::computeError in fp32: Hf (B, 8) float32, points (n,) float32 -> (B, n)."""
    h = [Hf[:, j:j + 1] for j in range(8)]
    one = np.float32(1.0)
    with np.errstate(all='ignore'):
        ww = one / ((h[6] * x + h[7] * y) + one)
        dx = ((h[0] * x + h[1] * y) + h[2]) * ww - xd
        dy = ((h[3] * x + h[4] * y) + h[5]) * ww - yd
        return dx * dx + dy * dy


def _collinear(px, py, a, b, c):
    """cv2's haveCollinearPoints test for the triple (a, b, c) with c as its last point: fp32 differences, fp64 rest."""
    dx1 = (px[:, b] - px[:, c]).astype(np.float64)
    dy1 = (py[:, b] - py[:, c]).astype(np.float64)
    dx2 = (px[:, a] - px[:, c]).astype(np.float64)
    dy2 = (py[:, a] - py[:, c]).astype(np.float64)
    with np.errstate(all='ignore'):
        lhs = np.abs(dx2 * dy1 - dy2 * dx1)
        rhs = FLT_EPSILON * (((np.abs(dx1) + np.abs(dy1)) + np.abs(dx2)) + np.abs(dy2))
    return lhs <= rhs


def _det3(px, py, t):
    x0, x1, x2 = (px[:, i].astype(np.float64) for i in t)
    y0, y1, y2 = (py[:, i].astype(np.float64) for i in t)
    with np.errstate(all='ignore'):
        return (x0 * (y1 - y2) - y0 * (x1 - x2)) + (x1 * y2 - x2 * y1)


def subset_ok(sx, sy, dx, dy):
    """checkSubset for (B, 4) samples: no three source or three destination points collinear (every triple, tested as
    cv2's haveCollinearPoints does), and the orientation of the four triangles agrees (0 or 4 negative det * det)."""
    bad = np.zeros(sx.shape[0], dtype=bool)
    for a, b, c in ((0, 1, 2), (0, 1, 3), (0, 2, 3), (1, 2, 3)):
        bad |= _collinear(sx, sy, a, b, c) | _collinear(dx, dy, a, b, c)
    neg = np.zeros(sx.shape[0], dtype=np.int64)
    for t in ((0, 1, 2), (1, 2, 3), (0, 2, 3), (0, 1, 3)):
        neg += (_det3(sx, sy, t) * _det3(dx, dy, t)) < 0
    return ~bad & ((neg == 0) | (neg == 4))


def draw_samples(seed, hyps, m, src, dst):
    """Samples of hypotheses `hyps` (int array): (idx (B, 4) int64, found (B,) bool)."""
    base = splitmix64(_U64(seed))
    hyps = np.asarray(hyps, dtype=np.int64)
    B = len(hyps)
    idx = np.zeros((B, 4), dtype=np.int64)
    found = np.zeros(B, dtype=bool)
    todo = np.arange(B)
    r = np.arange(MAX_RETRIES, dtype=_U64)
    mm = _U64(m)
    for a in range(MAX_ATTEMPTS):
        if len(todo) == 0:
            break
        att = hyps[todo].astype(_U64) * _U64(MAX_ATTEMPTS) + _U64(a)
        cur = np.zeros((len(todo), 4), dtype=np.int64)
        drew = np.ones(len(todo), dtype=bool)
        with np.errstate(over='ignore'):
            for k in range(4):
                key = ((att * _U64(4) + _U64(k)) * _U64(MAX_RETRIES))[:, None] + r[None, :]
                cand = (splitmix64(base + key) % mm).astype(np.int64)       # (T, 64)
                fresh = np.ones(cand.shape, dtype=bool)
                for j in range(k):
                    fresh &= cand != cur[:, j:j + 1]
                first = np.argmax(fresh, axis=1)
                drew &= fresh.any(axis=1)
                cur[:, k] = cand[np.arange(len(todo)), first]
        okk = drew.copy()
        if okk.any():
            sel = np.nonzero(okk)[0]
            c = cur[sel]
            okk[sel] = subset_ok(src[c, 0], src[c, 1], dst[c, 0], dst[c, 1])
        idx[todo[okk]] = cur[okk]
        found[todo[okk]] = True
        todo = todo[~okk]
    return idx, found


def _lm_terms(h, x, y, xd, yd):
    """Residuals and Jacobian rows of HomographyRefineCallback::compute (fp64) at the 8 parameters h."""
    X, Y = x.astype(np.float64), y.astype(np.float64)
    with np.errstate(all='ignore'):
        d = (h[6] * X + h[7] * Y) + 1.0
        ww = np.where(np.abs(d) > DBL_EPSILON, 1.0 / d, 0.0)
        xi = ((h[0] * X + h[1] * Y) + h[2]) * ww
        yi = ((h[3] * X + h[4] * Y) + h[5]) * ww
        ex = xi - xd.astype(np.float64)
        ey = yi - yd.astype(np.float64)
        zero = np.zeros_like(X)
        jx = [X * ww, Y * ww, ww, zero, zero, zero, -((X * ww) * xi), -((Y * ww) * xi)]
        jy = [zero, zero, zero, X * ww, Y * ww, ww, -((X * ww) * yi), -((Y * ww) * yi)]
    return ex, ey, jx, jy


def _lm_cost(h, x, y, xd, yd):
    ex, ey, _, _ = _lm_terms(h, x, y, xd, yd)
    with np.errstate(all='ignore'):
        return fixed_sum(ex * ex + ey * ey)


def _lm_normal(h, x, y, xd, yd):
    ex, ey, jx, jy = _lm_terms(h, x, y, xd, yd)
    A = np.zeros((8, 8))
    g = np.zeros(8)
    with np.errstate(all='ignore'):
        for a in range(8):
            for c in range(a, 8):
                A[a, c] = A[c, a] = fixed_sum(jx[a] * jx[c] + jy[a] * jy[c])
            g[a] = fixed_sum(jx[a] * ex + jy[a] * ey)
        cost = fixed_sum(ex * ex + ey * ey)
    return A, g, cost


def refine(H0, x, y, xd, yd):
    """LMSolver's schedule with maxIters 10 on the 8 parameters of H0 (h33 = 1): lambda from 1e-3, a step that lowers the
    cost is taken and lambda /= 10, otherwise lambda *= 10; each step solves (JtJ + lambda diag(JtJ)) d = -Jt r."""
    h = np.array(H0[:8], dtype=np.float64)
    A, g, cost = _lm_normal(h, x, y, xd, yd)
    lam = 1e-3
    for _ in range(LM_ITERS):
        Mx = A.copy()
        for j in range(8):
            Mx[j, j] = A[j, j] + lam * A[j, j]
        d, ok = _solve8(Mx[None], (-g)[None])
        if not ok[0]:
            lam = lam * 10.0
            continue
        with np.errstate(all='ignore'):
            hn = h + d[0]
        cn = _lm_cost(hn, x, y, xd, yd)
        if cn < cost:
            h = hn
            lam = lam / 10.0
            A, g, cost = _lm_normal(h, x, y, xd, yd)
        else:
            lam = lam * 10.0
    return np.concatenate([h, [1.0]])


def find_homography(src, dst, thresh=3.0, max_iters=2000, confidence=0.995, seed=0, wave=WAVE):
    """One pair.  src, dst: (M, 2) float32.  Returns (H (9,) fp64 or None, mask (M,) uint8, n_inliers, n_iters)."""
    src = np.ascontiguousarray(src, dtype=np.float32).reshape(-1, 2)
    dst = np.ascontiguousarray(dst, dtype=np.float32).reshape(-1, 2)
    m = src.shape[0]
    mask = np.zeros(m, dtype=np.uint8)
    if m < 4:
        return None, mask, 0, 0
    if m == 4:
        H, ok = dlt(src[None, :, 0], src[None, :, 1], dst[None, :, 0], dst[None, :, 1])
        if not ok[0]:
            return None, mask, 0, 0
        return H[0], np.ones(m, dtype=np.uint8), 4, 0
    thr2 = np.float32(float(thresh) * float(thresh))
    x, y, xd, yd = src[:, 0], src[:, 1], dst[:, 0], dst[:, 1]
    niters, best, best_h, i = int(max_iters), 0, None, 0
    stop = False
    while i < niters and not stop:
        hyps = np.arange(i, min(i + wave, niters))
        idx, found = draw_samples(seed, hyps, m, src, dst)
        H, ok = dlt(x[idx], y[idx], xd[idx], yd[idx])
        ok &= found
        counts = np.zeros(len(hyps), dtype=np.int64)
        if ok.any():
            sel = np.nonzero(ok)[0]
            err = reproj_err(H[sel, :8].astype(np.float32), x, y, xd, yd)
            counts[sel] = (err <= thr2).sum(axis=1)                 # integer counts
        for w, hi in enumerate(hyps):
            if hi >= niters:
                break
            if not found[w]:
                stop = True
                break
            i = hi + 1
            if counts[w] > max(best, 3):
                best, best_h = int(counts[w]), H[w]
                niters = min(niters, n_iters_bound(best, m, confidence, max_iters))
    if best == 0:
        return None, mask, 0, i
    H, n = best_h, best
    for _ in range(REFIT_ROUNDS):
        inl = reproj_err(H[None, :8].astype(np.float32), x, y, xd, yd)[0] <= thr2
        sel = np.nonzero(inl)[0]
        H0, ok = dlt(x[None, sel], y[None, sel], xd[None, sel], yd[None, sel])
        Hr = refine(H0[0] if ok[0] else H, x[sel], y[sel], xd[sel], yd[sel])
        mask = (reproj_err(Hr[None, :8].astype(np.float32), x, y, xd, yd)[0] <= thr2).astype(np.uint8)
        grew = int(mask.sum()) > len(sel)
        H, n = Hr, int(mask.sum())
        if not grew:
            break
    return H, mask, n, i

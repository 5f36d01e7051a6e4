"""CPU: the RANSAC homography restatement (oracle/ransac_oracle.py) — its primitives, its small-input behaviour, and its
outcome against cv2.findHomography(..., cv2.RANSAC, 3) on a fixed grid of synthetic pairs."""
import numpy as np
import pytest

cv2 = pytest.importorskip('cv2')

from gims_b200.synth import make_correspondences  # noqa: E402
from oracle import ransac_oracle as ro  # noqa: E402

CORNERS = np.array([[0, 0, 1], [800, 0, 1], [0, 600, 1], [800, 600, 1]], dtype=np.float64)


def corner_error(H, H_true):
    """Mean distance of the four 800x600 corners mapped by H and by the true H (eval_homography's score)."""
    a = CORNERS @ np.asarray(H, dtype=np.float64).reshape(3, 3).T
    b = CORNERS @ H_true.T
    return float(np.linalg.norm(a[:, :2] / a[:, 2:] - b[:, :2] / b[:, 2:], axis=1).mean())


def test_splitmix64_stream():
    # the reference splitmix64 sequence from state 0 (Vigna's splitmix64.c: state += gamma; mix)
    want = [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]
    state = np.uint64(0)
    with np.errstate(over='ignore'):
        for w in want:
            assert int(ro.splitmix64(state)) == w
            state = state + np.uint64(0x9E3779B97F4A7C15)
    v = ro.splitmix64(np.arange(4, dtype=np.uint64))
    assert v.dtype == np.uint64 and [int(t) for t in v] == [int(ro.splitmix64(np.uint64(i))) for i in range(4)]


def test_fixed_sum_order():
    t = np.arange(1000, dtype=np.float64) * 0.1
    part = [sum(t[p::256], 0.0) for p in range(256)]         # sequential from +0.0, points in order
    s = 128
    while s:
        part = [part[p] + part[p + s] for p in range(s)]
        s >>= 1
    assert ro.fixed_sum(t) == part[0]
    assert ro.fixed_sum(np.zeros(0)) == 0.0


@pytest.mark.parametrize('n', [4, 9, 300])
def test_dlt_exact_recovers_h(n):
    rng = np.random.default_rng(n)
    Ht = np.array([[1.02, 0.05, 13.0], [-0.03, 0.96, -7.0], [1.5e-5, -2e-5, 1.0]])
    src = (rng.random((n, 2)) * [800, 600]).astype(np.float32)
    p = np.c_[src.astype(np.float64), np.ones(n)] @ Ht.T
    dst = p[:, :2] / p[:, 2:]
    # the exact image of the fp32 source points under Ht, kept in fp64 through the DLT by feeding fp32 values that
    # are exact: scale the problem so that both sides are representable
    dst32 = dst.astype(np.float32)
    H, ok = ro.dlt(src[None, :, 0], src[None, :, 1], dst32[None, :, 0], dst32[None, :, 1])
    assert ok[0] and H[0, 8] == 1.0
    # fp32 rounding of dst is the only error: it moves the corners by well under a thousandth of a pixel
    assert corner_error(H[0], Ht) < 2e-3
    if n == 4:      # four points determine H: the solve reproduces the fp32 correspondences to the solver's precision
        q = np.c_[src.astype(np.float64), np.ones(4)] @ H[0].reshape(3, 3).T
        assert np.allclose(q[:, :2] / q[:, 2:], dst32, rtol=1e-9, atol=1e-9 * 800)


def test_dlt_exact_on_representable_points():
    # an affine H with power-of-two coefficients maps small integers to exact fp32 values: DLT recovers it to 1e-9
    Ht = np.array([[2.0, 0.5, 16.0], [-0.25, 1.0, 8.0], [0.0, 0.0, 1.0]])
    src = np.array([[0, 0], [64, 0], [0, 32], [64, 32], [16, 8], [40, 24]], dtype=np.float32)
    dst = (np.c_[src.astype(np.float64), np.ones(6)] @ Ht.T)[:, :2].astype(np.float32)
    H, ok = ro.dlt(src[None, :, 0], src[None, :, 1], dst[None, :, 0], dst[None, :, 1])
    assert ok[0]
    assert np.allclose(H[0], Ht.ravel(), rtol=1e-9, atol=1e-9)


def test_refit_matches_lstsq_on_noisy_data():
    src, dst, Ht = make_correspondences(400, 1.0, noise=0.8, seed=5)
    x, y, xd, yd = src[:, 0], src[:, 1], dst[:, 0], dst[:, 1]
    H0, ok = ro.dlt(x[None], y[None], xd[None], yd[None])
    assert ok[0]
    # algebraic least squares with h33 = 1 on the same normalised coordinates, in fp64 by LAPACK
    def norm(v):
        v = v.astype(np.float64)
        c = v.mean()
        return (v - c) * (len(v) / np.abs(v - c).sum()), c, len(v) / np.abs(v - c).sum()
    (X, cx, sx), (Y, cy, sy), (U, cu, su), (V, cv, sv) = (norm(v) for v in (x, y, xd, yd))
    z, o = np.zeros_like(X), np.ones_like(X)
    A = np.concatenate([np.stack([X, Y, o, z, z, z, -U * X, -U * Y], 1), np.stack([z, z, z, X, Y, o, -V * X, -V * Y], 1)])
    h = np.linalg.lstsq(A, np.concatenate([U, V]), rcond=None)[0]
    Hl = np.array([[1 / su, 0, cu], [0, 1 / sv, cv], [0, 0, 1]]) @ np.r_[h, 1].reshape(3, 3) @ \
        np.array([[sx, 0, -cx * sx], [0, sy, -cy * sy], [0, 0, 1]])
    assert np.allclose(H0[0], (Hl / Hl[2, 2]).ravel(), rtol=1e-8, atol=1e-12)
    assert corner_error(H0[0], Ht) < 0.5
    H = ro.refine(H0[0], x, y, xd, yd)
    cost = lambda hh: ro._lm_cost(hh, x, y, xd, yd)                      # noqa: E731
    assert cost(H) <= cost(H0[0])
    assert corner_error(H, Ht) < 0.5


def test_iteration_bound_vs_cv2_formula():
    for m in (12, 60, 300, 2048):
        for g in range(4, m + 1, max(1, m // 37)):
            for c in (0.9, 0.995, 0.999):
                ep = (m - g) / m
                denom = 1.0 - (1.0 - ep) ** 4
                if denom < np.finfo(np.float64).tiny:
                    cv = 0
                else:
                    num, den = np.log(max(1.0 - c, np.finfo(np.float64).tiny)), np.log(denom)
                    cv = 2000 if den >= 0 or -num >= 2000 * (-den) else int(np.floor(num / den + 0.5))
                ours = ro.n_iters_bound(g, m, c, 2000)
                assert ours == max(cv, 1) or ours == cv + 1, (m, g, c, ours, cv)


def test_small_inputs_like_cv2():
    rng = np.random.default_rng(1)
    s3 = (rng.random((3, 2)) * 100).astype(np.float32)
    with pytest.raises(cv2.error):
        cv2.findHomography(s3, s3 + 1, cv2.RANSAC, 3.0)
    assert ro.find_homography(s3, s3 + 1)[0] is None          # the drop-in raises on M < 4; the estimator says "not found"
    s4 = (rng.random((4, 2)) * 100).astype(np.float32)
    d4 = s4[::-1].copy()
    H, mask, n, it = ro.find_homography(s4, d4)
    Hc, mc = cv2.findHomography(s4, d4, cv2.RANSAC, 3.0)
    assert np.array_equal(mask, mc.ravel()) and n == 4 and it == 0
    assert np.allclose(H.reshape(3, 3), Hc, rtol=1e-6, atol=1e-6)
    for s, d in ((np.ones((10, 2), np.float32),) * 2, (np.ones((4, 2), np.float32),) * 2,
                 (np.stack([np.arange(10), 2 * np.arange(10)], 1).astype(np.float32),) * 2):
        H, mask, n, _ = ro.find_homography(s, d + 1)
        Hc, mc = cv2.findHomography(s, d + 1, cv2.RANSAC, 3.0)
        assert Hc is None and H is None and n == 0
        assert np.array_equal(mask, mc.ravel()) and not mask.any()


def _grid():
    cases = []
    for m in (12, 60, 300, 2048):
        for ratio in (0.9, 0.5, 0.25, 0.15):
            for noise in (0.5, 1.5):
                for rep in range(4):
                    cases.append((m, ratio, noise, 1000 * m + 100 * rep + int(ratio * 40) + int(noise * 2)))
    return cases


def outcome_vs_cv2():
    """The restatement and cv2 on the grid: per case (m, ratio, corner errors, mask Jaccard)."""
    rows = []
    for m, ratio, noise, seed in _grid():
        src, dst, Ht = make_correspondences(m, ratio, noise=noise, seed=seed)
        H, mask, _, _ = ro.find_homography(src, dst, 3.0)
        Hc, mc = cv2.findHomography(src, dst, cv2.RANSAC, 3.0)
        e = corner_error(H, Ht) if H is not None else np.inf
        ec = corner_error(Hc, Ht) if Hc is not None else np.inf
        a, b = mask.astype(bool), mc.ravel().astype(bool)
        jac = (a & b).sum() / max(1, (a | b).sum())
        rows.append((m, ratio, e, ec, jac))
    return rows


def test_restatement_vs_cv2_outcome():
    rows = outcome_vs_cv2()
    assert len(rows) >= 120
    ok = [r[2] <= 3.0 for r in rows]
    okc = [r[3] <= 3.0 for r in rows]
    both = [r for r, a, b in zip(rows, ok, okc) if a and b]
    med, medc = np.median([r[2] for r in both]), np.median([r[3] for r in both])
    jac = np.median([r[4] for r in rows if r[1] >= 0.5])
    print('\n[ransac vs cv2] %d cases: success %d (cv2 %d); median corner error on %d common successes %.4f px '
          '(cv2 %.4f); median mask Jaccard at inlier ratio >= 0.5: %.4f' % (len(rows), sum(ok), sum(okc), len(both),
                                                                            med, medc, jac))
    assert sum(ok) >= sum(okc) - 2
    assert med <= 1.10 * medc + 0.02
    assert jac >= 0.98

"""RANSAC homographies on the device (gims_find_homographies) against the numpy restatement oracle/ransac_oracle.py:
equal bit for bit — H as float64 bits, the mask, the inlier count and the number of hypotheses run."""
import threading

import numpy as np
import pytest
import torch

from gims_b200 import postprocess as pp
from gims_b200._lib import GimsError
from gims_b200.synth import make_correspondences
from oracle import ransac_oracle as ro

pytestmark = pytest.mark.gpu


def _case(m, ratio, seed, dirty=False):
    if m == 0:
        return np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32)
    src, dst, _ = make_correspondences(m, ratio, noise=1.0, seed=seed)
    if dirty and m >= 12:
        rng = np.random.default_rng(seed)
        j = rng.choice(m, 6, replace=False)
        src[j[0], 0], dst[j[1], 1], src[j[2], 1] = np.nan, np.inf, -np.inf
        src[j[3]], dst[j[3]] = src[j[4]], dst[j[4]]            # an exact duplicate correspondence
        src[j[5]] = src[j[4]]                                  # a repeated source point with another partner
    return src, dst


def _ref(src, dst, seed=0, **kw):
    H, mask, n, it = ro.find_homography(src, dst, seed=seed, **kw)
    return (np.zeros(9) if H is None else H), mask, n, it


def _device(pairs, seed=0, **kw):
    src = torch.from_numpy(np.concatenate([p[0] for p in pairs]).reshape(-1, 2)).cuda()
    dst = torch.from_numpy(np.concatenate([p[1] for p in pairs]).reshape(-1, 2)).cuda()
    offs = np.zeros(len(pairs) + 1, dtype=np.int32)
    np.cumsum([len(p[0]) for p in pairs], out=offs[1:])
    H, n, mask, it = pp.find_homographies_packed(src, dst, torch.from_numpy(offs).cuda(), seed=seed, **kw)
    torch.cuda.synchronize()
    H, n, mask, it = H.cpu().numpy().reshape(-1, 9), n.cpu().numpy(), mask.cpu().numpy(), it.cpu().numpy()
    return [(H[p], mask[offs[p]:offs[p + 1]], int(n[p]), int(it[p])) for p in range(len(pairs))]


def _assert_equal(got, want, what):
    assert np.array_equal(got[0].view(np.uint64), np.asarray(want[0], np.float64).view(np.uint64)), \
        (what, got[0], want[0])
    assert np.array_equal(got[1], want[1]), (what, 'mask')
    assert got[2] == want[2] and got[3] == want[3], (what, got[2:], want[2:])


CASES = [(m, r, s, dirty) for m in (4, 5, 12, 300, 2048, 16384) for r in (0.9, 0.5, 0.2, 0.05) for s in (0, 1)
         for dirty in ((False, True) if m >= 300 else (False,))]


@pytest.mark.parametrize('m,ratio,seed,dirty', CASES)
def test_device_equals_restatement(m, ratio, seed, dirty):
    src, dst = _case(m, ratio, 100 * m + int(ratio * 100) + seed, dirty)
    _assert_equal(_device([(src, dst)], seed=seed)[0], _ref(src, dst, seed=seed), (m, ratio, seed, dirty))


def test_parameters_follow_restatement():
    src, dst = _case(600, 0.4, 77)
    kw = dict(thresh=1.5, max_iters=150, confidence=0.9)
    got = _device([(src, dst)], seed=12345678901234567, threshold=1.5, max_iters=150, confidence=0.9)[0]
    _assert_equal(got, _ref(src, dst, seed=12345678901234567, **kw), 'parameters')


def test_ragged_batch_equals_single_pairs():
    rng = np.random.default_rng(3)
    sizes = [0, 1, 2, 3, 4, 5] + [int(v) for v in rng.integers(6, 700, 200)]
    pairs = [_case(m, float(rng.choice([0.9, 0.5, 0.25])), 5000 + i) for i, m in enumerate(sizes)]
    batch = _device(pairs)
    for i in [0, 1, 2, 3, 4, 5] + list(range(6, len(pairs), 17)):
        _assert_equal(batch[i], _device([pairs[i]])[0], ('single', i))
    for i in range(len(pairs)):
        _assert_equal(batch[i], _ref(*pairs[i]), ('restatement', i))


def test_repeated_and_threaded_calls_identical():
    pairs = [_case(m, 0.5, 900 + m) for m in (50, 300, 1200, 4000)]
    src = [torch.from_numpy(p[0]).cuda() for p in pairs]
    dst = [torch.from_numpy(p[1]).cuda() for p in pairs]

    def run():
        H, n, masks = pp.find_homographies(src, dst)
        torch.cuda.current_stream().synchronize()
        return H.cpu(), n.cpu(), [m.cpu() for m in masks]

    first = run()
    results = [None] * 4

    def worker(k):
        with torch.cuda.stream(torch.cuda.Stream()):
            results[k] = [run() for _ in range(3)]

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for res in [[run()]] + results:
        for H, n, masks in res:
            assert torch.equal(H, first[0]) and torch.equal(n, first[1])
            assert all(torch.equal(a, b) for a, b in zip(masks, first[2]))


def test_find_homography_drop_in():
    src, dst = _case(500, 0.6, 31)
    H, mask = pp.find_homography(src, dst, 8, 3.0)
    want = _ref(src, dst)
    assert H.dtype == np.float64 and H.shape == (3, 3) and mask.dtype == np.uint8 and mask.shape == (500, 1)
    assert np.array_equal(H.ravel().view(np.uint64), want[0].view(np.uint64))
    assert np.array_equal(mask.ravel(), want[1])
    H, mask = pp.find_homography(torch.from_numpy(src).cuda()[:, None], torch.from_numpy(dst).cuda()[:, None],
                                 method=8, ransacReprojThreshold=3.0)
    assert np.array_equal(H.ravel().view(np.uint64), want[0].view(np.uint64))
    same = np.ones((10, 2), np.float32)
    H, mask = pp.find_homography(same, same, 8)
    assert H is None and mask.shape == (10, 1) and not mask.any()


def test_bad_arguments_raise():
    src, dst = _case(20, 0.9, 1)
    with pytest.raises(GimsError):
        pp.find_homography(src[:3], dst[:3], 8)
    with pytest.raises(GimsError):
        pp.find_homography(src, dst, 0)                      # not cv2.RANSAC
    with pytest.raises(GimsError):
        pp.find_homography(src, dst[:19], 8)
    with pytest.raises(GimsError):
        pp.find_homography(src[:, :1], dst[:, :1], 8)
    for kw in (dict(ransacReprojThreshold=0.0), dict(confidence=1.0), dict(confidence=0.0), dict(maxIters=0)):
        with pytest.raises(GimsError):
            pp.find_homography(src, dst, 8, **kw)
    s, d = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
    with pytest.raises(GimsError):
        pp.find_homographies([s], [d[:10]])
    with pytest.raises(GimsError):
        pp.find_homographies([s], [])
    with pytest.raises(GimsError):
        pp.find_homographies([s.cpu()], [d.cpu()])
    with pytest.raises(GimsError):
        pp.find_homographies([s], [d], threshold=-1.0)


def test_matching_pipeline_to_homographies():
    """Images -> device SIFT -> the stand-in descriptor network -> the matcher -> matched_points -> find_homographies,
    all on the device, equal to the restatement run on the same matched points copied to the host."""
    import types
    pytest.importorskip('cv2')
    from gims_b200 import Matching
    from gims_b200.synth import make_state_dict, make_textured_image, warp_image
    from test_gpu_parity import _PatchNet
    dev = torch.device('cuda')
    torch.manual_seed(0)
    car = types.SimpleNamespace(model=_PatchNet().to(dev).eval(), batch_size=512)
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.01, 'max_keypoints': 700, 'detector': 'device'})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    matching = matching.eval().to(dev)
    img0 = make_textured_image(300, 400, seed=7)
    img1, _ = warp_image(img0, seed=8)
    with torch.no_grad():
        pred = matching({'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7,
                         'image0': img0[None], 'image1': img1[None], 'carhynet': car})
    mk0, mk1, _ = pp.matched_points(pred)
    assert mk0.is_cuda and mk0.shape[0] >= 4
    H, n, masks = pp.find_homographies([mk0], [mk1])
    got = (H[0].cpu().numpy().ravel(), masks[0].cpu().numpy(), int(n[0].cpu()))
    want = _ref(mk0.cpu().numpy().astype(np.float32), mk1.cpu().numpy().astype(np.float32))
    assert np.array_equal(got[0].view(np.uint64), want[0].view(np.uint64)) and np.array_equal(got[1], want[1])
    assert got[2] == want[2]

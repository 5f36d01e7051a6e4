"""The Gaussian pyramid on the GPU (gims_gaussian_pyramid, csrc/pyramid.cu) against the host pyramid OpenCV builds
(frontend.gaussian_pyramid): every level byte-identical, the patches cut from it identical, and the image-input Matching
call that now runs through it equal to the old route."""
import threading
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip('cv2')


def _image(h, w, channels, seed):
    from gims_b200.synth import make_textured_image
    img = make_textured_image(h, w, seed=seed)
    return cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if channels == 1 else img


class _Net(torch.nn.Module):
    """A stand-in descriptor network (colour 32x32 patches -> unit-norm 128-d): both routes run the same one."""

    def __init__(self):
        super().__init__()
        self.body = torch.nn.Sequential(torch.nn.Conv2d(3, 32, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(32, 64, 3, stride=2, padding=1), torch.nn.ReLU(),
                                        torch.nn.Conv2d(64, 128, 8))

    def forward(self, x):
        return torch.nn.functional.normalize(self.body(x).flatten(1), dim=1)


@pytest.mark.parametrize('h,w,channels,seed', [(600, 800, 3, 100), (301, 417, 3, 5), (240, 320, 1, 3), (40, 56, 3, 9),
                                               (40, 56, 1, 9)])
def test_device_pyramid_equals_host_pyramid(h, w, channels, seed):
    from gims_b200 import frontend as fe
    img = _image(h, w, channels, seed)
    want = fe.gaussian_pyramid(img)
    pyr = fe.gaussian_pyramid_device(img, 'cuda:0')
    assert len(pyr) == len(want)
    bad = []
    for i, lv in enumerate(want):
        got = pyr.level(i).cpu().numpy()
        if got.shape != lv.shape or not np.array_equal(got, lv):
            bad.append((i, lv.shape, int(np.abs(got.astype(int) - lv).max()) if got.shape == lv.shape else -1))
    assert not bad, bad


def test_device_pyramid_of_one_channel_image_equals_grey():
    from gims_b200 import frontend as fe
    img = _image(120, 90, 1, 4)
    a = fe.gaussian_pyramid_device(img, 'cuda:0')
    b = fe.gaussian_pyramid_device(img[:, :, None], 'cuda:0')
    want = fe.gaussian_pyramid(img[:, :, None])
    assert len(a) == len(b) == len(want)
    for i, lv in enumerate(want):
        assert np.array_equal(b.level(i).cpu().numpy(), lv) and torch.equal(a.level(i), b.level(i))


@pytest.mark.parametrize('h,w,channels,nkp,seed', [(600, 800, 3, 2048, 2), (240, 320, 1, 300, 3)])
def test_patches_from_device_pyramid_equal_host(h, w, channels, nkp, seed):
    from gims_b200 import frontend as fe
    img = _image(h, w, channels, seed)
    kps = fe.detect(img, nkp)
    want = fe.extract_patches(kps, fe.gaussian_pyramid(img))
    got = fe.extract_patches_device(kps, fe.gaussian_pyramid_device(img, 'cuda:0'), 'cuda:0')
    assert got.is_cuda and tuple(got.shape) == want.shape
    assert torch.equal(got.cpu(), torch.from_numpy(want.astype(np.float32)))


def _matching_and_car(dev):
    from gims_b200 import Matching
    from gims_b200.synth import make_state_dict
    torch.manual_seed(0)
    car = types.SimpleNamespace(model=_Net().to(dev).eval(), batch_size=512)
    matching = Matching({'sinkhorn_iterations': 20, 'match_threshold': 0.01, 'max_keypoints': 700})
    matching.gmodel.load_state_dict(make_state_dict(0, damped=True))
    return matching.eval().to(dev), car


def _pairs(n):
    from gims_b200.synth import make_textured_image, warp_image
    out = []
    for k in range(n):
        img0 = make_textured_image(300 + 20 * k, 400, seed=30 + k)
        img1, _ = warp_image(img0, seed=60 + k)
        out.append((img0[None], img1[None]))
    return out


def _call(matching, car, pair, dev):
    knobs = {'delaunay': False, 'device': dev, 'radius': 15, 'percentile': 2, 'min_size': 7}
    with torch.no_grad():
        pred = matching({**knobs, 'image0': pair[0], 'image1': pair[1], 'carhynet': car})
    return {k: v[0].cpu() for k, v in pred.items()}


def test_matching_with_images_equals_forced_host_pyramid_route(monkeypatch):
    dev = torch.device('cuda:0')
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)
    monkeypatch.setattr(torch.backends.cudnn, 'benchmark', False)
    matching, car = _matching_and_car(dev)
    pair = _pairs(1)[0]
    got = _call(matching, car, pair, dev)
    from gims_b200 import frontend as fe
    # the old route: host pyramid, levels uploaded by extract_patches_device
    monkeypatch.setattr(fe, '_use_device_pyramid', lambda image, device, detector: False)
    want = _call(matching, car, pair, dev)
    for s in '01':
        assert torch.equal(got['keypoints' + s], want['keypoints' + s])
        assert torch.equal(got['matches' + s], want['matches' + s])
        assert torch.allclose(got['descriptors' + s], want['descriptors' + s], rtol=0, atol=1e-6)
    assert int((got['matches0'] >= 0).sum()) > 0


def test_concurrent_image_callers_match_single_thread(monkeypatch):
    dev = torch.device('cuda:0')
    monkeypatch.setattr(torch.backends.cudnn, 'deterministic', True)
    monkeypatch.setattr(torch.backends.cudnn, 'benchmark', False)
    matching, car = _matching_and_car(dev)
    pairs = _pairs(4)
    single = [_call(matching, car, p, dev) for p in pairs]
    results = [None] * len(pairs)
    errors = []

    def worker(tid):
        try:
            with torch.cuda.stream(torch.cuda.Stream(dev)):
                for k in range(tid, len(pairs), 2):
                    results[k] = _call(matching, car, pairs[k], dev)
        except Exception as exc:                                      # noqa: BLE001
            errors.append(exc)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    torch.cuda.synchronize()
    assert not errors, errors
    for a, b in zip(single, results):
        for s in '01':
            assert torch.equal(a['keypoints' + s], b['keypoints' + s])
            assert torch.equal(a['matches' + s], b['matches' + s])
            assert torch.allclose(a['descriptors' + s], b['descriptors' + s], rtol=0, atol=1e-6)
